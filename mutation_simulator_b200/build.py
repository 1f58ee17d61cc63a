"""Builds libmutsim_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m mutation_simulator_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
OBJ = PKG / "_obj"
LIB = PKG / "libmutsim_b200.so"
SOURCES = ["ms_api.cu", "ms_apply.cu", "ms_sample.cu", "ms_genome.cu", "ms_ingest.cu", "ms_bgzf.cu", "ms_vcf_parse.cu", "ms_chain.cu",
           "ms_genotype.cu", "ms_reads.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
              "--extended-lambda", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-Wall", "-Xcudafe", "--diag_suppress=177"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (Path(cand).exists() or cand == "nvcc"):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    headers = list(CSRC.glob("*.h")) + list(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "mutsim_b200.h"]
    OBJ.mkdir(exist_ok=True)
    nvcc = _nvcc()
    jobs = []
    for s in SOURCES:
        src, obj = CSRC / s, OBJ / (s + ".o")
        if force or _stale(obj, [src] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", str(src), "-o", str(obj)]
            jobs.append(cmd)
    if jobs:
        with ThreadPoolExecutor(max_workers=4) as ex:
            for cmd, res in zip(jobs, ex.map(lambda c: subprocess.run(c, capture_output=True, text=True), jobs)):
                if verbose or res.returncode:
                    sys.stderr.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
                if res.returncode:
                    raise RuntimeError(f"nvcc failed for {cmd[-3]}")
    objs = [OBJ / (s + ".o") for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        cmd = [nvcc, "-arch=sm_100a", "-shared", "-o", str(LIB)] + [str(o) for o in objs] + ["-lcudart"]
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
