"""Paired-end reads (ms_reads_size + ms_reads_write) on the C2 run at --reads 1, and what --reads 1 does to the
file-to-file CLI time.

usage (GPU box): python profiles/reads_bench.py [--out FILE.json] [--reps 9] [--f2f-runs 3]

Prints one JSON object: the card's name and power limit (read in the same run); for C2 (bench.py's synthetic
GRCh38-shaped genome and ARGS mutation mix) the pairs and bytes of one FASTQ file at depth 1 (L = 150, fragments
500 +- 50, E = 0.001), the time of reads_size + reads_write as CUDA events on the engine's stream (warm, median of
--reps), the FASTQ rate (both files) and the HBM bound of the bytes the two kernels must move; and the wall time of the
whole CLI from a FASTA in /dev/shm to its outputs there, with and without --reads 1, alternated --f2f-runs times after
a warm-up pair."""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "profiles"))
import bench  # noqa: E402
from ploidy_bench import card, timed  # noqa: E402
from mutation_simulator_b200.engine import BUF_FASTA, BUF_READS, Engine  # noqa: E402
from mutation_simulator_b200.reads_writer import pair_counts, quality_char  # noqa: E402
from mutation_simulator_b200.records import REC_DTYPE  # noqa: E402

HBM_TBPS = 7.7     # NVIDIA data sheet, one B200 (HGX)


def kernels(reps):
    import torch
    wl = bench.WORKLOADS["c2"]
    lengths, names = list(wl["lengths"]), [n.encode() for n in wl["names"]]
    eng = Engine(0)
    stream = torch.cuda.Stream(device=0)
    eng.set_stream(stream.cuda_stream)
    eng.synth_genome(bench.GENOME_SEED, lengths, [60] * len(lengths), names, names, wl["n_fraction"], wl["telomere"])
    eng.set_ranges_array(bench.make_ranges(lengths, wl), len(lengths), [1] * 7, 1, wl["titv"] / (wl["titv"] + 1))
    eng.sample(7)
    eng.apply()
    L = 150
    cfg = dict(seed=7, hap=1, read_len=L, frag_mean=500, frag_sd=50, error_rate=0.001, qual=quality_char(0.001))
    n = pair_counts(1.0, eng.contig_out_len(), L, 1)
    total = int(n.sum())
    res = dict(pairs=total, read_len=L)
    nb = [0]

    def both():
        eng.reads_size(cfg, n, 0, total)
        nb[0] = eng.reads_write(cfg, n, 0, total)
    res["size_plus_write"] = timed(stream, both, reps)
    res["size_only"] = timed(stream, lambda: eng.reads_size(cfg, n, 0, total), reps)
    res["fastq_bytes_per_file"] = nb[0]
    ms = res["size_plus_write"]["ms_median"]
    res["fastq_GBps_both_files"] = round(2 * nb[0] / ms / 1e6, 2)
    # bytes the kernels must move at least: both template ends read twice (size check, write copy), 24 B of PairInfo
    # written and read, 8 B of offsets written and read, and both files' text written
    moved = total * (2 * 2 * L + 2 * 24 + 2 * 8) + 2 * nb[0]
    res["hbm_bytes_lower_bound"] = moved
    res["hbm_bound_ms"] = round(moved / (HBM_TBPS * 1e12) * 1e3, 3)
    res["fastq_hash"] = int(eng.hash_ranges(BUF_READS, [0], [2 * nb[0]])[0])
    eng.close()
    return res


def file_to_file(runs):
    wl = bench.WORKLOADS["c2"]
    lengths, names = list(wl["lengths"]), wl["names"]
    d = Path("/dev/shm/ms_reads_bench")
    d.mkdir(parents=True, exist_ok=True)
    try:
        g = Engine(0)
        g.synth_genome(4242, lengths, [60] * len(lengths), [n.encode() for n in names], [n.encode() for n in names],
                       wl["n_fraction"], wl["telomere"])
        g.load_records(np.zeros(0, dtype=REC_DTYPE))
        g.apply()
        with open(d / "genome.fa", "wb") as fh:
            fh.write(memoryview(g.download(BUF_FASTA)))
            fh.write(b"\n")
        g.close()
        env = dict(os.environ, PYTHONPATH=str(REPO))
        res = {"no_reads": [], "reads_1": []}
        sizes = {}
        for i in range(runs + 1):                 # run 0 of each arm is a warm-up (builds genome.fa.fai, page cache)
            for arm in res:
                extra = ["--reads", "1"] if arm == "reads_1" else []
                cmd = [sys.executable, "-m", "mutation_simulator_b200", str(d / "genome.fa"), "-o", str(d / "out"), "-q",
                       "--seed", "7"] + extra + bench.reference_cli_args(wl)
                t0 = time.perf_counter()
                subprocess.run(cmd, env=env, check=True)
                dt = time.perf_counter() - t0
                outs = sorted(d.glob("out_ms*"))
                sizes[arm] = {p.name: p.stat().st_size for p in outs}
                for p in outs:
                    p.unlink()
                if i:
                    res[arm].append(round(dt, 3))
        return dict(fasta_in_bytes=(d / "genome.fa").stat().st_size, wall_s=res,
                    median_s={k: statistics.median(v) for k, v in res.items()}, output_bytes=sizes)
    finally:
        shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", type=Path)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--f2f-runs", type=int, default=3)
    a = ap.parse_args()
    res = dict(card=card(), workload=bench.WORKLOADS["c2"]["desc"], kernels=kernels(a.reps))
    if a.f2f_runs:
        res["file_to_file"] = file_to_file(a.f2f_runs)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
