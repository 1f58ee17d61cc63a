"""BGZF encoder (ms_bgzf_compress) on the C2 outputs, and what --bgzip does to the file-to-file CLI time.

usage (GPU box): python profiles/bgzf_bench.py [--out FILE.json] [--reps 10] [--f2f-runs 3]

Prints one JSON object: the card's name and power limit (read in the same run); per output (FASTA image, VCF body
of C2: bench.py's synthetic GRCh38-shaped genome and ARGS mutation mix) the encoder's time as CUDA events around
Engine.bgzf_compress on the engine's stream (warm, median of --reps), input GB/s and ratio; and the wall time of
the whole CLI from a FASTA in /dev/shm to its outputs there, plain and --bgzip alternated --f2f-runs times."""
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
import bench  # noqa: E402
from mutation_simulator_b200.engine import BUF_FASTA, BUF_VCF, Engine  # noqa: E402
from mutation_simulator_b200.records import REC_DTYPE  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def encoder(reps):
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
    fo, vo, _, _ = eng.contig_layout()
    out = {}
    for name, which, lay in (("fasta", BUF_FASTA, fo), ("vcf", BUF_VCF, vo)):
        src, n = lay[:-1], np.diff(lay)
        for _ in range(2):
            eng.bgzf_compress(which, src, n, src)
        dev, wall = [], []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record(stream)
            _, tot = eng.bgzf_compress(which, src, n, src)
            e1.record(stream)
            e1.synchronize()
            wall.append((time.perf_counter() - t0) * 1e3)
            dev.append(e0.elapsed_time(e1))
        nin = int(lay[-1])
        ms = statistics.median(dev)
        out[name] = dict(input_bytes=nin, bgzf_bytes=int(tot), members=int(sum(-(-int(k) // 16384) for k in n)),
                         ratio=round(nin / tot, 3), encoder_ms_median=round(ms, 3), encoder_ms_min=round(min(dev), 3),
                         encoder_ms_max=round(max(dev), 3), host_wall_ms_median=round(statistics.median(wall), 3),
                         input_GBps=round(nin / ms / 1e6, 1), reps=reps)
    eng.close()
    return out


def file_to_file(runs):
    wl = bench.WORKLOADS["c2"]
    lengths, names = list(wl["lengths"]), wl["names"]
    d = Path("/dev/shm/ms_bgzf_bench")
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
        res = {"plain": [], "bgzip": []}
        sizes = {}
        for i in range(runs + 1):                 # run 0 of each arm is a warm-up (builds genome.fa.fai, page cache)
            for arm in ("plain", "bgzip"):
                cmd = [sys.executable, "-m", "mutation_simulator_b200", str(d / "genome.fa"), "-o", str(d / "out"), "-q",
                       "--seed", "7"] + (["--bgzip"] if arm == "bgzip" else []) + bench.reference_cli_args(wl)
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
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--f2f-runs", type=int, default=3)
    a = ap.parse_args()
    res = dict(card=card(), workload=bench.WORKLOADS["c2"]["desc"], encoder=encoder(a.reps))
    if a.f2f_runs:
        res["file_to_file"] = file_to_file(a.f2f_runs)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
