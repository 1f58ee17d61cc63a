"""Chain formatter (ms_chain_count + ms_chain_write) on the C2 run, and what --chain does to the file-to-file CLI time.

usage (GPU box): python profiles/chain_bench.py [--out FILE.json] [--reps 9] [--f2f-runs 3]

Prints one JSON object: the card's name and power limit (read in the same run); for C2 (bench.py's synthetic
GRCh38-shaped genome and ARGS mutation mix) the number of chains and text bytes, and the time of Engine.chain_count +
Engine.chain_write as CUDA events on the engine's stream (warm, median of --reps); and the wall time of the whole CLI
from a FASTA in /dev/shm to its outputs there, without and with --chain, alternated --f2f-runs times."""
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
from mutation_simulator_b200.chain_writer import first_ids  # noqa: E402
from mutation_simulator_b200.engine import BUF_CHAIN, BUF_FASTA, Engine  # noqa: E402
from mutation_simulator_b200.records import REC_DTYPE  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def formatter(reps):
    import torch
    wl = bench.WORKLOADS["c2"]
    lengths, names = list(wl["lengths"]), [n.encode() for n in wl["names"]]
    eng = Engine(0)
    stream = torch.cuda.Stream(device=0)
    eng.set_stream(stream.cuda_stream)
    eng.synth_genome(bench.GENOME_SEED, lengths, [60] * len(lengths), names, names, wl["n_fraction"], wl["telomere"])
    eng.set_ranges_array(bench.make_ranges(lengths, wl), len(lengths), [1] * 7, 1, wl["titv"] / (wl["titv"] + 1))
    eng.sample(7)
    fb, vb = eng.apply()
    recs = eng.records()
    n_sv = int((recs["kind"] != 1).sum())
    for _ in range(2):
        off = eng.chain_write(first_ids(eng.chain_count()))
    dev, wall = [], []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        n = eng.chain_count()
        off = eng.chain_write(first_ids(n))
        e1.record(stream)
        e1.synchronize()
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(e0.elapsed_time(e1))
    text_bytes = int(off[-1])
    ms = statistics.median(dev)
    h = eng.hash_ranges(BUF_CHAIN, [0], [text_bytes])
    res = dict(records=int(len(recs)), base_moving_records=n_sv, chains=int(n.sum()), chain_bytes=text_bytes,
               vcf_bytes=int(vb), fasta_bytes=int(fb), count_write_ms_median=round(ms, 3),
               count_write_ms_min=round(min(dev), 3), count_write_ms_max=round(max(dev), 3),
               host_wall_ms_median=round(statistics.median(wall), 3), output_GBps=round(text_bytes / ms / 1e6, 2),
               chain_hash=int(h[0]), reps=reps)
    eng.close()
    return res


def file_to_file(runs):
    wl = bench.WORKLOADS["c2"]
    lengths, names = list(wl["lengths"]), wl["names"]
    d = Path("/dev/shm/ms_chain_bench")
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
        res = {"plain": [], "chain": []}
        sizes = {}
        for i in range(runs + 1):                 # run 0 of each arm is a warm-up (builds genome.fa.fai, page cache)
            for arm in ("plain", "chain"):
                cmd = [sys.executable, "-m", "mutation_simulator_b200", str(d / "genome.fa"), "-o", str(d / "out"), "-q",
                       "--seed", "7"] + (["--chain"] if arm == "chain" else []) + bench.reference_cli_args(wl)
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
    res = dict(card=card(), workload=bench.WORKLOADS["c2"]["desc"], formatter=formatter(a.reps))
    if a.f2f_runs:
        res["file_to_file"] = file_to_file(a.f2f_runs)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
