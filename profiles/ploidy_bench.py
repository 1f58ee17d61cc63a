"""Polyploid stages (ms_genotype_draw, ms_select_haplotype, ms_vcf_phased) on the C2 run with P = 2, and what
--ploidy 2 does to the file-to-file CLI time.

usage (GPU box): python profiles/ploidy_bench.py [--out FILE.json] [--reps 9] [--f2f-runs 3]

Prints one JSON object: the card's name and power limit (read in the same run); for C2 (bench.py's synthetic
GRCh38-shaped genome and ARGS mutation mix) the records per haplotype and phased VCF bytes, the time of each stage as CUDA
events on the engine's stream (warm, median of --reps), and K7 (the haploid VCF formatter) from the engine's own stage
events of one apply for comparison; and the wall time of the whole CLI from a FASTA in /dev/shm to its outputs there,
with --ploidy 1 and --ploidy 2, alternated --f2f-runs times after a warm-up pair."""
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
from mutation_simulator_b200.engine import BUF_FASTA, BUF_VCF_PHASED, Engine  # noqa: E402
from mutation_simulator_b200.records import REC_DTYPE  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def timed(stream, fn, reps):
    import torch
    fn()
    fn()
    dev = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        dev.append(e0.elapsed_time(e1))
    return dict(ms_median=round(statistics.median(dev), 3), ms_min=round(min(dev), 3), ms_max=round(max(dev), 3))


def stages(reps):
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
    k7 = eng.stats()["stage_ms"]["vcf_format"]
    n_full = len(eng.records(True))
    res = dict(records=n_full, haploid_vcf_bytes=int(vb), k7_vcf_format_ms_one_apply=round(k7, 3))
    res["genotype"] = timed(stream, lambda: eng.genotype_draw(7, 2, 0.35), reps)
    masks = eng.genotypes()
    res["records_per_haplotype"] = [int((masks & 1).sum()), int((masks >> 1 & 1).sum())]
    res["hom_share"] = round(float((masks == 3).mean()), 5)

    def select():
        eng.select_haplotype(1)
        eng.select_haplotype(0)
    res["select_h1_and_restore"] = timed(stream, select, reps)
    res["vcf_phased"] = timed(stream, eng.vcf_phased, reps)
    off = eng.vcf_phased()
    res["phased_vcf_bytes"] = int(off[-1])
    res["vcf_phased_GBps"] = round(off[-1] / res["vcf_phased"]["ms_median"] / 1e6, 2)
    res["phased_vcf_hash"] = int(eng.hash_ranges(BUF_VCF_PHASED, [0], [int(off[-1])])[0])
    eng.close()
    return res


def file_to_file(runs):
    wl = bench.WORKLOADS["c2"]
    lengths, names = list(wl["lengths"]), wl["names"]
    d = Path("/dev/shm/ms_ploidy_bench")
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
        res = {"p1": [], "p2": []}
        sizes = {}
        for i in range(runs + 1):                 # run 0 of each arm is a warm-up (builds genome.fa.fai, page cache)
            for arm in ("p1", "p2"):
                cmd = [sys.executable, "-m", "mutation_simulator_b200", str(d / "genome.fa"), "-o", str(d / "out"), "-q",
                       "--seed", "7", "--ploidy", arm[1]] + bench.reference_cli_args(wl)
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
    res = dict(card=card(), workload=bench.WORKLOADS["c2"]["desc"], stages=stages(a.reps))
    if a.f2f_runs:
        res["file_to_file"] = file_to_file(a.f2f_runs)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
