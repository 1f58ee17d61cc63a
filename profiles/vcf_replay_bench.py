"""VCF replay input on the C2 VCF: the device parser (Engine.load_vcf), the host parser it replaces, and `vcf` mode
file to file.

usage (GPU box): python profiles/vcf_replay_bench.py [--out FILE.json] [--reps 7] [--host-lines 1000000] [--f2f-runs 2]

Prints one JSON object: the card's name and power limit (read in the same run); the C2 VCF (bench.py's synthetic
GRCh38-shaped genome and ARGS mutation mix, sampled and applied on the device, its body downloaded behind the header
VcfWriter writes); Engine.load_vcf on the whole text as CUDA events on the engine's stream (warm, median of --reps),
host-to-device copy included, with GB/s of text, next to a plain copy of the same pageable bytes; records_from_vcf + load_records on the first --host-lines lines of
the body (the host parser is linear in lines), scaled to the whole file; and the wall time of the whole CLI from
the C2 FASTA and VCF in /dev/shm to the outputs there, `vcf` mode next to an `args` run, alternated --f2f-runs times."""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
import bench  # noqa: E402
from mutation_simulator_b200.engine import BUF_FASTA, BUF_VCF, Engine  # noqa: E402
from mutation_simulator_b200.records import genome_offsets, records_from_vcf  # noqa: E402
from mutation_simulator_b200.vcf_writer import header_text  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def c2_engine():
    wl = bench.WORKLOADS["c2"]
    lengths, names = list(wl["lengths"]), [n.encode() for n in wl["names"]]
    eng = Engine(0)
    eng.synth_genome(bench.GENOME_SEED, lengths, [60] * len(lengths), names, names, wl["n_fraction"], wl["telomere"])
    return eng, lengths, names


def measure(d: Path, reps: int, host_lines: int):
    import torch
    wl = bench.WORKLOADS["c2"]
    eng, lengths, names = c2_engine()
    stream = torch.cuda.Stream(device=0)
    eng.set_stream(stream.cuda_stream)
    eng.set_ranges_array(bench.make_ranges(lengths, wl), len(lengths), [1] * 7, 1, wl["titv"] / (wl["titv"] + 1))
    eng.sample(7)
    eng.apply()
    # the VCF of this run, as the CLI would have written it
    head = header_text("genome.fa", [(n.decode(), ln) for n, ln in zip(names, lengths)], "Unknown", "Unknown",
                       "Unknown").encode("latin-1")
    body = eng.download(BUF_VCF)
    with open(d / "c2.vcf", "wb") as fh:
        fh.write(head)
        fh.write(memoryview(body))
    text = (d / "c2.vcf").read_bytes()
    for _ in range(2):
        assert eng.load_vcf(text)
    n_recs = int(eng.stats()["n_records"])
    dev, wall = [], []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        eng.load_vcf(text)
        e1.record(stream)
        e1.synchronize()
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(e0.elapsed_time(e1))
    ms = statistics.median(dev)
    # for scale: the plain host-to-device copy of the same pageable bytes, timed the same way
    src = torch.frombuffer(bytearray(text), dtype=torch.uint8)
    dst = torch.empty(len(text), dtype=torch.uint8, device="cuda")
    copy = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        with torch.cuda.stream(stream):
            dst.copy_(src)
        e1.record(stream)
        e1.synchronize()
        copy.append(e0.elapsed_time(e1))
    del src, dst
    lines = text.count(b"\n") - head.count(b"\n")
    device = dict(text_bytes=len(text), body_lines=lines, records=n_recs, load_vcf_ms_median=round(ms, 2),
                  load_vcf_ms_min=round(min(dev), 2), load_vcf_ms_max=round(max(dev), 2),
                  host_wall_ms_median=round(statistics.median(wall), 2), text_GBps=round(len(text) / ms / 1e6, 2), reps=reps,
                  pageable_h2d_copy_ms_median=round(statistics.median(copy), 2))
    # the host path on a fixed prefix: the first host_lines lines of the body
    cut, k = len(head), 0
    while k < host_lines and cut < len(text):
        cut = text.index(b"\n", cut) + 1
        k += 1
    sub = text[:cut]
    goff = genome_offsets(lengths)
    t0 = time.perf_counter()
    recs, lit = records_from_vcf(sub, names, goff, lengths)
    t1 = time.perf_counter()
    eng.load_records(recs, lit)
    t2 = time.perf_counter()
    host = dict(subset=f"header + the first {k} body lines", subset_bytes=len(sub), records_from_vcf_s=round(t1 - t0, 3),
                load_records_s=round(t2 - t1, 3), lines_per_s=round(k / (t2 - t0)),
                scaled_to_full_file_s=round((t2 - t0) * lines / k, 1))
    # the input genome for the file-to-file runs: an apply without records is its FASTA image
    eng.load_records(recs[:0])
    eng.apply()
    with open(d / "genome.fa", "wb") as fh:
        fh.write(memoryview(eng.download(BUF_FASTA)))
        fh.write(b"\n")
    eng.close()
    return device, host


def file_to_file(d: Path, runs: int):
    wl = bench.WORKLOADS["c2"]
    env = dict(os.environ, PYTHONPATH=str(REPO))
    res = {"args": [], "vcf": []}
    for i in range(runs + 1):                  # run 0 of each arm is a warm-up (genome.fa.fai, page cache)
        for arm in ("args", "vcf"):
            tail = bench.reference_cli_args(wl) if arm == "args" else ["vcf", str(d / "c2.vcf")]
            cmd = [sys.executable, "-m", "mutation_simulator_b200", str(d / "genome.fa"), "-o", str(d / "out"), "-q",
                   "--seed", "7"] + tail
            t0 = time.perf_counter()
            subprocess.run(cmd, env=env, check=True)
            dt = time.perf_counter() - t0
            for p in d.glob("out_ms*"):
                p.unlink()
            if i:
                res[arm].append(round(dt, 3))
    return dict(fasta_in_bytes=(d / "genome.fa").stat().st_size, vcf_in_bytes=(d / "c2.vcf").stat().st_size, wall_s=res,
                median_s={k: statistics.median(v) for k, v in res.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", type=Path)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--host-lines", type=int, default=1_000_000)
    ap.add_argument("--f2f-runs", type=int, default=2)
    a = ap.parse_args()
    d = Path("/dev/shm/ms_vcf_replay_bench")
    d.mkdir(parents=True, exist_ok=True)
    try:
        device, host = measure(d, a.reps, a.host_lines)
        res = dict(card=card(), workload=bench.WORKLOADS["c2"]["desc"], device_parser=device, host_parser=host)
        if a.f2f_runs:
            res["file_to_file"] = file_to_file(d, a.f2f_runs)
    finally:
        shutil.rmtree(d, ignore_errors=True)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
