#!/usr/bin/env python3
"""bench.py — mutated genome Gbp/s on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c2|c1|c3|c4|c4d|c5|c1g]
                    [--dump-outputs DIR]

A step = one pass of the hot path over the whole synthetic genome: sample -> resolve -> link -> plan ->
splice/emit FASTA image -> format VCF, all on the GPU (IT workloads: breakpoints -> exchange -> swap splice).
`value`   : input bases / device time with the genome already resident in HBM.
`e2e`     : the same through the C ABI with HOST buffers — pinned H2D of the genome, D2H of the FASTA image and
            the VCF body inside the timed region (ms_mutate_streamed).
`roofline`: the splice/emit kernel's algorithmic bytes / its CUDA-event time vs the measured HBM copy bandwidth
            (MEASURED_PEAKS.json); `roofline.emit` = splice + VCF kernels together (what the north star names).
`configs` : every BASELINE.json config (C1..C5, plus a 1 Gbp single contig) measured for a few steps each.
`cpu_baseline`: the UNMODIFIED reference (oracle/_ref, see oracle/make_ref.py) on C1 in full, one process (the
            reference is single-threaded Python); `cpu_baseline_port`: the C oracle port on a bounded sample.
`partition_invariant` (N > 1): every rank hashes its slices of the outputs on the device, rank 0 recomputes the
            whole genome alone with the same seed and compares — the N-GPU result IS the 1-GPU result.
`--impl reference`: the reference's own CPU implementation on all host cores (one process per contig).
`--dump-outputs DIR`: after the timed steps, the FASTA image and VCF body of the last one as float32 .npy files (see
            dump_outputs), so that two builds can be compared output for output on the same seeded inputs.
N > 1 (torchrun): contigs are partitioned over ranks (LPT by length, no data-path collective; for an IT pair that
straddles ranks the splice kernel reads the partner's intervals in place from the peer GPU over NVLink, or —
MS_IT_EXCHANGE=pull|nccl — they are copied / sent into a staging region); genomes with fewer contigs than ranks are cut at output
tile boundaries (ms_apply_window).  Total work is fixed, so scaling is "strong".
"""
from __future__ import annotations

import argparse
import json
import os
import random
import shutil
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

GRCH38 = [248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717,
          133797422, 135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285,
          58617616, 64444167, 46709983, 50818468, 156040895, 57227415]
GRCH38_NAMES = [f"chr{i}" for i in range(1, 23)] + ["chrX", "chrY"]
ALL_TYPES = dict(rates6=[0.01, 0.001, 0.001, 0.0005, 0.0005, 0.0005], minlen=[1, 1, 1, 2, 1, 1, 1],
                 maxlen=[1, 10, 10, 50, 50, 50, 50], titv=2.0)

WORKLOADS = {
    # BASELINE.json configs[1]: ARGS, all mutation types, GRCh38-shaped 3.1 Gbp / 24 contigs
    "c2": dict(kind="args", desc="C2: ARGS all types (sn .01 titv 2 in/de .001 len<=10, du/iv/tl .0005 len<=50) on synthetic GRCh38-shaped 3.088 Gbp, 24 contigs",
               lengths=GRCH38, names=GRCH38_NAMES, n_fraction=0.03, telomere=10000, **ALL_TYPES),
    # BASELINE.json configs[0]: the reference's CPU-runnable case
    "c1": dict(kind="args", desc="C1: ARGS sn .01 in/de .001 len 1-10 on a synthetic 10 Mbp contig",
               lengths=[10_000_000], names=["chr1"], rates6=[0.01, 0.001, 0.001, 0.0, 0.0, 0.0],
               minlen=[1, 1, 1, 2, 1, 1, 1], maxlen=[1, 10, 10, 3, 2, 2, 2], titv=1.0, n_fraction=0.0, telomere=0),
    # BASELINE.json configs[2]: RMT mode, 10 k hot/cold ranges + blocked centromeres, through from_rmt -> plan.build_ranges
    "c3": dict(kind="rmt", desc="C3: RMT on the GRCh38-shaped genome: 10k non-overlapping hot (sn .05 in/de .005 du/iv/tl .001) / cold (sn 1e-4) ranges, "
                                "std sn .001, one None range over each centromere",
               lengths=GRCH38, names=GRCH38_NAMES, n_fraction=0.03, telomere=10000, n_rmt_ranges=10_000),
    # BASELINE.json configs[3]: interchromosomal translocations on the 24-contig genome
    "c4": dict(kind="it", desc="C4: IT rate 1e-7 on the GRCh38-shaped genome (ceil(24/3) = 8 pairs like the reference's pairing; cross-GPU partners read in place over NVLink)",
               lengths=GRCH38, names=GRCH38_NAMES, n_fraction=0.03, telomere=10000, it_rate=1e-7),
    "c4d": dict(kind="it", desc="C4 dense: IT rate 1e-5 on the GRCh38-shaped genome (~2 k breakpoints per pair)",
                lengths=GRCH38, names=GRCH38_NAMES, n_fraction=0.03, telomere=10000, it_rate=1e-5),
    # BASELINE.json configs[4]: many small contigs
    "c5": dict(kind="args", desc="C5: ARGS all types on 200k contigs x 5 kbp",
               lengths=[5000] * 200_000, names=None, n_fraction=0.0, telomere=0, **ALL_TYPES),
    # the reference's own benchmark shape (README.md:441): ONE 1 Gbp contig — cut at tile boundaries over the GPUs
    "c1g": dict(kind="args", desc="C1G: ARGS all types on ONE synthetic 1 Gbp contig (README.md:441 shape); N > 1: tile-sharded apply",
                lengths=[1_000_000_000], names=["chr1"], n_fraction=0.0, telomere=0, **ALL_TYPES),
}
GENOME_SEED = 12345


def type_cdf(rates6):
    rates = list(rates6[:5]) + [rates6[5] / 2, rates6[5] / 2]     # rmt.py:91-94
    total = sum(rates)
    cdf = np.cumsum(np.array(rates) / total)
    return (cdf / cdf[-1]).tolist(), total


def make_ranges(lengths, wl):
    from mutation_simulator_b200._lib import MsRange
    cdf, total = type_cdf(wl["rates6"])
    arr = (MsRange * max(1, len(lengths)))()
    for i, L in enumerate(lengths):
        a = arr[i]
        a.contig, a.start, a.stop, a.k, a.limit = i, 0, L - 1, int(((L - 1) + 1) * total), L   # mutator.py:225
        for t in range(7):
            a.cdf[t], a.minlen[t], a.maxlen[t] = cdf[t], wl["minlen"][t], wl["maxlen"][t]
    return arr


class LenFasta:
    """The part of the Fasta surface SimulationSettings reads (contig names and lengths) for a synthetic genome."""

    class _Rec:
        def __init__(self, name, n):
            self.name, self.long_name, self._n = name, name, n

        def __len__(self):
            return self._n

    def __init__(self, names, lengths):
        self.names, self.long_names = list(names), list(names)
        self.lengths = np.asarray(lengths, dtype=np.int64)
        self.goff = np.concatenate(([0], np.cumsum(self.lengths)[:-1])).astype(np.int64)
        self._recs = [self._Rec(n, int(L)) for n, L in zip(names, lengths)]
        self._by_name = {r.name: r for r in self._recs}

    def keys(self):
        return list(self.names)

    def __getitem__(self, k):
        return self._recs[k] if isinstance(k, (int, np.integer)) else self._by_name[k]

    def close(self):
        pass


def c3_rmt_text(lengths, n_ranges, n_fraction, seed=3):
    """10 k sorted, non-overlapping 10-100 kbp ranges (alternating hot / cold) over the contigs in proportion to their
    length, and one None range over each contig's centromere-like N run (where ms_genome_synth puts it)."""
    rng = np.random.default_rng(seed)
    total = float(sum(lengths))
    hot = "sn 0.05 in 0.005 inmin 1 inmax 10 de 0.005 demin 1 demax 10 du 0.001 dumin 1 dumax 50 iv 0.001 ivmin 2 ivmax 50 tl 0.001 tlmin 1 tlmax 50"
    cold = "sn 0.0001"
    out = ["titv=2.0", "species_name=synthetic", "assembly_name=GRCh38-shaped", "sample_name=bench", "std", "it None", "sn 0.001", ""]
    n_total, flip = 0, 0
    for ci, L in enumerate(lengths):
        n_r = max(1, int(round(n_ranges * L / total)))
        slot = L // n_r
        cen_lo, cen_hi = (L * 2) // 5, (L * 2) // 5 + int(n_fraction * L)      # 0-based [lo, hi)
        rows = [(cen_lo + 1, cen_hi, "None")] if cen_hi > cen_lo else []
        for s in range(n_r):
            ln = int(rng.integers(10_000, min(100_000, slot - 2) + 1))
            a = s * slot + int(rng.integers(0, slot - ln)) + 1                  # 1-based inclusive
            b = a + ln - 1
            if b >= cen_lo + 1 and a <= cen_hi:                                # would touch the blocked centromere
                continue
            rows.append((a, b, hot if flip % 2 == 0 else cold))
            flip += 1
        rows.sort()
        out.append(f"chr {ci + 1}")
        out += [f"{a}-{b} {txt}" for a, b, txt in rows]
        n_total += len(rows)
    return "\n".join(out) + "\n", n_total


def lpt_partition(lengths, n):
    """Longest-processing-time bin packing of contigs onto n ranks (SURVEY.md §8e)."""
    from mutation_simulator_b200.distributed import lpt_partition as f
    return f(lengths, n)


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, polled through NVML every ~2 ms
    (the timed region is tens of milliseconds, too short for `nvidia-smi -lms`)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, device):
        self.device, self.samples, self.mask, self.max_mhz, self._stop, self._t = device, [], 0, None, False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            # torch's device order follows CUDA_VISIBLE_DEVICES; map through the UUID-less common case (same order)
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[device]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else device
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.nv, self.err = None, str(e)

    def _loop(self):
        nv = self.nv
        while not self._stop:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:  # noqa: BLE001
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"nvml unavailable: {getattr(self, 'err', '')}"], "samples": 0}
        self._stop = True
        self._t.join(timeout=2)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for bit, n in self.REASONS.items() if self.mask & bit), "samples": len(self.samples)}


def reduce_over_ranks(values, op, world):
    """max / sum of a list of floats over the ranks (device-timed numbers are the max over ranks)."""
    if world == 1:
        return list(values)
    import torch
    import torch.distributed as dist
    dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
    t = torch.tensor(values, dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return t.tolist()


def measured_peak():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------
# CPU arms: the unmodified reference (oracle/_ref) and the C oracle port
# ---------------------------------------------------------------------------------------
def cpu_run(lengths, names, wl, seed, threads):
    """One pass of the C oracle port (sample + walk + wrap + VCF) over a host genome."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import c_oracle
    c_oracle.lib()
    cdf, total = type_cdf(wl["rates6"])
    rng = np.random.default_rng(12345)
    seqs = [rng.choice(np.frombuffer(b"ACGT", np.uint8), L).tobytes() for L in lengths]

    def one(i):
        L = lengths[i]
        r = dict(start=0, stop=L - 1, k=int(L * total), cdf=cdf, minlen=wl["minlen"], maxlen=wl["maxlen"])
        fa, vcf, counts, _ = c_oracle.mutate_contig(seqs[i], names[i].encode(), names[i].encode(), 60, [r], [1] * 7, 1,
                                                    wl["titv"], seed + i)
        return len(fa) + len(vcf)

    def run():
        t0 = time.perf_counter()
        if threads > 1:
            with ThreadPoolExecutor(threads) as ex:
                list(ex.map(one, range(len(lengths))))
        else:
            for i in range(len(lengths)):
                one(i)
        return time.perf_counter() - t0
    return run


def scaled_sample(wl, target_bases):
    """Bounded sample of the workload: same contig count/shape, lengths scaled down."""
    lengths = wl["lengths"]
    tot = sum(lengths)
    if tot <= target_bases:
        return list(lengths), 1.0
    f = target_bases / tot
    return [max(1000, int(L * f)) for L in lengths], f


def reference_available() -> bool:
    return (REPO / "oracle" / "_ref" / "mutation_simulator" / "mutator.py").exists()


def reference_cli_args(wl):
    r6 = wl["rates6"]
    argv = ["args", "-sn", str(r6[0]), "-titv", str(wl["titv"])]
    for flag, rate, t in (("in", r6[1], 1), ("de", r6[2], 2), ("iv", r6[3], 3), ("du", r6[4], 4), ("tl", r6[5], 5)):
        if rate > 0:
            argv += [f"-{flag}", str(rate), f"-{flag}min", str(wl["minlen"][t]), f"-{flag}max", str(wl["maxlen"][t])]
    return argv


def write_host_fasta(path, name, L, seed):
    rng = np.random.default_rng(seed)
    seq = rng.choice(np.frombuffer(b"ACGT", np.uint8), L)
    full, rest = divmod(L, 60)
    with open(path, "wb") as fh:
        fh.write(b">" + name.encode() + b"\n")
        if full:
            body = np.empty((full, 61), np.uint8)
            body[:, :60] = seq[:full * 60].reshape(full, 60)
            body[:, 60] = 10
            fh.write(body.tobytes())
        if rest:
            fh.write(seq[full * 60:].tobytes() + b"\n")


def reference_processes(work, lengths, names, wl, seed):
    """One process of the UNMODIFIED reference CLI per contig file, all started together (the reference itself is
    single-threaded: this is the most the host's cores can do for it).  Returns the wall time."""
    cli = reference_cli_args(wl)
    t0 = time.perf_counter()
    procs = []
    for i in range(len(lengths)):
        cmd = [sys.executable, str(REPO / "oracle" / "ref_worker.py"), str(seed + i), str(work / f"{names[i]}.fa"), "-o",
               str(work / f"o_{names[i]}"), "-q"] + cli
        procs.append(subprocess.Popen(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE))
    for p in procs:
        _, err = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("reference run failed: " + err.decode(errors="replace")[-400:])
    return time.perf_counter() - t0


def reference_arm(args, wl, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores, on a bounded
    sample of the same workload (lengths scaled; the reference is linear in sequence length, README.md:438-441)."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    if wl["kind"] != "args":
        wl = dict(WORKLOADS["c2"], desc=wl["desc"] + " [reference arm runs the ARGS flags of C2 on the same genome shape]")
    base = {"impl": "reference", "metric": "mutated genome Gbp/s", "unit": "Gbp/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": {"workload": wl["desc"], "l2": "n/a (CPU)"}}
    n_runs = max(1, args.steps) + max(0, min(args.warmup, 1))
    if reference_available():
        # ~0.45 Mbp/s per process with all mutation types; the whole arm should end within ~3 minutes
        procs = min(cores, len(wl["lengths"]))
        budget_s = 150.0 / n_runs
        per_proc = max(20_000, int(0.45e6 * budget_s))
        lengths, f = scaled_sample(wl, min(sum(wl["lengths"]), per_proc * procs))
        if len(lengths) > cores:          # many small contigs: one file per core, contigs concatenated per file
            lengths, f = [sum(lengths) // cores] * cores, sum(lengths) / sum(wl["lengths"])
        names = (wl["names"] or [f"ctg{i}" for i in range(len(lengths))])[:len(lengths)]
        work = Path(tempfile.mkdtemp(prefix="ms_ref_", dir="/dev/shm" if Path("/dev/shm").is_dir() else None))
        try:
            for i, L in enumerate(lengths):
                write_host_fasta(work / f"{names[i]}.fa", names[i], L, 100 + i)
            for _ in range(max(0, min(args.warmup, 1))):
                reference_processes(work, lengths, names, wl, 1)
            ts = [reference_processes(work, lengths, names, wl, 10 + s) for s in range(max(1, args.steps))]
        finally:
            shutil.rmtree(work, ignore_errors=True)
        t = float(np.mean(ts))
        val = sum(lengths) / t / 1e9
        kind, used = "reference", len(lengths)
        sample = (f"UNMODIFIED reference (oracle/_ref = /root/reference 3.0.2, pyfaidx served by the in-memory stand-in), one "
                  f"`mutation-simulator FILE args ...` process per contig, all {used} started together on a {cores}-core host; "
                  f"workload scaled x{f:.4f} = {sum(lengths)/1e6:.1f} Mbp per step (FASTA in /dev/shm -> .fa + .vcf)")
    else:
        threads = min(cores, len(wl["lengths"]))
        lengths, f = scaled_sample(wl, 400_000_000)
        names = wl["names"] or [f"ctg{i}" for i in range(len(lengths))]
        run = cpu_run(lengths, names, wl, 1, threads)
        for _ in range(max(0, min(args.warmup, 1))):
            run()
        ts = [run() for _ in range(max(1, args.steps))]
        t = float(np.mean(ts))
        val = sum(lengths) / t / 1e9
        kind, used = "port", threads
        sample = (f"oracle/_ref absent: oracle/ms_oracle.c (C port of the reference's path) on the workload scaled x{f:.3f} = "
                  f"{sum(lengths)/1e6:.0f} Mbp, one contig per thread")
    line = dict(base, value=val, ms_per_step=t * 1e3,
                cpu_baseline={"value": val, "unit": "Gbp/s", "cores": used, "kind": kind, "sample": sample},
                e2e={"value": val, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    print(json.dumps(line))


def cpu_baselines(wl):
    """Rank 0, N = 1: (a) the unmodified reference on C1 IN FULL (10 Mbp, one process = one core; the reference cannot
    use more), (b) the C oracle port on a bounded sample of this workload, one thread."""
    out = {}
    c1 = WORKLOADS["c1"]
    if reference_available():
        work = Path(tempfile.mkdtemp(prefix="ms_ref_", dir="/dev/shm" if Path("/dev/shm").is_dir() else None))
        try:
            write_host_fasta(work / "chr1.fa", "chr1", c1["lengths"][0], 100)
            t = reference_processes(work, c1["lengths"], ["chr1"], c1, 42)
        finally:
            shutil.rmtree(work, ignore_errors=True)
        out["cpu_baseline"] = {"value": c1["lengths"][0] / t / 1e9, "unit": "Gbp/s", "cores": 1, "kind": "reference",
                               "sample": f"UNMODIFIED reference (oracle/_ref, pyfaidx stand-in) on C1 in full: 10 Mbp, `args -sn .01 -in .001 -de .001 "
                                         f"len 1-10 -q`, FASTA in /dev/shm -> .fa + .vcf, {t:.1f} s wall incl. interpreter start, one process "
                                         f"(the reference is single-threaded; host has {os.cpu_count()} cores; it is linear in sequence "
                                         f"length, README.md:438-441, so this rate is what {wl['desc'].split(':')[0]} would see)"}
    if wl["kind"] == "args":
        lens_s, f = scaled_sample(wl, 200_000_000)
        nm = wl["names"] or [f"ctg{i}" for i in range(len(lens_s))]
        run = cpu_run(lens_s, nm, wl, 1, 1)
        tcpu = run()
        port = {"value": sum(lens_s) / tcpu / 1e9, "unit": "Gbp/s", "cores": 1, "kind": "port",
                "sample": f"oracle/ms_oracle.c (C restatement of the path), 1 thread, workload scaled x{f:.3f} = {sum(lens_s)/1e6:.0f} Mbp in {tcpu:.1f} s"}
        out["cpu_baseline_port"] = port
        out.setdefault("cpu_baseline", port)
    return out


# ---------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------
class Run:
    """One workload on this rank's GPU: genome synthesis (keyed by GLOBAL contig id), ranges, step()."""

    def __init__(self, name, rank, world, local_rank, stream):
        from mutation_simulator_b200 import distributed as D
        from mutation_simulator_b200.engine import Engine
        self.name, self.wl, self.rank, self.world = name, WORKLOADS[name], rank, world
        wl = self.wl
        self.lengths_all = list(wl["lengths"])
        self.names_all = wl["names"] or [f"ctg{i}" for i in range(len(self.lengths_all))]
        self.total_bases = sum(self.lengths_all)
        self.mode = D.shard_mode(self.lengths_all, world) if wl["kind"] != "it" else "contigs"
        self.tiles = world > 1 and self.mode == "tiles"
        self.mine = lpt_partition(self.lengths_all, world)[rank] if world > 1 and not self.tiles else list(range(len(self.lengths_all)))
        self.eng = Engine(local_rank)
        self.eng.set_stream(stream.cuda_stream)
        self.n_ranges = None
        self.it = None
        self._setup(self.eng, self.mine)

    def _synth(self, eng, ids):
        wl = self.wl
        names = [self.names_all[i].encode() for i in ids]
        eng.synth_genome(GENOME_SEED, [self.lengths_all[i] for i in ids], [60] * len(ids), names, names, wl["n_fraction"],
                         wl["telomere"], gid=ids)

    def _setup(self, eng, ids):
        """Make `ids` (global contig indices) resident on `eng` and install the sampling table."""
        from mutation_simulator_b200 import plan
        wl = self.wl
        self.lengths = [self.lengths_all[i] for i in ids]
        if wl["kind"] == "it":
            self._setup_it(eng, ids)
            return
        self._synth(eng, ids)
        if wl["kind"] == "args":
            self._ranges = (make_ranges(self.lengths, wl), len(ids), [1] * 7, 1, wl["titv"] * (1 / (wl["titv"] + 1)))
            self.n_ranges = len(self.lengths_all)
        else:   # rmt: the real parser and planner (from_rmt -> plan.build_ranges), on the global contig table
            from mutation_simulator_b200.rmt import SimulationSettings
            if not hasattr(self, "_sim"):
                text, _ = c3_rmt_text(self.lengths_all, wl["n_rmt_ranges"], wl["n_fraction"])
                with tempfile.NamedTemporaryFile("w", suffix=".rmt", delete=False) as fh:
                    fh.write(text)
                try:
                    self._sim = SimulationSettings.from_rmt(Path(fh.name), LenFasta(self.names_all, self.lengths_all), True)
                finally:
                    os.unlink(fh.name)
            sim = self._sim
            arr, n = plan.build_ranges(sim, self.lengths_all, ids)
            self._ranges = (arr, n, plan.block_list(sim), min(sim.mut_block.values()), plan.p_transition(sim.titv))
            self.n_ranges = sum(len(c.range_definitions) for c in sim.chromosomes)
        eng.set_ranges_array(*self._ranges)

    # -- IT ------------------------------------------------------------------------------
    def _setup_it(self, eng, ids):
        from argparse import Namespace
        from mutation_simulator_b200.it_mutator import ITMutator
        from mutation_simulator_b200.rmt import SimulationSettings
        run = self

        class SynthFasta(LenFasta):
            def upload(self, engine, contig_ids=None):
                run._synth(engine, list(range(len(self.names))) if contig_ids is None else list(contig_ids))
        fasta = SynthFasta(self.names_all, self.lengths_all)
        sim = SimulationSettings.from_it(self.wl["it_rate"], fasta, True)
        args = Namespace(outfastait=os.devnull, outbedpe=os.devnull, ignore_warnings=True, no_color=True, seed=777, device=eng.device)
        it = ITMutator.__new__(ITMutator)            # no output files: the bench keeps the image in HBM
        it._args, it._fasta, it._sim = args, fasta, sim
        it._rank, it._world = (self.rank, self.world) if eng is self.eng else (0, 1)
        it._fasta_writer = it._bedpe_writer = None
        it._seed = 777
        it._rng = random.Random(777)
        from mutation_simulator_b200.it_mutator import assign_partners
        it._partners = assign_partners([c.number for c in sim.chromosomes if c.it_rate is not None and len(fasta[c.number]) > 2], it._rng)
        it._engine, it.breakpoints, it._replay = eng, {}, None
        fasta.engine = eng
        if it._world > 1:
            it.setup_partitioned()
        else:
            fasta.upload(eng)
        if eng is self.eng:
            self.it = it
        else:
            self._it_full = it
        self.n_ranges = len(it._partners) // 2

    def _it_step(self, it, seed):
        it._seed = seed
        if it._world > 1:
            it.step_partitioned()
        else:
            bps = it.breakpoints = it._generate_all_breakpoints(it._engine)
            it._engine.load_records(it._records(bps))
            it._engine.apply()

    # -- one step --------------------------------------------------------------------------
    def step(self, seed):
        if self.it is not None:
            self._it_step(self.it, seed)
            return self.eng.size_of(0), 0
        self.eng.sample(seed)
        if self.tiles:
            w = self.eng.apply_window(self.rank, self.world)
            self.window = w
            return w["fasta_bytes"], w["vcf_bytes"]
        return self.eng.apply()

    # -- partition invariance ----------------------------------------------------------------
    def output_hashes(self, eng, ids, window=None):
        """{"fasta:<global contig>" | "vcf:<global contig>" | "<kind>:<lo>:<hi>": hash}: per contig (header + body of the
        FASTA slice, VCF lines) or, for a tile-sharded run, per window of the (rank-independent) output layout."""
        from mutation_simulator_b200.engine import BUF_FASTA, BUF_VCF
        out = {}
        if window is not None:
            for kind, buf in (("fasta", BUF_FASTA), ("vcf", BUF_VCF)):
                lo, hi = window[kind]
                if hi > lo:
                    out[f"{kind}:{lo}:{hi}"] = int(eng.hash_ranges(buf, [lo], [hi])[0])
            return out
        fo, vo, sep, _ = eng.contig_layout()
        hf = eng.hash_ranges(BUF_FASTA, fo[:-1], fo[1:] - sep.astype(np.int64))
        for i, g in enumerate(ids):
            out[f"fasta:{int(g)}"] = int(hf[i])
        if self.wl["kind"] != "it":
            hv = eng.hash_ranges(BUF_VCF, vo[:-1], vo[1:])
            for i, g in enumerate(ids):
                out[f"vcf:{int(g)}"] = int(hv[i])
        return out

    def partition_invariant(self, seed, local_rank):
        """All ranks hash the outputs of step(seed) on their devices; rank 0 recomputes the WHOLE genome alone with the
        same seed (untimed) and compares.  True iff every slice of every rank equals the single-GPU result."""
        import torch.distributed as dist
        from mutation_simulator_b200.engine import BUF_FASTA, BUF_VCF, Engine
        self.step(seed)
        mine = self.output_hashes(self.eng, self.mine, self.window if self.tiles else None)
        gathered = [None] * self.world
        dist.all_gather_object(gathered, mine)
        got = {}
        for g in gathered:
            got.update(g)
        verdict = [None]
        if self.rank == 0:
            full = Engine(local_rank)
            keep = getattr(self, "_ranges", None)
            try:
                all_ids = list(range(len(self.lengths_all)))
                self._setup(full, all_ids)
                if self.wl["kind"] == "it":
                    self._it_step(self._it_full, seed)
                else:
                    full.sample(seed)
                    full.apply()
                if self.tiles:
                    want = {}
                    for k in got:
                        kind, lo, hi = k.split(":")
                        want[k] = int(full.hash_ranges(BUF_FASTA if kind == "fasta" else BUF_VCF, [int(lo)], [int(hi)])[0])
                    covered = sorted((int(k.split(":")[1]), int(k.split(":")[2])) for k in got if k.startswith("fasta:"))
                    whole = bool(covered) and covered[0][0] == 0 and covered[-1][1] == full.size_of(BUF_FASTA) and \
                        all(a[1] == b[0] for a, b in zip(covered, covered[1:]))
                else:
                    want = self.output_hashes(full, all_ids)
                    whole = True
                verdict[0] = bool(whole and len(got) == len(want) and all(got.get(k) == v for k, v in want.items()))
            finally:
                full.close()
                self._ranges = keep
                self.lengths = [self.lengths_all[i] for i in self.mine]
        dist.broadcast_object_list(verdict, src=0)
        return verdict[0]

    def close(self):
        self.eng.close()


def measure(run: Run, steps, warmup, barrier, stream, local_rank, with_clocks=False):
    """W warm-up steps, then exactly K timed steps bracketed by barrier + synchronize; CUDA events on the engine's
    stream; max over ranks."""
    import torch
    eng, world = run.eng, run.world
    for w in range(warmup):
        run.step(1000 + w)
    barrier()
    sampler = ClockSampler(local_rank) if with_clocks else None
    if sampler:
        sampler.start()
    launches0 = eng.stats()["kernel_launches"]
    stage_acc, ex_ms, ex_bytes = {}, 0.0, 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    t0 = time.perf_counter()
    sizes = (0, 0)
    for s in range(steps):
        sizes = run.step(2000 + s)
        st = eng.stats()
        for k, v in st["stage_ms"].items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v
        if run.it is not None and world > 1:
            ex_ms += run.it.exchange_ms
            ex_bytes += run.it.exchange_bytes
    ev1.record(stream)
    barrier()
    wall = time.perf_counter() - t0
    dev_ms = ev0.elapsed_time(ev1)
    if run.it is not None:       # IT steps contain host work (breakpoint download, record build): wall clock is the honest one
        dev_ms = max(dev_ms, wall * 1e3)
    clocks = sampler.stop() if sampler else None
    st = eng.stats()
    launches = st["kernel_launches"] - launches0
    dev_ms = reduce_over_ranks([dev_ms], "max", world)[0]
    launches = int(reduce_over_ranks([float(launches)], "sum", world)[0])
    ms_per_step = dev_ms / steps
    res = {"value": run.total_bases / (ms_per_step * 1e-3) / 1e9, "ms_per_step": ms_per_step, "launches": launches,
           "stage_ms": {k: v / steps for k, v in stage_acc.items()}, "sizes": sizes, "stats": st, "clocks": clocks,
           "wall_ms_per_step": wall / steps * 1e3}
    if run.it is not None and world > 1:
        exm, exb = reduce_over_ranks([ex_ms / steps], "max", world)[0], reduce_over_ranks([float(ex_bytes) / steps], "sum", world)[0]
        route = getattr(run.it, "_route", "nccl")
        res["exchange"] = {"ms_per_step": exm if route == "nccl" else None, "bytes_per_step": int(exb), "route": route,
                           "transport": {"nccl": "NCCL P2P (batch_isend_irecv) into a staging region, odd intervals only",
                                         "pull": "copy engine, peer genome mapped with CUDA IPC -> staging region, odd intervals only",
                                         "direct": "none: k_splice gathers the odd intervals from the peer's HBM (CUDA IPC "
                                                   "mapping) over NVLink; bytes_per_step = bytes read remotely"}[route]}
    return res


DUMP_SEED = 2024
DUMP_WINDOWS, DUMP_WINDOW = 1024, 4096        # per output: 4 MiB of bytes, 16 MiB as float32


def dump_outputs(eng, out_dir: Path):
    """Write what a caller of the last step receives: the FASTA image and the VCF body.  An output of at most
    DUMP_WINDOWS * DUMP_WINDOW bytes is written whole, as one row; a larger one as DUMP_WINDOWS rows of DUMP_WINDOW
    consecutive bytes at offsets drawn from its size with a fixed seed.  Files: fasta.npy / vcf.npy (byte values as
    float32, one row per window), fasta_offsets.npy / vcf_offsets.npy (float64, where each row starts), sizes.npy
    (float64: FASTA bytes, VCF bytes).  Under 33 MiB in all."""
    from mutation_simulator_b200.engine import BUF_FASTA, BUF_VCF
    out_dir.mkdir(parents=True, exist_ok=True)
    sizes = []
    for name, buf in (("fasta", BUF_FASTA), ("vcf", BUF_VCF)):
        data = eng.download(buf)
        sizes.append(len(data))
        if len(data) <= DUMP_WINDOWS * DUMP_WINDOW:
            offsets, rows = np.zeros(1, np.int64), data[None, :]
        else:
            rng = np.random.default_rng([DUMP_SEED, buf])
            offsets = np.sort(rng.integers(0, len(data) - DUMP_WINDOW + 1, DUMP_WINDOWS))
            rows = data[offsets[:, None] + np.arange(DUMP_WINDOW)]
        np.save(out_dir / f"{name}.npy", rows.astype(np.float32))
        np.save(out_dir / f"{name}_offsets.npy", offsets.astype(np.float64))
    np.save(out_dir / "sizes.npy", np.array(sizes, np.float64))


def roofline_of(run: Run, res):
    """k_splice: algorithmic bytes (SURVEY.md §8d: L + L' + ceil(L'/bpl) + 32 M + sum of TLI sources) / CUDA-event time
    of the stage, this rank's share; `emit` adds the VCF kernel (32 M read + line bytes written)."""
    st, wl = res["stats"], run.wl
    fasta_bytes, vcf_bytes = res["sizes"]
    my_bases = sum(run.lengths) if not run.tiles else run.total_bases / run.world
    share = 1.0 if not run.tiles else 1.0 / run.world
    hdr_bytes = sum(len(run.names_all[i]) + 2 for i in run.mine) * share
    recs_n = st["n_records"] * share
    counts = st["counts"]
    splice_ms = res["stage_ms"].get("splice_emit_fasta", 0.0)
    vcf_ms = res["stage_ms"].get("vcf_format", 0.0)
    tli_src = 25.5 * counts[6] * share if wl.get("maxlen", [0] * 7)[5] == 50 else 0.0          # E[len] of the TLI gathers
    alg = my_bases + (fasta_bytes * share - hdr_bytes) + 32 * recs_n + tli_src
    alg_vcf = 32 * recs_n + vcf_bytes * share
    peak, peak_src = measured_peak()
    ach = alg / (splice_ms * 1e-3) / 1e9 if splice_ms > 0 else 0.0
    both_ms = splice_ms + vcf_ms
    ach_both = (alg + alg_vcf) / (both_ms * 1e-3) / 1e9 if both_ms > 0 else 0.0
    traffic, traffic_src = None, None
    tf = REPO / "profiles" / "k_splice_traffic.json"
    if tf.exists() and run.name == "c2" and run.world == 1:   # ncu --set full capture of this kernel on this workload
        t_ = json.loads(tf.read_text())
        traffic = t_["dram_bytes_read"] + t_["dram_bytes_write"]
        traffic_src = t_.get("capture")
    return {"bound": "hbm", "kernel": "k_splice", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak if peak else None,
            "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "alg_bytes_per_launch": alg, "kernel_ms": splice_ms,
            "emit": {"kernels": "k_splice + k_vcf_write", "alg_bytes": alg + alg_vcf, "ms": both_ms, "achieved": ach_both,
                     "frac": ach_both / peak if peak else None},
            "all_kernels_frac": ((my_bases + fasta_bytes * share + vcf_bytes * share + 64 * recs_n) / (res["ms_per_step"] * 1e-3) / 1e9) / peak}


def file_to_file(args, wl, rank, world, lengths_all, names_all, total_bases):
    """The drop-in path end to end on files.  The input FASTA is the synthetic genome wrapped at 60 columns
    (built once, untimed, by applying an empty mutation table); the timed part is what a CLI user waits for."""
    import torch
    from mutation_simulator_b200 import Mutator, SimulationSettings, get_args, load_fasta
    from mutation_simulator_b200.engine import BUF_FASTA, Engine
    from mutation_simulator_b200.records import REC_DTYPE
    base = Path("/dev/shm") if Path("/dev/shm").is_dir() else Path(tempfile.gettempdir())
    d = base / f"ms_bench_{os.environ.get('MASTER_PORT', '0')}_{os.getppid() if world > 1 else os.getpid()}"
    src = d / "genome.fa"
    try:
        if rank == 0:
            d.mkdir(parents=True, exist_ok=True)
            g = Engine(int(os.environ.get("LOCAL_RANK", "0")))
            g.synth_genome(4242, lengths_all, [60] * len(lengths_all), [n.encode() for n in names_all],
                           [n.encode() for n in names_all], wl["n_fraction"], wl["telomere"])
            g.load_records(np.zeros(0, dtype=REC_DTYPE))
            g.apply()
            with open(src, "wb") as fh:
                fh.write(memoryview(g.download(BUF_FASTA)))
                fh.write(b"\n")
            g.close()
        if world > 1:
            torch.distributed.barrier()
        argv = [str(src), "-o", str(d / "out"), "-q", "--seed", "7"] + reference_cli_args(wl)
        a = get_args(argv)
        a.device = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fasta = load_fasta(a.infile, device=a.device)   # FASTA ingest on the device
        t1 = time.perf_counter()
        sim = SimulationSettings.from_args(a, fasta, True)
        m = Mutator(a, fasta, sim)
        m.mutate()
        m.close()
        fasta.close()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        dt, parse = reduce_over_ranks([t2 - t0, t1 - t0], "max", world)
        out_bytes = (d / "out_ms.fa").stat().st_size + (d / "out_ms.vcf").stat().st_size if rank == 0 else 0
        return {"value": total_bases / dt / 1e9, "unit": "Gbp/s", "seconds": dt, "parse_seconds": parse,
                "in_bytes": src.stat().st_size if rank == 0 else 0, "out_bytes": out_bytes,
                "note": f"{base}: load_fasta + Mutator.mutate() writing .fa and .vcf, wall clock, max over ranks"}
    except Exception as e:  # noqa: BLE001 - the figure is auxiliary; never lose the main line over it
        return {"value": None, "error": f"{type(e).__name__}: {e}"}
    finally:
        if world > 1:
            try:
                torch.distributed.barrier()
            except Exception:  # noqa: BLE001
                pass
        if rank == 0:
            shutil.rmtree(d, ignore_errors=True)


def e2e_measure(run: Run, args, barrier, fasta_bytes, vcf_bytes):
    """HOST buffers through the C ABI: pinned genome in, FASTA image + VCF body out."""
    import torch
    from mutation_simulator_b200.engine import BUF_FASTA, BUF_VCF
    eng, world, lengths, mine = run.eng, run.world, run.lengths, run.mine
    names = [run.names_all[i].encode() for i in mine]
    my_bases = sum(lengths)
    g = torch.empty(my_bases, dtype=torch.uint8, pin_memory=True)
    gn = g.numpy()
    gn[:] = eng.download_genome()
    fa_host = torch.empty(int(fasta_bytes * 1.02) + 4096, dtype=torch.uint8, pin_memory=True).numpy()
    vcf_host = torch.empty(int(vcf_bytes * 1.05) + 4096, dtype=torch.uint8, pin_memory=True).numpy()
    n_e2e = max(2, min(args.steps, 4))

    def e2e_serial(seed):     # the same work as four separate C-ABI calls, no overlap (reported for comparison)
        eng.upload_genome(gn, lengths, [60] * len(lengths), names, names, gid=mine)
        eng.set_ranges_array(*run._ranges)
        eng.sample(seed)
        fb, vb = eng.apply()
        eng.download(BUF_FASTA, fa_host)
        eng.download(BUF_VCF, vcf_host)
        return fb, vb

    def e2e_step(seed):       # ms_mutate_streamed: H2D / kernels / D2H of successive contig groups overlap
        eng.declare_genome(lengths, [60] * len(lengths), names, names, gid=mine)
        eng.set_ranges_array(*run._ranges)
        return eng.mutate_streamed(seed, gn, fa_host, vcf_host)
    e2e_serial(1)
    barrier()
    t0 = time.perf_counter()
    e2e_serial(2)
    barrier()
    serial_ms = reduce_over_ranks([(time.perf_counter() - t0) * 1e3], "max", world)[0]
    e2e_step(1)
    barrier()
    t0 = time.perf_counter()
    for s in range(n_e2e):
        fb, vb = e2e_step(3000 + s)
    barrier()
    dt = (time.perf_counter() - t0) / n_e2e
    dt = reduce_over_ranks([dt], "max", world)[0]
    return {"value": run.total_bases / dt / 1e9, "unit": "Gbp/s", "h2d_bytes_per_step": int(my_bases),
            "d2h_bytes_per_step": int(fb + vb), "steps": n_e2e, "ms_per_step": dt * 1e3, "serial_ms_per_step": serial_ms,
            "note": "per-rank bytes; pinned host genome in, FASTA image + VCF body out; one ms_mutate_streamed call per "
                    "step (copies of successive contig groups overlap the kernels); serial_ms_per_step = the same work "
                    "as upload/sample/apply/download calls without overlap"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-f2f", action="store_true", help="skip the file-to-file measurement")
    ap.add_argument("--no-configs", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--no-invariance", action="store_true", help="skip the N-GPU == 1-GPU hash check")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write the FASTA image and VCF body of the last timed step into DIR as .npy files")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs is not None and (world > 1 or args.impl == "reference"):
        ap.error("--dump-outputs needs the GPU implementation in a single process")

    if args.impl == "reference":
        reference_arm(args, wl, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.Stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    run = Run(args.workload, rank, world, local_rank, stream)
    res = measure(run, args.steps, args.warmup, barrier, stream, local_rank, with_clocks=True)
    if args.dump_outputs is not None:          # before anything below runs more steps on the same engine
        dump_outputs(run.eng, args.dump_outputs)
    roofline = roofline_of(run, res)
    fasta_bytes, vcf_bytes = res["sizes"]
    invariant = None
    if world > 1 and not args.no_invariance:
        try:
            invariant = run.partition_invariant(2000 + args.steps - 1, local_rank)
        except Exception as e:  # noqa: BLE001
            invariant = f"error: {type(e).__name__}: {e}"

    e2e = None
    if not args.no_e2e and wl["kind"] != "it" and not run.tiles:
        e2e = e2e_measure(run, args, barrier, fasta_bytes, vcf_bytes)
    run.close()

    # every other BASELINE config, a few steps each (device-resident), same timing rules
    configs = None
    if not args.no_configs and args.workload == "c2":
        configs = {"c2": {"value": res["value"], "unit": "Gbp/s", "ms_per_step": res["ms_per_step"], "roofline_frac": roofline["frac"],
                          "emit_frac": roofline["emit"]["frac"], "n_ranges": run.n_ranges, "records_per_step": int(res["stats"]["n_records"]),
                          "partition_invariant": invariant, "workload": wl["desc"]}}
        for name in ("c1", "c3", "c4", "c4d", "c5", "c1g"):
            try:
                r2 = Run(name, rank, world, local_rank, stream)
                m2 = measure(r2, max(3, min(args.steps, 5)), 3, barrier, stream, local_rank)
                rf = roofline_of(r2, m2)
                inv = None
                if world > 1 and not args.no_invariance:
                    try:
                        inv = r2.partition_invariant(2002, local_rank)
                    except Exception as e:  # noqa: BLE001
                        inv = f"error: {type(e).__name__}: {e}"
                entry = {"value": m2["value"], "unit": "Gbp/s", "ms_per_step": m2["ms_per_step"], "roofline_frac": rf["frac"],
                         "emit_frac": rf["emit"]["frac"], "n_ranges": r2.n_ranges, "records_per_step": int(m2["stats"]["n_records"]),
                         "sharding": r2.mode if world > 1 else "single GPU", "partition_invariant": inv,
                         "stage_ms": m2["stage_ms"], "workload": r2.wl["desc"]}
                if "exchange" in m2:
                    entry["exchange"] = m2["exchange"]
                if r2.it is not None:
                    entry["timing"] = "wall clock per step (breakpoints come back to the host to build the swap records), max over ranks"
                configs[name] = entry
                r2.close()
            except Exception as e:  # noqa: BLE001
                configs[name] = {"value": None, "error": f"{type(e).__name__}: {e}"}

    # file-to-file: FASTA on (RAM-backed) disk -> load_fasta -> Mutator.mutate() -> *_ms.fa + *_ms.vcf on disk, wall clock
    f2f = None
    if not args.no_f2f and wl["kind"] == "args":
        f2f = file_to_file(args, wl, rank, world, run.lengths_all, run.names_all, run.total_bases)

    cpu = {}
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baselines(wl)

    if rank == 0:
        line = {"metric": "mutated genome Gbp/s", "value": res["value"], "unit": "Gbp/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": wl["desc"],
                           "partition": (f"output tiles over {world} rank(s) (ms_apply_window; sampling replicated)" if run.tiles
                                         else f"contigs LPT over {world} rank(s)"),
                           "l2": "inputs (>=1 GB per rank) larger than the 126 MB L2; fresh seed every step",
                           "timing": "CUDA events on the engine's stream, max over ranks"},
                "roofline": roofline, "cpu_baseline": cpu.get("cpu_baseline"), "cpu_baseline_port": cpu.get("cpu_baseline_port"),
                "e2e": e2e, "file_to_file": f2f, "gpu_launches": int(res["launches"]), "clocks": res["clocks"],
                "partition_invariant": invariant, "configs": configs,
                "stage_ms": res["stage_ms"], "records_per_step": int(res["stats"]["n_records"]),
                "wall_ms_per_step": res["wall_ms_per_step"]}
        if "exchange" in res:
            line["exchange"] = res["exchange"]
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
