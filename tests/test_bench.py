"""bench.py --dump-outputs: what the last timed step computed, written so that two builds can be compared."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import bench
from mutation_simulator_b200.engine import BUF_FASTA, BUF_VCF

REPO = Path(__file__).resolve().parent.parent


class FakeEngine:
    """The one Engine call dump_outputs makes, over host arrays."""

    def __init__(self, fasta_bytes, vcf_bytes):
        rng = np.random.default_rng(0)
        self.bufs = {BUF_FASTA: rng.integers(0, 256, fasta_bytes, dtype=np.uint8),
                     BUF_VCF: rng.integers(0, 256, vcf_bytes, dtype=np.uint8)}

    def download(self, which):
        return self.bufs[which].copy()


def load_dump(d):
    return {p.name: np.load(p) for p in sorted(d.iterdir())}


@pytest.mark.parametrize("fasta_bytes,vcf_bytes", [(30_000_000, 5_000_000), (1000, 0)])
def test_dump_is_a_fixed_sample_of_the_outputs(tmp_path, fasta_bytes, vcf_bytes):
    eng = FakeEngine(fasta_bytes, vcf_bytes)
    bench.dump_outputs(eng, tmp_path / "a")
    bench.dump_outputs(eng, tmp_path / "b")
    a, b = load_dump(tmp_path / "a"), load_dump(tmp_path / "b")
    assert sorted(a) == ["fasta.npy", "fasta_offsets.npy", "sizes.npy", "vcf.npy", "vcf_offsets.npy"]
    assert all(a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k]) for k in a)
    assert sum(v.nbytes for v in a.values()) <= 64 * 2**20
    assert a["sizes.npy"].tolist() == [fasta_bytes, vcf_bytes]
    for name, buf in (("fasta", BUF_FASTA), ("vcf", BUF_VCF)):
        data, rows, offsets = eng.bufs[buf], a[f"{name}.npy"], a[f"{name}_offsets.npy"].astype(np.int64)
        if data.size <= bench.DUMP_WINDOWS * bench.DUMP_WINDOW:
            assert offsets.tolist() == [0] and np.array_equal(rows[0], data)
        else:
            assert rows.shape == (bench.DUMP_WINDOWS, bench.DUMP_WINDOW) and (np.diff(offsets) >= 0).all()
            for off, row in zip(offsets, rows):
                assert np.array_equal(row.astype(np.uint8), data[off:off + bench.DUMP_WINDOW])


def run_bench(out_dir, steps):
    cmd = [sys.executable, str(REPO / "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--workload", "c1",
           "--no-e2e", "--no-cpu", "--no-f2f", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return load_dump(out_dir)


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    """Same arguments, same dump; one more timed step draws a new seed, so the last step's outputs change."""
    a, b, c = run_bench(tmp_path / "a", 2), run_bench(tmp_path / "b", 2), run_bench(tmp_path / "c", 3)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert a["sizes.npy"][0] > 10_000_000 and a["sizes.npy"][1] > 0
    assert not np.array_equal(a["vcf.npy"], c["vcf.npy"])
