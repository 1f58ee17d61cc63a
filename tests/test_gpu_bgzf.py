"""BGZF output encoded on the GPU (ms_bgzf_compress, --bgzip): members inflate to the plain outputs, sit on the
16 KiB-cell x contig-slice grid, equal the host encoder's bytes, and every CLI mode writes the plain run's content."""
import gzip
import json
import os
import shutil
import struct
import subprocess
import sys
import zlib
from pathlib import Path

import numpy as np
import pytest

from tests.helpers import GOLDEN

pytestmark = pytest.mark.gpu
REPO = Path(__file__).resolve().parent.parent
CELL = 16384


def members(z: bytes):
    """-> [(offset, member bytes)] of a BGZF stream, checking every header."""
    out, o = [], 0
    while o < len(z):
        assert z[o:o + 4] == b"\x1f\x8b\x08\x04" and z[o + 12:o + 16] == b"BC\x02\x00", o
        size = struct.unpack("<H", z[o + 16:o + 18])[0] + 1
        out.append((o, z[o:o + size]))
        o += size
    assert o == len(z)
    return out


def check_grid(z: bytes, plain: bytes, cuts, eof=True):
    """Every member's extent is a 16 KiB cell of `plain` intersected with a segment [cuts[i], cuts[i+1])."""
    from mutation_simulator_b200.bgzf import EOF
    if eof:
        assert z.endswith(EOF)
        z = z[:-len(EOF)]
    want = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        p = a
        while p < b:
            q = min(b, (p // CELL + 1) * CELL)
            want.append((p, q))
            p = q
    got, p = [], 0
    for _, m in members(z):
        isize = struct.unpack("<I", m[-4:])[0]
        crc = struct.unpack("<I", m[-8:-4])[0]
        data = zlib.decompressobj(-15).decompress(m[18:-8])
        assert len(data) == isize and zlib.crc32(data) == crc and len(m) <= isize + 31
        assert data == plain[p:p + isize]
        got.append((p, p + isize))
        p += isize
    assert got == want and p == len(plain)


def _genome(seed=3, lens=(70_001, 16_384, 5, 40_000, 1, 33_000, 16_383)):
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(b"ACGTACGTACGTN", np.uint8)
    return [(b"c%d" % i, b"c%d len=%d" % (i, n), rng.choice(alpha, n).tobytes(), 60 if i % 2 else 70) for i, n in enumerate(lens)]


def _sampled_engine():
    from tests.helpers import engine_for
    eng, _, _, lens = engine_for(_genome())
    rates = [0.01, 0.002, 0.002, 0.0005, 0.0005, 0.00025, 0.00025]
    cdf = (np.cumsum(rates) / sum(rates)).tolist()
    cdf[-1] = 1.0
    ranges = [dict(contig=i, start=0, stop=int(n) - 1, k=int(int(n) * sum(rates)), limit=int(n), cdf=cdf,
                   minlen=[1, 1, 1, 2, 1, 1, 1], maxlen=[1, 10, 10, 50, 50, 50, 50]) for i, n in enumerate(lens)]
    eng.set_ranges(ranges, [1] * 7, 1, 2.0 / 3.0)
    eng.sample(99)
    eng.apply()
    return eng


def test_engine_members_inflate_to_the_buffers_on_the_grid(tmp_path):
    from mutation_simulator_b200 import bgzf
    from mutation_simulator_b200.engine import BUF_BGZF, BUF_FASTA, BUF_VCF, bgzf_compress_host
    eng = _sampled_engine()
    fo, vo, _, _ = eng.contig_layout()
    for which, lay in ((BUF_FASTA, fo), (BUF_VCF, vo)):
        plain = eng.download(which).tobytes()
        assert len(plain) > CELL
        with open(tmp_path / "o.gz", "w+b") as fh:
            bgzf.write_from_engine(fh, eng, which)
        z = (tmp_path / "o.gz").read_bytes()
        assert gzip.decompress(z) == plain
        check_grid(z, plain, [int(x) for x in lay])
        # the device's members are the host encoder's bytes for the same blocks
        host = b"".join(bgzf_compress_host(zlib.decompress(m[18:-8], -15)) for _, m in members(z[:-len(bgzf.EOF)]))
        assert host == z[:-len(bgzf.EOF)]
        seg, tot = eng.bgzf_compress(which, lay[:-1], np.diff(lay), lay[:-1])
        assert tot == len(z) - len(bgzf.EOF) == int(seg.sum()) == eng.size_of(BUF_BGZF)
        assert eng.hash_ranges(BUF_BGZF, [0], [tot]).size == 1
    # segments at arbitrary file offsets, with the separator '\n' appended (the multi-GPU FASTA slices)
    plain = eng.download(BUF_FASTA).tobytes()
    src, n, foff, nl = [0, 100, 30_000], [100, 29_000, 50_000], [5, 16_000, 60_000], [1, 0, 1]
    seg, tot = eng.bgzf_compress(BUF_FASTA, src, n, foff, nl)
    z = eng.download(BUF_BGZF).tobytes()
    o = 0
    for s, k, f, e, zs in zip(src, n, foff, nl, seg):
        part = z[o:o + int(zs)]
        text = plain[s:s + k] + b"\n" * e
        assert gzip.decompress(part) == text
        cuts = []
        p = f
        while p < f + len(text):
            q = min(f + len(text), (p // CELL + 1) * CELL)
            cuts.append(q - p)
            p = q
        assert [struct.unpack("<I", m[-4:])[0] for _, m in members(part)] == cuts
        o += int(zs)
    assert o == tot
    with pytest.raises(Exception):
        eng.bgzf_compress(BUF_FASTA, [len(plain) - 10], [11], [0])
    eng.close()


def run_main(argv, env=None):
    from mutation_simulator_b200.__main__ import main
    old, saved = sys.argv, {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    sys.argv = ["mutation-simulator"] + [str(a) for a in argv]
    try:
        main()
    finally:
        sys.argv = old
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _no_date(vcf: bytes) -> bytes:
    return b"".join(l for l in vcf.splitlines(keepends=True) if not l.startswith(b"##filedate"))


def _body(z: bytes) -> bytes:
    """The members of a VCF.gz after the header's (header members hold only '#' lines)."""
    return b"".join(m for _, m in members(z) if not zlib.decompress(m[18:-8], -15).startswith(b"#") and len(m) > 28)


def _compare(tmp_path, base_plain, base_z, names):
    from mutation_simulator_b200.bgzf import EOF
    for nm in names:
        p = (tmp_path / f"{base_plain}{nm}").read_bytes()
        z = (tmp_path / f"{base_z}{nm}.gz").read_bytes()
        assert z.endswith(EOF), nm
        members(z)
        u = gzip.decompress(z)
        if nm.endswith(".vcf"):
            assert _no_date(u) == _no_date(p), nm
        else:
            assert u == p, nm


@pytest.mark.parametrize("mode", ["args", "rmt", "it", "rmt_it", "rmt_it_nochain"])
def test_cli_bgzip_equals_plain_run(tmp_path, mode):
    rmt_it = ["std", "it 0.002", "sn 0.01 in 0.004 inmin 1 inmax 9 de 0.004 demin 1 demax 30 du 0.002 dumin 2 dumax 12",
              "chr 2", "it 0.05", "1-41 de 0.1 demin 1 demax 3"]
    if mode == "args":
        shutil.copy(GOLDEN / "args_all" / "in.fa", tmp_path / "in.fa")
        tail = json.loads((GOLDEN / "args_all" / "cmd.json").read_text())["argv"][4:]
        outs = ["_ms.fa", "_ms.vcf"]
    elif mode == "rmt":
        shutil.copy(GOLDEN / "rmt_ranges" / "in.fa", tmp_path / "in.fa")
        shutil.copy(GOLDEN / "rmt_ranges" / "in.rmt", tmp_path / "in.rmt")
        tail = ["rmt", tmp_path / "in.rmt"]
        outs = ["_ms.fa", "_ms.vcf"]
    elif mode == "it":
        shutil.copy(GOLDEN / "it_basic" / "in.fa", tmp_path / "in.fa")
        tail = ["it", "0.004"]
        outs = ["_ms_it.fa"]
    else:
        rng = np.random.default_rng(11)
        with open(tmp_path / "in.fa", "wb") as f:
            for i, n in enumerate((50_000, 41, 73_000, 3, 61_000, 2500)):
                s = rng.choice(list(b"ACGT"), size=n).astype(np.uint8).tobytes()
                f.write(b">c%d some text\n" % i + b"".join(s[o:o + 50] + b"\n" for o in range(0, n, 50)))
        (tmp_path / "in.rmt").write_text("\n".join(rmt_it) + "\n")
        tail = ["rmt", tmp_path / "in.rmt"]
        outs = ["_ms.fa", "_ms.vcf", "_ms_it.fa"]
    env = {"MS_NO_CHAIN": "1"} if mode == "rmt_it_nochain" else {}
    common = ["-q", "-w", "--seed", "17"]
    run_main([tmp_path / "in.fa", "-o", tmp_path / "p"] + common + tail, env)
    run_main([tmp_path / "in.fa", "-o", tmp_path / "z", "--bgzip"] + common + tail, env)
    _compare(tmp_path, "p", "z", outs)
    if "it" in mode:
        assert (tmp_path / "z_ms_it.bedpe").read_bytes() == (tmp_path / "p_ms_it.bedpe").read_bytes()
    first = {nm: (tmp_path / f"z{nm}.gz").read_bytes() for nm in outs}
    run_main([tmp_path / "in.fa", "-o", tmp_path / "z", "--bgzip"] + common + tail, env)
    for nm in outs:
        b = (tmp_path / f"z{nm}.gz").read_bytes()
        if nm.endswith(".vcf"):       # the header carries the date: its members may differ, the body's may not
            assert _body(b) == _body(first[nm]) and len(_body(b)) > 0
        else:
            assert b == first[nm], nm


@pytest.mark.slow
def test_full_size_c2_shaped_genome():
    """GRCh38-shaped synthetic genome (3.1 Gbp, 24 contigs, bench.py's C2 mutation mix): the compressed outputs inflate
    to the plain ones and the FASTA shrinks at least 3.3x."""
    sys.path.insert(0, str(REPO))
    import bench
    from mutation_simulator_b200.engine import BUF_BGZF, BUF_FASTA, BUF_VCF, Engine
    wl = bench.WORKLOADS["c2"]
    lengths, names = list(wl["lengths"]), [n.encode() for n in wl["names"]]
    eng = Engine(0)
    eng.synth_genome(bench.GENOME_SEED, lengths, [60] * len(lengths), names, names, wl["n_fraction"], wl["telomere"])
    eng.set_ranges_array(bench.make_ranges(lengths, wl), len(lengths), [1] * 7, 1, wl["titv"] / (wl["titv"] + 1))
    eng.sample(7)
    eng.apply()
    fo, vo, _, _ = eng.contig_layout()
    for which, lay, ratio in ((BUF_FASTA, fo, 3.3), (BUF_VCF, vo, 1.5)):
        plain = eng.download(which)
        _, tot = eng.bgzf_compress(which, lay[:-1], np.diff(lay), lay[:-1])
        z = eng.download(BUF_BGZF).tobytes()
        assert len(z) == tot and plain.size / tot >= ratio, (which, plain.size / tot)
        out, o = [], 0
        while o < len(z):            # member by member (gzip.decompress of 1 GB holds several copies)
            size = struct.unpack("<H", z[o + 16:o + 18])[0] + 1
            out.append(zlib.decompress(z[o + 18:o + size - 8], -15))
            o += size
        assert b"".join(out) == plain.tobytes(), which
    eng.close()


def _ngpu():
    import torch
    return torch.cuda.device_count()


def _cli(argv, nproc, port, **extra_env):
    env = dict(os.environ, PYTHONPATH=str(REPO), **extra_env)
    cmd = [sys.executable, "-m", "mutation_simulator_b200"] + argv if nproc == 1 else \
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
         f"--master-port={port}", "-m", "mutation_simulator_b200"] + argv
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]


@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
def test_multi_gpu_bgzip_equals_single_gpu(tmp_path):
    from tests.test_gpu_multi import make_genome
    n = min(_ngpu(), 4)
    lens = [90_000, 70_011, 65_000, 40_000, 33_333, 20_000, 7, 1_000]
    make_genome(tmp_path / "g.fa", lens, 1)
    common = ["-q", "--seed", "77", "--bgzip", "args", "-sn", "0.01", "-in", "0.002", "-inmax", "9", "-de", "0.002", "-demax", "9",
              "-du", "0.001", "-dumax", "30", "-iv", "0.001", "-ivmax", "30", "-tl", "0.002", "-tlmax", "20"]
    for d, k, env, port in (("a", 1, {}, 0), ("b", n, {}, 29641), ("c", n, {"MS_SHARD": "tiles"}, 29642)):
        (tmp_path / d).mkdir()
        _cli([str(tmp_path / "g.fa"), "-o", str(tmp_path / d / "g")] + common, k, port, **env)
    a = {f: (tmp_path / "a" / f).read_bytes() for f in ("g_ms.fa.gz", "g_ms.vcf.gz")}
    b = {f: (tmp_path / "b" / f).read_bytes() for f in a}
    c = {f: (tmp_path / "c" / f).read_bytes() for f in a}
    assert b["g_ms.fa.gz"] == a["g_ms.fa.gz"] and c["g_ms.fa.gz"] == a["g_ms.fa.gz"]
    # contig mode: byte-identical after the header's members; tile mode: the same text
    assert _no_date(gzip.decompress(b["g_ms.vcf.gz"])) == _no_date(gzip.decompress(a["g_ms.vcf.gz"]))
    assert _no_date(gzip.decompress(c["g_ms.vcf.gz"])) == _no_date(gzip.decompress(a["g_ms.vcf.gz"]))
    assert _body(b["g_ms.vcf.gz"]) == _body(a["g_ms.vcf.gz"])
