"""The genotype rule and the phased VCF line (ms_genotype_core.h, host build in tests/emu/genotype_emu.cpp) against a
plain restatement, the GT parse of both parsers, and the ``--ploidy`` command line — without a GPU."""
import ctypes as C
import math
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
from scipy import stats

from mutation_simulator_b200 import records as R
from tests.helpers import GOLDEN, MS_CASES, load_muts, read_fasta_simple, vcf_body

HERE = Path(__file__).resolve().parent
CSRC = HERE.parent / "mutation_simulator_b200" / "csrc"
P_GENOTYPE = 9
MASK32 = 0xFFFFFFFF


@pytest.fixture(scope="module")
def core():
    src, lib = HERE / "emu" / "genotype_emu.cpp", HERE / "emu" / "_build" / "libgenotype.so"
    lib.parent.mkdir(exist_ok=True)
    deps = [src] + list(CSRC.glob("*.h"))
    if not lib.exists() or lib.stat().st_mtime < max(p.stat().st_mtime for p in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", str(lib), str(src)])
    L = C.CDLL(str(lib))
    L.genotype_emu.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_uint64, C.c_int32, C.c_double, C.c_void_p]
    L.phased_line_emu.restype = C.c_int64
    L.phased_line_emu.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                  C.c_int32, C.c_uint32, C.c_void_p, C.POINTER(C.c_int64)]
    L.parse_gt_emu.argtypes = [C.c_char_p, C.c_int64, C.c_int32, C.POINTER(C.c_uint8)]
    return L


P = lambda a: a.ctypes.data_as(C.c_void_p)


def core_masks(core, recs, lens, seed, ploidy, f):
    recs = np.ascontiguousarray(recs, dtype=R.REC_DTYPE)
    lens = np.ascontiguousarray(lens, dtype=np.int64)
    out = np.zeros(max(1, len(recs)), np.uint8)
    core.genotype_emu(P(recs), len(recs), P(lens), len(lens), seed, ploidy, f, P(out))
    return out[:len(recs)]


# ---- the rule, restated -----------------------------------------------------------------------------------------------
def philox(ctr, k0, k1):
    x, y, z, w = ctr
    for _ in range(10):
        p0, p1 = 0xD2511F53 * x, 0xCD9E8D57 * z
        x, y, z, w = (p1 >> 32) ^ y ^ k0, p1 & MASK32, (p0 >> 32) ^ w ^ k1, p0 & MASK32
        k0, k1 = (k0 + 0x9E3779B9) & MASK32, (k1 + 0xBB67AE85) & MASK32
    return x, y, z, w


def restate_mask(seed, gid, key, ploidy, f):
    x, y, _, _ = philox((gid, P_GENOTYPE, key & MASK32, key >> 32), seed & MASK32, seed >> 32)
    thr = min(2 ** 32, math.floor(f * 2 ** 32 + 0.5))
    full = (1 << ploidy) - 1
    return full if x < thr else 1 + ((y * (full - 1)) >> 32)


def random_table(rng, n_contigs=3, L=5000, n=300):
    """Records at distinct positions per contig, every TL paired with a TLI elsewhere in its contig whose source is the
    TL's span (what the sampler links)."""
    lens = [L] * n_contigs
    goff = R.genome_offsets(lens)
    rows = []
    for c in range(n_contigs):
        pos = np.sort(rng.choice(np.arange(0, L - 20, 10), n, replace=False))
        types = rng.choice([R.T_SN, R.T_IN, R.T_DE, R.T_IV, R.T_DU, R.T_TL], n)
        tl = [int(p) for p, t in zip(pos, types) if t == R.T_TL]
        free = [int(p) + 5 for p in pos]                       # positions no record uses
        partner = rng.choice(free, len(tl), replace=False)
        for p, t in zip(pos, types):
            t = int(t)
            kind = {R.T_SN: R.K_SNP, R.T_IN: R.K_LIT, R.T_DE: R.K_NONE, R.T_IV: R.K_RC, R.T_DU: R.K_RAW, R.T_TL: R.K_NONE}[t]
            rows.append((int(p), 3 if t in (R.T_DE, R.T_TL, R.T_IV) else 1 if t == R.T_SN else 0, 3, 0, int(goff[c]) + int(p),
                         kind, t, 65, 67, c))
        for s, q in zip(tl, partner):
            rows.append((int(q), 0, 3, 0, int(goff[c]) + s, int(rng.choice([R.K_CONV, R.K_RC])), R.T_TLI, 0, 0, c))
    rows.sort(key=lambda r: (r[9], r[0]))
    return np.array(rows, dtype=R.REC_DTYPE), lens, goff


@pytest.mark.parametrize("ploidy", range(2, 9))
@pytest.mark.parametrize("f", [0.0, 0.35, 1.0])
def test_masks_match_the_restated_rule(core, ploidy, f):
    rng = np.random.default_rng(ploidy * 10 + int(f * 100))
    recs, lens, goff = random_table(rng)
    seed = int(rng.integers(0, 2 ** 63))
    got = core_masks(core, recs, lens, seed, ploidy, f)
    for r, m in zip(recs, got):
        c = int(r["contig"])
        key = int(r["src"]) - int(goff[c]) if r["type"] == R.T_TLI else int(r["pos"])
        assert m == restate_mask(seed, c, key, ploidy, f)
    full = (1 << ploidy) - 1
    assert ((got >= 1) & (got <= full)).all()
    if f == 1.0:
        assert (got == full).all()
    if f == 0.0:
        assert (got != full).all()


def test_tli_shares_its_tl_mask(core):
    rng = np.random.default_rng(3)
    for ploidy in (2, 3, 5, 8):
        recs, lens, goff = random_table(rng)
        m = core_masks(core, recs, lens, 77 + ploidy, ploidy, 0.35)
        pos_mask = {(int(r["contig"]), int(r["pos"])): int(x) for r, x in zip(recs, m) if r["type"] == R.T_TL}
        tli = np.flatnonzero(recs["type"] == R.T_TLI)
        assert len(tli) > 10
        for i in tli:
            c = int(recs[i]["contig"])
            assert m[i] == pos_mask[(c, int(recs[i]["src"]) - int(goff[c]))]


def test_hom_fraction_and_het_uniformity(core):
    """Family-wise at alpha = 1e-3 (Bonferroni over 2 tests x 7 ploidies): the hom share is F, and the het masks are
    uniform over the 2^P - 2 masks that are neither empty nor full."""
    n, f, alpha = 200_000, 0.35, 1e-3 / 14
    recs = np.zeros(n, dtype=R.REC_DTYPE)
    recs["pos"] = np.arange(n)
    recs["type"] = R.T_SN
    for ploidy in range(2, 9):
        m = core_masks(core, recs, [n + 1], 1234 + ploidy, ploidy, f)
        full = (1 << ploidy) - 1
        hom = int((m == full).sum())
        assert stats.binomtest(hom, n, f).pvalue > alpha
        het = m[m != full]
        counts = np.bincount(het, minlength=full)[1:full]
        assert stats.chisquare(counts).pvalue > alpha
    m2 = core_masks(core, recs, [n + 1], 9, 2, 0.0)
    assert set(np.unique(m2)) == {1, 2}


# ---- the phased line --------------------------------------------------------------------------------------------------
def golden_table(case):
    contigs = read_fasta_simple(GOLDEN / case / "in.fa")
    seqs = [c[2] for c in contigs]
    genome, goff = R.pack_genome(seqs)
    recs, lit = R.build_records(genome, goff, [len(s) for s in seqs], load_muts(case))
    names = [c[0] for c in contigs]
    noff = np.concatenate(([0], np.cumsum([len(x) for x in names]))).astype(np.int64)
    return genome, np.array([len(s) for s in seqs], np.int64), b"".join(names) + b"\0", noff, recs, lit


def line(core, g, i, ploidy, mask):
    genome, lens, blob, noff, recs, lit = g
    out = C.create_string_buffer(1 << 16)
    closed = C.c_int64()
    n = core.phased_line_emu(P(genome), P(lens), len(lens), blob, P(noff), P(lit), P(recs), i, ploidy, mask, out, C.byref(closed))
    assert n >= 0
    return out.raw[:n], closed.value


@pytest.mark.parametrize("case", MS_CASES)
def test_phased_line_size_and_gt(core, case):
    g = golden_table(case)
    recs = g[4]
    body = []
    for i in range(len(recs)):
        hap, closed1 = line(core, g, i, 0, 0)
        assert len(hap) == closed1
        body.append(hap)
        assert line(core, g, i, 1, 1)[0] == hap                    # P = 1 is today's line
        for ploidy in range(2, 9):
            mask = (i * 37 + ploidy) % (1 << ploidy)
            txt, closed = line(core, g, i, ploidy, mask)
            assert len(txt) == closed
            if not hap:
                assert not txt
                continue
            gt = "|".join("1" if mask >> h & 1 else "0" for h in range(ploidy)).encode()
            assert txt == hap[:-len(b"1\n")] + gt + b"\n"
    assert b"".join(body) == vcf_body((GOLDEN / case / "out.vcf").read_bytes())


# ---- GT parse -----------------------------------------------------------------------------------------------------------
REC = "chr1\t5\t.\tA\tC\t.\t.\t.\tGT\t"


@pytest.mark.parametrize("gt,ploidy,mask", [("1|0", 2, 1), ("0|1", 2, 2), ("1|1", 2, 3), ("0|0", 2, 0), ("0|1|1", 3, 6),
                                            ("1|0|0|0|0|0|0|1", 8, 129), ("1", 1, 1),
                                            ("1", 2, None), ("1|0|1", 2, None), ("1/0", 2, None), ("2|0", 2, None),
                                            ("1||0", 3, None), ("", 2, None), ("10", 2, None), ("1|0\r", 2, None)])
def test_gt_parse(core, gt, ploidy, mask):
    text = (REC + gt).encode()
    m = C.c_uint8()
    ok = core.parse_gt_emu(text, len(text), ploidy, C.byref(m))
    assert ok == (mask is not None)
    if ok:
        assert m.value == mask
        assert R.parse_gt(gt, ploidy) == mask
    elif not gt.endswith("\r"):
        with pytest.raises(ValueError):
            R.parse_gt(gt, ploidy)


def test_gt_parse_missing_field_and_trailing_fields(core):
    m = C.c_uint8()
    for text in (b"chr1\t5\t.\tA\tC\t.\t.\t.\tGT", b"chr1\t5\t.\tA\tC\t.\t.\t."):
        assert core.parse_gt_emu(text, len(text), 2, C.byref(m)) == 0
    text = (REC + "0|1\textra").encode()
    assert core.parse_gt_emu(text, len(text), 2, C.byref(m)) == 1 and m.value == 2


def test_host_parser_reads_masks_and_names_the_line():
    text = ("##h\n" + REC + "0|1\n" + "chr1\t2\t.\tA\tG\t.\t.\t.\tGT\t1|1\r\n" + "chr1\t9\t.\tA\tG\t.\t.\t.\tGT\t0|0\n")
    recs, lit, masks = R.records_from_vcf(text, [b"chr1"], [0], [20], ploidy=2)
    assert list(recs["pos"]) == [1, 4, 8] and list(masks) == [3, 2, 0]      # sorted with their records; CRLF accepted
    recs1, _ = R.records_from_vcf(text, [b"chr1"], [0], [20])                # without ploidy GT is ignored
    assert (recs1 == recs).all()
    with pytest.raises(ValueError, match="line 2.*ploidy 2"):
        R.records_from_vcf("##h\n" + REC + "1\n", [b"chr1"], [0], [20], ploidy=2)
    with pytest.raises(ValueError, match="line 1: no GT field"):
        R.records_from_vcf("chr1\t5\t.\tA\tC\t.\t.\t.\n", [b"chr1"], [0], [20], ploidy=2)


# ---- command line -----------------------------------------------------------------------------------------------------
def test_ploidy_options_and_output_names():
    from mutation_simulator_b200.argument_parser import get_args
    a = get_args(["g.fa", "-o", "out/run", "args"])
    assert (a.ploidy, a.hom_fraction, a.outfastas, a.outchains) == (1, 0.35, [], [])
    b = get_args(["g.fa", "-o", "out/run", "--ploidy", "3", "--hom-fraction", "0", "--chain", "args"])
    assert [p.name for p in b.outfastas] == ["run_ms_h1.fa", "run_ms_h2.fa", "run_ms_h3.fa"]
    assert [p.name for p in b.outchains] == ["run_ms_h1.chain", "run_ms_h2.chain", "run_ms_h3.chain"]
    assert (b.outvcf.name, b.hom_fraction) == ("run_ms.vcf", 0.0)
    c = get_args(["g.fa", "--ploidy", "2", "--bgzip", "vcf", "x.vcf"])
    assert [p.name for p in c.outfastas] == ["g_ms_h1.fa.gz", "g_ms_h2.fa.gz"]
    assert [p.name for p in c.outchains] == ["g_ms_h1.chain.gz", "g_ms_h2.chain.gz"] and c.outvcf.name == "g_ms.vcf.gz"


def run_cli(tmp_path, *argv):
    (tmp_path / "g.fa").write_bytes(b">c\nACGTACGTAC\n")
    r = subprocess.run([sys.executable, "-m", "mutation_simulator_b200", str(tmp_path / "g.fa"), "-o", str(tmp_path / "r"), *argv],
                       capture_output=True, text=True, cwd=HERE.parent)
    assert sorted(p.name for p in tmp_path.iterdir()) == ["g.fa"]       # nothing written
    return r


@pytest.mark.parametrize("argv", [["--ploidy", "0", "args"], ["--ploidy", "9", "args"], ["--hom-fraction", "1.5", "args"],
                                  ["--hom-fraction", "-0.1", "args"]])
def test_cli_refuses_out_of_range(tmp_path, argv):
    r = run_cli(tmp_path, *argv)
    assert r.returncode == 2 and ("ploidy" in r.stderr or "hom-fraction" in r.stderr)


def test_cli_refuses_it_mode(tmp_path):
    r = run_cli(tmp_path, "--ploidy", "2", "it", "0.1")
    assert r.returncode == 1 and "interchromosomal" in r.stderr


def test_ploidy_refuses_rmt_with_it():
    from mutation_simulator_b200.__main__ import PloidyError, check_ploidy
    from mutation_simulator_b200.argument_parser import get_args
    from mutation_simulator_b200.fasta import Fasta
    from mutation_simulator_b200.rmt import SimulationSettings
    fa = Fasta(GOLDEN / "rmt_it" / "in.fa", build_index=False)
    sim = SimulationSettings.from_rmt(GOLDEN / "rmt_it" / "in.rmt", fa, True)
    assert sim.has_it
    with pytest.raises(PloidyError):
        check_ploidy(get_args(["g.fa", "--ploidy", "2", "rmt", "x.rmt"]), sim.has_it)
    check_ploidy(get_args(["g.fa", "rmt", "x.rmt"]), sim.has_it)
    check_ploidy(get_args(["g.fa", "--ploidy", "2", "args"]), False)


def test_replay_guard_covers_the_haplotypes(tmp_path):
    from mutation_simulator_b200.__main__ import check_replay_paths
    from mutation_simulator_b200.argument_parser import get_args
    from mutation_simulator_b200.vcf_writer import VcfWriterError
    for name, extra in (("r_ms_h2.fa", []), ("r_ms_h1.chain", ["--chain"])):
        vcf = tmp_path / name
        vcf.write_bytes(b"")
        with pytest.raises(VcfWriterError):
            check_replay_paths(get_args([str(tmp_path / "g.fa"), "-o", str(tmp_path / "r"), "--ploidy", "2", *extra, "vcf", str(vcf)]))
        check_replay_paths(get_args([str(tmp_path / "g.fa"), "-o", str(tmp_path / "r"), *extra, "vcf", str(vcf)]))
