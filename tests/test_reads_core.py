"""The read-pair rule (ms_reads_core.h, host build in tests/emu/reads_emu.cpp) against a plain restatement, its
statistics, the truth in the read names against the oracle's mutated contigs and the chain emitter, and the
``--reads`` command line — without a GPU."""
import ctypes as C
import math
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
from scipy import stats

from mutation_simulator_b200 import records as R
from mutation_simulator_b200.reads_writer import pair_counts, quality_char
from oracle import c_oracle
from tests.helpers import GOLDEN, MS_CASES, load_muts, read_fasta_simple

HERE = Path(__file__).resolve().parent
CSRC = HERE.parent / "mutation_simulator_b200" / "csrc"
P_READS = 10
MASK32 = 0xFFFFFFFF
COMP = bytes(range(256)).translate(bytes.maketrans(b"ACGTUMRWSYKVHDB", b"TGCAAKYWSRMBDHV"))


@pytest.fixture(scope="module")
def core():
    src, lib = HERE / "emu" / "reads_emu.cpp", HERE / "emu" / "_build" / "libreads.so"
    lib.parent.mkdir(exist_ok=True)
    deps = [src] + list(CSRC.glob("*.h"))
    if not lib.exists() or lib.stat().st_mtime < max(p.stat().st_mtime for p in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", str(lib), str(src)])
    L = C.CDLL(str(lib))
    L.reads_emu.restype = C.c_int64
    L.reads_emu.argtypes = [C.c_char_p, C.c_int64, C.c_int32, C.c_int64, C.c_char_p, C.c_int32, C.c_uint32, C.c_void_p,
                            C.c_int64, C.c_uint64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_uint8,
                            C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lift_emu.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    return L


P = lambda a: a.ctypes.data_as(C.c_void_p)


def wrap(seq: bytes, bpl: int) -> bytes:
    return b"".join(seq[i:i + bpl] + b"\n" for i in range(0, len(seq), bpl))


def with_out(recs):
    """Records of one contig with ``out`` filled in (what the delta scan of an apply computes)."""
    recs = np.array(recs, dtype=R.REC_DTYPE, copy=True)
    shift = 0
    for r in recs:
        r["out"] = int(r["pos"]) + shift
        shift += int(r["prod"]) - int(r["cons"])
    return recs


def run_core(core, mseq, recs, name, gid, seed, hap, L, M, S, E, first, n, bpl=60, head=b">x\n"):
    """-> (R1 bytes, R2 bytes, info[n, 6] = s, f, strand, attempt, lift1, lift2) from the host build"""
    img = head + wrap(mseq, bpl)
    recs = np.ascontiguousarray(recs, dtype=R.REC_DTYPE)
    cap = max(1, n * (len(name) + 2 * L + 80))
    o1, o2 = C.create_string_buffer(cap), C.create_string_buffer(cap)
    info = np.zeros((max(n, 1), 6), np.int64)
    k = core.reads_emu(img, len(head), bpl, len(mseq), name, len(name), gid, P(recs) if len(recs) else None, len(recs), seed,
                       hap, L, M, S, E, quality_char(E), first, n, o1, o2, P(info))
    assert k >= 0
    return o1.raw[:k], o2.raw[:k], info[:n]


# ---- the rule, restated -----------------------------------------------------------------------------------------------
def philox(ctr, k0, k1):
    x, y, z, w = ctr
    for _ in range(10):
        p0, p1 = 0xD2511F53 * x, 0xCD9E8D57 * z
        x, y, z, w = (p1 >> 32) ^ y ^ k0, p1 & MASK32, (p0 >> 32) ^ w ^ k1, p0 & MASK32
        k0, k1 = (k0 + 0x9E3779B9) & MASK32, (k1 + 0xBB67AE85) & MASK32
    return x, y, z, w


class Words:
    """w0, w1, ... of pair i, attempt a"""

    def __init__(self, seed, gid, hap, i, a):
        self.key, self.ctr, self.blocks = (seed & MASK32, seed >> 32), (gid, hap, i * 16 + a), {}

    def __getitem__(self, k):
        b = k // 4
        if b not in self.blocks:
            gid, hap, idx = self.ctr
            self.blocks[b] = philox((gid, P_READS | hap << 8 | b << 12, idx & MASK32, idx >> 32), *self.key)
        return self.blocks[b][k % 4]


def restate_lift(recs, q):
    r = None
    for x in recs:
        if int(x["out"]) <= q:
            r = x
        else:
            break
    if r is None:
        return q
    out, prod = int(r["out"]), int(r["prod"])
    if q < out + prod:
        return int(r["pos"]) if r["kind"] == R.K_SNP else None
    return int(r["pos"]) + int(r["cons"]) + q - out - prod


def restate(mseq, recs, name, gid, seed, hap, L, M, S, E, first, n):
    """The records of pairs [first, first + n) of one contig as the rule describes them, written out plainly."""
    Lp, thr, q = len(mseq), math.floor(E * 2 ** 32 + 0.5), quality_char(E)
    r1, r2 = [], []
    for i in range(first, first + n):
        for a in range(8):
            w = Words(seed, gid, hap, i, a)
            z = sum(w[k] for k in range(12)) - 6 * 2 ** 32
            f = min(max(M + ((S * z + 2 ** 31) >> 32), L), Lp)
            s = (w[12] * (Lp - f + 1)) >> 32
            minus = w[13] & 1
            left, right = mseq[s:s + L], mseq[s + f - L:s + f]
            if a == 7 or all(c in b"ACGT" for c in left + right):
                break
        fwd_l, rc_r = left, right[::-1].translate(COMP)
        reads = (rc_r, fwd_l) if minus else (fwd_l, rc_r)
        x1, x2 = (s + f - L, s) if minus else (s, s + f - L)
        lifts = [restate_lift(recs, x) for x in (x1, x2)]
        head = b"@%s:%d:%d:%d:%d:%s:%s:%s" % (name, hap, i, s + 1, f, b"-" if minus else b"+",
                                             *[b"*" if v is None else b"%d" % (v + 1) for v in lifts])
        for m, (read, out) in enumerate(zip(reads, (r1, r2))):
            seq = bytearray(read)
            for j, b in enumerate(read):
                v = w[16 + m * L + j]
                if chr(b) in "ACGT" and v < thr:
                    seq[j] = ord([c for c in "ACGT" if c != chr(b)][v % 3])
            out.append(head + b"/%d\n" % (m + 1) + bytes(seq) + b"\n+\n" + bytes([q]) * L + b"\n")
    return b"".join(r1), b"".join(r2)


def golden_contigs(case):
    """-> [(name, input seq, mutated seq, records of the contig with out)] through the C oracle"""
    contigs = read_fasta_simple(GOLDEN / case / "in.fa")
    seqs = [c[2] for c in contigs]
    genome, goff = R.pack_genome(seqs)
    muts = load_muts(case)
    recs, _ = R.build_records(genome, goff, [len(s) for s in seqs], muts)
    out = []
    for c, (name, _, seq, _) in enumerate(contigs):
        mseq, _ = c_oracle.walk(seq, name, muts[c])
        out.append((name, seq, mseq, with_out(recs[recs["contig"] == c])))
    return out


def random_contig(rng, n_len=3000):
    """A contig with records at position 0, adjacent records, a no-op record, N runs and a deletion to the end."""
    seq = bytearray(rng.choice(list(b"ACGT"), n_len).astype(np.uint8).tobytes())
    seq[700:760] = b"N" * 60
    seq[1500:1503] = b"RYN"
    rows, pos = [], 0
    for t, cons, prod, kind in ((R.T_SN, 1, 1, R.K_SNP), (R.T_IN, 0, 4, R.K_LIT), (R.T_DE, 5, 0, R.K_NONE),
                                (R.T_SN, 1, 1, R.K_SNP), (R.T_DU, 0, 30, R.K_RAW), (255, 0, 0, R.K_NONE),
                                (R.T_IV, 40, 40, R.K_RC), (R.T_SN, 1, 1, R.K_SNP), (R.T_IN, 0, 12, R.K_LIT)):
        rows.append((pos, cons, prod, 0, pos, kind, t, 65, 71, 0))
        pos += max(cons, 1) + (0 if len(rows) % 3 else int(rng.integers(1, 200)))
    rows.append((n_len - 100, 100, 0, 0, 0, R.K_NONE, R.T_DE, 0, 0, 0))
    recs = with_out(np.array(rows, dtype=R.REC_DTYPE))
    # the mutated sequence that these records describe (payload bytes are arbitrary here: the rule only reads them)
    m, at = bytearray(), 0
    for r in recs:
        p, cons, prod = int(r["pos"]), int(r["cons"]), int(r["prod"])
        m += seq[at:p] + (b"G" if r["kind"] == R.K_SNP else bytes(rng.choice(list(b"ACGT"), prod).astype(np.uint8)))
        at = p + cons
    m += seq[at:]
    return bytes(seq), bytes(m), recs


@pytest.mark.parametrize("case", MS_CASES)
@pytest.mark.parametrize("hap", [1, 2, 3])
def test_core_matches_the_restated_rule_on_golden_tables(core, case, hap):
    L, M, S, E = 30, 80, 15, 0.05
    for gid, (name, _, mseq, recs) in enumerate(golden_contigs(case)):
        n = pair_counts(3.0, [len(mseq)], L, 1)[0]
        n = min(int(n), 25)
        a1, a2, _ = run_core(core, mseq, recs, name, gid, 99 + hap, hap, L, M, S, E, 3, n)
        b1, b2 = restate(mseq, recs, name, gid, 99 + hap, hap, L, M, S, E, 3, n)
        assert (a1, a2) == (b1, b2)


@pytest.mark.parametrize("hap", [1, 2, 3])
def test_core_matches_the_restated_rule_on_random_tables(core, hap):
    rng = np.random.default_rng(hap)
    seq, mseq, recs = random_contig(rng)
    for L, M, S, E in ((50, 200, 40, 0.02), (1, 1, 0, 0.3), (100, 150, 100, 0.0), (200, 100, 20, 0.001)):
        seed = int(rng.integers(0, 2 ** 63))
        a1, a2, info = run_core(core, mseq, recs, b"chr:1", 5, seed, hap, L, M, S, E, 0, 60, bpl=7)
        assert (a1, a2) == restate(mseq, recs, b"chr:1", 5, seed, hap, L, M, S, E, 0, 60)
        assert (info[:, 1] >= L).all() and (info[:, 1] <= len(mseq)).all()
    # a contig of exactly L bases: one fragment, the whole contig
    a1, a2, info = run_core(core, b"ACGTTGCA", with_out(np.zeros(0, R.REC_DTYPE)), b"t", 0, 1, hap, 8, 500, 50, 0.0, 0, 3)
    assert (info[:, 0] == 0).all() and (info[:, 1] == 8).all()
    assert a1 == restate(b"ACGTTGCA", [], b"t", 0, 1, hap, 8, 500, 50, 0.0, 0, 3)[0]


def test_redraw_and_the_kept_eighth_attempt(core):
    rng = np.random.default_rng(8)
    seq = bytearray(rng.choice(list(b"ACGT"), 4000).astype(np.uint8).tobytes())
    for k in range(0, 4000, 200):
        seq[k:k + 120] = b"N" * 120          # 60 % N: many pairs redraw
    seq = bytes(seq)
    none = with_out(np.zeros(0, R.REC_DTYPE))
    a1, a2, info = run_core(core, seq, none, b"n", 1, 3, 1, 40, 60, 5, 0.01, 0, 80)
    assert (a1, a2) == restate(seq, [], b"n", 1, 3, 1, 40, 60, 5, 0.01, 0, 80)
    assert (info[:, 3] > 0).any() and (info[:, 3] < 7).any()
    allN = b"N" * 500
    n1, _, info_n = run_core(core, allN, none, b"n", 1, 3, 1, 40, 60, 5, 0.5, 0, 10)
    assert (info_n[:, 3] == 7).all()
    assert n1 == restate(allN, [], b"n", 1, 3, 1, 40, 60, 5, 0.5, 0, 10)[0]
    assert b"NNNN\n+\n" in n1                                  # N bases are never changed by errors
    ok = [i for i in range(80) if info[i, 3] < 7]
    for i in ok:                                               # a kept draw before the 8th has A/C/G/T templates only
        s, f = info[i, 0], info[i, 1]
        assert all(c in b"ACGT" for c in seq[s:s + 40] + seq[s + f - 40:s + f])


# ---- statistics --------------------------------------------------------------------------------------------------------
def test_fragment_start_strand_statistics(core):
    """Family-wise at alpha = 1e-3: fragment mean and SD as Irwin-Hall(12) gives them (within 5 sigma), start uniform
    over [0, Lp - f] (KS on the scaled start), strand 1/2."""
    n, L, M, S, Lp = 100_000, 100, 500, 50, 200_000
    mseq = bytes(np.random.default_rng(1).choice(list(b"ACGT"), Lp).astype(np.uint8))
    _, _, info = run_core(core, mseq, with_out(np.zeros(0, R.REC_DTYPE)), b"c", 2, 17, 1, L, M, S, 0.0, 0, n)
    f = info[:, 1].astype(float)
    assert f.min() >= L and f.max() <= Lp and f.min() >= M - 6 * S and f.max() <= M + 6 * S + 1
    assert abs(f.mean() - M) < 5 * S / math.sqrt(n)
    sd_of_sd = S * math.sqrt(0.5 / n * (1 + 0.4 / 2))          # Irwin-Hall(12) excess kurtosis -0.1
    assert abs(f.std() - S) < 5 * sd_of_sd + 0.5                 # + rounding of f to integers
    u = (info[:, 0] + 0.5) / (Lp - info[:, 1] + 1)
    assert stats.kstest(u, "uniform").pvalue > 1e-3 / 3
    assert stats.binomtest(int(info[:, 2].sum()), n, 0.5).pvalue > 1e-3 / 3


@pytest.mark.parametrize("E", [0.0, 0.01, 0.2])
def test_error_share_and_substitutions(core, E):
    n, L, Lp = 4000, 150, 100_000
    mseq = bytes(np.random.default_rng(2).choice(list(b"ACGT"), Lp).astype(np.uint8))
    a1, a2, info = run_core(core, mseq, with_out(np.zeros(0, R.REC_DTYPE)), b"c", 0, 5, 2, L, 400, 40, E, 0, n)
    seqs = a1.split(b"\n")[1::4] + a2.split(b"\n")[1::4]
    errs, subst = 0, {c: np.zeros(4, np.int64) for c in b"ACGT"}
    for k, read in enumerate(seqs):
        i, mate = k % n, 1 + k // n
        s, f, minus = info[i, :3]
        fwd = (mate == 1) == (minus == 0)
        tmpl = mseq[s:s + L] if fwd else mseq[s + f - L:s + f][::-1].translate(COMP)
        a = np.frombuffer(read, np.uint8)
        b = np.frombuffer(tmpl, np.uint8)
        d = a != b
        errs += int(d.sum())
        for x, y in zip(b[d], a[d]):
            subst[int(x)][b"ACGT".index(bytes([y]))] += 1
    total = 2 * n * L
    if E == 0:
        assert errs == 0
        return
    assert abs(errs - E * total) < 5 * math.sqrt(total * E * (1 - E))
    for c, cnt in subst.items():
        other = np.delete(cnt, b"ACGT".index(bytes([c])))
        assert cnt[b"ACGT".index(bytes([c]))] == 0
        assert stats.chisquare(other).pvalue > 1e-3 / 8


# ---- the truth in the names ---------------------------------------------------------------------------------------------
def parse_name(line: bytes):
    f = line[1:].rsplit(b"/", 1)[0].rsplit(b":", 7)
    lift = lambda x: None if x == b"*" else int(x) - 1
    return f[0], int(f[1]), int(f[2]), int(f[3]) - 1, int(f[4]), f[5], lift(f[6]), lift(f[7])


@pytest.mark.parametrize("case", MS_CASES)
def test_reads_at_named_coordinates_and_lift_against_input(core, case):
    L = 25
    for gid, (name, seq, mseq, recs) in enumerate(golden_contigs(case)):
        n = min(int(pair_counts(2.0, [len(mseq)], L, 2)[0]), 40)
        a1, a2, _ = run_core(core, mseq, recs, name, gid, 7, 2, L, 60, 10, 0.0, 0, n)
        snp_out = {int(r["out"]) for r in recs if r["kind"] == R.K_SNP}
        for text, mate in ((a1, 1), (a2, 2)):
            lines = text.split(b"\n")
            for k in range(n):
                nm, h, i, s, f, strand, l1, l2 = parse_name(lines[4 * k])
                assert (nm, h, i) == (name, 2, k) and lines[4 * k].endswith(b"/%d" % mate)
                fwd = (mate == 1) == (strand == b"+")
                x = s if fwd else s + f - L
                assert lines[4 * k + 1] == (mseq[x:x + L] if fwd else mseq[x:x + L][::-1].translate(COMP))
                lift = l1 if mate == 1 else l2
                if lift is not None and x not in snp_out:
                    assert seq[lift] == mseq[x] or mseq[x] == ord("N")


def run_lift(core, recs, qs):
    recs = np.ascontiguousarray(recs, dtype=R.REC_DTYPE)
    q = np.ascontiguousarray(qs, dtype=np.int64)
    out = np.zeros(len(q), np.int64)
    core.lift_emu(P(recs) if len(recs) else None, len(recs), P(q), len(q), P(out))
    return out


@pytest.mark.parametrize("case", MS_CASES)
def test_lift_is_the_primary_chain(core, case):
    """Every mutated position lifts to what the primary chain of the chain emitter (tests/emu/chain_emu.cpp) maps it
    to, and to '*' where no block covers it."""
    from tests import test_chain_core as T
    src, lib = HERE / "emu" / "chain_emu.cpp", HERE / "emu" / "_build" / "libchain_reads.so"
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", str(lib), str(src)])
    chain_lib = C.CDLL(str(lib))
    chain_lib.chain_emu.restype = C.c_int64
    chain_lib.chain_emu.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32] + [C.c_void_p] * 6
    all_recs, lens, names = T.golden_table(case)
    text, n_chains, off = T.run_core(chain_lib, all_recs, lens, names)
    for c, (name, seq, mseq, recs) in enumerate(golden_contigs(case)):
        want = np.full(len(mseq), -1, np.int64)
        chains = T.parse_chains(text[off[c]:off[c + 1]])
        copies = int(((np.isin(recs["kind"], T.COPY_KINDS)) & (recs["prod"] > 0)).sum())
        if n_chains[c] > copies:                      # the contig has a primary chain: its first
            ch = chains[0]
            t, q = ch["t0"], ch["q0"]
            for n, dt, dq in ch["blocks"]:
                want[q:q + n] = np.arange(t, t + n)
                t, q = t + n + dt, q + n + dq
        got = run_lift(core, recs, np.arange(len(mseq)))
        assert (got == want).all(), (case, c)


# ---- command line -----------------------------------------------------------------------------------------------------
def test_count_rule_and_quality():
    assert list(pair_counts(1.0, [299, 300, 301, 3000, 10], 150, 1)) == [0, 1, 1, 10, 0]
    assert list(pair_counts(30.0, [1000], 100, 2)) == [75]
    assert list(pair_counts(0.5, [100], 100, 1)) == [0]           # rounds to 0
    assert quality_char(0.0) == ord("!") + 41 and quality_char(0.001) == ord("!") + 30
    assert quality_char(0.9) == ord("!") + 2 and quality_char(1e-9) == ord("!") + 41


NEW_KEYS = {"reads", "read_length", "fragment_mean", "fragment_sd", "read_error_rate", "outreads1", "outreads2"}


def test_namespace_and_names_without_reads_are_unchanged():
    from mutation_simulator_b200.argument_parser import get_args
    for argv in (["g.fa", "-o", "out/run", "args"], ["g.fa", "--bgzip", "--ploidy", "2", "rmt", "x.rmt"], ["g.fa", "vcf", "v.vcf"]):
        a = vars(get_args(argv))
        assert not NEW_KEYS & set(a), argv


def test_reads_options_and_output_names():
    from mutation_simulator_b200.argument_parser import get_args
    a = get_args(["g.fa", "-o", "out/run", "--reads", "30", "args"])
    assert (a.reads, a.read_length, a.fragment_mean, a.fragment_sd, a.read_error_rate) == (30.0, 150, 500, 50, 0.001)
    assert (str(a.outreads1), str(a.outreads2)) == ("out/run_ms_R1.fq", "out/run_ms_R2.fq")
    b = get_args(["g.fa", "--reads", "0.5", "--read-length", "100", "--fragment-mean", "100", "--fragment-sd", "0",
                  "--read-error-rate", "0", "--bgzip", "--ploidy", "2", "vcf", "v.vcf"])
    assert (b.outreads1.name, b.outreads2.name, b.read_length, b.fragment_mean) == ("g_ms_R1.fq.gz", "g_ms_R2.fq.gz", 100, 100)


def run_cli(tmp_path, *argv):
    (tmp_path / "g.fa").write_bytes(b">c\nACGTACGTAC\n")
    r = subprocess.run([sys.executable, "-m", "mutation_simulator_b200", str(tmp_path / "g.fa"), "-o", str(tmp_path / "r"), *argv],
                       capture_output=True, text=True, cwd=HERE.parent)
    assert sorted(p.name for p in tmp_path.iterdir()) == ["g.fa"]       # nothing written
    return r


@pytest.mark.parametrize("argv,word", [(["--reads", "0"], "reads"), (["--reads", "nan"], "reads"), (["--reads", "inf"], "reads"),
                                       (["--reads", "-1"], "reads"), (["--reads", "1", "--read-length", "0"], "read-length"),
                                       (["--reads", "1", "--read-length", "1001"], "read-length"),
                                       (["--reads", "1", "--fragment-mean", "149"], "fragment-mean"),
                                       (["--reads", "1", "--fragment-mean", "1000001"], "fragment-mean"),
                                       (["--reads", "1", "--fragment-sd", "-1"], "fragment-sd"),
                                       (["--reads", "1", "--fragment-sd", "100001"], "fragment-sd"),
                                       (["--reads", "1", "--read-error-rate", "1"], "read-error-rate"),
                                       (["--reads", "1", "--read-error-rate", "-0.1"], "read-error-rate"),
                                       (["--reads", "1", "--read-length", "abc"], "read-length"),
                                       (["--reads", "1", "--read-error-rate", "x"], "read-error-rate")])
def test_cli_refuses_out_of_range(tmp_path, argv, word):
    r = run_cli(tmp_path, *argv, "args")
    assert r.returncode == 2 and word in r.stderr


def test_read_options_are_ignored_without_reads():
    from mutation_simulator_b200.argument_parser import get_args
    a = vars(get_args(["g.fa", "--read-length", "5000", "--fragment-mean", "1", "--fragment-sd", "abc", "args"]))
    assert not NEW_KEYS & set(a)


def test_cli_refuses_it_mode(tmp_path):
    r = run_cli(tmp_path, "--reads", "1", "it", "0.1")
    assert r.returncode == 1 and "interchromosomal" in r.stderr and "--reads" in r.stderr


def test_reads_refuse_rmt_with_it():
    from mutation_simulator_b200.__main__ import ReadsError, check_reads
    from mutation_simulator_b200.argument_parser import get_args
    from mutation_simulator_b200.fasta import Fasta
    from mutation_simulator_b200.rmt import SimulationSettings
    fa = Fasta(GOLDEN / "rmt_it" / "in.fa", build_index=False)
    sim = SimulationSettings.from_rmt(GOLDEN / "rmt_it" / "in.rmt", fa, True)
    with pytest.raises(ReadsError):
        check_reads(get_args(["g.fa", "--reads", "2", "rmt", "x.rmt"]), sim.has_it)
    check_reads(get_args(["g.fa", "rmt", "x.rmt"]), sim.has_it)
    check_reads(get_args(["g.fa", "--reads", "2", "args"]), False)
