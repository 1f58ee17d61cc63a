"""The chain emitter (ms_chain_core.h, host build in tests/emu/chain_emu.cpp) against a plain restatement of the
chain format, a lift check of the chains against the golden FASTA files, the interchromosomal step's chain, and the
``--chain`` command line — without a GPU."""
import ctypes as C
import json
import subprocess
from pathlib import Path

import numpy as np
import pytest

from mutation_simulator_b200 import records as R
from mutation_simulator_b200.chain_writer import first_ids, it_chain_text
from tests.helpers import GOLDEN, MS_CASES, load_muts, read_fasta_simple

HERE = Path(__file__).resolve().parent
CSRC = HERE.parent / "mutation_simulator_b200" / "csrc"
COPY_KINDS = (R.K_RAW, R.K_CONV, R.K_RC)
COMP = np.arange(256, dtype=np.uint8)
for _a, _b in zip(b"ACGTUMRWSYKVHDB", b"TGCAAKYWSRMBDHV"):
    COMP[_a] = _b


@pytest.fixture(scope="module")
def core():
    src, lib = HERE / "emu" / "chain_emu.cpp", HERE / "emu" / "_build" / "libchain.so"
    lib.parent.mkdir(exist_ok=True)
    deps = [src] + list(CSRC.glob("*.h"))
    if not lib.exists() or lib.stat().st_mtime < max(p.stat().st_mtime for p in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", str(lib), str(src)])
    L = C.CDLL(str(lib))
    L.chain_emu.restype = C.c_int64
    L.chain_emu.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                            C.c_void_p, C.c_void_p]
    return L


def run_core(core, recs, lens, names, first=None):
    """-> (text, chains per contig, chain_off) from the host build of the emitter"""
    recs = np.ascontiguousarray(recs, dtype=R.REC_DTYPE)
    lens = np.ascontiguousarray(lens, dtype=np.int64)
    blob = b"".join(names) + b"\0"
    noff = np.concatenate(([0], np.cumsum([len(n) for n in names]))).astype(np.int64)
    n = len(lens)
    nch, off = np.zeros(n, np.int64), np.zeros(n + 1, np.int64)
    fid = None if first is None else np.ascontiguousarray(first, dtype=np.int64)
    P = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    size = core.chain_emu(P(recs), len(recs), P(lens), n, blob, P(noff), P(fid), P(nch), None, P(off))
    assert size >= 0, size
    out = C.create_string_buffer(max(1, size))
    assert core.chain_emu(P(recs), len(recs), P(lens), n, blob, P(noff), P(fid), P(nch), out, P(off)) == size
    return out.raw[:size], nch, off


# ---- the format, restated from its description ---------------------------------------------------------------------
def restate(recs, lens, names, start_id=1):
    """Primary chain per contig (blocks = the non-empty runs between the base-moving records), then one chain per
    record that copies bases (DU, TLI, IV) in record order.  Records with cons = prod = 0 move nothing."""
    goff = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    text, cid = [], start_id
    for c, (L, name) in enumerate(zip(lens, names)):
        L, name = int(L), name.decode()
        sel = recs[recs["contig"] == c]
        moving, shift = [], 0
        for r in sel:
            pos, cons, prod, kind = int(r["pos"]), int(r["cons"]), int(r["prod"]), int(r["kind"])
            if kind != R.K_SNP and (cons or prod):
                moving.append((pos, cons, prod, pos + shift, kind, int(r["src"]) - int(goff[c])))
            shift += prod - cons
        Lq = L + shift
        starts = [(0, 0)] + [(p + cn, o + pr) for p, cn, pr, o, _, _ in moving]
        ends = [(p, o) for p, _, _, o, _, _ in moving] + [(L, Lq)]
        blocks = [(ts, qs, te - ts) for (ts, qs), (te, qe) in zip(starts, ends) if te > ts]
        for (ts, qs), (te, qe) in zip(starts, ends):
            assert te - ts == qe - qs >= 0
        if blocks:
            score = sum(n for _, _, n in blocks)
            assert score == L - sum(cn for _, cn, _, _, _, _ in moving)
            t0, q0, _ = blocks[0]
            tl, ql, nl = blocks[-1]
            text.append(f"chain {score} {name} {L} + {t0} {tl + nl} {name} {Lq} + {q0} {ql + nl} {cid}\n")
            for (t, q, n), (tn, qn, _) in zip(blocks, blocks[1:]):
                text.append(f"{n}\t{tn - t - n}\t{qn - q - n}\n")
            text.append(f"{nl}\n\n")
            cid += 1
        for p, cn, pr, o, kind, s in moving:
            if kind in COPY_KINDS and pr > 0:
                q0 = Lq - o - pr if kind == R.K_RC else o
                strand = "-" if kind == R.K_RC else "+"
                text.append(f"chain {pr} {name} {L} + {s} {s + pr} {name} {Lq} {strand} {q0} {q0 + pr} {cid}\n{pr}\n\n")
                cid += 1
    return "".join(text).encode()


def parse_chains(text: bytes):
    chains = []
    for part in text.decode().split("\n\n"):
        if not part:
            continue
        lines = part.split("\n")
        h = lines[0].split(" ")
        assert h[0] == "chain" and len(h) == 13, lines[0]
        blocks = []
        for i, ln in enumerate(lines[1:]):
            f = [int(x) for x in ln.split("\t")]
            assert len(f) == (1 if i == len(lines) - 2 else 3), ln
            blocks.append((f[0], f[1] if len(f) == 3 else 0, f[2] if len(f) == 3 else 0))
        chains.append(dict(score=int(h[1]), tname=h[2], tsize=int(h[3]), t0=int(h[5]), t1=int(h[6]), qname=h[7],
                           qsize=int(h[8]), qstrand=h[9], q0=int(h[10]), q1=int(h[11]), id=int(h[12]), blocks=blocks))
    return chains


def golden_table(case):
    d = GOLDEN / case
    contigs = read_fasta_simple(d / "in.fa")
    seqs = [c[2] for c in contigs]
    genome, goff = R.pack_genome(seqs)
    recs, _ = R.build_records(genome, goff, [len(s) for s in seqs], load_muts(case))
    return recs, [len(s) for s in seqs], [c[0] for c in contigs]


@pytest.mark.parametrize("case", MS_CASES)
def test_core_matches_restatement_on_goldens(core, case):
    recs, lens, names = golden_table(case)
    text, nch, off = run_core(core, recs, lens, names)
    assert text == restate(recs, lens, names)
    chains = parse_chains(text)
    assert [c["id"] for c in chains] == list(range(1, len(chains) + 1))
    assert int(nch.sum()) == len(chains)
    for c, name in enumerate(names):     # each contig's slice holds its chains
        part = parse_chains(text[off[c]:off[c + 1]])
        assert all(x["qname"] == name.decode() for x in part) and len(part) == nch[c]


def random_table(rng, n_contigs=7):
    """Contigs with: a record at pos 0, a deletion reaching the end, adjacent records (empty runs), a wholly deleted
    contig, a contig without records, IV / reversed TLI ('-'), forward TLI, DU, inserts, SNPs and no-op records."""
    lens = [int(rng.integers(1, 3000)) for _ in range(n_contigs)]
    lens[1] = 0 if rng.random() < 0.3 else lens[1]
    goff = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    rows = []
    for c, L in enumerate(lens):
        if c == 2 and L:                       # wholly deleted
            rows.append((0, L, 0, 0, 0, R.K_NONE, R.T_DE, 0, 0, c))
            continue
        if c == 3 or L < 4:                    # no records
            continue
        pos = 0 if rng.random() < 0.7 else int(rng.integers(0, 5))
        while pos < L:
            room = L - pos
            t = int(rng.integers(0, 8))
            src = 0
            if t == 0:
                row = (pos, 1, 1, R.K_SNP, R.T_SN, 65, 67)
            elif t == 1:
                row = (pos, 0, int(rng.integers(1, 9)), R.K_LIT, R.T_IN, 0, 0)
            elif t == 2:
                row = (pos, int(rng.integers(1, min(room, 12) + 1)), 0, R.K_NONE, R.T_DE, 0, 0)
            elif t == 3:
                n = int(rng.integers(1, min(room, 12) + 1))
                row = (pos, n, n, R.K_RC, R.T_IV, 0, 0)
                src = int(goff[c]) + pos
            elif t == 4:
                n = int(rng.integers(1, min(room, 12) + 1))
                row = (pos, 0, n, R.K_RAW, R.T_DU, 0, 0)
                src = int(goff[c]) + pos
            elif t == 5:
                n = int(rng.integers(1, min(L, 12) + 1))
                s = int(rng.integers(0, L - n + 1))
                row = (pos, 0, n, R.K_RC if rng.random() < 0.5 else R.K_CONV, R.T_TLI, 0, 0)
                src = int(goff[c]) + s
            elif t == 6:
                row = (pos, 0, 0, R.K_NONE, 255, 0, 0)
            else:
                row = (pos, room, 0, R.K_NONE, R.T_TL, 0, 0)      # reaches the contig end
            p, cons, prod, kind, typ, ref, alt = row
            rows.append((p, cons, prod, 0, src if kind in COPY_KINDS else 0, kind, typ, ref, alt, c))
            step = max(cons, 1)
            pos += step + (0 if rng.random() < 0.4 else int(rng.integers(1, 40)))   # adjacent records give empty runs
    recs = np.array(rows, dtype=R.REC_DTYPE) if rows else np.zeros(0, dtype=R.REC_DTYPE)
    names = [b"ctg%d" % i for i in range(n_contigs)]
    return recs, lens, names


@pytest.mark.parametrize("seed", range(40))
def test_core_matches_restatement_on_random_tables(core, seed):
    rng = np.random.default_rng(seed)
    recs, lens, names = random_table(rng)
    text, nch, off = run_core(core, recs, lens, names)
    assert text == restate(recs, lens, names)
    # ids running across contigs from any first ids (as several GPUs pass them)
    start = int(rng.integers(1, 1 << 30))
    text2, _, _ = run_core(core, recs, lens, names, first=first_ids(nch, start))
    assert text2 == restate(recs, lens, names, start)
    chains = parse_chains(text)
    assert any(c["qstrand"] == "-" for c in chains) or not (recs["kind"] == R.K_RC).any()
    if lens[2]:                             # the wholly deleted contig has no chain at all
        assert nch[2] == 0
    if lens[3]:                             # a contig without records: the identity chain
        assert text[off[3]:off[4]] == (f"chain {lens[3]} ctg3 {lens[3]} + 0 {lens[3]} ctg3 {lens[3]} + 0 {lens[3]} "
                                       f"{first_ids(nch)[3]}\n{lens[3]}\n\n").encode()


def test_core_rejects_a_copy_from_another_contig(core):
    lens = [100, 100]
    recs = np.zeros(2, dtype=R.REC_DTYPE)
    recs[0] = (10, 0, 5, 0, 150, R.K_RAW, R.T_DU, 0, 0, 0)     # source in contig 1
    recs[1] = (10, 0, 5, 0, 110, R.K_RAW, R.T_DU, 0, 0, 1)
    blob = b"ab\0"
    noff = np.array([0, 1, 2], np.int64)
    nch, off = np.zeros(2, np.int64), np.zeros(3, np.int64)
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    assert core.chain_emu(P(recs), 2, P(np.array(lens, np.int64)), 2, blob, P(noff), None, P(nch), None, P(off)) == -1


# ---- the lift check: every block names the same bases in the two FASTA files ---------------------------------------
def lift_check(chains, t_seqs, q_seqs, snps=None, inserts=None, partition=True):
    """t_seqs / q_seqs: name -> bytes.  Blocks must hold equal bytes up to SNPs (snps[name] = t positions), IUPAC
    conversion and '-' written as 'N' ('+' copies), reverse complement ('-').  Then (partition) the q intervals of
    every contig's chains and its insert payloads (inserts[name] = [(q, n)]) must partition the contig."""
    cover = {n: [] for n in q_seqs}
    for ch in chains:
        t = np.frombuffer(t_seqs[ch["tname"]], np.uint8)
        q = np.frombuffer(q_seqs[ch["qname"]], np.uint8)
        assert ch["tsize"] == len(t) and ch["qsize"] == len(q)
        tp, qp = ch["t0"], ch["q0"]
        bt = bq = 0
        for n, dt, dq in ch["blocks"]:
            a = t[tp:tp + n]
            if ch["qstrand"] == "-":
                b = q[len(q) - qp - n:len(q) - qp]
                want = COMP[R.CONV[a]][::-1]
                assert np.array_equal(b, want), (ch["id"], tp, qp)
                cover[ch["qname"]].append((len(q) - qp - n, n))
            else:
                b = q[qp:qp + n]
                bad = np.flatnonzero((a != b) & (R.CONV[a] != b))
                ok = set(snps.get(ch["tname"], ())) if snps and ch["tname"] == ch["qname"] else set()
                assert all(tp + int(i) in ok for i in bad), (ch["id"], [tp + int(i) for i in bad][:5])
                cover[ch["qname"]].append((qp, n))
            tp += n + dt; qp += n + dq
            bt += n + dt; bq += n + dq
        assert (bt, bq) == (ch["t1"] - ch["t0"], ch["q1"] - ch["q0"])
        assert sum(n for n, _, _ in ch["blocks"]) == ch["score"]
    for name, q in q_seqs.items() if partition else ():
        iv = sorted(cover[name] + list((inserts or {}).get(name, ())))
        at = 0
        for s, n in iv:
            assert s == at, (name, s, at)
            at += n
        assert at == len(q), name


@pytest.mark.parametrize("case", MS_CASES)
def test_lift_check_on_golden_replays(core, case):
    """Replay the reference's own out.vcf, build the chain, and check it against the reference's in.fa / out.fa."""
    d = GOLDEN / case
    ins, outs = read_fasta_simple(d / "in.fa"), read_fasta_simple(d / "out.fa")
    names = [c[0] for c in ins]
    lens = [len(c[2]) for c in ins]
    goff = R.genome_offsets(lens)
    recs, lit = R.records_from_vcf((d / "out.vcf").read_bytes(), [n.decode() for n in names], goff, lens)
    text, _, _ = run_core(core, recs, lens, names)
    assert text == restate(recs, lens, names)
    snps, inserts = {}, {}
    for c, name in enumerate(names):
        sel = recs[recs["contig"] == c]
        shift = 0
        for r in sel:
            o = int(r["pos"]) + shift
            if r["kind"] == R.K_SNP:
                snps.setdefault(name.decode(), []).append(int(r["pos"]))
            elif r["kind"] == R.K_LIT:
                inserts.setdefault(name.decode(), []).append((o, int(r["prod"])))
            shift += int(r["prod"]) - int(r["cons"])
    lift_check(parse_chains(text), {n.decode(): c[2] for n, c in zip(names, ins)},
               {c[0].decode(): c[2] for c in outs}, snps, inserts)


def test_lift_check_covers_random_tables(core):
    """Random tables applied by a plain Python walk: blocks, copies and inserts tile every mutated contig."""
    rng = np.random.default_rng(99)
    for _ in range(20):
        recs, lens, names = random_table(rng)
        seqs = [bytes(rng.choice(np.frombuffer(b"ACGTRYN", np.uint8), L)) for L in lens]
        genome = b"".join(seqs)
        outs, inserts = {}, {}
        for c, s in enumerate(seqs):
            o, at = bytearray(), 0
            for r in recs[recs["contig"] == c]:
                p, cons, prod, kind, src = int(r["pos"]), int(r["cons"]), int(r["prod"]), int(r["kind"]), int(r["src"])
                o += s[at:p]
                if kind == R.K_SNP:
                    o += b"C"
                elif kind == R.K_LIT:
                    inserts.setdefault(names[c].decode(), []).append((len(o), prod))
                    o += b"G" * prod
                elif kind == R.K_RAW:
                    o += genome[src:src + prod]
                elif kind == R.K_CONV:
                    o += bytes(R.CONV[np.frombuffer(genome[src:src + prod], np.uint8)])
                elif kind == R.K_RC:
                    o += bytes(COMP[R.CONV[np.frombuffer(genome[src:src + prod], np.uint8)]][::-1])
                at = p + cons
            outs[names[c].decode()] = bytes(o + s[at:])
        snps = {names[c].decode(): [int(r["pos"]) for r in recs[(recs["contig"] == c) & (recs["kind"] == R.K_SNP)]]
                for c in range(len(lens))}
        text, _, _ = run_core(core, recs, lens, names)
        lift_check(parse_chains(text), {n.decode(): s for n, s in zip(names, seqs)}, outs, snps, inserts)


# ---- the interchromosomal step ---------------------------------------------------------------------------------------
def it_output(seqs, partners, bps):
    out = []
    for c, s in enumerate(seqs):
        if c not in bps:
            out.append(s)
            continue
        p = partners[c]
        a = [0] + list(bps[c]["self"]) + [len(s)]
        b = [0] + list(bps[c]["partner"]) + [len(seqs[p])]
        out.append(b"".join(s[a[i]:a[i + 1]] if i % 2 == 0 else seqs[p][b[i]:b[i + 1]] for i in range(len(a) - 1)))
    return out


@pytest.mark.parametrize("case", ["it_basic", "rmt_it"])
def test_it_chain_on_goldens(case):
    d = GOLDEN / case
    bp = json.loads((d / "bp.json").read_text())
    src = read_fasta_simple(d / ("out.fa" if (d / "out.fa").exists() else "in.fa"))
    out = read_fasta_simple(d / "out_it.fa")
    names = [c[0].decode() for c in src]
    partners = {int(k): int(v) for k, v in bp["partners"].items() if k in bp["breakpoints"]}
    bps = {int(k): {"self": np.array(v["self"]), "partner": np.array(v["partner"])} for k, v in bp["breakpoints"].items()}
    text = it_chain_text(names, [len(c[2]) for c in src], partners, bps)
    chains = parse_chains(text)
    assert [c["id"] for c in chains] == list(range(1, len(chains) + 1))
    lift_check(chains, {c[0].decode(): c[2] for c in src}, {c[0].decode(): c[2] for c in out})


def test_it_chain_with_breakpoints_at_the_ends():
    rng = np.random.default_rng(5)
    seqs = [bytes(rng.choice(np.frombuffer(b"ACGT", np.uint8), n)) for n in (50, 40, 30, 0)]
    names = ["a", "b", "c", "d"]
    partners = {0: 1, 1: 0}
    for sa, sb in (([10, 20, 50], [5, 15, 40]), ([10, 50], [3, 40]), ([1, 2, 3], [1, 2, 3]), ([10], [39])):
        bps = {0: {"self": np.array(sa), "partner": np.array(sb)}, 1: {"self": np.array(sb), "partner": np.array(sa)}}
        out = it_output(seqs, partners, bps)
        text = it_chain_text(names, [len(s) for s in seqs], partners, bps)
        chains = parse_chains(text)
        lift_check(chains, dict(zip(names, seqs)), dict(zip(names, out)))
        assert [c["qname"] for c in chains if c["tname"] == c["qname"] == "c"] == ["c"]      # identity chain
        assert not any(c["qname"] == "d" for c in chains)                                     # empty contig: none
        assert all(c["blocks"][0][0] > 0 for c in chains)                                     # no empty interval


# ---- command line ----------------------------------------------------------------------------------------------------
def test_chain_flag_and_output_names():
    from mutation_simulator_b200.argument_parser import get_args
    a = get_args(["g.fa", "-o", "out/run", "args"])
    assert a.chain is False
    b = get_args(["g.fa", "-o", "out/run", "--chain", "rmt", "x.rmt"])
    assert b.chain and (b.outchain.name, b.outchainit.name) == ("run_ms.chain", "run_ms_it.chain")
    c = get_args(["g.fa", "--chain", "--bgzip", "it", "0.1"])
    assert (c.outchain.name, c.outchainit.name) == ("g_ms.chain.gz", "g_ms_it.chain.gz")
    assert (c.outfasta.name, c.outvcf.name, c.outbedpe.name) == ("g_ms.fa.gz", "g_ms.vcf.gz", "g_ms_it.bedpe")


def test_replay_guard_covers_the_chain(tmp_path):
    from mutation_simulator_b200.__main__ import check_replay_paths
    from mutation_simulator_b200.argument_parser import get_args
    from mutation_simulator_b200.vcf_writer import VcfWriterError
    vcf = tmp_path / "r_ms.chain"
    vcf.write_bytes(b"")
    args = get_args([str(tmp_path / "g.fa"), "-o", str(tmp_path / "r"), "--chain", "vcf", str(vcf)])
    with pytest.raises(VcfWriterError):
        check_replay_paths(args)
    check_replay_paths(get_args([str(tmp_path / "g.fa"), "-o", str(tmp_path / "r"), "vcf", str(vcf)]))
