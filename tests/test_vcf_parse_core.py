"""The device VCF parser's per-line core (ms_vcf_parse_core.h, host build in tests/emu/vcf_parse_emu.cpp) against the
host parser records_from_vcf, and the `vcf` sub-command's command line, without a GPU."""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from mutation_simulator_b200.records import CONV, REC_DTYPE, genome_offsets, records_from_vcf
from tests.helpers import MS_CASES, load_case

HERE = Path(__file__).resolve().parent
CSRC = HERE.parent / "mutation_simulator_b200" / "csrc"


@pytest.fixture(scope="module")
def core():
    src, lib = HERE / "emu" / "vcf_parse_emu.cpp", HERE / "emu" / "_build" / "libvcfparse.so"
    lib.parent.mkdir(exist_ok=True)
    deps = [src, CSRC / "ms_vcf_parse_core.h", CSRC / "ms_records.h", CSRC / "ms_rng.h"]
    if not lib.exists() or lib.stat().st_mtime < max(p.stat().st_mtime for p in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", str(lib), str(src)])
    L = C.CDLL(str(lib))
    L.vcf_parse.restype = C.c_int
    L.vcf_parse.argtypes = [C.c_char_p, C.c_int64, C.c_char_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                            C.c_void_p, C.POINTER(C.c_int64), C.c_void_p, C.POINTER(C.c_int64)]
    return L


def core_parse(core, text: bytes, names, lengths, skip_unknown=False):
    """-> (recs, pool) like records_from_vcf, or None when the core declares the text irregular."""
    blob = b"".join(names)
    off = np.zeros(len(names) + 1, np.int64)
    np.cumsum([len(n) for n in names], out=off[1:])
    lens = np.asarray(lengths, np.int64)
    out = np.zeros(text.count(b"\n") + 1, REC_DTYPE)
    lit = np.zeros(len(text) + 1, np.uint8)
    n, nl = C.c_int64(), C.c_int64()
    reg = core.vcf_parse(text, len(text), blob, off.ctypes.data, lens.ctypes.data, len(names), int(skip_unknown),
                         out.ctypes.data, C.byref(n), lit.ctypes.data, C.byref(nl))
    if not reg:
        return None
    return out[:n.value], lit[:nl.value].tobytes()


def host_parse(text: bytes, names, lengths, skip_unknown=False):
    recs, lit = records_from_vcf(text, names, genome_offsets(lengths), lengths, skip_unknown)
    n = 0
    if (recs["kind"] == 2).any():
        k = recs[recs["kind"] == 2]
        n = int((k["src"] + k["prod"]).max())
    return recs, lit[:n].tobytes()


def assert_same(got, want):
    assert got is not None, "regular text declared irregular"
    assert got[0].tobytes() == want[0].tobytes()
    assert got[1] == want[1]


@pytest.mark.parametrize("case", MS_CASES)
def test_golden_vcfs_parse_like_the_host(core, case):
    d, contigs = load_case(case)
    names, lens = [c[0] for c in contigs], [len(c[2]) for c in contigs]
    text = (d / "out.vcf").read_bytes()
    assert_same(core_parse(core, text, names, lens), host_parse(text, names, lens))


# ---- random VCFs in this package's output format -----------------------------------------------------------------
_COMP = bytes.maketrans(b"ACGTUMRWSYKVHDB", b"TGCAAKYWSRMBDHV")


def random_genome(rng, n_contigs=6, iupac=True):
    alphabet = np.frombuffer(b"ACGTNRYKMSWBDHV" if iupac else b"ACGT", np.uint8)
    lens = [int(x) for x in rng.integers(1, 3000, n_contigs)]
    lens[0] = max(lens[0], 500)
    return [(b"ctg%d" % i, rng.choice(alphabet, n).tobytes()) for i, n in enumerate(lens)]


def _contig_lines(rng, name: bytes, seq: bytes):
    """VCF lines of non-overlapping records on one contig, as VcfWriter.write words them (records.py:119-134)."""
    L, out, p = len(seq), [], int(rng.integers(0, 3))
    conv = lambda s: bytes(CONV[np.frombuffer(s, np.uint8)])
    while p < L:
        t = rng.choice(["SN", "IN", "DE", "IV", "DU", "TL", "TLI"], p=[0.4, 0.12, 0.12, 0.09, 0.09, 0.09, 0.09])
        d = int(rng.integers(1, 12))
        ins = rng.choice(np.frombuffer(b"ACGTN", np.uint8), d).tobytes()
        nm = name.decode()
        if t == "SN":
            line, cons = f"{p + 1}\t.\t{chr(CONV[seq[p]])}\t{'ACGT'[int(rng.integers(4))]}\t.\t.\t.", 1
        elif t in ("IN", "TLI"):
            sv = "INS" if t == "IN" else "INS:ME"
            if p == 0:
                ref = conv(seq[0:1]).decode()
                line = f"1\t.\t{ref}\t{ins.decode()}{ref}\t.\t.\tSVTYPE={sv};END=1;SVLEN={d}"
            else:
                ref = conv(seq[p - 1:p]).decode()
                line = f"{p}\t.\t{ref}\t{ref}{ins.decode()}\t.\t.\tSVTYPE={sv};END={p};SVLEN={d}"
            cons = 0
        elif t in ("DE", "TL"):
            sv = "DEL" if t == "DE" else "DEL:ME"
            d = min(d, L - p)
            if p == 0:
                ref = conv(seq[0:d + 1]).decode()
                line = f"1\t.\t{ref}\t{ref[-1]}\t.\t.\tSVTYPE={sv};END={d};SVLEN={d}"
                d = min(d, L)
            else:
                ref = conv(seq[p - 1:p + d]).decode()
                line = f"{p}\t.\t{ref}\t{ref[0]}\t.\t.\tSVTYPE={sv};END={p + d};SVLEN={d}"
            cons = d
        else:
            d = min(d, L - p)
            ref = conv(seq[p:p + d])
            alt = ref[::-1].translate(_COMP) if t == "IV" else ref * 2
            sv, svlen = ("INV", 0) if t == "IV" else ("DUP", d)
            line = f"{p + 1}\t.\t{ref.decode()}\t{alt.decode()}\t.\t.\tSVTYPE={sv};END={p + d};SVLEN={svlen}"
            cons = d if t == "IV" else 0
        out.append(f"{nm}\t{line}\tGT\t1\n".encode())
        p += max(cons, 1) + int(rng.integers(1, 40))
    return out


def random_vcf(rng, contigs, shuffle=True, header=True):
    """Text of a VCF over contigs [(name, seq)], one block of lines per contig, blocks in shuffled order."""
    blocks = [_contig_lines(rng, n, s) for n, s in contigs]
    order = rng.permutation(len(blocks)) if shuffle else range(len(blocks))
    head = b"##fileformat=VCFv4.3\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tUnknown\n" if header else b""
    return head + b"".join(b"".join(blocks[i]) for i in order)


@pytest.mark.parametrize("seed", range(12))
def test_random_vcfs_parse_like_the_host(core, seed):
    rng = np.random.default_rng(seed)
    contigs = random_genome(rng, iupac=seed % 2 == 0)
    text = random_vcf(rng, contigs)
    if seed % 3 == 0:
        text = text.rstrip(b"\n")          # last line without a line break
    names, lens = [n for n, _ in contigs], [len(s) for _, s in contigs]
    assert_same(core_parse(core, text, names, lens), host_parse(text, names, lens))
    # one rank of a contig-sharded run: the lines of other ranks' contigs are dropped
    keep = sorted(rng.choice(len(contigs), 3, replace=False))
    sub_n, sub_l = [names[i] for i in keep], [lens[i] for i in keep]
    assert_same(core_parse(core, text, sub_n, sub_l, True), host_parse(text, sub_n, sub_l, True))
    assert core_parse(core, text, sub_n, sub_l, False) is None     # unknown contigs: the host raises


def test_pos_one_anchors_and_iupac_refs(core):
    seq = b"RACGTNKACGTACGTTTGCA" * 5
    text = (b"c\t1\t.\tR\tGGR\t.\t.\tSVTYPE=INS;END=1;SVLEN=2\tGT\t1\n"
            b"c\t3\t.\tCG\tC\t.\t.\tSVTYPE=DEL;END=4;SVLEN=1\tGT\t1\n"
            b"c\t6\t.\tN\tA\t.\t.\t.\tGT\t1\n"
            b"c\t8\t.\tACGT\tACGT\t.\t.\tSVTYPE=INV;END=11;SVLEN=0\tGT\t1\n")
    want = host_parse(text, [b"c"], [len(seq)])
    assert_same(core_parse(core, text, [b"c"], [len(seq)]), want)
    assert list(want[0]["pos"]) == [0, 3, 5, 7]
    text2 = b"d\t1\t.\tAAC\tC\t.\t.\tSVTYPE=DEL:ME;END=2;SVLEN=2\tGT\t1\n"
    assert_same(core_parse(core, text2, [b"d"], [10]), host_parse(text2, [b"d"], [10]))


# ---- fuzz: single edits of valid files ------------------------------------------------------------------------------
def _edit(rng, text: bytes, names):
    lines = text.split(b"\n")
    body = [i for i, l in enumerate(lines) if l and not l.startswith(b"#")]
    kind = int(rng.integers(0, 9))
    if kind == 0:                                  # a byte swapped
        i = int(rng.integers(len(text)))
        b = [b"\r", b"\x85", b" ", b"+", b"_", bytes([int(rng.integers(65, 91))]), bytes([int(rng.integers(97, 123))])]
        return text[:i] + b[int(rng.integers(len(b)))] + text[i + 1:]
    if kind == 1:                                  # a tab removed
        tabs = [i for i, ch in enumerate(text) if ch == 9]
        i = tabs[int(rng.integers(len(tabs)))]
        return text[:i] + text[i + 1:]
    if kind == 2:                                  # a tab added
        i = int(rng.integers(len(text)))
        return text[:i] + b"\t" + text[i:]
    li = body[int(rng.integers(len(body)))]
    f = lines[li].split(b"\t")
    if kind == 3:                                  # INFO keys reordered or one added
        if f[7] == b".":
            f[7] = b"SVTYPE=INS;END=3;SVLEN=1" if rng.integers(2) else b".;X=1"
        else:
            kv = f[7].split(b";")
            f[7] = b";".join(kv[::-1]) if rng.integers(2) else f[7] + b";IMPRECISE=1"
    elif kind == 4:                                # a line moved
        ln = lines.pop(li)
        lines.insert(body[int(rng.integers(len(body)))], ln)
        return b"\n".join(lines)
    elif kind == 5:                                # a duplicated POS
        prev = [i for i in body if i < li]
        if prev:
            f[1] = lines[prev[-1]].split(b"\t")[1]
    elif kind == 6:                                # an unknown contig
        f[0] = b"chrUn"
    elif kind == 7:                                # another contig's name
        f[0] = names[int(rng.integers(len(names)))]
    else:                                          # POS off by a little
        f[1] = str(max(0, int(f[1]) + int(rng.integers(-3, 4)))).encode()
    lines[li] = b"\t".join(f)
    return b"\n".join(lines)


def test_fuzzed_edits_are_irregular_or_parse_like_the_host(core):
    rng = np.random.default_rng(2024)
    outcomes = {"irregular": 0, "same": 0, "host_raised": 0}
    for it in range(3000):
        if it % 100 == 0:
            contigs = random_genome(rng, n_contigs=3)
            names, lens = [n for n, _ in contigs], [len(s) for _, s in contigs]
            base = random_vcf(rng, contigs)
        text = _edit(rng, base, names)
        skip = bool(it % 2)
        got = core_parse(core, text, names, lens, skip)
        try:
            want = host_parse(text, names, lens, skip)
        except ValueError:
            outcomes["host_raised"] += 1
            assert got is None, text
            continue
        if got is None:
            outcomes["irregular"] += 1
        else:
            outcomes["same"] += 1
            assert_same(got, want)
    assert outcomes["irregular"] > 100 and outcomes["same"] > 100 and outcomes["host_raised"] > 100, outcomes


# ---- the `vcf` sub-command -----------------------------------------------------------------------------------------
def test_vcf_subcommand_and_output_names(tmp_path):
    from mutation_simulator_b200.argument_parser import get_args
    a = get_args([str(tmp_path / "g.fa"), "-o", str(tmp_path / "out"), "vcf", str(tmp_path / "t.vcf")])
    assert a.mode == "vcf" and a.vcffile == tmp_path / "t.vcf"
    assert (a.outfasta.name, a.outvcf.name) == ("out_ms.fa", "out_ms.vcf")
    b = get_args([str(tmp_path / "g.fa"), "--bgzip", "-o", str(tmp_path / "out"), "vcf", str(tmp_path / "t.vcf.gz")])
    assert (b.outfasta.name, b.outvcf.name) == ("out_ms.fa.gz", "out_ms.vcf.gz")
    with pytest.raises(SystemExit):
        get_args([str(tmp_path / "g.fa"), "vcf"])


@pytest.mark.parametrize("bgzip", [False, True])
def test_replaying_into_the_input_vcf_is_refused_before_any_output(tmp_path, bgzip):
    (tmp_path / "in.fa").write_bytes(b">c\nACGT\n")
    vcf = tmp_path / ("in_ms.vcf.gz" if bgzip else "in_ms.vcf")
    vcf.write_bytes(b"keep me")
    argv = [str(tmp_path / "in.fa"), "-o", str(tmp_path / "in")] + (["--bgzip"] if bgzip else []) + ["vcf", str(vcf)]
    r = subprocess.run([sys.executable, "-m", "mutation_simulator_b200"] + argv, capture_output=True, text=True,
                       cwd=str(HERE.parent))
    assert r.returncode == 1
    assert "ERROR:" in r.stderr and "overwrite" in r.stderr
    assert vcf.read_bytes() == b"keep me"
    assert not (tmp_path / ("in_ms.fa.gz" if bgzip else "in_ms.fa")).exists()
