"""The BGZF encoder core (ms_bgzf_core.h, host build in tests/emu/bgzf_emu.cpp), the --bgzip output names and
BGZF FASTA input, without a GPU."""
import ctypes as C
import gzip
import struct
import subprocess
import zlib
from pathlib import Path

import numpy as np
import pytest

HERE = Path(__file__).resolve().parent
CORE = HERE.parent / "mutation_simulator_b200" / "csrc" / "ms_bgzf_core.h"


@pytest.fixture(scope="module")
def core():
    src, lib = HERE / "emu" / "bgzf_emu.cpp", HERE / "emu" / "_build" / "libbgzf.so"
    lib.parent.mkdir(exist_ok=True)
    if not lib.exists() or lib.stat().st_mtime < max(src.stat().st_mtime, CORE.stat().st_mtime):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", str(lib), str(src)])
    L = C.CDLL(str(lib))
    L.bgzf_crc32.restype = C.c_uint32
    L.bgzf_crc32.argtypes = [C.c_char_p, C.c_int64]
    L.bgzf_crc32_combine.restype = C.c_uint32
    L.bgzf_crc32_combine.argtypes = [C.c_uint32, C.c_uint32, C.c_uint64]
    L.bgzf_crc32_raw_finish.restype = C.c_uint32
    L.bgzf_crc32_raw_finish.argtypes = [C.c_char_p, C.c_int64]
    return L


def encode(core, data: bytes) -> bytes:
    dst = C.create_string_buffer(core.bgzf_max_member())
    n = core.bgzf_encode_member(data, len(data), dst)
    return dst.raw[:n]


def parse_member(z: bytes):
    """-> (BSIZE + 1, CRC32, ISIZE, deflate bytes) of one BGZF member, checking the fixed header fields."""
    assert z[:4] == b"\x1f\x8b\x08\x04" and z[4:8] == b"\0\0\0\0" and z[9] == 255
    xlen, = struct.unpack("<H", z[10:12])
    assert xlen == 6 and z[12:14] == b"BC" and z[14:16] == b"\x02\x00"
    bsize, = struct.unpack("<H", z[16:18])
    crc, isize = struct.unpack("<II", z[-8:])
    return bsize + 1, crc, isize, z[18:-8]


def _fasta_lines(rng, n):
    seq = rng.choice(np.frombuffer(b"ACGT", np.uint8), n).tobytes()
    return b"".join(seq[i:i + 60] + b"\n" for i in range(0, n, 60))


def _vcf_lines(rng, n):
    out = []
    pos = 1000
    for _ in range(n):
        pos += int(rng.integers(1, 200))
        ref = rng.choice(np.frombuffer(b"ACGT", np.uint8), int(rng.integers(1, 8))).tobytes().decode()
        out.append(f"chr7\t{pos}\t.\t{ref}\t{ref[0]}\t.\t.\tSVTYPE=DEL;END={pos + len(ref) - 1};SVLEN={len(ref) - 1}\tGT\t1\n")
    return "".join(out).encode()


def _cases():
    rng = np.random.default_rng(7)
    return {
        "empty": b"",
        "one_byte": b"A",
        "n_block": b"N" * 16384,
        "acgt_fasta": _fasta_lines(rng, 16000)[:16384],
        "vcf": _vcf_lines(rng, 400)[:16384],
        "all_bytes": bytes(range(256)) * 64,
        "random": rng.integers(0, 256, 16384, dtype=np.uint8).tobytes(),
        "header_text": b">chr1 some description\n" + _fasta_lines(rng, 900),
    }


@pytest.mark.parametrize("name", list(_cases()))
def test_member_inflates_to_its_input(core, name):
    data = _cases()[name]
    z = encode(core, data)
    assert gzip.decompress(z) == data
    size, crc, isize, deflate = parse_member(z)
    assert size == len(z) and isize == len(data) and crc == zlib.crc32(data)
    assert zlib.decompressobj(-15).decompress(deflate) == data
    assert len(z) <= len(data) + 31


def test_stored_fallback_and_ratios(core):
    c = _cases()
    for name in ("random", "all_bytes", "empty", "one_byte"):
        assert core.bgzf_is_stored(c[name], len(c[name])) == 1, name
        assert len(encode(core, c[name])) == len(c[name]) + 31
    for name in ("acgt_fasta", "vcf", "n_block"):
        assert core.bgzf_is_stored(c[name], len(c[name])) == 0, name
    # uniform ACGT text with line breaks: about 2 bits per base
    assert len(c["acgt_fasta"]) / len(encode(core, c["acgt_fasta"])) > 3.3
    # the code is dynamic Huffman (BTYPE=10) for compressible blocks
    assert parse_member(encode(core, c["vcf"]))[3][0] & 7 == 0b101


def test_length_limited_code_is_complete(core):
    """Fibonacci frequencies make plain Huffman codes as deep as the alphabet; limited to 15 (and 7) bits the code
    must still be complete: Kraft sum exactly 1."""
    fib = [1, 1]
    while len(fib) < 40:
        fib.append(fib[-1] + fib[-2])
    for nsym, limit in ((40, 15), (19, 7), (257, 15)):
        f = (fib * 7)[:nsym] if nsym > 40 else fib[:nsym]
        freq = (C.c_uint32 * nsym)(*f)
        out = (C.c_uint32 * nsym)()
        core.bgzf_huff_lengths(freq, nsym, limit, out)
        lens = list(out)
        assert max(lens) <= limit and min(lens) >= 1
        assert sum(2.0 ** -l for l in lens) == 1.0
        # more frequent symbols never get longer codes
        order = sorted(range(nsym), key=lambda s: (f[s], s))
        assert all(lens[order[i]] >= lens[order[i + 1]] for i in range(nsym - 1))
    # a single used symbol still yields a complete two-codeword code
    freq = (C.c_uint32 * 4)(0, 0, 9, 0)
    out = (C.c_uint32 * 4)()
    core.bgzf_huff_lengths(freq, 4, 15, out)
    assert sorted(out) == [0, 0, 1, 1]


def test_crc_combine(core):
    data = _cases()["vcf"][:3000]
    for k in range(0, len(data) + 1, 7):
        a, b = data[:k], data[k:]
        assert core.bgzf_crc32_combine(zlib.crc32(a), zlib.crc32(b), len(b)) == zlib.crc32(data)
    for n in (0, 1, 63, 64, 65, 16384):
        d = np.random.default_rng(n).integers(0, 256, n, dtype=np.uint8).tobytes()
        assert core.bgzf_crc32_raw_finish(d, n) == zlib.crc32(d) == core.bgzf_crc32(d, n)


def test_output_names_with_and_without_bgzip(tmp_path):
    from mutation_simulator_b200.argument_parser import get_args
    base = ["-o", str(tmp_path / "out"), "args", "-sn", "0.01"]
    a = get_args([str(tmp_path / "in.fa")] + base)
    assert (a.outfasta.name, a.outfastait.name, a.outvcf.name, a.outbedpe.name) == \
        ("out_ms.fa", "out_ms_it.fa", "out_ms.vcf", "out_ms_it.bedpe")
    assert a.bgzip is False
    b = get_args([str(tmp_path / "in.fa"), "--bgzip"] + base)
    assert (b.outfasta.name, b.outfastait.name, b.outvcf.name, b.outbedpe.name) == \
        ("out_ms.fa.gz", "out_ms_it.fa.gz", "out_ms.vcf.gz", "out_ms_it.bedpe")


def _bgzf_file(core, data: bytes) -> bytes:
    from mutation_simulator_b200.bgzf import EOF
    return b"".join(encode(core, data[i:i + 16384]) for i in range(0, len(data), 16384)) + EOF


def test_bgzf_fasta_loads_like_the_plain_file_and_plain_gzip_is_refused(core, tmp_path):
    from mutation_simulator_b200 import load_fasta
    from mutation_simulator_b200.fasta import FastaIndexingError
    rng = np.random.default_rng(5)
    text = b"".join(b">c%d desc\n" % i + _fasta_lines(rng, n) for i, n in enumerate((50_000, 61, 7, 33_333)))
    (tmp_path / "p.fa").write_bytes(text)
    (tmp_path / "z.fa.gz").write_bytes(_bgzf_file(core, text))
    assert gzip.decompress((tmp_path / "z.fa.gz").read_bytes()) == text
    plain, z = load_fasta(tmp_path / "p.fa"), load_fasta(tmp_path / "z.fa.gz")
    assert z.names == plain.names and z.long_names == plain.long_names
    assert (z.lengths == plain.lengths).all() and (z.bpl == plain.bpl).all()
    assert all(str(z[i]) == str(plain[i]) for i in range(4))
    # the index side effect uses offsets into the uncompressed text, as samtools faidx does
    assert (tmp_path / "z.fa.gz.fai").read_text() == (tmp_path / "p.fa.fai").read_text()
    plain.close(); z.close()
    (tmp_path / "g.fa.gz").write_bytes(gzip.compress(text))
    with pytest.raises(FastaIndexingError, match="only supported in BGZF format"):
        load_fasta(tmp_path / "g.fa.gz")
