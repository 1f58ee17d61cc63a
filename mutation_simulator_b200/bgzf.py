"""BGZF output (``--bgzip``): the device encoder's members streamed into a file, and reading BGZF FASTA back.

BGZF is a series of independent gzip members of at most 64 KiB of input each (SAM/BAM specification §4.1), which
``bgzip``, ``samtools faidx``, ``tabix`` and ``bcftools`` read.  The members written here are cut on 16 KiB cells of
the uncompressed file and never span two contigs (ms_bgzf_compress), so the compressed bytes do not depend on how
many GPUs wrote the file."""
from __future__ import annotations

import gzip

import numpy as np

# the empty member that ends every BGZF file
EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")

NOT_BGZF = ("Compressed FASTA is only supported in BGZF format. Use the samtools bgzip utility (instead of gzip) to "
            "compress your FASTA.")


def contig_segments(engine, which: int):
    """(src_off, nbytes) of every contig's slice of the FASTA image (which=0) or VCF body (which=1) of the last
    apply(); on one GPU the buffer is the file, so the file offsets are src_off."""
    fo, vo, _, _ = engine.contig_layout()
    lay = fo if which == 0 else vo
    return lay[:-1].copy(), np.diff(lay)


def window_segments(engine, which: int, lo: int, hi: int):
    """The contig slices of bytes [lo, hi) of the buffer (a tile-sharded rank's window), clipped to it."""
    src, n = contig_segments(engine, which)
    a = np.maximum(src, lo)
    b = np.minimum(src + n, hi)
    keep = b > a
    return a[keep], (b - a)[keep]


def write_from_engine(fh, engine, which: int):
    """Compress the whole buffer `which` of a one-GPU run into the open file at its position, then the EOF member."""
    from .engine import BUF_BGZF
    src, n = contig_segments(engine, which)
    _, tot = engine.bgzf_compress(which, src, n, src)
    fh.flush()
    off = fh.tell()
    if tot:
        engine.download_to_fd(BUF_BGZF, fh.fileno(), off, 0, tot)
    fh.seek(off + tot)
    fh.write(EOF)


def compress_host(data: bytes) -> bytes:
    """BGZF members of small host bytes (the VCF header), from the same encoder as the device's."""
    from .engine import bgzf_compress_host
    return bgzf_compress_host(data) if data else b""


def inflate_if_compressed(path):
    """None for a file that is not gzip-compressed; the inflated bytes of a BGZF file; FastaIndexingError for any
    other gzip file (what pyfaidx raises)."""
    from .fasta import FastaIndexingError
    with open(path, "rb") as fh:
        head = fh.read(16)
        if head[:2] != b"\x1f\x8b":
            return None
        # FLG.FEXTRA, then the BC subfield (SI1 'B', SI2 'C', SLEN 2) that bgzip and this package put first
        if len(head) < 16 or not head[3] & 4 or head[12:14] != b"BC" or head[14:16] != b"\x02\x00":
            raise FastaIndexingError(NOT_BGZF)
        fh.seek(0)
        return gzip.decompress(fh.read())
