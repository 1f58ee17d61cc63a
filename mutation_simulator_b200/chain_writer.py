"""Chain output (``--chain``): a UCSC chain file from the input genome to the mutated genome.

``liftOver``, CrossMap and the rest of the liftover ecosystem read it, so annotations (a GFF of the input, e.g. the
genes ``tools/gff_genes_2_rmt.py`` mutated) can be carried over to ``*_ms.fa`` and reads simulated from ``*_ms.fa``
mapped back to input coordinates.  Per contig in FASTA order the file holds its primary chain (the runs of bases the
mutated contig copies unchanged from the input; SNPs stay inside blocks) and then one single-block chain per stretch
that is copied from elsewhere: a duplication's copy (``+``), a translocation insert (``+``, or ``-`` when reversed) and
an inversion (``-``).  So a duplicated source maps to two places, an inversion to a gap of the primary chain plus a
``-`` chain, and a translocated source is a gap whose insert is a chain of its own.  Blocks may hold mismatches: SNPs,
the IUPAC conversion of translocation inserts, and '-' written as 'N'.  Chain ids run 1, 2, 3, ... through the file.

The mutation step's file is formatted on the GPU from the records of the apply (ms_chain_write).  The
interchromosomal step's file (``*_ms_it.chain``) maps that step's input to ``*_ms_it.fa`` and is built here from the
breakpoints, as the BEDPE is."""
from __future__ import annotations

import numpy as np


class ChainWriterError(Exception):
    """Raised when the chain file can not be written."""


def first_ids(n_chains, start: int = 1) -> np.ndarray:
    """Id of each contig's first chain when the contigs' chains are numbered consecutively from `start`."""
    n = np.asarray(n_chains, dtype=np.int64)
    return start + np.concatenate(([0], np.cumsum(n)[:-1])).astype(np.int64) if n.size else np.zeros(0, np.int64)


def _open(path):
    try:
        return open(path, "w+b")   # read-write: libmutsim_b200 maps the file for its parallel writers
    except OSError as e:
        raise ChainWriterError(f"Cannot write to chain file {path} {e}")


def write_from_engine(path, engine, bgzip: bool = False):
    """One GPU: format the chain file of the engine's last apply on the device and write it (BGZF with bgzip)."""
    from .engine import BUF_CHAIN
    off = engine.chain_write(first_ids(engine.chain_count()))
    with _open(path) as fh:
        if bgzip:
            from .bgzf import write_from_engine as write_bgzf
            write_bgzf(fh, engine, BUF_CHAIN)
        elif off[-1]:
            engine.download_to_fd(BUF_CHAIN, fh.fileno(), 0)


def write_text(path, data: bytes):
    """A chain file built on the host (the interchromosomal step's), already encoded."""
    with _open(path) as fh:
        fh.write(data)


def encode(text: bytes, bgzip: bool) -> bytes:
    """The file's bytes: the text, or its BGZF members and the end-of-file member."""
    if not bgzip:
        return text
    from .bgzf import EOF, compress_host
    return compress_host(text) + EOF


def _header(score, tname, tsize, t0, t1, qname, qsize, q0, q1, cid) -> str:
    return f"chain {score} {tname} {tsize} + {t0} {t1} {qname} {qsize} + {q0} {q1} {cid}\n"


def it_chain_text(names, lengths, partners, breakpoints) -> bytes:
    """The interchromosomal step's chain file.  names / lengths: the step's input contigs in FASTA order; partners[c]
    and breakpoints[c] = {"self": [...], "partner": [...]} as ITMutator keeps them.  A paired contig's output is its own
    even intervals with the partner's odd intervals between them (it_mutator.py:133-142): the own intervals are the
    blocks of its primary chain, and each non-empty partner interval is a '+' chain whose tName is the partner.
    Unpaired contigs get the identity chain; a contig of length 0 gets none."""
    out = []
    cid = 1
    for c, (name, L) in enumerate(zip(names, lengths)):
        L = int(L)
        if c not in breakpoints:
            if L > 0:
                out.append(_header(L, name, L, 0, L, name, L, 0, L, cid) + f"{L}\n\n")
                cid += 1
            continue
        p = partners[c]
        a = [0] + [int(x) for x in breakpoints[c]["self"]] + [L]
        b = [0] + [int(x) for x in breakpoints[c]["partner"]] + [int(lengths[p])]
        blocks, copies, q = [], [], 0
        for i in range(len(a) - 1):
            if i % 2 == 0:
                if a[i + 1] > a[i]:
                    blocks.append((a[i], q, a[i + 1] - a[i]))
                q += a[i + 1] - a[i]
            else:
                if b[i + 1] > b[i]:
                    copies.append((b[i], q, b[i + 1] - b[i]))
                q += b[i + 1] - b[i]
        Lq = q
        if blocks:
            (t0, q0, _), (tl, ql, nl) = blocks[0], blocks[-1]
            lines = [_header(sum(n for _, _, n in blocks), name, L, t0, tl + nl, name, Lq, q0, ql + nl, cid)]
            for (t, qq, n), (tn, qn, _) in zip(blocks, blocks[1:]):
                lines.append(f"{n}\t{tn - (t + n)}\t{qn - (qq + n)}\n")
            lines.append(f"{nl}\n\n")
            out.append("".join(lines))
            cid += 1
        pname, pl = names[p], int(lengths[p])
        for t, qq, n in copies:
            out.append(_header(n, pname, pl, t, t + n, name, Lq, qq, qq + n, cid) + f"{n}\n\n")
            cid += 1
    return "".join(out).encode("latin-1")
