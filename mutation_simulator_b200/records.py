"""Host-side construction of splice descriptors (``Rec``, csrc/ms_records.h) from
a typed mutation table — the replay input of Gate A (SURVEY.md §4.2) and the
hand-off format of ``ms_load_records``.

A typed mutation is what the reference's walk receives in its ``muts`` dict
(mutator.py:26-47, :318-426): key, type, start, stop, reverse, plus the two RNG
outputs the walk would draw itself (SNP ALT base, insert string).
"""
from __future__ import annotations

import numpy as np

REC_DTYPE = np.dtype([("pos", "<u4"), ("cons", "<u4"), ("prod", "<u4"), ("out", "<u4"), ("src", "<i8"),
                      ("kind", "u1"), ("type", "u1"), ("ref", "u1"), ("alt", "u1"), ("contig", "<u4")])
assert REC_DTYPE.itemsize == 32

T_SN, T_IN, T_DE, T_IV, T_DU, T_TL, T_TLI, T_IT = range(8)
TYPE_CODE = {"SN": T_SN, "IN": T_IN, "DE": T_DE, "IV": T_IV, "DU": T_DU, "TL": T_TL, "TLI": T_TLI, "IT": T_IT}
TYPE_NAME = {v: k for k, v in TYPE_CODE.items()}
K_NONE, K_SNP, K_LIT, K_RAW, K_CONV, K_RC = range(6)

# mutator.py:75 non_ambiguous as a 256-entry table
CONV = np.arange(256, dtype=np.uint8)
for _a, _b in zip(b"KSYMWRBDHV-", b"GCCAAACAAAN"):
    CONV[_a] = _b


def align16(n: int) -> int:
    return (n + 15) & ~15


def genome_offsets(lengths) -> np.ndarray:
    """Index of base 0 of each contig in the genome array (contigs are simply concatenated;
    the device copy carries 64 pad bytes after the last base)."""
    goff = np.zeros(len(lengths) + 1, dtype=np.int64)
    np.cumsum(np.asarray(lengths, dtype=np.int64), out=goff[1:])
    return goff


def pack_genome(seqs) -> tuple[np.ndarray, np.ndarray]:
    """seqs: list of upper-cased uint8 arrays/bytes -> (padded genome with 64 trailing pad bytes, goff)."""
    goff = genome_offsets([len(s) for s in seqs])
    g = np.full(int(goff[-1]) + 64, ord("N"), dtype=np.uint8)
    for i, s in enumerate(seqs):
        a = np.frombuffer(s, dtype=np.uint8) if isinstance(s, (bytes, bytearray)) else np.asarray(s, dtype=np.uint8)
        g[goff[i]:goff[i] + len(a)] = a
    return g, goff


def build_records(genome: np.ndarray, goff: np.ndarray, lengths, tables) -> tuple[np.ndarray, np.ndarray]:
    """tables: per contig a list of dicts/objects with key,type,start,stop,reverse,alt,insert
    (already restricted to the mutations the walk visits).  Returns (recs sorted by
    (contig, pos) with ``out`` = 0, literal pool)."""
    rows = []
    lit = bytearray()
    for ci, muts in enumerate(tables):
        g0 = int(goff[ci])
        L = int(lengths[ci])
        for m in sorted(muts, key=lambda x: _get(x, "key")):
            key, typ = int(_get(m, "key")), _get(m, "type")
            t = TYPE_CODE[typ] if isinstance(typ, str) else int(typ)
            start, stop = int(_get(m, "start")), int(_get(m, "stop"))
            if not (0 <= key < L):
                raise ValueError(f"mutation key {key} outside contig {ci} (length {L})")
            ref = alt = 0
            src = 0
            if t == T_SN:
                cons, prod, kind = 1, 1, K_SNP
                ref = int(CONV[genome[g0 + key]])
                a = _get(m, "alt")
                alt = a[0] if isinstance(a, (bytes, bytearray)) else (ord(a) if isinstance(a, str) else int(a))
            elif t == T_IN:
                ins = _get(m, "insert")
                ins = ins.encode() if isinstance(ins, str) else bytes(ins)
                cons, prod, kind, src = 0, len(ins), K_LIT, len(lit)
                lit += ins
            elif t in (T_DE, T_TL):
                cons, prod, kind = stop - start + 1, 0, K_NONE
            elif t == T_IV:
                n = stop - start + 1
                cons, prod, kind, src = n, n, K_RC, g0 + key
            elif t == T_DU:
                cons, prod, kind, src = 0, stop - start + 1, K_RAW, g0 + key
            elif t == T_TLI:
                ins = _get(m, "insert", None)
                if ins is not None:  # literal insert (VCF replay: the source TL is not recorded in the VCF)
                    ins = ins.encode() if isinstance(ins, str) else bytes(ins)
                    cons, prod, kind, src = 0, len(ins), K_LIT, len(lit)
                    lit += ins
                else:
                    cons, prod, src = 0, stop - start + 1, g0 + start
                    kind = K_RC if _get(m, "reverse", False) else K_CONV
            else:
                raise ValueError(f"unknown mutation type {typ}")
            if key + cons > L:
                raise ValueError(f"mutation at {key} of contig {ci} runs past the contig end")
            rows.append((key, cons, prod, 0, src, kind, t, ref, alt, ci))
    recs = np.array(rows, dtype=REC_DTYPE) if rows else np.zeros(0, dtype=REC_DTYPE)
    return recs, np.frombuffer(bytes(lit) + b"\0" * 16, dtype=np.uint8).copy()


def _get(m, name, default=KeyError):
    if isinstance(m, dict):
        if default is KeyError:
            return m[name]
        return m.get(name, default)
    if default is KeyError:
        return getattr(m, name)
    return getattr(m, name, default)


# ---------------------------------------------------------------------------------------
# Replay of the reference's FILES: a VCF written by VcfWriter.write (vcf_writer.py:118-126,
# info string :44-52) back into splice descriptors.  Record wording per type: mutator.py:334-421.
# ---------------------------------------------------------------------------------------
_SVTYPE = {"INS": T_IN, "DEL": T_DE, "INV": T_IV, "DUP": T_DU, "DEL:ME": T_TL, "INS:ME": T_TLI}


def parse_gt(field: str, ploidy: int) -> int:
    """A phased genotype of `ploidy` alleles from {0, 1} joined by '|' -> its haplotype mask (bit h-1 = allele h is 1);
    ValueError for anything else."""
    alleles = field.split("|")
    if len(alleles) != ploidy or any(a not in ("0", "1") for a in alleles):
        raise ValueError(f"GT {field!r} is not a phased genotype of ploidy {ploidy} ({ploidy} alleles of 0 or 1 joined by '|')")
    return sum(1 << h for h, a in enumerate(alleles) if a == "1")


def records_from_vcf(text, names, goff, lengths, skip_unknown: bool = False, ploidy=None):
    """VCF text (header lines are skipped) -> (recs sorted by (contig, pos), literal pool) for ``ms_load_records``.
    With `ploidy` (a phased VCF of a polyploid run) -> (recs, literal pool, haplotype masks in record order): field 10 of
    every record must be a GT of exactly `ploidy` alleles of 0 / 1 joined by '|' (:func:`parse_gt`).

    names: contig names (VCF CHROM) in genome order; goff/lengths as in :func:`build_records`.
    The replay rule is "replace REF by ALT at POS" (SURVEY.md §8c) expressed without touching the anchor base of
    INS / INS:ME / DEL / DEL:ME records (their REF shows the IUPAC-converted anchor, the FASTA keeps the raw one):
      SNP     POS=pos+1                                     -> substitute ALT
      INS     ALT = REF + insert (pos > 0, POS = pos)       -> insert before base POS   (mutator.py:343-358)
              ALT = insert + REF (pos = 0, POS = END = 1)   -> insert before base 0
      INS:ME  same, the inserted (already converted / reverse-complemented) string is literal  (:401-421)
      DEL / DEL:ME  ALT = REF[0] (pos > 0, POS = pos)       -> drop SVLEN bases from POS       (:360-377)
                    ALT = REF[-1] (pos = 0, POS = 1)        -> drop SVLEN bases from 0
      INV     POS=pos+1, SVLEN is 0                          -> reverse complement of len(REF) bases  (:379-387)
      DUP     POS=pos+1                                      -> the SVLEN bases at POS twice           (:389-399)
    A record whose ALT both starts and ends with REF (or, for DEL, REF[0] == REF[-1] at POS 1) is read as anchored
    before; both readings give the same output except for an IUPAC anchor at the very first base of a contig."""
    if isinstance(text, (bytes, bytearray)):
        text = bytes(text).decode("latin-1")
    index = {(n.decode("latin-1") if isinstance(n, (bytes, bytearray)) else str(n)): i for i, n in enumerate(names)}
    rows, lit, masks = [], bytearray(), {}
    for ln, line in enumerate(text.splitlines(), 1):
        if not line or line[0] == "#":
            continue
        f = line.split("\t")
        if len(f) < 8:
            raise ValueError(f"VCF line {ln}: expected at least 8 tab-separated fields")
        if f[0] not in index:
            if skip_unknown:      # several GPUs: the contig belongs to another rank
                continue
            raise ValueError(f"VCF line {ln}: unknown contig {f[0]!r}")
        ci = index[f[0]]
        if ploidy is not None:
            if len(f) < 10:
                raise ValueError(f"VCF line {ln}: no GT field (field 10) for ploidy {ploidy}")
            try:
                masks[len(rows)] = parse_gt(f[9], ploidy)
            except ValueError as e:
                raise ValueError(f"VCF line {ln}: {e}") from None
        g0, L = int(goff[ci]), int(lengths[ci])
        pos1, ref, alt = int(f[1]), f[3].encode("latin-1"), f[4].encode("latin-1")
        if f[7] == ".":
            if len(ref) != 1 or len(alt) != 1:
                raise ValueError(f"VCF line {ln}: a record without INFO must be a single-base substitution")
            if not (1 <= pos1 <= L):
                raise ValueError(f"VCF line {ln}: record outside contig {f[0]!r} (length {L})")
            rows.append((pos1 - 1, 1, 1, 0, 0, K_SNP, T_SN, ref[0], alt[0], ci))
            continue
        info = dict(kv.split("=", 1) for kv in f[7].split(";") if "=" in kv)
        try:
            t, svlen = _SVTYPE[info["SVTYPE"]], int(info["SVLEN"])
        except KeyError:
            raise ValueError(f"VCF line {ln}: unsupported INFO {f[7]!r}") from None
        if t in (T_IN, T_TLI):
            if alt.startswith(ref):
                pos, ins = pos1, alt[len(ref):]
            elif alt.endswith(ref) and pos1 == 1:
                pos, ins = 0, alt[:len(alt) - len(ref)]
            else:
                raise ValueError(f"VCF line {ln}: ALT of an insertion must extend REF")
            rows.append((pos, 0, len(ins), 0, len(lit), K_LIT, t, 0, 0, ci))
            lit += ins
        elif t in (T_DE, T_TL):
            if alt == ref[:1]:
                pos = pos1
            elif alt == ref[-1:] and pos1 == 1:
                pos = 0
            else:
                raise ValueError(f"VCF line {ln}: ALT of a deletion must be the first (or, at POS 1, the last) base of REF")
            cons = min(svlen, L - pos)
            rows.append((pos, cons, 0, 0, 0, K_NONE, t, 0, 0, ci))
        elif t == T_IV:
            rows.append((pos1 - 1, len(ref), len(ref), 0, g0 + pos1 - 1, K_RC, t, 0, 0, ci))
        else:   # DUP
            rows.append((pos1 - 1, 0, len(ref), 0, g0 + pos1 - 1, K_RAW, t, 0, 0, ci))
        p, c = rows[-1][0], rows[-1][1]
        if not (0 <= p < L) or p + c > L:
            raise ValueError(f"VCF line {ln}: record outside contig {f[0]!r} (length {L})")
    order = sorted(range(len(rows)), key=lambda i: (rows[i][9], rows[i][0]))
    rows = [rows[i] for i in order]
    recs = np.array(rows, dtype=REC_DTYPE) if rows else np.zeros(0, dtype=REC_DTYPE)
    pool = np.frombuffer(bytes(lit) + b"\0" * 16, dtype=np.uint8).copy()
    if ploidy is None:
        return recs, pool
    return recs, pool, np.array([masks[i] for i in order], dtype=np.uint8)
