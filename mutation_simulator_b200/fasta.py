"""Bulk FASTA loader with the ``pyfaidx.Fasta`` surface the reference uses.

Replaces util.load_fasta's ``pyfaidx.Fasta(..., as_raw=True,
sequence_always_upper=True)`` (util.py:77-91).  The whole file is parsed at once
with numpy into one upper-cased base array (what the GPU consumes); the objects
below are thin host views over it exposing exactly what reference-style code
reads: ``fasta[int|str]``, ``keys()``, ``get_seq(name, start1, end1)``,
``faidx.index[name].lenc``, ``close()``; records: ``len()``, ``[int]``, ``[a:b]``,
``.name``, ``.long_name``, iteration by line (SURVEY.md §8b/§8c).
"""
from __future__ import annotations

import mmap
import os
from pathlib import Path

import numpy as np

from .bgzf import inflate_if_compressed

_UPPER = np.arange(256, dtype=np.uint8)
_UPPER[ord("a"):ord("z") + 1] -= 32


class FastaIndexingError(Exception):
    """Malformed FASTA (same role as pyfaidx.FastaIndexingError)."""


class FastaNotFoundError(Exception):
    """FASTA file cannot be read (same role as pyfaidx.FastaNotFoundError)."""


class IndexEntry:
    __slots__ = ("rlen", "offset", "lenc", "lenb")

    def __init__(self, rlen, offset, lenc, lenb):
        self.rlen, self.offset, self.lenc, self.lenb = rlen, offset, lenc, lenb


class _Faidx:
    def __init__(self):
        self.index = {}


class FastaRecord:
    """One contig; a view into the genome array (upper-cased on access when the loader kept the file's case)."""

    def __init__(self, name: str, long_name: str, bases, lenc: int, is_upper: bool = True, length: int = None):
        """bases: a uint8 array, or a zero-argument callable that produces it on first use (lazy contigs)."""
        self.name = name
        self.long_name = long_name
        self._raw = bases
        self._lenc = lenc
        self._is_upper = is_upper
        self._length = int(length) if length is not None else int(bases.size)

    @property
    def _b(self) -> np.ndarray:
        if callable(self._raw):
            self._raw = self._raw()
        if not self._is_upper:
            self._raw = _UPPER[self._raw]
            self._is_upper = True
        return self._raw

    def __len__(self):
        return self._length

    def __getitem__(self, n):
        if isinstance(n, slice):
            start, stop, step = n.start, n.stop, n.step
            size = len(self)
            if not start:
                start = 0
            if not stop:  # pyfaidx: a falsy stop means "to the end"
                stop = size
            if stop < 0:
                stop += size
            if start < 0:
                start += size
            return self._b[start:stop][::step].tobytes().decode("latin-1")
        if n < 0:
            n += len(self)
        return chr(self._b[n])

    def __iter__(self):
        w = self._lenc if self._lenc > 0 else max(1, len(self))
        for i in range(0, len(self), w):
            yield self._b[i:i + w].tobytes().decode("latin-1")

    def __str__(self):
        return self._b.tobytes().decode("latin-1")

    @property
    def array(self) -> np.ndarray:
        """The upper-cased bases as uint8 (no copy)."""
        return self._b


class Fasta:
    """All contigs of one FASTA file, upper-cased, resident in host memory."""

    def __init__(self, filename, one_based_attributes=False, as_raw=True, sequence_always_upper=True,
                 read_ahead=None, build_index=True, device=None, **_):
        """A BGZF-compressed file (``--bgzip`` output, or ``bgzip``) is inflated on the host and parsed there; the .fai
        then holds offsets into the uncompressed text, as ``samtools faidx`` writes them.
        device: CUDA device index — the file is then ingested on that GPU (ms_fasta_ingest_fd: raw bytes to HBM,
        records / line layout / stripping / upper-casing there) and `self.engine` holds the resident genome for the
        Mutator / ITMutator that follows; host views of the bases are fetched from the device on demand.  Files that
        are not regularly wrapped, and device=None, go through the host parsers."""
        self.filename = str(filename)
        self.genome_is_upper = True
        self._lazy = None          # (mmap, uint8 view, spans, layout) of a regularly wrapped file: bases are copied on demand
        self._genome = None
        self.engine = None
        try:
            inflated = inflate_if_compressed(self.filename)     # BGZF input: inflated on the host, then the host parser
            if inflated is not None:
                self._parse(np.frombuffer(inflated, dtype=np.uint8), sequence_always_upper)
            elif device is not None and self._ingest_device(int(device)):
                pass
            elif not self._parse_regular():
                self._parse(np.fromfile(self.filename, dtype=np.uint8), sequence_always_upper)
        except (FileNotFoundError, IsADirectoryError, PermissionError):
            raise FastaNotFoundError(f"Cannot read FASTA from file {self.filename}")
        self.faidx = _Faidx()
        self._records = {}
        for i, nm in enumerate(self.names):
            if nm in self._records:
                raise ValueError(f"Duplicate key \"{nm}\"")  # util.py:89-91 maps this to FastaDuplicateHeaderError
            if self._lazy is not None or self.engine is not None:
                src = (lambda k=i: self.gather([k]))
            else:
                src = self._genome[self.goff[i]:self.goff[i + 1]]
            self._records[nm] = FastaRecord(nm, self.long_names[i], src, int(self.bpl[i]), self.genome_is_upper, int(self.lengths[i]))
            self.faidx.index[nm] = IndexEntry(int(self.lengths[i]), int(self._seq_off[i]), int(self.bpl[i]), int(self._lenb[i]))
        if build_index:
            self._write_fai()

    # -- parsing -----------------------------------------------------------
    def _ingest_device_sliced(self, device: int, rank: int, world: int):
        """One process per GPU: every rank looks for record starts in its 1/world slice of the file, the ranks exchange
        them, and each reads and indexes only the records of its own contigs (ms_fasta_ingest_ranges); names, lengths
        and line layout of all contigs are then gathered, so the object describes the whole file while only this rank's
        bases are resident.  Returns True / None (None: use the whole-file path — a genome that will be sharded by
        tiles, or a file the device indexer declines; decided identically on all ranks)."""
        from . import distributed as D
        from .engine import Engine
        D.init()
        size = os.path.getsize(self.filename)
        if size == 0:
            return None
        with open(self.filename, "rb") as fh:
            mm = mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ)
            try:
                lo, hi = size * rank // world, size * (rank + 1) // world
                starts = [0] if (rank == 0 and mm[0:1] == b">") else []
                pos = max(lo - 1, 0)
                while True:                       # "\n>" whose '>' lies in [lo, hi)
                    k = mm.find(b"\n>", pos, hi)
                    if k < 0:
                        break
                    starts.append(k + 1)
                    pos = k + 1
            finally:
                mm.close()
            every = sorted(set(x for part in D.all_gather_object(starts) for x in part))
            if not every or every[0] != 0:
                return None
            sizes = [b - a for a, b in zip(every, every[1:] + [size])]
            if D.shard_mode(sizes, world) != "contigs":
                return None
            parts = D.lpt_partition(sizes, world)
            mine = parts[rank]
            ranges = []                           # consecutive records become one read
            for g in mine:
                if ranges and ranges[-1][0] + ranges[-1][1] == every[g]:
                    ranges[-1][1] += sizes[g]
                else:
                    ranges.append([every[g], sizes[g]])
            eng = Engine(device)
            ok, info, names, long_names = False, None, [], []
            try:
                info = eng.ingest_fasta(fh.fileno(), size, ranges)
                if info is not None and len(info["long_names"]) == len(mine):
                    long_names = info["long_names"]
                    names = [(ln.split() or [""])[0] for ln in long_names]
                    ok = eng.commit_fasta(info["length"], info["lenc"], [ln.encode("latin-1") for ln in long_names],
                                          [nm.encode("latin-1") for nm in names], gid=mine)
            except Exception:
                eng.close()
                raise
        mine_off = np.concatenate(([0], np.cumsum([sizes[g] for g in mine])[:-1])).astype(np.int64) if mine else np.zeros(0, np.int64)
        payload = None
        if ok:
            payload = (mine, names, long_names, info["length"].tolist(), info["lenc"].tolist(), info["lenb"].tolist(),
                       [int(every[g] + (so - mo)) for g, so, mo in zip(mine, info["seq_off"].tolist(), mine_off.tolist())])
        gathered = D.all_gather_object(payload)
        n = len(every)
        all_names = [None] * n
        if any(p is None for p in gathered):
            eng.close()
            return None
        all_long = [None] * n
        length = np.zeros(n, np.int64); lenc = np.zeros(n, np.int32); lenb = np.zeros(n, np.int64); seq_off = np.zeros(n, np.int64)
        for ids, nm, ln, L, lc, lb, so in gathered:
            for j, g in enumerate(ids):
                all_names[g], all_long[g], length[g], lenc[g], lenb[g], seq_off[g] = nm[j], ln[j], L[j], lc[j], lb[j], so[j]
        if len(set(all_names)) != n:              # duplicate keys: the host parser owns pyfaidx's error message
            eng.close()
            return None
        self.engine = eng
        self.names, self.long_names = all_names, all_long
        self.lengths, self.bpl, self._lenb, self._seq_off = length, lenc, lenb, seq_off
        self.goff = np.zeros(n + 1, np.int64)
        np.cumsum(self.lengths, out=self.goff[1:])
        self.partition, self.shard = parts, "contigs"     # Mutator / ITMutator keep this partition
        self._resident_ids = list(mine)
        return True

    def _ingest_device(self, device: int) -> bool:
        from .engine import Engine
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if world > 1 and not os.environ.get("MS_FULL_INGEST"):
            if self._ingest_device_sliced(device, int(os.environ.get("RANK", "0")), world):
                return True
        with open(self.filename, "rb") as fh:
            size = os.fstat(fh.fileno()).st_size
            if size == 0:
                return False
            eng = Engine(device)
            try:
                info = eng.ingest_fasta(fh.fileno(), size)
                if info is None:
                    eng.close()
                    return False
                long_names = info["long_names"]
                names = [(ln.split() or [""])[0] for ln in long_names]
                if len(set(names)) != len(names):        # (raised as a duplicate-key error by the caller's loop)
                    eng.close()
                    return False
                ok = eng.commit_fasta(info["length"], info["lenc"], [ln.encode("latin-1") for ln in long_names],
                                      [nm.encode("latin-1") for nm in names])
            except Exception:
                eng.close()
                raise
            if not ok:
                eng.close()
                return False
        self.engine = eng
        self.names, self.long_names = names, long_names
        self.lengths = info["length"].astype(np.int64)
        self.bpl = info["lenc"].astype(np.int32)
        self._lenb = info["lenb"].astype(np.int64)
        self._seq_off = info["seq_off"].astype(np.int64)
        self.goff = np.zeros(len(names) + 1, np.int64)
        np.cumsum(self.lengths, out=self.goff[1:])
        return True

    def _parse_regular(self) -> bool:
        """Fast path for regularly wrapped files (every line of a record but the last has the same width, LF line
        ends): contig boundaries by memmem, bases by one strided 2-D copy per contig, no per-byte masking.  The
        file's case is kept; the GPU upper-cases at upload (ms_genome_upload) and host views upper-case lazily.
        Returns False when the layout is not regular (the general parser then decides whether it is an error)."""
        with open(self.filename, "rb") as fh:
            size = os.fstat(fh.fileno()).st_size
            if size == 0:
                return False
            mm = mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ)
        keep_open = False
        try:
            if mm[0:1] != b">":
                return False
            data = np.frombuffer(mm, dtype=np.uint8)
            keep_open = False
            spans = []      # (header start, header end, seq_lo, seq_hi)
            pos = 0
            while pos < size:
                he = mm.find(b"\n", pos)
                if he < 0:
                    he = size
                nxt = mm.find(b"\n>", he) if he < size else -1
                seq_lo = min(he + 1, size)
                seq_hi = nxt + 1 if nxt >= 0 else size
                spans.append((pos, he, seq_lo, seq_hi))
                pos = seq_hi
            n = len(spans)
            lengths = np.zeros(n, np.int64); lenc = np.zeros(n, np.int64); lenb = np.zeros(n, np.int64)
            layout = []
            for i, (_, _, lo, hi) in enumerate(spans):
                R = hi - lo
                if R == 0:
                    layout.append((0, 0, 0))
                    continue
                nl = mm.find(b"\n", lo, hi)
                if nl < 0:                       # one line, no line break at the end of the file
                    if mm.find(b"\r", lo, hi) >= 0:
                        return False
                    lenb[i] = R; lenc[i] = R; lengths[i] = R
                    layout.append((0, R, R))
                    continue
                if nl > lo and mm[nl - 1] == 13:
                    return False                 # CRLF files go through the general parser
                b = nl - lo + 1
                nfull = R // b
                tail = R - nfull * b
                tail_bases = tail
                # the partial last line may end with line breaks (blank lines at EOF are tolerated)
                while tail_bases > 0 and mm[lo + nfull * b + tail_bases - 1] == 10:
                    tail_bases -= 1
                if tail_bases and mm.find(b"\n", lo + nfull * b, lo + nfull * b + tail_bases) >= 0:
                    return False
                lenb[i] = b; lenc[i] = b - 1
                lengths[i] = nfull * (b - 1) + tail_bases
                layout.append((nfull, tail_bases, b))
            goff = np.zeros(n + 1, np.int64)
            np.cumsum(lengths, out=goff[1:])
            # validate the line structure now (cheap: one strided compare per contig), copy bases lazily
            for i, (_, _, lo, hi) in enumerate(spans):
                nfull, tail_bases, b = layout[i]
                if nfull and not (data[lo + b - 1:lo + nfull * b:b] == 10).all():
                    return False             # ragged lines
            self.names, self.long_names = [], []
            for hs, he, _, _ in spans:
                line = mm[hs + 1:he].decode("latin-1").rstrip("\r")
                self.long_names.append(line)
                tok = line.split()
                self.names.append(tok[0] if tok else "")
            self.lengths = lengths
            self.bpl = lenc.astype(np.int32)
            self._lenb = lenb
            self._seq_off = np.array([sp[2] for sp in spans], dtype=np.int64)
            self.goff = goff
            self.genome_is_upper = False
            self._lazy = (mm, data, spans, layout)
            keep_open = True
            return True
        finally:
            if not keep_open:
                try:
                    del data
                except NameError:
                    pass
                try:
                    mm.close()
                except BufferError:       # a view is still alive (early return paths): the GC closes it
                    pass

    def _copy_contig(self, i: int, dest: np.ndarray):
        """Bases of contig i (file case) into dest: one strided 2-D copy for the full lines + the partial last line."""
        _, data, spans, layout = self._lazy
        lo = spans[i][2]
        nfull, tail_bases, b = layout[i]
        o = 0
        if nfull:
            dest[:nfull * (b - 1)].reshape(nfull, b - 1)[:] = data[lo:lo + nfull * b].reshape(nfull, b)[:, :b - 1]
            o = nfull * (b - 1)
        if tail_bases:
            dest[o:o + tail_bases] = data[lo + nfull * b:lo + nfull * b + tail_bases]

    def gather(self, ids) -> np.ndarray:
        """Concatenated bases of the given contigs (file case for lazily loaded files; the GPU upper-cases)."""
        ids = list(ids)
        if self.engine is not None and self._genome is None:      # resident on the GPU: fetch the slices
            res = getattr(self, "_resident_ids", None)
            if res is not None:                                   # reduced to a rank's share (ms_genome_subset)
                loc = {g: k for k, g in enumerate(res)}
                off = np.concatenate(([0], np.cumsum([int(self.lengths[g]) for g in res])))
                parts = [self.engine.read_genome(int(off[loc[i]]), int(self.lengths[i])) for i in ids]
                return np.concatenate(parts) if parts else np.zeros(0, np.uint8)
            parts = [self.engine.read_genome(int(self.goff[i]), int(self.lengths[i])) for i in ids]
            return np.concatenate(parts) if parts else np.zeros(0, np.uint8)
        if self._lazy is None:
            if len(ids) == len(self.names) and ids == list(range(len(self.names))):
                return self._genome
            return np.concatenate([self._genome[self.goff[i]:self.goff[i + 1]] for i in ids]) if ids else np.zeros(0, np.uint8)
        off = np.zeros(len(ids) + 1, np.int64)
        np.cumsum([int(self.lengths[i]) for i in ids], out=off[1:])
        out = np.empty(int(off[-1]), dtype=np.uint8)
        jobs = [(i, out[off[k]:off[k + 1]]) for k, i in enumerate(ids) if self.lengths[i] > 0]
        big = sum(int(self.lengths[i]) for i in ids) > (64 << 20)
        if big and len(jobs) > 1:
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(min(len(jobs), os.cpu_count() or 1, 16)) as ex:   # numpy copies release the GIL
                list(ex.map(lambda j: self._copy_contig(*j), jobs))
        else:
            for j in jobs:
                self._copy_contig(*j)
        return out

    @property
    def genome(self) -> np.ndarray:
        """All contigs concatenated (materialised on first use for lazily loaded files)."""
        if self._genome is None:
            self._genome = self.gather(range(len(self.names)))
        return self._genome

    @genome.setter
    def genome(self, value):
        self._genome = value

    def _parse(self, data: np.ndarray, upper: bool):
        n = data.size
        nl = np.flatnonzero(data == 10)
        gt = np.flatnonzero(data == ord(">"))
        if gt.size:
            at_line_start = np.ones(gt.size, dtype=bool)
            nz = gt > 0
            at_line_start[nz] = data[gt[nz] - 1] == 10
            hdr = gt[at_line_start]
        else:
            hdr = gt
        if hdr.size == 0:
            raise FastaIndexingError(f"No sequences found in {self.filename}")
        # end of each header line
        k = np.searchsorted(nl, hdr)
        hdr_end = np.where(k < nl.size, nl[np.minimum(k, max(nl.size - 1, 0))] if nl.size else n, n).astype(np.int64)
        seq_lo = np.minimum(hdr_end + 1, n)
        seq_hi = np.append(hdr[1:], n).astype(np.int64)
        keep = (data != 10) & (data != 13)
        for a, b in zip(hdr.tolist(), seq_lo.tolist()):
            keep[a:b] = False
        if hdr[0] > 0:
            keep[:hdr[0]] = False  # anything before the first header is ignored
        lengths = np.add.reduceat(keep, hdr.astype(np.intp)).astype(np.int64) if n else np.zeros(0, np.int64)
        genome = data[keep]
        if upper:
            genome = _UPPER[genome]
        # bases per line of the first sequence line (pyfaidx lenc) and bytes per line (lenb)
        k1 = np.searchsorted(nl, seq_lo)
        first_nl = np.where(k1 < nl.size, nl[np.minimum(k1, max(nl.size - 1, 0))] if nl.size else n, n)
        first_end = np.minimum(first_nl, seq_hi)
        lenb = np.where(first_nl < seq_hi, first_end - seq_lo + 1, first_end - seq_lo)
        cr = np.zeros(hdr.size, dtype=np.int64)
        has = first_end > seq_lo
        cr[has] = data[np.maximum(first_end[has] - 1, 0)] == 13
        lenc = np.maximum(first_end - seq_lo - cr, 0)
        self._check_line_widths(data, nl, seq_lo, seq_hi, lenb)
        self.names, self.long_names = [], []
        for a, b in zip(hdr.tolist(), hdr_end.tolist()):
            line = data[a + 1:b].tobytes().decode("latin-1").rstrip("\r")
            self.long_names.append(line)
            tok = line.split()
            self.names.append(tok[0] if tok else "")
        self.lengths = lengths
        self.bpl = lenc.astype(np.int32)
        self._lenb = lenb
        self._seq_off = seq_lo
        self.goff = np.zeros(hdr.size + 1, dtype=np.int64)
        np.cumsum(lengths, out=self.goff[1:])
        self.genome = genome

    def _check_line_widths(self, data, nl, seq_lo, seq_hi, lenb):
        """pyfaidx refuses records whose lines (all but the last) differ in length."""
        if nl.size == 0:
            return
        starts = np.concatenate(([0], nl[:-1] + 1))
        widths = nl - starts + 1                       # bytes per line incl. '\n'
        rec = np.searchsorted(seq_lo, starts, side="right") - 1
        ok = (rec >= 0)
        inside = ok & (starts >= seq_lo[np.maximum(rec, 0)]) & (starts < seq_hi[np.maximum(rec, 0)])
        if not inside.any():
            return
        r = rec[inside]
        w = widths[inside]
        e = nl[inside] + 1
        last = e >= seq_hi[r]                          # last line of the record may be shorter
        bad = (~last) & (w != lenb[r])
        long_last = last & (w > lenb[r])
        if bad.any() or long_last.any():
            i = int(r[np.flatnonzero(bad | long_last)[0]])
            raise FastaIndexingError(f"Line length of fasta file is not consistent! Inconsistent line found in record {i + 1}")

    def _write_fai(self):
        """pyfaidx leaves <file>.fai next to the input (README 'Notes') and rebuilds it when it is older than the FASTA;
        keep that side effect when the directory is writable.  One process per GPU: only rank 0 writes it, through a
        temporary file, so that concurrent readers never see a partial index."""
        if int(os.environ.get("RANK", "0")) != 0:
            return
        p = Path(self.filename + ".fai")
        try:
            if p.exists() and p.stat().st_mtime >= Path(self.filename).stat().st_mtime:
                return
            tmp = Path(f"{p}.{os.getpid()}.tmp")
            with open(tmp, "w") as fh:
                for nm in self.names:
                    e = self.faidx.index[nm]
                    fh.write(f"{nm}\t{e.rlen}\t{e.offset}\t{e.lenc}\t{e.lenb}\n")
            os.replace(tmp, p)
        except OSError:
            pass

    # -- pyfaidx surface ---------------------------------------------------
    def keys(self):
        return list(self.names)

    def __len__(self):
        return len(self.names)

    def __iter__(self):
        return iter(self._records[nm] for nm in self.names)

    def __contains__(self, key):
        return key in self._records

    def __getitem__(self, key):
        if isinstance(key, (int, np.integer)):
            return self._records[self.names[key]]
        return self._records[key]

    def get_seq(self, name, start, end, rc=False):
        return self._records[name]._b[start - 1:end].tobytes().decode("latin-1")

    def detach_engine(self):
        """Hand the engine that holds the ingested genome to the caller (who then owns and closes it)."""
        eng, self.engine = self.engine, None
        return eng

    def close(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None
        if self._lazy is not None:
            mm = self._lazy[0]
            self._lazy = None
            try:
                mm.close()
            except BufferError:
                pass

    # -- engine side -------------------------------------------------------
    def upload(self, engine, contig_ids=None):
        """Make this genome (or a subset of its contigs) resident on the engine's GPU."""
        # (the engine upper-cases on the device, so a mixed-case host array is fine)
        ids = list(range(len(self.names))) if contig_ids is None else list(contig_ids)
        if engine is self.engine and self.engine is not None:     # ingested on this engine: already resident
            if ids != list(range(len(self.names))):
                if self._genome is None and getattr(self, "_resident_ids", None) is None:
                    self._resident_ids = ids                      # host views of the other contigs are gone from now on
                    engine.subset_genome(ids)
                elif getattr(self, "_resident_ids", None) != ids:
                    raise ValueError("the resident genome was already reduced to a different set of contigs")
            return ids
        bases = self.gather(ids)
        engine.upload_genome(bases, [int(self.lengths[i]) for i in ids], [int(self.bpl[i]) for i in ids],
                             [self.long_names[i].encode("latin-1") for i in ids],
                             [self.names[i].encode("latin-1") for i in ids], gid=ids)
        return ids


class ResidentFasta:
    """The mutated genome of a finished Mutator run, still resident on its engine: what the reference obtains by
    load_fasta(args.outfasta) between Mutator and ITMutator (__main__.py:88-95), without the trip through the file.
    Exposes the part of the Fasta surface ITMutator uses (names, lengths, records with len()/name)."""

    def __init__(self, engine, source: "Fasta", my_ids=None, parts=None):
        """my_ids / parts: one process per GPU — the engine holds the contigs my_ids (global indices) of the partition
        `parts`; the mutated lengths of the others are gathered from their ranks, and the IT step keeps the partition."""
        lens = np.asarray(engine.adopt_output(), dtype=np.int64)
        self.engine = engine
        self.names = list(source.names)
        self.long_names = list(source.long_names)
        if my_ids is None:
            self.lengths = lens
            self._my_ids = None
        else:
            from . import distributed as D
            self.lengths = np.zeros(len(self.names), dtype=np.int64)
            for ids, ln in D.all_gather_object((list(my_ids), lens.tolist())):
                if len(ids):
                    self.lengths[ids] = ln
            self._my_ids = list(my_ids)
            self.partition, self.shard = parts, "contigs"
        self.goff = np.concatenate(([0], np.cumsum(self.lengths)[:-1])).astype(np.int64)
        self._records = {nm: FastaRecord(nm, ln, None, 0, length=int(n))
                         for nm, ln, n in zip(self.names, self.long_names, self.lengths)}

    def keys(self):
        return list(self.names)

    def __len__(self):
        return len(self.names)

    def __getitem__(self, key):
        if isinstance(key, (int, np.integer)):
            return self._records[self.names[key]]
        return self._records[key]

    def close(self):
        pass

    def upload(self, engine, contig_ids=None):
        mine = getattr(self, "_my_ids", None)
        if engine is not self.engine or (contig_ids is not None and list(contig_ids) != (mine if mine is not None else list(range(len(self.names))))):
            raise ValueError("a resident genome lives on the engine that produced it")
        return mine if mine is not None else list(range(len(self.names)))
