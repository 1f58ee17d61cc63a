"""Paired-end reads (``--reads``): FASTQ pairs drawn on the GPU from the mutated genome that is still in HBM after its
FASTA is written, with the truth of every pair in its name.

The draw is a pure function of (seed, contig gid, haplotype, pair index) (ms_reads_core.h), so the files do not depend
on how the pairs are batched or on the number of GPUs.  Contig c of haplotype h gets ``pair_counts`` pairs; pairs come
in file order: haplotype 1..P, contigs in FASTA order, pair index.  The device formats one batch of pairs at a time into
buffer 9 (R1 records, then the R2 records of the same pairs, of equal size), bounded by a budget of FASTQ bytes per
call: 30x of a human diploid sample is about 220 GB of FASTQ, more than HBM holds.  With ``--bgzip`` each batch is
compressed on the device into BGZF members that continue at the file's uncompressed offset."""
from __future__ import annotations

import math
import os

import numpy as np

DEFAULT_BATCH_BYTES = 4 << 30     # FASTQ text (R1 + R2) formatted in HBM per call
_HEADER_FIXED = 64                # bytes of a record's name line besides the contig name (7 fields of <= 10 digits, ...)


class ReadsWriterError(Exception):
    """Raised when a FASTQ file can not be written."""


def pair_counts(coverage: float, out_lens, read_len: int, ploidy: int) -> np.ndarray:
    """Pairs of each contig of one haplotype: floor(C * Lp / (2 L P)) in float64, 0 when the mutated length Lp < L."""
    lp = np.asarray(out_lens, dtype=np.int64)
    n = np.floor(float(coverage) * lp.astype(np.float64) / (2.0 * read_len * ploidy)).astype(np.int64)
    n[lp < read_len] = 0
    return n


def quality_char(error_rate: float) -> int:
    """The quality character of every base: '!' + Q, Q = 41 for E = 0, else -10 log10 E rounded half up, within 2..41."""
    if error_rate <= 0:
        return ord("!") + 41
    q = math.floor(-10.0 * math.log10(error_rate) + 0.5)
    return ord("!") + min(max(q, 2), 41)


def config(args, seed: int, hap: int) -> dict:
    """The ms_reads_cfg of haplotype `hap` (1-based) of a run."""
    return dict(seed=seed, hap=hap, read_len=args.read_length, frag_mean=args.fragment_mean, frag_sd=args.fragment_sd,
                error_rate=args.read_error_rate, qual=quality_char(args.read_error_rate))


def _batches(first: int, count: int, per_pair: int, budget: int):
    step = max(1, int(budget) // per_pair)
    for f in range(first, first + count, step):
        yield f, min(step, first + count - f)


def _per_pair_bytes(engine, read_len: int) -> int:
    """An upper bound of the bytes one pair takes in buffer 9 (R1 + R2 record)."""
    longest = max((len(n) for n in engine.names), default=0)
    return 2 * (longest + _HEADER_FIXED + 2 * read_len + 4)


def _open(path):
    try:
        return open(path, "w+b")       # read-write: libmutsim_b200 maps the file for its parallel writers
    except OSError as e:
        raise ReadsWriterError(f"Cannot write to FASTQ file {path} {e}")


class ReadsWriter:
    """Both FASTQ files of a run.  One GPU: write() appends each haplotype's pairs.  Several GPUs:
    write_partitioned() places every rank's slices at offsets gathered from all ranks.  close() ends BGZF files with
    the EOF member.  budget: FASTQ bytes (R1 + R2) formatted in HBM per call."""

    def __init__(self, paths, bgzip: bool = False, budget: int = DEFAULT_BATCH_BYTES, create: bool = True):
        self.paths, self.bgzip, self.budget = list(paths), bool(bgzip), int(budget)
        self.plain = 0                 # uncompressed bytes of each file so far (R1 and R2 records have equal sizes)
        self.z = [0, 0]                # compressed bytes of each file so far (bgzip)
        self._fh = [_open(p) for p in self.paths] if create else []      # several GPUs: rank 0 creates them in _grow
        self._grown = False

    # -- one GPU -----------------------------------------------------------------------------------------------------
    def write(self, engine, cfg: dict, n_pairs):
        """All pairs of the engine's contigs (n_pairs per contig), batch by batch, at the end of both files."""
        n_pairs = np.ascontiguousarray(n_pairs, dtype=np.int64)
        per = _per_pair_bytes(engine, cfg["read_len"])
        for first, count in _batches(0, int(n_pairs.sum()), per, self.budget):
            nb = engine.reads_write(cfg, n_pairs, first, count)
            for m, fh in enumerate(self._fh):
                self.z[m] += self._put(engine, fh.fileno(), m, nb, self.plain, self.z[m])
            self.plain += nb

    def _put(self, engine, fd, m, nb, file_off, zoff) -> int:
        """Mate m's records of the batch in buffer 9 into fd: plain at file_off, or compressed at zoff.  -> compressed
        bytes (bgzip) or nb."""
        from .engine import BUF_BGZF, BUF_READS
        if not nb:
            return 0
        if not self.bgzip:
            engine.download_to_fd(BUF_READS, fd, file_off, m * nb, nb)
            return nb
        _, tot = engine.bgzf_compress(BUF_READS, [m * nb], [nb], [file_off])
        if tot:
            engine.download_to_fd(BUF_BGZF, fd, zoff, 0, tot)
        return tot

    # -- several GPUs ------------------------------------------------------------------------------------------------
    def write_partitioned(self, engine, cfg: dict, n_pairs, slices, n_slots: int):
        """slices: [(slot, local contig, lo, hi)] = pairs [lo, hi) of that contig, written at the file position of
        `slot` (slots in file order over all ranks; each rank sends its own).  The batches of every slice are planned
        once and sized once; the sizes are gathered from every rank; with bgzip the compressed sizes too, by a first
        compression pass whose bytes are dropped."""
        from . import distributed as D
        from .engine import BUF_READS
        n_pairs = np.ascontiguousarray(n_pairs, dtype=np.int64)
        pre = np.concatenate(([0], np.cumsum(n_pairs))).astype(np.int64)
        per = _per_pair_bytes(engine, cfg["read_len"]) if engine is not None else 1

        plan = [list(_batches(int(pre[c] + lo), int(hi - lo), per, self.budget)) for _, c, lo, hi in slices]
        sizes = [sum(int(engine.reads_size(cfg, n_pairs, f, n)[s[1]]) for f, n in plan[k]) for k, s in enumerate(slices)]
        off = self._gather(D, slices, sizes, n_slots, self.plain)
        total = int(off[-1])
        if self.bgzip:
            # members are cut at the uncompressed file offsets, and the compressed offsets need every rank's compressed
            # sizes while buffer 9 holds one batch: the slices are formatted and compressed once for their sizes, and
            # again to be written
            zsz = [[0, 0] for _ in slices]
            for k, s in enumerate(slices):
                at = int(off[s[0]])
                for first, count in plan[k]:
                    nb = engine.reads_write(cfg, n_pairs, first, count)
                    for m in range(2):
                        zsz[k][m] += int(engine.bgzf_compress(BUF_READS, [m * nb], [nb], [at])[1]) if nb else 0
                    at += nb
            zoff = [self._gather(D, slices, [z[m] for z in zsz], n_slots, self.z[m]) for m in range(2)]
        self._grow(D, [total] * 2 if not self.bgzip else [int(zoff[0][-1]), int(zoff[1][-1])])
        fds = [os.open(p, os.O_RDWR) for p in self.paths]
        try:
            for k, s in enumerate(slices):
                at = int(off[s[0]])
                za = [int(zoff[m][s[0]]) for m in range(2)] if self.bgzip else [0, 0]
                for first, count in plan[k]:
                    nb = engine.reads_write(cfg, n_pairs, first, count)
                    for m in range(2):
                        za[m] += self._put(engine, fds[m], m, nb, at, za[m])
                    at += nb
        finally:
            for fd in fds:
                os.close(fd)
        D.barrier()
        self.plain = total
        if self.bgzip:
            self.z = [int(zoff[0][-1]), int(zoff[1][-1])]

    @staticmethod
    def _gather(D, slices, sizes, n_slots, base):
        per_slot = np.zeros(n_slots, dtype=np.int64)
        for r_slots, r_sizes in D.all_gather_object(([s[0] for s in slices], [int(x) for x in sizes])):
            for s, b in zip(r_slots, r_sizes):
                per_slot[s] = b
        off = np.zeros(n_slots + 1, dtype=np.int64)
        np.cumsum(per_slot, out=off[1:])
        return off + int(base)

    def _grow(self, D, ends):
        """Rank 0 creates both files on the first call and grows them to `ends`; the outcome is broadcast so that all
        ranks leave together on an error."""
        err = None
        if D.rank_world()[0] == 0:
            try:
                for p, e in zip(self.paths, ends):
                    with open(p, "r+b" if self._grown else "wb") as fh:
                        fh.truncate(int(e))
            except OSError as e:
                err = f"Cannot write to FASTQ file {p} {e}"
        self._grown = True
        err = D.broadcast_object(err)
        if err is not None:
            raise ReadsWriterError(err)

    def close(self):
        """Ends BGZF files with the EOF member (rank 0 with several GPUs) and closes them."""
        from .bgzf import EOF
        from . import distributed as D
        if self._fh:
            if self.bgzip:
                for m, fh in enumerate(self._fh):
                    fh.seek(self.z[m])
                    fh.write(EOF)
            for fh in self._fh:
                fh.close()
        elif self._grown and self.bgzip and D.rank_world()[0] == 0:
            for m, p in enumerate(self.paths):
                with open(p, "r+b") as fh:
                    fh.seek(self.z[m])
                    fh.write(EOF)
        self._fh, self._grown = [], False

