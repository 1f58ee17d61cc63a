"""Thin object wrapper over the C ABI: one ``Engine`` = one ms_ctx on one GPU.

Host arrays go in as numpy arrays; every method maps 1:1 onto an entry point of
include/mutsim_b200.h.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import MsRange, MsReadsCfg, MsStats, MutSimError
from .records import REC_DTYPE

BUF_FASTA, BUF_VCF, BUF_RECS, BUF_LIT, BUF_GENOME, BUF_BGZF, BUF_CHAIN, BUF_VCF_PHASED, BUF_GT, BUF_READS = range(10)


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def bgzf_compress_host(data: bytes) -> bytes:
    """BGZF members (16 KiB of input each) of small host data with the device's encoder (ms_bgzf_compress_host);
    needs the library, not a GPU."""
    lib = _lib.load()
    src = np.frombuffer(bytes(data), dtype=np.uint8)
    cap = C.c_int64()
    rc = lib.ms_bgzf_compress_host(None, _ptr(src), src.size, None, 0, C.byref(cap))
    out = np.empty(max(cap.value, 1), dtype=np.uint8)
    n = C.c_int64()
    rc = rc or lib.ms_bgzf_compress_host(None, _ptr(src), src.size, _ptr(out), out.size, C.byref(n))
    if rc:
        raise MutSimError(rc, "ms_bgzf_compress_host failed")
    return out[:n.value].tobytes()


def _blob(items: Sequence[bytes]):
    off = np.zeros(len(items) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in items], out=off[1:])
    return np.frombuffer(b"".join(items) + b"\0", dtype=np.uint8).copy(), off


class Engine:
    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        h = C.c_void_p()
        rc = self._lib.ms_create(device, C.byref(h))
        if rc:
            raise MutSimError(rc, (self._lib.ms_last_error(None) or b"").decode())
        self._h = h
        self.device = device
        self.n_contigs = 0
        self.total_bases = 0

    # -- lifecycle ---------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.ms_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int):
        if rc:
            raise MutSimError(rc, (self._lib.ms_last_error(self._h) or b"").decode())

    def set_stream(self, cuda_stream: int):
        self._check(self._lib.ms_set_stream(self._h, C.c_void_p(cuda_stream)))

    def synchronize(self):
        self._check(self._lib.ms_synchronize(self._h))

    # -- genome ------------------------------------------------------------
    def _contig_args(self, lengths, bpl, headers, names, gid):
        self._len = np.ascontiguousarray(lengths, dtype=np.int64)
        self._bpl = np.ascontiguousarray(bpl, dtype=np.int32)
        self._hdr, self._hoff = _blob(headers)
        self._nam, self._noff = _blob(names)
        self._gid = None if gid is None else np.ascontiguousarray(gid, dtype=np.uint32)
        self.n_contigs = len(self._len)
        self.total_bases = int(self._len.sum())
        self.names = list(names)

    def upload_genome(self, bases: np.ndarray, lengths, bpl, headers: Sequence[bytes], names: Sequence[bytes], gid=None):
        """bases: uint8, all contigs concatenated, upper-cased (ms_genome_upload)."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        self._contig_args(lengths, bpl, headers, names, gid)
        self._check(self._lib.ms_genome_upload(self._h, _ptr(bases), self.total_bases, self.n_contigs, _ptr(self._len),
                                               _ptr(self._bpl), _ptr(self._gid), _ptr(self._hdr), _ptr(self._hoff),
                                               _ptr(self._nam), _ptr(self._noff)))

    def adopt_genome(self, device_ptr: int, lengths, bpl, headers, names, gid=None):
        self._contig_args(lengths, bpl, headers, names, gid)
        self._check(self._lib.ms_genome_adopt(self._h, C.c_void_p(device_ptr), self.total_bases, self.n_contigs,
                                              _ptr(self._len), _ptr(self._bpl), _ptr(self._gid), _ptr(self._hdr),
                                              _ptr(self._hoff), _ptr(self._nam), _ptr(self._noff)))

    def synth_genome(self, seed: int, lengths, bpl, headers, names, n_fraction=0.0, telomere_n=0, gid=None):
        """Synthetic genome on the device; gid = global index of each contig (the bases of a contig depend on
        (seed, gid) only, so a rank's share equals the same contigs of a single-GPU genome)."""
        self._contig_args(lengths, bpl, headers, names, gid)
        self._check(self._lib.ms_genome_synth(self._h, seed, self.n_contigs, _ptr(self._len), _ptr(self._bpl), _ptr(self._gid),
                                              float(n_fraction), int(telomere_n), _ptr(self._hdr), _ptr(self._hoff),
                                              _ptr(self._nam), _ptr(self._noff)))

    def hash_ranges(self, which: int, start, end) -> np.ndarray:
        """64-bit content hashes of byte ranges of an output buffer, computed on the device (ms_hash_ranges)."""
        start = np.ascontiguousarray(start, dtype=np.int64); end = np.ascontiguousarray(end, dtype=np.int64)
        out = np.zeros(len(start), dtype=np.uint64)
        if len(start):
            self._check(self._lib.ms_hash_ranges(self._h, which, len(start), _ptr(start), _ptr(end), _ptr(out)))
        return out

    def ingest_fasta(self, fd: int, nbytes: int, ranges=None):
        """Raw FASTA file -> device image + record index (ms_fasta_ingest_fd / ms_fasta_index).  Returns None when the
        file is not regularly wrapped (the host parser then takes over), else a dict with length, seq_off, lenc, lenb
        (numpy arrays) and long_names (deflines without '>').  ranges = [(file offset, bytes)] of whole records: only
        those are read (ms_fasta_ingest_ranges); seq_off is then relative to their concatenation."""
        n, reg = C.c_int32(0), C.c_int32(0)
        if ranges is None:
            self._check(self._lib.ms_fasta_ingest_fd(self._h, int(fd), int(nbytes), C.byref(n), C.byref(reg)))
        else:
            off = np.ascontiguousarray([r[0] for r in ranges], dtype=np.int64)
            ln = np.ascontiguousarray([r[1] for r in ranges], dtype=np.int64)
            self._check(self._lib.ms_fasta_ingest_ranges(self._h, int(fd), len(ranges), _ptr(off), _ptr(ln), C.byref(n), C.byref(reg)))
        if not reg.value:
            return None
        n = n.value
        hoff = np.zeros(n + 1, np.int64)
        seq_off, length = np.zeros(n, np.int64), np.zeros(n, np.int64)
        lenc, lenb = np.zeros(n, np.int32), np.zeros(n, np.int32)
        self._check(self._lib.ms_fasta_index(self._h, _ptr(hoff), _ptr(seq_off), _ptr(length), _ptr(lenc), _ptr(lenb), None, 0))
        blob = np.zeros(int(hoff[-1]) + 1, np.uint8)
        self._check(self._lib.ms_fasta_index(self._h, _ptr(hoff), None, None, None, None, _ptr(blob), blob.size))
        raw = blob.tobytes()
        long_names = [raw[hoff[i]:hoff[i + 1]].decode("latin-1") for i in range(n)]
        return dict(length=length, seq_off=seq_off, lenc=lenc, lenb=lenb, long_names=long_names)

    def commit_fasta(self, lengths, bpl, headers: Sequence[bytes], names: Sequence[bytes], gid=None) -> bool:
        """Strip + upper-case + verify the ingested image into the resident genome (ms_fasta_commit)."""
        self._contig_args(lengths, bpl, headers, names, gid)
        reg = C.c_int32(0)
        self._check(self._lib.ms_fasta_commit(self._h, _ptr(self._gid), _ptr(self._hdr), _ptr(self._hoff), _ptr(self._nam),
                                              _ptr(self._noff), C.byref(reg)))
        return bool(reg.value)

    def subset_genome(self, ids):
        """Keep only contigs `ids` (local indices) of the resident genome, in that order (ms_genome_subset)."""
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        self._check(self._lib.ms_genome_subset(self._h, _ptr(ids), int(ids.size)))
        self._len = self._len[ids].copy()
        self._bpl = self._bpl[ids].copy()
        self.names = [self.names[int(i)] for i in ids]
        self.n_contigs = int(ids.size)
        self.total_bases = int(self._len.sum())

    def read_genome(self, off: int, n: int) -> np.ndarray:
        out = np.empty(int(n), dtype=np.uint8)
        self._check(self._lib.ms_genome_read(self._h, int(off), int(n), _ptr(out)))
        return out

    def declare_genome(self, lengths, bpl, headers: Sequence[bytes], names: Sequence[bytes], gid=None):
        """Contig table without bases (they arrive with mutate_streamed)."""
        self._contig_args(lengths, bpl, headers, names, gid)
        self._check(self._lib.ms_genome_declare(self._h, self.total_bases, self.n_contigs, _ptr(self._len), _ptr(self._bpl),
                                                _ptr(self._gid), _ptr(self._hdr), _ptr(self._hoff), _ptr(self._nam),
                                                _ptr(self._noff)))

    def mutate_streamed(self, seed: int, bases: np.ndarray, fasta_out: np.ndarray, vcf_out: np.ndarray, group_min_bases: int = 0):
        """Host genome in, host FASTA image + VCF body out, copies overlapped with the kernels (ms_mutate_streamed).
        Returns (fasta_bytes, vcf_bytes).  Pass pinned arrays for the overlap."""
        if bases.dtype != np.uint8 or not bases.flags.c_contiguous or bases.size != self.total_bases:
            raise ValueError("bases must be a contiguous uint8 array of total_bases elements")
        fb, vb = C.c_int64(0), C.c_int64(0)
        self._check(self._lib.ms_mutate_streamed(self._h, C.c_uint64(seed & (2**64 - 1)), _ptr(bases), _ptr(fasta_out),
                                                 fasta_out.nbytes, _ptr(vcf_out), vcf_out.nbytes, C.byref(fb), C.byref(vb),
                                                 int(group_min_bases)))
        return fb.value, vb.value

    def reserve_foreign(self, nbytes: int):
        """Staging space behind the genome for partner contigs owned by another GPU (call before upload)."""
        self._check(self._lib.ms_genome_reserve(self._h, int(nbytes)))

    def export_genome(self):
        """-> (64-byte CUDA IPC handle of the resident genome buffer, its size): another process maps it with open_peer."""
        h = np.zeros(64, dtype=np.uint8)
        n = C.c_int64(0)
        self._check(self._lib.ms_genome_export(self._h, _ptr(h), C.byref(n)))
        return h.tobytes(), n.value

    def open_peer(self, handle: bytes, nbytes: int) -> int:
        """Map another GPU's genome buffer; -> offset of its base relative to this engine's genome (for Rec.src)."""
        h = np.frombuffer(handle, dtype=np.uint8).copy()
        rel = C.c_int64(0)
        self._check(self._lib.ms_peer_open(self._h, _ptr(h), int(nbytes), C.byref(rel)))
        return rel.value

    def pull_peer(self, src, dst, nbytes):
        """Async copies peer window -> staging region on the engine's stream (src relative like open_peer's offset)."""
        src, dst, nbytes = (np.ascontiguousarray(a, dtype=np.int64) for a in (src, dst, nbytes))
        self._check(self._lib.ms_peer_pull(self._h, len(src), _ptr(src), _ptr(dst), _ptr(nbytes)))

    def close_peers(self):
        self._check(self._lib.ms_peer_close(self._h))

    def adopt_output(self) -> np.ndarray:
        """The mutated genome of the last apply() becomes the resident genome; returns the new contig lengths."""
        self._check(self._lib.ms_genome_adopt_output(self._h))
        lens = self.contig_out_len()
        self._len = lens.copy()
        self.total_bases = int(lens.sum())
        return lens

    def download_genome(self) -> np.ndarray:
        out = np.empty(self.total_bases, dtype=np.uint8)
        self._check(self._lib.ms_genome_download(self._h, _ptr(out), out.size))
        return out

    # -- sampling ----------------------------------------------------------
    def set_ranges(self, ranges: Sequence[dict], block: Sequence[int], min_dist: int, p_ti: float):
        """ranges: dicts with contig,start,stop,k,limit,cdf[7],minlen[7],maxlen[7] sorted by (contig,start)."""
        arr = (MsRange * max(1, len(ranges)))()
        for i, r in enumerate(ranges):
            a = arr[i]
            a.contig, a.start, a.stop, a.k, a.limit = r["contig"], r["start"], r["stop"], r["k"], r.get("limit", 0)
            for t in range(7):
                a.cdf[t], a.minlen[t], a.maxlen[t] = r["cdf"][t], r["minlen"][t], r["maxlen"][t]
        blk = (C.c_int32 * 7)(*block)
        self._check(self._lib.ms_set_ranges(self._h, arr, len(ranges), blk, int(min_dist), float(p_ti)))

    def set_ranges_array(self, arr, n: int, block, min_dist: int, p_ti: float):
        blk = (C.c_int32 * 7)(*block)
        self._check(self._lib.ms_set_ranges(self._h, arr, n, blk, int(min_dist), float(p_ti)))

    def sample(self, seed: int):
        self._check(self._lib.ms_sample(self._h, C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF)))

    def debug_candidates(self):
        n = C.c_int64()
        self._check(self._lib.ms_debug_candidates(self._h, 0, None, None, None, None, C.byref(n)))
        k = n.value
        gpos = np.empty(k, np.int64); typ = np.empty(k, np.uint8); ln = np.empty(k, np.uint32); acc = np.empty(k, np.uint8)
        self._check(self._lib.ms_debug_candidates(self._h, k, _ptr(gpos), _ptr(typ), _ptr(ln), _ptr(acc), C.byref(n)))
        return gpos, typ, ln, acc

    # -- replay / apply ----------------------------------------------------
    def load_records(self, recs: np.ndarray, lit: Optional[np.ndarray] = None):
        recs = np.ascontiguousarray(recs, dtype=REC_DTYPE)
        lit = np.zeros(16, np.uint8) if lit is None else np.ascontiguousarray(lit, dtype=np.uint8)
        nlit = int((recs["src"][recs["kind"] == 2] + recs["prod"][recs["kind"] == 2]).max()) if (recs["kind"] == 2).any() else 0
        self._check(self._lib.ms_load_records(self._h, _ptr(recs), len(recs), _ptr(lit), max(nlit, 0)))

    def load_vcf(self, text, skip_unknown: bool = False) -> bool:
        """Parse VCF text (bytes-like or mmap, read in place) on the device into the record table (ms_load_vcf).
        Returns False when the text is not of the regular shape: nothing was loaded and records.records_from_vcf +
        load_records must take it.  skip_unknown: drop the lines of contigs this engine does not hold."""
        buf = np.frombuffer(text, dtype=np.uint8) if len(text) else np.zeros(1, np.uint8)
        reg, n = C.c_int32(0), C.c_int64(0)
        self._check(self._lib.ms_load_vcf(self._h, _ptr(buf), len(text), int(bool(skip_unknown)), C.byref(reg), C.byref(n)))
        return bool(reg.value)

    def load_vcf_phased(self, text, ploidy: int, skip_unknown: bool = False) -> bool:
        """load_vcf that also reads each record's haplotype mask from its GT field (ms_load_vcf_phased).  False: the text
        (a GT included) is not of the regular shape and records.records_from_vcf(..., ploidy=) must take it."""
        buf = np.frombuffer(text, dtype=np.uint8) if len(text) else np.zeros(1, np.uint8)
        reg, n = C.c_int32(0), C.c_int64(0)
        self._check(self._lib.ms_load_vcf_phased(self._h, _ptr(buf), len(text), int(bool(skip_unknown)), int(ploidy), C.byref(reg),
                                                 C.byref(n)))
        return bool(reg.value)

    # -- polyploid runs ----------------------------------------------------
    def genotype_draw(self, seed: int, ploidy: int, hom_fraction: float):
        """Draw the haplotype mask of every record of the full table (ms_genotype_draw)."""
        self._check(self._lib.ms_genotype_draw(self._h, C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), int(ploidy), float(hom_fraction)))

    def genotype_load(self, masks, ploidy: int):
        """Host-supplied haplotype masks, one per record of the full table (ms_genotype_load)."""
        m = np.ascontiguousarray(masks, dtype=np.uint8)
        self._check(self._lib.ms_genotype_load(self._h, _ptr(m) if m.size else None, int(m.size), int(ploidy)))

    def select_haplotype(self, h: int):
        """Make haplotype h's records (1..P) the active table; 0 restores the full table (ms_select_haplotype)."""
        self._check(self._lib.ms_select_haplotype(self._h, int(h)))

    def vcf_phased(self) -> np.ndarray:
        """Format the phased VCF body of the full table into buffer BUF_VCF_PHASED (ms_vcf_phased).  Returns each
        contig's slice, n_contigs + 1 offsets (kept as vcf_phased_off)."""
        off = np.zeros(self.n_contigs + 1, dtype=np.int64)
        self._check(self._lib.ms_vcf_phased(self._h, _ptr(off)))
        self.vcf_phased_off = off
        return off

    def genotypes(self) -> np.ndarray:
        """Haplotype masks of the full table (bit h-1: haplotype h carries the record)."""
        return self.download(BUF_GT)

    def apply(self) -> tuple[int, int]:
        fb, vb = C.c_int64(), C.c_int64()
        self._check(self._lib.ms_apply(self._h, C.byref(fb), C.byref(vb)))
        return fb.value, vb.value

    def apply_window(self, part: int, n_parts: int) -> dict:
        """ms_apply for one part of the output (tiles / records [part/n_parts, (part+1)/n_parts)); every part must run on
        a context holding the same genome and record table.  Returns the sizes of the whole outputs and the byte
        ranges this part produced."""
        w = np.zeros(6, dtype=np.int64)
        self._check(self._lib.ms_apply_window(self._h, int(part), int(n_parts), _ptr(w)))
        return dict(fasta_bytes=int(w[0]), vcf_bytes=int(w[1]), fasta=(int(w[2]), int(w[3])), vcf=(int(w[4]), int(w[5])))

    def download(self, which: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        n = C.c_int64()
        self._check(self._lib.ms_download(self._h, which, None, 0, C.byref(n)))
        if out is None:
            out = np.empty(n.value, dtype=np.uint8)
        self._check(self._lib.ms_download(self._h, which, _ptr(out), out.nbytes, C.byref(n)))
        return out[:n.value] if out.dtype == np.uint8 else out

    def size_of(self, which: int) -> int:
        n = C.c_int64()
        self._check(self._lib.ms_download(self._h, which, None, 0, C.byref(n)))
        return n.value

    def download_to_fd(self, which: int, fd: int, file_off: int = 0, src_off: int = 0, nbytes: Optional[int] = None) -> int:
        """Stream (a slice of) an output buffer into an open file descriptor at file_off; returns the bytes written."""
        if nbytes is None:
            nbytes = self.size_of(which) - src_off
        self._check(self._lib.ms_download_to_fd(self._h, which, int(src_off), int(nbytes), int(fd), int(file_off)))
        return int(nbytes)

    def bgzf_compress(self, which: int, src_off, nbytes, file_off, add_nl=None):
        """BGZF members of segments of the FASTA image (which=0), the VCF body (which=1), the chain text (6), the phased
        VCF body (7) or the FASTQ records (9), cut on 16 KiB cells of
        the uncompressed file (ms_bgzf_compress); they become buffer BUF_BGZF.  Returns (compressed bytes of each
        segment, total)."""
        src_off, nbytes, file_off = (np.ascontiguousarray(a, dtype=np.int64) for a in (src_off, nbytes, file_off))
        nl = None if add_nl is None else np.ascontiguousarray(add_nl, dtype=np.uint8)
        seg = np.zeros(len(src_off), dtype=np.int64)
        tot = C.c_int64()
        self._check(self._lib.ms_bgzf_compress(self._h, int(which), len(src_off), _ptr(src_off), _ptr(nbytes), _ptr(file_off),
                                               _ptr(nl), _ptr(seg), C.byref(tot)))
        return seg, tot.value

    def chain_count(self) -> np.ndarray:
        """Chains of each contig in the chain file of the last apply (ms_chain_count)."""
        out = np.zeros(self.n_contigs, dtype=np.int64)
        self._check(self._lib.ms_chain_count(self._h, _ptr(out)))
        return out

    def chain_write(self, first_id) -> np.ndarray:
        """Format the chain file of the last apply into buffer BUF_CHAIN, numbering contig c's chains from first_id[c]
        (ms_chain_write).  Returns each contig's slice of the buffer, n_contigs + 1 offsets (kept as chain_off)."""
        first = np.ascontiguousarray(first_id, dtype=np.int64)
        if first.size != self.n_contigs:
            raise ValueError("first_id needs one entry per contig")
        off = np.zeros(self.n_contigs + 1, dtype=np.int64)
        self._check(self._lib.ms_chain_write(self._h, _ptr(first), _ptr(off)))
        self.chain_off = off
        return off

    @staticmethod
    def _reads_cfg(cfg: dict) -> MsReadsCfg:
        return MsReadsCfg(C.c_uint64(int(cfg["seed"]) & 0xFFFFFFFFFFFFFFFF).value, int(cfg["hap"]), int(cfg["read_len"]),
                          int(cfg["frag_mean"]), int(cfg["frag_sd"]), float(cfg["error_rate"]), int(cfg["qual"]))

    def reads_size(self, cfg: dict, n_pairs, first: int, count: int) -> np.ndarray:
        """Bytes one FASTQ file's records of pairs [first, first + count) take in each contig (ms_reads_size).  cfg: seed,
        hap, read_len, frag_mean, frag_sd, error_rate, qual; n_pairs: pairs of each contig, numbered contig-major."""
        n = np.ascontiguousarray(n_pairs, dtype=np.int64)
        out = np.zeros(self.n_contigs, dtype=np.int64)
        c = self._reads_cfg(cfg)
        self._check(self._lib.ms_reads_size(self._h, C.byref(c), _ptr(n), int(first), int(count), _ptr(out)))
        return out

    def reads_write(self, cfg: dict, n_pairs, first: int, count: int) -> int:
        """Format pairs [first, first + count) into buffer BUF_READS: R1 records at [0, n), R2 records at [n, 2n)
        (ms_reads_write).  Returns n."""
        n = np.ascontiguousarray(n_pairs, dtype=np.int64)
        nb = C.c_int64()
        c = self._reads_cfg(cfg)
        self._check(self._lib.ms_reads_write(self._h, C.byref(c), _ptr(n), int(first), int(count), C.byref(nb)))
        return nb.value

    def fasta(self) -> bytes:
        return self.download(BUF_FASTA).tobytes()

    def vcf(self) -> bytes:
        return self.download(BUF_VCF).tobytes()

    def records(self, include_dead: bool = False) -> np.ndarray:
        """Applied mutations as splice descriptors.  Unpaired translocation halves stay in the device table as
        no-op records (type 255); they are filtered here unless asked for."""
        r = self.download(BUF_RECS).view(REC_DTYPE)
        return r if include_dead else r[r["type"] != 255]

    def literals(self) -> np.ndarray:
        return self.download(BUF_LIT)

    def device_ptr(self, which: int) -> tuple[int, int]:
        p, n = C.c_void_p(), C.c_int64()
        self._check(self._lib.ms_device_ptr(self._h, which, C.byref(p), C.byref(n)))
        return (p.value or 0), n.value

    def contig_out_len(self) -> np.ndarray:
        out = np.empty(self.n_contigs, dtype=np.int64)
        self._check(self._lib.ms_contig_out_len(self._h, _ptr(out)))
        return out

    def contig_records(self) -> np.ndarray:
        out = np.empty(self.n_contigs, dtype=np.int64)
        self._check(self._lib.ms_contig_records(self._h, _ptr(out)))
        return out

    def contig_layout(self):
        """-> (fasta_off[n+1], vcf_off[n+1], sep[n], partial[n]) of the last apply()."""
        n = self.n_contigs
        fo = np.empty(n + 1, np.int64); vo = np.empty(n + 1, np.int64)
        sep = np.empty(n, np.uint8); par = np.empty(n, np.uint8)
        self._check(self._lib.ms_contig_layout(self._h, _ptr(fo), _ptr(vo), _ptr(sep), _ptr(par)))
        return fo, vo, sep, par

    def sample_positions(self, seed: int, gid, start, stop, k, min_dist: int):
        """util.sample_with_minimum_distance for many ranges; returns the concatenated sorted positions."""
        gid = np.ascontiguousarray(gid, np.uint32); start = np.ascontiguousarray(start, np.uint32)
        stop = np.ascontiguousarray(stop, np.uint32); k = np.ascontiguousarray(k, np.uint32)
        out = np.empty(max(1, int(k.sum())), np.uint32)
        self._check(self._lib.ms_sample_positions(self._h, C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), len(gid), _ptr(gid), _ptr(start),
                                                  _ptr(stop), _ptr(k), int(min_dist), _ptr(out)))
        return out[:int(k.sum())]

    # -- IT ----------------------------------------------------------------
    def it_breakpoints(self, seed: int, contig_a, contig_b, n):
        a = np.ascontiguousarray(contig_a, dtype=np.uint32)
        b = np.ascontiguousarray(contig_b, dtype=np.uint32)
        n = np.ascontiguousarray(n, dtype=np.uint32)
        tot = int(n.sum())
        bpa = np.empty(max(tot, 1), np.uint32)
        bpb = np.empty(max(tot, 1), np.uint32)
        self._check(self._lib.ms_it_breakpoints(self._h, C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), len(a), _ptr(a), _ptr(b),
                                                _ptr(n), _ptr(bpa), _ptr(bpb)))
        return bpa[:tot], bpb[:tot]

    # -- stats -------------------------------------------------------------
    def stats(self) -> dict:
        s = MsStats()
        self._check(self._lib.ms_get_stats(self._h, C.byref(s)))
        stages = {}
        for i in range(16):
            name = self._lib.ms_stage_name(i)
            if name:
                stages[name.decode()] = float(s.stage_ms[i])
        return {"n_candidates": s.n_candidates, "n_accepted": s.n_accepted, "n_records": s.n_records,
                "lit_bytes": s.lit_bytes, "fasta_bytes": s.fasta_bytes, "vcf_bytes": s.vcf_bytes,
                "kernel_launches": s.kernel_launches, "counts": list(s.counts), "stage_ms": stages}
