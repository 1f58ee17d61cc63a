"""One process per GPU (torchrun): contig partitioning, peer exchange and output assembly.

ARGS/RMT need no data-path collective: contigs are independent (mutator.py:111 carries no
state between them) and the RNG is keyed by the global contig index, so every rank simply
processes its share and the ranks' slices are written into one file at offsets derived
from an all-gather of their sizes.  IT needs the partner's odd intervals: for a pair whose
members live on different GPUs the reader maps the owner's genome buffer (CUDA IPC) and its
raw far-copy records point straight into the peer's HBM (it_mutator.py:133-142; SURVEY.md
§8e); exchange_contigs() below is the NCCL send/recv route into a staging region that the
`nccl` setting of MS_IT_EXCHANGE keeps available."""
from __future__ import annotations

import os

import numpy as np

_pg_ready = False


def rank_world():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def local_device(default: int = 0) -> int:
    return int(os.environ.get("LOCAL_RANK", default))


def init():
    """Initialise torch.distributed (NCCL) when launched with WORLD_SIZE > 1."""
    global _pg_ready
    rank, world = rank_world()
    if world > 1 and not _pg_ready:
        import torch
        import torch.distributed as dist
        if not dist.is_initialized():
            torch.cuda.set_device(local_device())
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_device()))
        _pg_ready = True
    return rank, world


def barrier():
    if rank_world()[1] > 1:
        import torch.distributed as dist
        dist.barrier()


def broadcast_object(obj):
    if rank_world()[1] == 1:
        return obj
    import torch.distributed as dist
    box = [obj]
    dist.broadcast_object_list(box, src=0)
    return box[0]


def all_gather_object(obj):
    world = rank_world()[1]
    if world == 1:
        return [obj]
    import torch.distributed as dist
    out = [None] * world
    dist.all_gather_object(out, obj)
    return out


def lpt_partition(lengths, n):
    """Longest-processing-time bin packing of contigs onto n ranks; deterministic."""
    bins = [[] for _ in range(n)]
    load = [0] * n
    for i in sorted(range(len(lengths)), key=lambda i: (-int(lengths[i]), i)):
        b = load.index(min(load))
        bins[b].append(i)
        load[b] += int(lengths[i])
    return [sorted(b) for b in bins]


def shard_mode(lengths, n) -> str:
    """How n ranks split one run.  'contigs': LPT partition of whole contigs — every stage, sampling included, is
    sharded and nothing is exchanged.  'tiles': when that would leave a rank idle or overloaded (fewer contigs than
    ranks, or one contig far larger than a rank's share — the reference's own benchmark is a single 1 Gbp contig,
    README.md:441) every rank keeps the whole genome, draws the same mutation table, and the byte-moving stages are
    cut at 16 KiB tile boundaries of the output (ms_apply_window).  MS_SHARD=contigs|tiles overrides."""
    forced = os.environ.get("MS_SHARD")
    if forced in ("contigs", "tiles"):
        return forced
    if n <= 1:
        return "contigs"
    parts = lpt_partition(lengths, n)
    loads = [sum(int(lengths[i]) for i in p) for p in parts]
    total = sum(loads)
    if min(len(p) for p in parts) == 0 or (total > 0 and max(loads) > 1.25 * total / n):
        return "tiles"
    return "contigs"


def partition_of(fasta, n):
    """The contig partition of a run: the one the FASTA was ingested with (every rank read only its own records), else
    LPT on the contig lengths."""
    return getattr(fasta, "partition", None) or lpt_partition(fasta.lengths, n)


def shard_of(fasta, n) -> str:
    return getattr(fasta, "shard", None) or shard_mode(fasta.lengths, n)


def owners(parts, n_contigs):
    own = np.zeros(n_contigs, dtype=np.int64)
    for r, ids in enumerate(parts):
        own[ids] = r
    return own


class _DevMem:
    """Zero-copy torch view of engine-owned device memory (for NCCL send/recv)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def device_view(ptr: int, nbytes: int, device: int):
    import torch
    return torch.as_tensor(_DevMem(ptr, nbytes), device=f"cuda:{device}")


def exchange_contigs(engine, device, sends, recvs):
    """sends: [(peer, genome_index, nbytes)], recvs: [(peer, genome_index, nbytes)] in a globally agreed order.
    One grouped NCCL call (ncclGroupStart/End under batch_isend_irecv).  Returns the device time of the exchange in ms."""
    if not sends and not recvs:
        return 0.0
    import torch
    import torch.distributed as dist
    from .engine import BUF_GENOME
    base, _ = engine.device_ptr(BUF_GENOME)
    ops = []
    keep = []
    for peer, idx, n in sends:
        t = device_view(base + idx, n, device)
        keep.append(t)
        ops.append(dist.P2POp(dist.isend, t, peer))
    for peer, idx, n in recvs:
        t = device_view(base + idx, n, device)
        keep.append(t)
        ops.append(dist.P2POp(dist.irecv, t, peer))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    engine.synchronize()                      # the engine's stream may still be reading the staging region
    ev0.record()
    for w in dist.batch_isend_irecv(ops):
        w.wait()
    ev1.record()
    torch.cuda.synchronize()
    return float(ev0.elapsed_time(ev1))


def write_partitioned(path, my_ids, chunks, n_contigs, prefix: bytes = b""):
    """Every rank writes the byte chunks of its contigs (chunks[i] belongs to global contig my_ids[i]) into
    one file, contigs in global order, after `prefix` (written by rank 0)."""
    off = _global_offsets(my_ids, [len(c) for c in chunks], n_contigs, len(prefix))
    _create(path, prefix, off[-1])
    fd = os.open(path, os.O_RDWR)
    try:
        for g, c in zip(my_ids, chunks):
            if len(c):
                os.pwrite(fd, c, int(off[g]))
    finally:
        os.close(fd)
    barrier()


def fasta_chunks(engine, my_ids, n_contigs_global):
    """Per-contig slices of the engine's FASTA image with the separator fixed up for the global file:
    a '\\n' follows a partial last line unless the contig is the last one of the whole file."""
    from .engine import BUF_FASTA
    image = engine.download(BUF_FASTA)
    fo, vo, sep, partial = engine.contig_layout()
    out = []
    for i, g in enumerate(my_ids):
        a, b = int(fo[i]), int(fo[i + 1])
        if sep[i]:
            b -= 1
        chunk = image[a:b].tobytes()
        if partial[i] and g != n_contigs_global - 1:
            chunk += b"\n"
        out.append(chunk)
    return out, vo


def vcf_chunks(engine, my_ids, vcf_off):
    from .engine import BUF_VCF
    body = engine.download(BUF_VCF)
    return [body[int(vcf_off[i]):int(vcf_off[i + 1])].tobytes() for i in range(len(my_ids))]


def _global_offsets(my_ids, my_sizes, n_contigs, prefix_len):
    sizes = np.zeros(n_contigs, dtype=np.int64)
    for r_ids, r_sizes in all_gather_object((list(my_ids), [int(x) for x in my_sizes])):
        if len(r_ids):
            sizes[r_ids] = r_sizes
    off = np.zeros(n_contigs + 1, dtype=np.int64)
    np.cumsum(sizes, out=off[1:])
    return off + prefix_len


class OutputCreateError(OSError):
    """Rank 0 could not create an output file; raised on EVERY rank so that all of them leave together."""


def _create(path, prefix: bytes, total: int):
    """Rank 0 creates the file (prefix + room for `total` bytes); the outcome is broadcast, so an unwritable path
    fails all ranks with the same exception instead of leaving the others at a barrier."""
    err = None
    if rank_world()[0] == 0:
        try:
            with open(path, "wb") as fh:
                fh.write(prefix)
                fh.truncate(int(total))
        except OSError as e:
            err = str(e)
    err = broadcast_object(err)
    if err is not None:
        raise OutputCreateError(err)


def write_window(path, engine, which, lo: int, hi: int, total: int, prefix: bytes = b"", bgzip: bool = False):
    """Tile-sharded runs: this rank produced bytes [lo, hi) of device buffer `which`, whose layout is the same on every
    rank; all ranks stream their ranges into one file of `total` bytes after `prefix`.  bgzip: each rank compresses
    the contig slices of its window (the FASTA windows start on 16 KiB cells, so the members are the 1-GPU run's),
    the compressed sizes are gathered in rank order, and the last rank appends the EOF member."""
    if bgzip:
        return _write_window_bgzf(path, engine, which, lo, hi, prefix)
    _create(path, prefix, len(prefix) + int(total))
    if hi > lo:
        fd = os.open(path, os.O_RDWR)
        try:
            engine.download_to_fd(which, fd, len(prefix) + int(lo), int(lo), int(hi - lo))
        finally:
            os.close(fd)
    barrier()


def write_slices_partitioned(path, engine, which, my_ids, slice_off, n_contigs, prefix: bytes = b"", bgzip: bool = False):
    """Contig i of this rank owns bytes [slice_off[i], slice_off[i+1]) of device buffer `which`; all ranks stream
    their slices into one file, contigs in global order, without passing through Python."""
    sizes = [int(slice_off[i + 1] - slice_off[i]) for i in range(len(my_ids))]
    if bgzip:
        off = _global_offsets(my_ids, sizes, n_contigs, 0)
        return _write_contigs_bgzf(path, engine, which, my_ids, [int(slice_off[i]) for i in range(len(my_ids))], sizes,
                                   off, [0] * len(my_ids), n_contigs, prefix)
    off = _global_offsets(my_ids, sizes, n_contigs, len(prefix))
    _create(path, prefix, off[-1])
    fd = os.open(path, os.O_RDWR)
    try:
        # consecutive local contigs that are also consecutive in the file go out as one transfer
        i = 0
        while i < len(my_ids):
            j = i
            while j + 1 < len(my_ids) and my_ids[j + 1] == my_ids[j] + 1:
                j += 1
            n = int(slice_off[j + 1] - slice_off[i])
            if n:
                engine.download_to_fd(which, fd, int(off[my_ids[i]]), int(slice_off[i]), n)
            i = j + 1
    finally:
        os.close(fd)
    barrier()


def write_fasta_partitioned(path, engine, my_ids, n_contigs_global, bgzip: bool = False):
    """FASTA image slices with the separator fixed up for the global file order (a '\\n' follows a partial last
    line unless the contig is the last one of the whole file).  Returns the per-contig VCF offsets of the layout."""
    if len(my_ids) == 0:      # more ranks than contigs: this rank only takes part in the collectives
        fo, vo, sep, partial = np.zeros(1, np.int64), np.zeros(1, np.int64), [], []
    else:
        fo, vo, sep, partial = engine.contig_layout()
    body = [int(fo[i + 1] - fo[i]) - int(sep[i]) for i in range(len(my_ids))]
    extra = [1 if (partial[i] and g != n_contigs_global - 1) else 0 for i, g in enumerate(my_ids)]
    off = _global_offsets(my_ids, [b + e for b, e in zip(body, extra)], n_contigs_global, 0)
    if bgzip:
        _write_contigs_bgzf(path, engine, 0, my_ids, [int(fo[i]) for i in range(len(my_ids))], body, off, extra,
                            n_contigs_global, b"")
        return vo
    _create(path, b"", off[-1])
    from .engine import BUF_FASTA
    fd = os.open(path, os.O_RDWR)
    try:
        for i, g in enumerate(my_ids):
            if body[i]:
                engine.download_to_fd(BUF_FASTA, fd, int(off[g]), int(fo[i]), body[i])
            if extra[i]:
                os.pwrite(fd, b"\n", int(off[g]) + body[i])
    finally:
        os.close(fd)
    barrier()
    return vo


def _write_contigs_bgzf(path, engine, which, my_ids, src, nbytes, file_off, add_nl, n_contigs, prefix: bytes):
    """Contig-sharded BGZF: contig i of this rank is nbytes[i] bytes of buffer `which` at src[i] (+ '\\n' if
    add_nl[i]) and starts at file_off[global id] of the uncompressed file (the first all-gather); each rank compresses
    its contigs, a second all-gather of the compressed sizes places them, rank 0 writes the compressed prefix and the
    owner of the last contig the EOF member."""
    from .bgzf import EOF, compress_host
    from .engine import BUF_BGZF
    zhead = compress_host(prefix)
    if len(my_ids):
        zseg, _ = engine.bgzf_compress(which, src, nbytes, [int(file_off[g]) for g in my_ids], add_nl)
    else:
        zseg = np.zeros(0, np.int64)
    zoff = _global_offsets(my_ids, [int(z) for z in zseg], n_contigs, len(zhead))
    _create(path, zhead, int(zoff[-1]) + len(EOF))
    fd = os.open(path, os.O_RDWR)
    try:
        local = np.concatenate(([0], np.cumsum(zseg))).astype(np.int64)
        i = 0
        while i < len(my_ids):          # consecutive contigs are consecutive in buffer 5 and in the file
            j = i
            while j + 1 < len(my_ids) and my_ids[j + 1] == my_ids[j] + 1:
                j += 1
            n = int(local[j + 1] - local[i])
            if n:
                engine.download_to_fd(BUF_BGZF, fd, int(zoff[my_ids[i]]), int(local[i]), n)
            i = j + 1
        if n_contigs - 1 in my_ids:
            os.pwrite(fd, EOF, int(zoff[-1]))
    finally:
        os.close(fd)
    barrier()


def _write_window_bgzf(path, engine, which, lo: int, hi: int, prefix: bytes):
    from .bgzf import EOF, compress_host, window_segments
    from .engine import BUF_BGZF
    zhead = compress_host(prefix)
    tot = 0
    if hi > lo:
        src, n = window_segments(engine, which, int(lo), int(hi))
        _, tot = engine.bgzf_compress(which, src, n, src)
    sizes = all_gather_object(int(tot))
    rank = rank_world()[0]
    at = len(zhead) + sum(sizes[:rank])
    end = len(zhead) + sum(sizes)
    _create(path, zhead, end + len(EOF))
    fd = os.open(path, os.O_RDWR)
    try:
        if tot:
            engine.download_to_fd(BUF_BGZF, fd, at, 0, tot)
        if rank == len(sizes) - 1:
            os.pwrite(fd, EOF, end)
    finally:
        os.close(fd)
    barrier()
