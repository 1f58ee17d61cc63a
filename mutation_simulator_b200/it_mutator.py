"""``ITMutator`` — interchromosomal translocations (it_mutator.py:20-220) on the B200 path.

Pairing of contigs is a host decision over at most a few thousand integers; breakpoints
are sampled on the GPU with the same position sampler as mutations
(sample_with_minimum_distance(1, len, n, 1), it_mutator.py:108-111); the alternating
own/partner concatenation is the splice kernel with raw far-copy records, and the output
FASTA image comes back complete.  Contigs without a partner are written once with normal
line wrapping (SURVEY.md Q1: the reference's duplicated header is treated as a bug)."""
from __future__ import annotations

import os
import random

import numpy as np

from . import distributed as D
from .bedpe_writer import BedpeWriter, rows
from .engine import BUF_FASTA, Engine
from .fasta_writer import FastaWriter
from .mutator import run_seed
from .records import K_RAW, REC_DTYPE, T_IT
from ._lib import MS_ERR_ARG, MutSimError
from .util import print_warning


def assign_partners(avail, rng) -> dict:
    """it_mutator.py:59-70 ``__assign_parters``.  The reference iterates ``__avail_chroms`` while removing from the
    SAME list (``remain_chr`` is an alias): every pass drops the current element and its partner and the iterator's
    index still advances by one, so the element that slid into the vacated slot is skipped and the loop ends after
    ceil(n/3) passes.  n eligible contigs therefore give ceil(n/3) pairs (24 -> 8, not 12); the rest stay unpaired
    and are written unchanged.  Reproduced here step for step (tests/golden/it_pairs.json pins the counts)."""
    pool = list(avail)
    rng.shuffle(pool)
    partners = {}
    i = 0
    while i < len(pool):
        chrom = pool.pop(i)                                 # remain_chr.remove(chrom)
        if pool:
            partner = pool.pop(rng.randrange(len(pool)))    # choice(remain_chr); remain_chr.remove(partner)
            partners[partner] = chrom
            partners[chrom] = partner
        i += 1                                              # the list iterator moves on over the shrunken list
    return partners


class ITMutator:
    def __init__(self, args, fasta, sim):
        self._args, self._fasta, self._sim = args, fasta, sim
        self._rank, self._world = D.init()
        if self._world == 1:
            self._fasta_writer = FastaWriter(args.outfastait, getattr(args, "bgzip", False))
            self._bedpe_writer = BedpeWriter(args.outbedpe)
        else:
            self._fasta_writer = self._bedpe_writer = None
        self._seed = D.broadcast_object(run_seed(args))
        self._rng = random.Random(self._seed)
        # it_mutator.py:51-57: eligible contigs
        avail = [c.number for c in sim.chromosomes if c.it_rate is not None and len(fasta[c.number]) > 2]
        self._partners = assign_partners(avail, self._rng)
        self._engine = None
        self.breakpoints = {}
        self._replay = None

    def load_bedpe(self, text):
        """Replay instead of sampling: take the pairing and the breakpoints from a BEDPE file written by the reference
        (bedpe_writer.py:36-55) or by this package; mutate() then reproduces that run's *_it.fa and .bedpe."""
        from .bedpe_writer import breakpoints_from_rows
        self._partners, self._replay = breakpoints_from_rows(text, self._fasta.names, self._fasta.lengths)

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def close(self):
        if self._fasta_writer is not None:
            self._fasta_writer.close()
            self._bedpe_writer.close()
        if self._engine is not None:
            if getattr(self, "_peer_src", None):     # mapped peer buffers go before their owners free them
                self._engine.close_peers()
            if getattr(self, "_route", "nccl") != "nccl":
                D.barrier()
            self._engine.close()
            self._engine = None

    def _pairs_once(self):
        seen, out = set(), []
        for a, b in self._partners.items():
            if a not in seen:
                out.append((a, b))
                seen.update((a, b))
        return out

    def _generate_all_breakpoints(self, eng):
        if self._replay is not None:
            return self._replay
        fasta, sim, args = self._fasta, self._sim, self._args
        pairs, counts = [], []
        for a, b in self._pairs_once():
            la, lb = len(fasta[a]), len(fasta[b])
            n = int((la + lb - 4) / 2 * ((sim.chromosomes[a].it_rate + sim.chromosomes[b].it_rate) / 2))   # it_mutator.py:92
            ok = True
            if n > 0 and (n > la - n or n > lb - n or la - n <= 0 or lb - n <= 0):   # random.sample would raise (util.py:104)
                ok = False
                if not args.ignore_warnings:
                    print_warning(f"Interchromosomal translocation rate too high for sequence {a+1} and {b+1}.", args.no_color)
            if n <= 0 or not ok:
                if not args.ignore_warnings:
                    print_warning(f"No interchromosomal translocations could be generated between sequence {a+1} and {b+1} (it rates too low).",
                                  args.no_color)
                continue
            pairs.append((a, b))
            counts.append(n)
        bps = {}
        if pairs:
            # sample_with_minimum_distance(1, len, n, 1) for both members of every pair (it_mutator.py:108-111);
            # keyed by the global contig index, so every rank computes the same breakpoints
            gid, stop, k = [], [], []
            for (a, b), n in zip(pairs, counts):
                gid += [a, b]; stop += [len(fasta[a]), len(fasta[b])]; k += [n, n]
            pos = eng.sample_positions(self._seed, gid, [1] * len(gid), stop, k, 1)
            o = 0
            for (a, b), n in zip(pairs, counts):
                pa, pb = pos[o:o + n], pos[o + n:o + 2 * n]
                bps[a] = {"self": pa, "partner": pb}
                bps[b] = {"self": pb, "partner": pa}
                o += 2 * n
        return bps

    def _records(self, bps, my_ids=None, src_of=None):
        """One raw far-copy record per interval taken from the partner.  my_ids: global contigs resident on this
        engine (local index = position); src_of[p]: genome index of partner p's first base on this engine."""
        fasta = self._fasta
        parts = []
        local = None if my_ids is None else {g: i for i, g in enumerate(my_ids)}
        for c in sorted(bps):
            if local is not None and c not in local:
                continue
            p = self._partners[c]
            a = np.concatenate(([0], bps[c]["self"].astype(np.int64), [len(fasta[c])]))
            b = np.concatenate(([0], bps[c]["partner"].astype(np.int64), [len(fasta[p])]))
            odd = np.arange(1, len(a) - 1, 2)          # intervals taken from the partner (it_mutator.py:133-137)
            r = np.zeros(len(odd), dtype=REC_DTYPE)
            r["pos"] = a[odd]
            r["cons"] = a[odd + 1] - a[odd]
            r["prod"] = b[odd + 1] - b[odd]
            r["src"] = (fasta.goff[p] if src_of is None else src_of[p]) + b[odd]
            r["kind"] = K_RAW
            r["type"] = T_IT
            r["contig"] = c if local is None else local[c]
            parts.append(r)
        return np.concatenate(parts) if parts else np.zeros(0, dtype=REC_DTYPE)

    def mutate(self):
        """Creates interchromosomal translocations and writes them to a Fasta and BEDPE file."""
        fasta = self._fasta
        if self._world > 1:
            return self._mutate_partitioned()
        eng = self._engine = getattr(fasta, "engine", None) or Engine(getattr(self._args, "device", 0))
        fasta.upload(eng)
        bps = self.breakpoints = self._generate_all_breakpoints(eng)
        eng.load_records(self._records(bps))
        eng.apply()
        self._fasta_writer.write_from_engine(eng, BUF_FASTA)
        for chrom in self._sim.chromosomes:            # FASTA order, one block of rows per paired contig
            c = chrom.number
            if c in bps:
                p = self._partners[c]
                self._bedpe_writer._f.write(rows(fasta[c].name, bps[c]["self"], len(fasta[c]), fasta[p].name,
                                                 bps[c]["partner"], len(fasta[p])))

    def _mutate_tiles(self):
        """Fewer (or far more uneven) contigs than GPUs: every rank holds the genome and the same breakpoints (they are
        keyed by the global contig id) and writes its share of the output tiles (ms_apply_window); no exchange."""
        fasta, rank, world = self._fasta, self._rank, self._world
        eng = self._engine = getattr(fasta, "engine", None) or Engine(D.local_device())
        fasta.upload(eng)
        bps = self.breakpoints = self._generate_all_breakpoints(eng)
        eng.load_records(self._records(bps))
        w = eng.apply_window(rank, world)
        D.write_window(self._args.outfastait, eng, BUF_FASTA, *w["fasta"], w["fasta_bytes"], bgzip=getattr(self._args, "bgzip", False))
        bed = b""
        if rank == 0:
            for chrom in self._sim.chromosomes:
                c = chrom.number
                if c in bps:
                    p = self._partners[c]
                    bed += rows(fasta[c].name, bps[c]["self"], len(fasta[c]), fasta[p].name, bps[c]["partner"], len(fasta[p]))
        D.write_partitioned(self._args.outbedpe, [0] if rank == 0 else [], [bed] if rank == 0 else [], 1)

    def _mutate_partitioned(self):
        """One process per GPU: contigs are partitioned; for a pair that straddles two GPUs each member reads the
        intervals it takes from the other out of the peer's HBM (see setup_partitioned; SURVEY.md §8e)."""
        if D.shard_of(self._fasta, self._world) == "tiles":
            return self._mutate_tiles()
        self.setup_partitioned()
        self.step_partitioned()
        self.write_partitioned()

    # The three phases are separate so that bench.py can time the step (breakpoints -> exchange -> splice) alone.
    def setup_partitioned(self):
        """Partition, upload of this rank's contigs, and the route to partner contigs owned by a peer:
        ``direct`` (default) maps the owner's genome buffer (CUDA IPC) so the splice kernel gathers the swapped intervals
        in place over NVLink; ``pull`` copies them from the mapped buffer into a staging region behind this rank's genome;
        ``nccl`` has the owner send them there (MS_IT_EXCHANGE selects; all three write identical files)."""
        fasta, rank, world = self._fasta, self._rank, self._world
        n_contigs = len(fasta.names)
        parts = D.partition_of(fasta, world)
        self._own = own = D.owners(parts, n_contigs)
        self._my_ids = my_ids = parts[rank]
        self._device = device = D.local_device()
        self._route = route = os.environ.get("MS_IT_EXCHANGE", "direct")
        if route not in ("direct", "pull", "nccl"):
            raise MutSimError(MS_ERR_ARG, f"MS_IT_EXCHANGE={route}: expected direct, pull or nccl")
        eng = self._engine = getattr(fasta, "engine", None) or Engine(device)
        foreign = sorted(self._partners[c] for c in my_ids if c in self._partners and own[self._partners[c]] != rank)
        # staging (pull, nccl): a slot per foreign partner, sized for the whole contig — an interval lands at its own
        # coordinate, so the records' sources need no translation table
        stage_off, acc = {}, 0
        if route != "direct":
            for p in foreign:
                stage_off[p] = acc
                acc += int(fasta.lengths[p]) + 64
        eng.reserve_foreign(acc)
        if my_ids:
            fasta.upload(eng, my_ids)
        total = int(sum(int(fasta.lengths[g]) for g in my_ids))
        goff_on = {}                       # contig -> index of its base 0 in its owner's genome
        for part in parts:
            o = 0
            for g in part:
                goff_on[g] = o
                o += int(fasta.lengths[g])
        self._local_goff = {g: goff_on[g] for g in my_ids}
        self._src_of = {p: goff_on[p] for p in my_ids}
        self._peer_src = {}
        if route == "nccl":
            self._src_of.update({p: total + 64 + off for p, off in stage_off.items()})
        else:
            # every rank with contigs exports its buffer; a reader maps only the owners of its foreign partners
            mine = eng.export_genome() if my_ids else None
            handles = D.all_gather_object(mine)
            rel = {}
            if my_ids:
                for r in sorted({int(own[p]) for p in foreign}):
                    rel[r] = eng.open_peer(*handles[r])
            self._peer_src = {p: rel[int(own[p])] + goff_on[p] for p in foreign}
            if route == "direct":
                self._src_of.update(self._peer_src)
            else:
                self._src_of.update({p: total + 64 + off for p, off in stage_off.items()})
        self.exchange_bytes = self.exchange_ms = 0

    MAX_INTERVAL_OPS = 64      # beyond this many intervals per direction the whole contig goes as one transfer

    def step_partitioned(self):
        """Breakpoints (identical on every rank: keyed by the global contig id), exchange, records, splice."""
        fasta, rank = self._fasta, self._rank
        own, my_ids, src_of, local_goff = self._own, self._my_ids, self._src_of, self._local_goff
        eng, route = self._engine, self._route
        bps = self.breakpoints = self._generate_all_breakpoints(eng)
        # globally agreed order: ascending (min, max) of each straddling pair; for each member the intervals the
        # OTHER one takes from it (odd-numbered intervals of its own breakpoint list, it_mutator.py:133-137)
        sends, recvs, pulls, remote = [], [], [], 0
        for a in sorted(bps):
            b = self._partners[a]
            if a < b and own[a] != own[b]:
                for mine, theirs in ((a, b), (b, a)):
                    if own[mine] != rank:
                        continue
                    peer = int(own[theirs])
                    cut = np.concatenate(([0], bps[mine]["self"].astype(np.int64), [int(fasta.lengths[mine])]))
                    cut_t = np.concatenate(([0], bps[theirs]["self"].astype(np.int64), [int(fasta.lengths[theirs])]))
                    odd = np.arange(1, len(cut) - 1, 2)
                    remote += int(sum(int(cut_t[i + 1] - cut_t[i]) for i in odd))
                    if route == "pull" and len(odd) <= self.MAX_INTERVAL_OPS:
                        pulls += [(self._peer_src[theirs] + int(cut_t[i]), src_of[theirs] + int(cut_t[i]),
                                   int(cut_t[i + 1] - cut_t[i])) for i in odd]
                    elif route == "pull":
                        pulls.append((self._peer_src[theirs], src_of[theirs], int(fasta.lengths[theirs])))
                    elif len(odd) <= self.MAX_INTERVAL_OPS:
                        sends += [(peer, local_goff[mine] + int(cut[i]), int(cut[i + 1] - cut[i])) for i in odd]
                        recvs += [(peer, src_of[theirs] + int(cut_t[i]), int(cut_t[i + 1] - cut_t[i])) for i in odd]
                    else:
                        sends.append((peer, local_goff[mine], int(fasta.lengths[mine])))
                        recvs.append((peer, src_of[theirs], int(fasta.lengths[theirs])))
        if route == "nccl":
            self.exchange_bytes = sum(n for _, _, n in recvs)
            self.exchange_ms = D.exchange_contigs(eng, self._device, sends, recvs)
        elif route == "pull":
            self.exchange_bytes = sum(n for _, _, n in pulls)
            if pulls:
                eng.pull_peer(*zip(*pulls))        # on the engine's stream, ahead of the splice that reads the staging
        else:                                      # direct: the splice kernel reads the peers' HBM (bytes it gathers remotely)
            self.exchange_bytes = remote
        if my_ids:
            eng.load_records(self._records(bps, my_ids, src_of))
            eng.apply()

    def write_partitioned(self):
        fasta, my_ids, bps = self._fasta, self._my_ids, self.breakpoints
        n_contigs = len(fasta.names)
        D.write_fasta_partitioned(self._args.outfastait, self._engine, my_ids, n_contigs, bgzip=getattr(self._args, "bgzip", False))
        bed = []
        for g in my_ids:
            if g in bps:
                p = self._partners[g]
                bed.append(rows(fasta[g].name, bps[g]["self"], len(fasta[g]), fasta[p].name, bps[g]["partner"], len(fasta[p])))
            else:
                bed.append(b"")
        D.write_partitioned(self._args.outbedpe, my_ids, bed, n_contigs)
