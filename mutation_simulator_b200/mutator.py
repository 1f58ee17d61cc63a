"""``Mutator`` — the reference's class API (mutator.py:73-142) on the B200 path.

``Mutator(args, fasta, sim).mutate()`` samples positions, types and lengths for every
range of every contig, resolves overlaps, links translocations, splices the genome and
formats FASTA + VCF — all on the GPU through libmutsim_b200 — then writes the two files.
Nothing here touches a base on the host.

With ``--ploidy P`` >= 2 the same table is sampled, every record draws its haplotype mask on the GPU, the phased VCF of
the whole table is written, and then each haplotype's records are selected on the device and applied in turn: one
FASTA (and chain) per haplotype.

With ``--reads`` each haplotype's read pairs are drawn right after its FASTA (and chain) is written, while its mutated
genome is still in HBM, and appended to ``*_ms_R1.fq`` / ``*_ms_R2.fq`` (reads_writer.py)."""
from __future__ import annotations

import os
import secrets
import sys
import time

import numpy as np

from . import distributed as D
from .engine import BUF_FASTA, BUF_VCF, BUF_VCF_PHASED, Engine
from .fasta_writer import FastaWriter
from .plan import block_list, build_ranges, p_transition
from .util import format_warning
from .vcf_writer import VcfWriter


def run_seed(args) -> int:
    """--seed if given; otherwise a fresh 64-bit seed (the reference's RNGs are unseeded too)."""
    s = getattr(args, "seed", None)
    return secrets.randbits(63) if s is None else int(s)


class Mutator:
    def __init__(self, args, fasta, sim, reads_budget=None):
        """reads_budget: FASTQ bytes formatted in HBM per call with --reads (default reads_writer.DEFAULT_BATCH_BYTES)."""
        self._args, self._fasta, self._sim = args, fasta, sim
        self._rank, self._world = D.init()
        self._engine = None
        self.stats = None
        self._replay = None
        self._ploidy = getattr(args, "ploidy", 1)
        self._hap_writers = []
        self._reads_writer = None
        self._reads_pairs = None         # pairs per contig over the haplotypes written so far (for the empty-contig warning)
        from .reads_writer import DEFAULT_BATCH_BYTES
        self._reads_budget = reads_budget or DEFAULT_BATCH_BYTES
        # plan the ranges (and reject overlapping ones) BEFORE any output file is opened and truncated: a settings
        # error must not leave partial *_ms.fa / *_ms.vcf behind (the reference dies later, with both files cut)
        self._planned = build_ranges(sim, fasta.lengths, None) if sim.has_mutations else None
        if getattr(args, "reads", None) is not None:
            from .reads_writer import ReadsWriter
            self._reads_writer = ReadsWriter([args.outreads1, args.outreads2], getattr(args, "bgzip", False), self._reads_budget,
                                             create=self._world == 1)
        if self._world > 1:      # one process per GPU: files are assembled by write_partitioned()
            self._fasta_writer = self._vcf_writer = None
            return
        bgzip = getattr(args, "bgzip", False)
        if self._ploidy > 1:     # one FASTA per haplotype instead of *_ms.fa
            self._fasta_writer = None
            self._hap_writers = [FastaWriter(p, bgzip) for p in args.outfastas]
        else:
            self._fasta_writer = FastaWriter(args.outfasta, bgzip)
        self._vcf_writer = VcfWriter(args.outvcf, bgzip)
        if getattr(args, "chain", False):
            from .chain_writer import write_text
            for p in (args.outchains if self._ploidy > 1 else [args.outchain]):
                write_text(p, b"")      # created (and checked) up front like the other outputs
        self._vcf_writer.write_header(args.infile.name, fasta, sim.assembly_name, sim.species_name, sim.sample_name)

    def load_vcf(self, text):
        """Replay instead of sampling: apply the records of a VCF written by the reference (vcf_writer.py:118-126) or by
        this package to the same FASTA; mutate() then reproduces that run's *_ms.fa and re-emits the VCF.  text: str,
        a bytes-like object or an mmap (parsed in place on the GPU)."""
        self._replay = text

    def detach_engine(self):
        """Hand the engine (with the mutated genome's FASTA image still in HBM) to the caller; close() then
        leaves it alone."""
        eng, self._engine = self._engine, None
        return eng

    def close(self):
        for w in self._hap_writers:
            w.close()
        if self._reads_writer is not None:
            self._reads_writer.close()
            self._reads_writer = None
        if self._fasta_writer is not None:
            self._fasta_writer.close()
        if self._vcf_writer is not None:
            self._vcf_writer.close()
        if self._engine is not None:
            self._engine.close()
            self._engine = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def mutate(self):
        """Creates random mutations and writes them to a Fasta and VCF file."""
        args, fasta, sim = self._args, self._fasta, self._sim
        world = self._world
        marks = [("start", time.perf_counter())]
        lap = lambda name: marks.append((name, time.perf_counter()))
        n_contigs = len(fasta.names)
        # several GPUs: whole contigs per rank (every stage sharded, no exchange), or — when contigs are too few or too
        # uneven for that — the same table on every rank and the output cut at tile boundaries (distributed.shard_mode)
        mode = D.shard_of(fasta, world)
        tiles = world > 1 and mode == "tiles"
        my_ids = D.partition_of(fasta, world)[self._rank] if world > 1 and not tiles else list(range(n_contigs))
        self.shard, self.my_ids = ("tiles" if tiles else "contigs"), my_ids
        self.parts = D.partition_of(fasta, world) if world > 1 and not tiles else None
        seed = self._seed = D.broadcast_object(run_seed(args))
        eng = self._engine = getattr(fasta, "engine", None) or \
            Engine(D.local_device(getattr(args, "device", 0)) if world > 1 else getattr(args, "device", 0))
        lap("engine")
        window = None
        if my_ids:      # (more ranks than contigs in MS_SHARD=contigs mode: an idle rank only joins the collectives)
            fasta.upload(eng, my_ids if world > 1 and not tiles else None)
            lap("gather+upload")
            if self._replay is not None:
                # parsed on the device; a VCF of another shape than VcfWriter's goes through the host parser
                text, skip = self._replay, world > 1 and not tiles
                if isinstance(text, str):
                    try:
                        text = text.encode("latin-1")
                    except UnicodeEncodeError:
                        pass
                ploidy = self._ploidy if self._ploidy > 1 else None
                loaded = not isinstance(text, str) and \
                    (eng.load_vcf_phased(text, ploidy, skip) if ploidy else eng.load_vcf(text, skip))
                if not loaded:
                    from .records import genome_offsets, records_from_vcf
                    lens = [int(fasta.lengths[g]) for g in my_ids]
                    if not isinstance(text, (str, bytes, bytearray)):
                        text = bytes(text)
                    recs, lit, *masks = records_from_vcf(text, [fasta.names[g] for g in my_ids], genome_offsets(lens), lens,
                                                         skip_unknown=skip, ploidy=ploidy)
                    eng.load_records(recs, lit)
                    if ploidy:
                        eng.genotype_load(masks[0], ploidy)
            else:
                ranges, n = self._planned if (self._planned is not None and len(my_ids) == n_contigs) \
                    else build_ranges(sim, fasta.lengths, my_ids)
                eng.set_ranges_array(ranges, n, block_list(sim), min(sim.mut_block.values()), p_transition(sim.titv))
                eng.sample(seed)
                if self._ploidy > 1:
                    eng.genotype_draw(seed, self._ploidy, getattr(args, "hom_fraction", 0.35))
            if self._ploidy > 1:
                eng.vcf_phased()
            elif tiles:
                window = eng.apply_window(self._rank, world)
            else:
                eng.apply()
            lap("sample+apply")
            if self._ploidy == 1 and not args.ignore_warnings and (not tiles or self._rank == 0) \
                    and getattr(args, "mode", None) != "vcf":      # (a polyploid run warns after its haplotypes)
                self._warn_empty(eng.contig_records(), my_ids)
        if self._ploidy > 1:
            return self._mutate_haplotypes(eng, tiles, my_ids, n_contigs, lap, marks)
        chain = getattr(args, "chain", False)
        if world == 1:
            self._fasta_writer.write_from_engine(eng, BUF_FASTA)
            self._vcf_writer.write_from_engine(eng, BUF_VCF)
            if chain:
                from .chain_writer import write_from_engine
                write_from_engine(args.outchain, eng, getattr(args, "bgzip", False))
        else:
            from .fasta_writer import FastaWriterError
            from .vcf_writer import VcfWriterError, header_text
            head = header_text(args.infile.name, [(fasta[k].name, len(fasta[k])) for k in fasta.keys()], sim.assembly_name,
                               sim.species_name, sim.sample_name).encode("latin-1")
            bgzip = getattr(args, "bgzip", False)
            try:
                if tiles:
                    D.write_window(args.outfasta, eng, BUF_FASTA, *window["fasta"], window["fasta_bytes"], bgzip=bgzip)
                else:
                    vcf_off = D.write_fasta_partitioned(args.outfasta, eng, my_ids, n_contigs, bgzip=bgzip)
            except D.OutputCreateError as e:
                raise FastaWriterError(f"Cannot write to Fasta file {args.outfasta} {e}")
            try:
                if tiles:
                    D.write_window(args.outvcf, eng, BUF_VCF, *window["vcf"], window["vcf_bytes"], prefix=head, bgzip=bgzip)
                else:
                    D.write_slices_partitioned(args.outvcf, eng, BUF_VCF, my_ids, vcf_off, n_contigs, prefix=head, bgzip=bgzip)
            except D.OutputCreateError as e:
                raise VcfWriterError(f"Cannot write to VCF file {args.outvcf} {e}")
            if chain:
                self._write_chain_partitioned(eng, tiles, my_ids, n_contigs, bgzip)
        lap("download+write")
        if self._reads_writer is not None:
            self._write_reads(eng, 1, tiles, my_ids, n_contigs)
            self._warn_no_reads(tiles, my_ids)
            lap("reads")
        self._finish(eng, my_ids, marks)

    def _finish(self, eng, my_ids, marks):
        self.stats = eng.stats() if my_ids else None
        self.host_seconds = {b[0]: b[1] - a[1] for a, b in zip(marks, marks[1:])}
        if os.environ.get("MS_TIMING"):
            print(f"[rank {self._rank}] " + " ".join(f"{k}={v:.3f}s" for k, v in self.host_seconds.items()), file=sys.stderr)

    def _mutate_haplotypes(self, eng, tiles, my_ids, n_contigs, lap, marks):
        """Polyploid run, after the table and its genotypes are in place and the phased VCF is formatted: write the VCF,
        then select, apply and write each haplotype in turn.  Several GPUs: in contig mode each rank writes its contigs'
        slices (ms_vcf_phased's per-contig offsets); in tile mode every rank formatted the whole VCF and writes its byte
        window, and applies its window of each haplotype."""
        args, fasta, sim = self._args, self._fasta, self._sim
        world, bgzip, chain = self._world, getattr(args, "bgzip", False), getattr(args, "chain", False)
        from .fasta_writer import FastaWriterError
        from .vcf_writer import VcfWriterError
        if world == 1:
            self._vcf_writer.write_from_engine(eng, BUF_VCF_PHASED)
        else:
            from .vcf_writer import header_text
            head = header_text(args.infile.name, [(fasta[k].name, len(fasta[k])) for k in fasta.keys()], sim.assembly_name,
                               sim.species_name, sim.sample_name).encode("latin-1")
            off = eng.vcf_phased_off if my_ids else np.zeros(1, np.int64)
            try:
                if tiles:
                    total = int(off[-1])
                    D.write_window(args.outvcf, eng, BUF_VCF_PHASED, total * self._rank // world,
                                   total * (self._rank + 1) // world, total, prefix=head, bgzip=bgzip)
                else:
                    D.write_slices_partitioned(args.outvcf, eng, BUF_VCF_PHASED, my_ids, off, n_contigs, prefix=head, bgzip=bgzip)
            except D.OutputCreateError as e:
                raise VcfWriterError(f"Cannot write to VCF file {args.outvcf} {e}")
        per = np.zeros(len(my_ids), dtype=np.int64)
        for h in range(1, self._ploidy + 1):
            path = args.outfastas[h - 1]
            if my_ids:
                eng.select_haplotype(h)
                window = eng.apply_window(self._rank, world) if tiles else None
                if not tiles:
                    eng.apply()
                per += eng.contig_records()
            try:
                if world == 1:
                    self._hap_writers[h - 1].write_from_engine(eng, BUF_FASTA)
                elif tiles:
                    D.write_window(path, eng, BUF_FASTA, *window["fasta"], window["fasta_bytes"], bgzip=bgzip)
                else:
                    D.write_fasta_partitioned(path, eng, my_ids, n_contigs, bgzip=bgzip)
            except D.OutputCreateError as e:
                raise FastaWriterError(f"Cannot write to Fasta file {path} {e}")
            if chain:
                if world == 1:
                    from .chain_writer import write_from_engine
                    write_from_engine(args.outchains[h - 1], eng, bgzip)
                else:
                    self._write_chain_partitioned(eng, tiles, my_ids, n_contigs, bgzip, args.outchains[h - 1])
            if self._reads_writer is not None:
                self._write_reads(eng, h, tiles, my_ids, n_contigs)
        lap("haplotypes")
        if self._reads_writer is not None:
            self._warn_no_reads(tiles, my_ids)
        if my_ids and not args.ignore_warnings and (not tiles or self._rank == 0) and getattr(args, "mode", None) != "vcf":
            self._warn_empty(per, my_ids)        # a contig that no haplotype mutates got no records at all
        self._finish(eng, my_ids, marks)

    def _write_reads(self, eng, h, tiles, my_ids, n_contigs):
        """Haplotype h's read pairs from the mutated genome of its apply, appended to both FASTQ files.  Tile mode: every
        rank applies the whole haplotype (the window apply leaves buffer 0 partly valid) and writes pairs
        [n r / W, n (r + 1) / W) of each contig; contig mode: each rank writes its contigs' pairs."""
        from .reads_writer import config, pair_counts
        args, world, rank = self._args, self._world, self._rank
        cfg = config(args, self._seed, h)
        n = np.zeros(len(my_ids), dtype=np.int64)
        if my_ids:
            if tiles:
                eng.apply()
            n = pair_counts(args.reads, eng.contig_out_len(), args.read_length, self._ploidy)
        self._reads_pairs = n if self._reads_pairs is None else self._reads_pairs + n
        if world == 1:
            self._reads_writer.write(eng, cfg, n)
        elif tiles:
            slices = [(g * world + rank, g, int(n[g]) * rank // world, int(n[g]) * (rank + 1) // world) for g in range(len(my_ids))]
            self._reads_writer.write_partitioned(eng, cfg, n, slices, n_contigs * world)
        else:
            self._reads_writer.write_partitioned(eng, cfg, n, [(g, i, 0, int(n[i])) for i, g in enumerate(my_ids)], n_contigs)

    def _warn_no_reads(self, tiles, my_ids):
        if not my_ids or self._args.ignore_warnings or (tiles and self._rank != 0):
            return
        for i in np.flatnonzero(self._reads_pairs == 0):
            print(format_warning(f"No reads could be simulated on sequence {my_ids[int(i)]+1} (shorter than the read length or "
                                 "depth too low)", self._args.no_color), file=sys.stderr)

    def _warn_empty(self, per_contig, my_ids):
        for i in np.flatnonzero(per_contig == 0):
            print(format_warning(f"No mutations could be generated on sequence {my_ids[int(i)]+1} (mutation rates too low)",
                                 self._args.no_color), file=sys.stderr)

    def _write_chain_partitioned(self, eng, tiles, my_ids, n_contigs, bgzip, path=None):
        """Several GPUs.  Tiles: every rank holds the whole table, formats the whole file and writes its byte window.
        Contigs: the ranks gather the per-contig chain counts to number the chains, then write their contigs' slices.
        path: the chain file (default *_ms.chain; a polyploid run writes one per haplotype)."""
        from .chain_writer import ChainWriterError, first_ids
        from .engine import BUF_CHAIN
        path = path or self._args.outchain
        try:
            if tiles:
                off = eng.chain_write(first_ids(eng.chain_count()))
                total = int(off[-1])
                lo, hi = total * self._rank // self._world, total * (self._rank + 1) // self._world
                D.write_window(path, eng, BUF_CHAIN, lo, hi, total, bgzip=bgzip)
            else:
                mine = eng.chain_count() if my_ids else np.zeros(0, np.int64)
                counts = np.zeros(n_contigs, dtype=np.int64)
                for ids, cnt in D.all_gather_object((list(my_ids), [int(x) for x in mine])):
                    if len(ids):
                        counts[ids] = cnt
                off = eng.chain_write(first_ids(counts)[list(my_ids)]) if my_ids else np.zeros(1, np.int64)
                D.write_slices_partitioned(path, eng, BUF_CHAIN, my_ids, off, n_contigs, bgzip=bgzip)
        except D.OutputCreateError as e:
            raise ChainWriterError(f"Cannot write to chain file {path} {e}")
