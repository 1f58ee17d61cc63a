"""``Mutator`` — the reference's class API (mutator.py:73-142) on the B200 path.

``Mutator(args, fasta, sim).mutate()`` samples positions, types and lengths for every
range of every contig, resolves overlaps, links translocations, splices the genome and
formats FASTA + VCF — all on the GPU through libmutsim_b200 — then writes the two files.
Nothing here touches a base on the host."""
from __future__ import annotations

import os
import secrets
import sys
import time

import numpy as np

from . import distributed as D
from .engine import BUF_FASTA, BUF_VCF, Engine
from .fasta_writer import FastaWriter
from .plan import block_list, build_ranges, p_transition
from .util import format_warning
from .vcf_writer import VcfWriter


def run_seed(args) -> int:
    """--seed if given; otherwise a fresh 64-bit seed (the reference's RNGs are unseeded too)."""
    s = getattr(args, "seed", None)
    return secrets.randbits(63) if s is None else int(s)


class Mutator:
    def __init__(self, args, fasta, sim):
        self._args, self._fasta, self._sim = args, fasta, sim
        self._rank, self._world = D.init()
        self._engine = None
        self.stats = None
        self._replay = None
        # plan the ranges (and reject overlapping ones) BEFORE any output file is opened and truncated: a settings
        # error must not leave partial *_ms.fa / *_ms.vcf behind (the reference dies later, with both files cut)
        self._planned = build_ranges(sim, fasta.lengths, None) if sim.has_mutations else None
        if self._world > 1:      # one process per GPU: files are assembled by write_partitioned()
            self._fasta_writer = self._vcf_writer = None
            return
        bgzip = getattr(args, "bgzip", False)
        self._fasta_writer = FastaWriter(args.outfasta, bgzip)
        self._vcf_writer = VcfWriter(args.outvcf, bgzip)
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
        if self._fasta_writer is not None:
            self._fasta_writer.close()
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
        seed = D.broadcast_object(run_seed(args))
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
                if isinstance(text, str) or not eng.load_vcf(text, skip):
                    from .records import genome_offsets, records_from_vcf
                    lens = [int(fasta.lengths[g]) for g in my_ids]
                    if not isinstance(text, (str, bytes, bytearray)):
                        text = bytes(text)
                    recs, lit = records_from_vcf(text, [fasta.names[g] for g in my_ids], genome_offsets(lens), lens,
                                                 skip_unknown=skip)
                    eng.load_records(recs, lit)
            else:
                ranges, n = self._planned if (self._planned is not None and len(my_ids) == n_contigs) \
                    else build_ranges(sim, fasta.lengths, my_ids)
                eng.set_ranges_array(ranges, n, block_list(sim), min(sim.mut_block.values()), p_transition(sim.titv))
                eng.sample(seed)
            if tiles:
                window = eng.apply_window(self._rank, world)
            else:
                eng.apply()
            lap("sample+apply")
            if not args.ignore_warnings and (not tiles or self._rank == 0) and getattr(args, "mode", None) != "vcf":
                per = eng.contig_records()
                for i in np.flatnonzero(per == 0):
                    print(format_warning(f"No mutations could be generated on sequence {my_ids[int(i)]+1} (mutation rates too low)",
                                         args.no_color), file=sys.stderr)
        if world == 1:
            self._fasta_writer.write_from_engine(eng, BUF_FASTA)
            self._vcf_writer.write_from_engine(eng, BUF_VCF)
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
        lap("download+write")
        self.stats = eng.stats() if my_ids else None
        self.host_seconds = {b[0]: b[1] - a[1] for a, b in zip(marks, marks[1:])}
        if os.environ.get("MS_TIMING"):
            print(f"[rank {self._rank}] " + " ".join(f"{k}={v:.3f}s" for k, v in self.host_seconds.items()), file=sys.stderr)
