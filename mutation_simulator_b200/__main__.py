"""``python -m mutation_simulator_b200`` / ``mutation-simulator``: the reference's
entry point (__main__.py:34-107) — same modes, messages and exit codes."""
from __future__ import annotations

import gzip
import mmap
import os
import zlib
from timeit import default_timer as timer

from . import (BedpeWriterError, ChromNotExistError, FastaDuplicateHeaderError, FastaIndexingError, FastaNotFoundError,
               FastaWriterError, ITMutator, ITNotEnoughAvailChromsError, ItRateTooHighError, ItRateTooLowError,
               MinimumLengthHigherThanMaximumError, MinimumLengthTooLowError, MissingLengthError, Mutator, MutSimError,
               RangeDefinitionOutOfBoundsError, RangeOverlapError, RatesTooHighError, RatesTooLowError, RMTParseError,
               SimulationSettings, TitvTooLowError, VcfWriterError, exit_with_error, get_args, get_md5, load_fasta,
               print_success, print_warning)
from .rmt import MutationSettings

_SETUP_ERRORS = (FileNotFoundError, ITNotEnoughAvailChromsError, RatesTooHighError, RatesTooLowError, FastaIndexingError,
                 FastaNotFoundError, ItRateTooHighError, ItRateTooLowError, RMTParseError, MissingLengthError,
                 MinimumLengthTooLowError, TitvTooLowError, ChromNotExistError, RangeDefinitionOutOfBoundsError,
                 FastaDuplicateHeaderError, MinimumLengthHigherThanMaximumError)


def check_replay_paths(args):
    """`vcf` mode: the VCF to replay must not be one of the files this run writes (e.g. `-o in vcf in_ms.vcf`), which
    would be truncated before it is read."""
    src = args.vcffile
    for out in (args.outvcf, args.outfasta):
        if out.resolve() == src.resolve() or (out.exists() and src.exists() and os.path.samefile(out, src)):
            raise VcfWriterError(f"The output file {out} would overwrite the input VCF {src}; choose another -o")


def read_replay_vcf(path):
    """The VCF text of `vcf` mode: a plain file is memory-mapped (the engine parses it in place); gzip or BGZF input is
    inflated on the host, as load_fasta does."""
    with open(path, "rb") as fh:
        if fh.read(2) == b"\x1f\x8b":
            fh.seek(0)
            return gzip.decompress(fh.read())
        if os.fstat(fh.fileno()).st_size == 0:
            return b""
        return mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ)


def initialize():
    args = get_args()
    if args.mode == "vcf":      # before any output file is opened
        try:
            check_replay_paths(args)
        except VcfWriterError as e:
            exit_with_error(e, args.no_color)
    try:
        from . import distributed
        # the file is parsed on the GPU and stays there for the engines (SURVEY.md §8 f1); with several GPUs every
        # rank ingests it and later keeps its share of the contigs
        multi = distributed.rank_world()[1] > 1
        fasta = load_fasta(args.infile, device=distributed.local_device(getattr(args, "device", 0)) if multi
                           else getattr(args, "device", 0))
        if args.mode == "args":
            sim = SimulationSettings.from_args(args, fasta, args.ignore_warnings)
        elif args.mode == "it":
            sim = SimulationSettings.from_it(args.interchromosomalrate, fasta, args.ignore_warnings)
        elif args.mode == "rmt":
            sim = SimulationSettings.from_rmt(args.rmtfile, fasta, args.ignore_warnings)
        else:   # vcf: the records come from the file; no ranges, no IT
            sim = SimulationSettings(MutationSettings(None, None), None, [], None, ignore_warnings=args.ignore_warnings)
    except _SETUP_ERRORS + (MutSimError,) as e:   # MutSimError: no usable CUDA device / library (there is no CPU fallback)
        exit_with_error(e, args.no_color)
    if not args.ignore_warnings:
        warn_user(args, sim)
    return args, fasta, sim


def warn_user(args, sim):
    if sim.fasta and args.infile.name != sim.fasta:
        print_warning("Fasta filename does not match RMT", args.no_color)
    if sim.md5 and get_md5(args.infile) != sim.md5:
        print_warning("Fasta md5 hash does not match RMT", args.no_color)


def main():
    start = timer()
    args, fasta, sim = initialize()
    from . import distributed
    resident = None
    replay = None
    if args.mode == "vcf":
        try:
            replay = read_replay_vcf(args.vcffile)
        except (OSError, EOFError, zlib.error) as e:
            exit_with_error(e, args.no_color)
    if sim.has_mutations or replay is not None:
        try:
            mutator = Mutator(args, fasta, sim)
            if replay is not None:
                mutator.load_vcf(replay)
            mutator.mutate()
            # the mutated genome stays in HBM for the IT step (MS_NO_CHAIN=1 forces the reference's reload of *_ms.fa);
            # with several GPUs every rank keeps the contigs it mutated and the IT step reuses the partition
            if sim.has_it and not os.environ.get("MS_NO_CHAIN"):
                world = distributed.rank_world()[1]
                ok = mutator._engine is not None and mutator.shard == "contigs" and len(mutator.my_ids) > 0 \
                    and int(mutator._engine.contig_out_len().min()) > 0
                if world > 1:
                    ok = all(distributed.all_gather_object(bool(ok)))
                if ok:
                    from .fasta import ResidentFasta
                    resident = ResidentFasta(mutator.detach_engine(), fasta, mutator.my_ids if world > 1 else None, mutator.parts)
                    fasta.detach_engine()
            mutator.close()
            fasta.close()
        except (FastaWriterError, VcfWriterError, MutSimError, RangeOverlapError) as e:
            exit_with_error(e, args.no_color)
        except ValueError as e:     # a VCF line the replay cannot read (records.records_from_vcf)
            if replay is None:
                raise
            exit_with_error(e, args.no_color)
    if sim.has_it:
        if resident is not None:
            fasta = resident
        elif sim.has_mutations:   # IT runs on the mutated genome (__main__.py:88-95)
            distributed.barrier()   # all ranks have written their slices of *_ms.fa
            try:
                fasta = load_fasta(args.outfasta)
            except (FastaDuplicateHeaderError, FastaIndexingError, FastaNotFoundError) as e:
                exit_with_error(e, args.no_color)
        try:
            it_mutator = ITMutator(args, fasta, sim)
            it_mutator.mutate()
            it_mutator.close()
            fasta.close()
        except (FastaWriterError, BedpeWriterError, MutSimError) as e:
            exit_with_error(e, args.no_color)
    runtime = round(timer() - start, 4)
    if distributed.rank_world()[0] != 0:
        return
    if not args.quiet:
        print_success(f"Mutation-Simulator finished in: {runtime}s", args.no_color)


if __name__ == "__main__":
    main()
