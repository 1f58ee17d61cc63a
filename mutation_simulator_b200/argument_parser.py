"""Command line of ``mutation-simulator`` — flag for flag the reference's
(argument_parser.py:31-240) plus three extensions that default to the reference's
behaviour: ``--seed`` (reproducible runs; default: a fresh random seed, like the
reference's unseeded RNGs), ``--device`` (CUDA device index), ``--bgzip``
(BGZF-compressed FASTA and VCF output, encoded on the GPU), ``--chain`` (a UCSC
chain file from the input to the mutated genome, built on the GPU) and ``--ploidy`` /
``--hom-fraction`` (a diploid or polyploid sample: one FASTA per haplotype and a phased
VCF, genotypes drawn on the GPU), ``--reads`` (paired-end reads of the mutated sample,
drawn on the GPU), and the ``vcf`` mode (replay a VCF the reference or this package wrote
onto the same FASTA).

With ``--ploidy P`` >= 2 the record table is sampled as for one haplotype; each record then
carries haplotype h with a drawn genotype: homozygous (on all P haplotypes) with probability
``--hom-fraction``, else on a uniformly drawn non-empty proper subset of them.  The run writes
``*_ms_h1.fa`` .. ``*_ms_hP.fa`` (and ``*_ms_h1.chain`` .. with ``--chain``) instead of
``*_ms.fa``, and one phased ``*_ms.vcf`` (GT ``1|0``, ``0|1``, ``1|1``, ...).

With ``--reads C`` each haplotype gets C / P of the sample's mean depth as read pairs
(``--read-length``, ``--fragment-mean``, ``--fragment-sd``, ``--read-error-rate``), written
to ``*_ms_R1.fq`` and ``*_ms_R2.fq`` next to ``*_ms.vcf``; every read name carries the pair's
position on the mutated contig and where its reads start on the input genome.  The read
options are ignored (and absent from the namespace) without ``--reads``.

The option table below drives argparse; the derived output names follow
argument_parser.py:14-28."""
from __future__ import annotations

import math
from argparse import SUPPRESS, ArgumentParser, ArgumentTypeError, Namespace
from pathlib import Path

from ._version import __version__
from .defaults import Defaults as D

# (short, long, dest kind, type, default, help) for the `args` sub-command, in the reference's order
_KINDS = [("sn", "snp", "SNP", "SNP"), ("in", "insert", "Insert", "insert"), ("de", "deletion", "Deletion", "deletion"),
          ("iv", "inversion", "Inversion", "inversion"), ("du", "duplication", "Duplication", "duplication"),
          ("tl", "translocation", "Translocation", "translocations")]
_PLURAL = {"in": "inserts", "de": "deletions", "iv": "inversion", "du": "duplications", "tl": "translocations"}


def add_outfile_names(args: Namespace) -> Namespace:
    """outfasta / outfastait / outvcf / outbedpe / outchain / outchainit from the output base; outfastas / outchains:
    the per-haplotype FASTA and chain files of a polyploid run (empty lists for ploidy 1)."""
    base = args.outbase
    try:
        base = base.with_stem(base.stem + "_ms")
    except ValueError:  # '.' or a bare directory: use the input's stem inside it
        base = base / (args.infile.stem + "_ms")
    args.outbase = base
    args.outfasta = base.with_suffix(args.infile.suffix)
    args.outfastait = args.outfasta.with_stem(args.outfasta.stem + "_it")
    args.outvcf = args.outfasta.with_suffix(".vcf")
    args.outbedpe = args.outfastait.with_suffix(".bedpe")
    args.outchain = args.outfasta.with_suffix(".chain")
    args.outchainit = args.outfastait.with_suffix(".chain")
    hap = range(1, getattr(args, "ploidy", 1) + 1) if getattr(args, "ploidy", 1) > 1 else ()
    args.outfastas = [args.outfasta.with_stem(f"{args.outfasta.stem}_h{h}") for h in hap]
    args.outchains = [args.outchain.with_stem(f"{args.outchain.stem}_h{h}") for h in hap]
    if getattr(args, "reads", None) is not None:
        args.outreads1, args.outreads2 = (args.outvcf.with_name(f"{args.outvcf.stem}_R{m}.fq") for m in (1, 2))
    if getattr(args, "bgzip", False):      # after the derivation: *_it, .bedpe and .chain keep their names
        for k in ("outfasta", "outfastait", "outvcf", "outchain", "outchainit"):
            p = getattr(args, k)
            setattr(args, k, p.with_name(p.name + ".gz"))
        args.outfastas = [p.with_name(p.name + ".gz") for p in args.outfastas]
        args.outchains = [p.with_name(p.name + ".gz") for p in args.outchains]
        if getattr(args, "reads", None) is not None:
            args.outreads1, args.outreads2 = (p.with_name(p.name + ".gz") for p in (args.outreads1, args.outreads2))
    return args


MAX_PLOIDY = 8


def _ploidy(text: str) -> int:
    v = int(text)
    if not 1 <= v <= MAX_PLOIDY:
        raise ArgumentTypeError(f"ploidy must be between 1 and {MAX_PLOIDY}, got {v}")
    return v


def _fraction(text: str) -> float:
    v = float(text)
    if not 0.0 <= v <= 1.0:
        raise ArgumentTypeError(f"hom-fraction must be between 0 and 1, got {text}")
    return v


# --reads options: (flag, dest, type, default, lowest, highest or None, help); checked only when --reads is given
_READS = [("--read-length", "read_length", int, D.READ_LENGTH, 1, 1000, "bases per read"),
          ("--fragment-mean", "fragment_mean", int, D.FRAGMENT_MEAN, None, 1_000_000,
           "mean fragment (insert) length, from the read length"),
          ("--fragment-sd", "fragment_sd", int, D.FRAGMENT_SD, 0, 100_000, "fragment length standard deviation"),
          ("--read-error-rate", "read_error_rate", float, D.READ_ERROR_RATE, 0.0, None, "per-base substitution error rate, below 1")]


def _check_reads(p: ArgumentParser, args: Namespace):
    """Fill in the read options' defaults and check them; exits with status 2 like any argparse error."""
    if not (math.isfinite(args.reads) and args.reads > 0):
        p.error(f"argument --reads: the depth must be finite and > 0, got {args.reads}")
    for flag, dest, typ, default, lo, hi, _ in _READS:
        v = getattr(args, dest, default)
        try:                    # taken as text by argparse, so that without --reads nothing about them is checked
            v = typ(v)
        except ValueError:
            p.error(f"argument {flag}: invalid {typ.__name__} value: {v!r}")
        setattr(args, dest, v)
        lo = args.read_length if dest == "fragment_mean" else lo
        if v < lo or (hi is not None and v > hi) or (dest == "read_error_rate" and not v < 1.0):
            top = "below 1" if hi is None else f"at most {hi}"
            p.error(f"argument {flag}: must be at least {lo} and {top}, got {v}")


def build_parser() -> ArgumentParser:
    p = ArgumentParser(prog="mutation-simulator",
                       description="See https://github.com/mkpython3/Mutation-Simulator for more information about this program.")
    p.add_argument("infile", type=Path, help="Path of the reference Fasta file")
    p.add_argument("-o", "--output", type=Path, default=D.OUTBASE, dest="outbase",
                   help="Path/Basename for the output files (without file extension)")
    for flags, hlp, default in ((("-w", "--ignore-warnings"), "Silences warnings", D.IGNORE_WARNINGS),
                                (("-c", "--no-color"), "Always disable color", D.NO_COLOR),
                                (("-p", "--no-progress"), "Disable progressbars", D.NO_PROGRESS),
                                (("-q", "--quiet"), "Disable all output except errors", D.QUIET)):
        p.add_argument(*flags, help=hlp, action="store_true", default=default)
    p.add_argument("-v", "--version", action="version", version=f"Mutation-Simulator {__version__}")
    p.add_argument("--seed", type=int, default=None,
                   help="[extension] seed of the counter-based RNG; default: a fresh random seed per run")
    p.add_argument("--device", type=int, default=0, help="[extension] CUDA device index. Default = 0")
    p.add_argument("--bgzip", action="store_true", default=False,
                   help="[extension] write the FASTA and VCF outputs BGZF-compressed (names get .gz); the BEDPE stays plain")
    p.add_argument("--chain", action="store_true", default=False,
                   help="[extension] also write a UCSC chain file from the input to the mutated genome (*_ms.chain, "
                        "*_ms_it.chain for the interchromosomal step; .gz with --bgzip) for liftOver and CrossMap")
    p.add_argument("--ploidy", type=_ploidy, default=D.PLOIDY,
                   help=f"[extension] haplotypes of the simulated sample (1..{MAX_PLOIDY}); >= 2 writes *_ms_h1.fa .. *_ms_hP.fa and a "
                        f"phased *_ms.vcf, and in vcf mode reads the GT of a phased VCF. Default = {D.PLOIDY}")
    p.add_argument("--hom-fraction", type=_fraction, default=D.HOM_FRACTION, dest="hom_fraction",
                   help=f"[extension] probability that a record of a polyploid sample is on every haplotype (homozygous); "
                        f"the others go to a uniformly drawn proper subset. Default = {D.HOM_FRACTION}")
    p.add_argument("--reads", type=float, default=SUPPRESS, metavar="C",
                   help="[extension] also simulate paired-end reads of the mutated sample at mean depth C (each haplotype "
                        "gets C / ploidy) into *_ms_R1.fq and *_ms_R2.fq (.gz with --bgzip), with the truth in every read name")
    for flag, dest, typ, default, _, _, hlp in _READS:
        p.add_argument(flag, dest=dest, default=SUPPRESS, help=f"[extension] with --reads: {hlp}. Default = {default}")

    sub = p.add_subparsers(dest="mode", help="Generate mutations or interchromosomal translocations via RMT or arguments")
    sub.required = True
    a = sub.add_parser("args", help="Use commandline arguments for mutations instead of RMT")
    for short, long_, title, noun in _KINDS:
        a.add_argument(f"-{short}", f"--{long_}", type=float, default=D.RATE, help=f"{title} rate. Default = {D.RATE}")
        if short == "sn":
            a.add_argument("-snb", "--snpblock", type=int, default=D.BLOCK, help=f"Amount of bases blocked after SNP. Default = {D.BLOCK}")
            a.add_argument("-titv", "--transitionstransversions", type=float, default=D.TITV,
                           help=f"Ratio of transitions:transversions likelihood. Default = {D.TITV}")
            continue
        lo, hi = (D.IV_MINLEN, D.IV_MAXLEN) if short == "iv" else (D.MINLEN, D.MAXLEN)
        a.add_argument(f"-{short}min", f"--{long_}minlength", type=int, default=lo, help=f"Minimum length of {_PLURAL[short]}. Default = {lo}")
        a.add_argument(f"-{short}max", f"--{long_}maxlength", type=int, default=hi, help=f"Maximum length of {_PLURAL[short]}. Default = {hi}")
        a.add_argument(f"-{short}b", f"--{long_}block", type=int, default=D.BLOCK, help=f"Amount of bases blocked after {noun}. Default = {D.BLOCK}")
    for flag, long_, what, default in (("-a", "--assembly", "Assembly", D.ASSEMBLY_NAME), ("-s", "--species", "Species", D.SPECIES_NAME),
                                       ("-n", "--sample", "Sample", D.SAMPLE_NAME)):
        a.add_argument(flag, long_, default=default, help=f"{what} name for the VCF file. Default = '{default}'")
    it = sub.add_parser("it", help="Generate interchromosomal translocations via the command line")
    it.add_argument("interchromosomalrate", type=float, help="Rate of interchromosomal translocations")
    rmt = sub.add_parser("rmt", help="Use random mutation table instead of arguments")
    rmt.add_argument("rmtfile", type=Path, help="Path to the RMT file")
    vcf = sub.add_parser("vcf", help="[extension] Apply the mutations of a VCF written by Mutation-Simulator to the Fasta "
                                     "(writes the *_ms.fa it describes and re-emits the VCF)")
    vcf.add_argument("vcffile", type=Path, help="Path to the VCF file (plain, gzip or BGZF)")
    return p


def get_args(argv=None) -> Namespace:
    p = build_parser()
    args = p.parse_args(argv)
    if hasattr(args, "reads"):
        _check_reads(p, args)
    else:                       # the read options mean nothing without --reads
        for _, dest, *_ in _READS:
            if hasattr(args, dest):
                delattr(args, dest)
    if args.quiet:
        args.ignore_warnings = True
        args.no_progress = True
    return add_outfile_names(args)
