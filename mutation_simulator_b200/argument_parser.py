"""Command line of ``mutation-simulator`` — flag for flag the reference's
(argument_parser.py:31-240) plus three extensions that default to the reference's
behaviour: ``--seed`` (reproducible runs; default: a fresh random seed, like the
reference's unseeded RNGs), ``--device`` (CUDA device index) and ``--bgzip``
(BGZF-compressed FASTA and VCF output, encoded on the GPU), and the ``vcf`` mode
(replay a VCF the reference or this package wrote onto the same FASTA).

The option table below drives argparse; the derived output names follow
argument_parser.py:14-28."""
from __future__ import annotations

from argparse import ArgumentParser, Namespace
from pathlib import Path

from ._version import __version__
from .defaults import Defaults as D

# (short, long, dest kind, type, default, help) for the `args` sub-command, in the reference's order
_KINDS = [("sn", "snp", "SNP", "SNP"), ("in", "insert", "Insert", "insert"), ("de", "deletion", "Deletion", "deletion"),
          ("iv", "inversion", "Inversion", "inversion"), ("du", "duplication", "Duplication", "duplication"),
          ("tl", "translocation", "Translocation", "translocations")]
_PLURAL = {"in": "inserts", "de": "deletions", "iv": "inversion", "du": "duplications", "tl": "translocations"}


def add_outfile_names(args: Namespace) -> Namespace:
    """outfasta / outfastait / outvcf / outbedpe from the output base."""
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
    if getattr(args, "bgzip", False):      # after the derivation: *_it and .bedpe keep their names
        for k in ("outfasta", "outfastait", "outvcf"):
            p = getattr(args, k)
            setattr(args, k, p.with_name(p.name + ".gz"))
    return args


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
    args = build_parser().parse_args(argv)
    if args.quiet:
        args.ignore_warnings = True
        args.no_progress = True
    return add_outfile_names(args)
