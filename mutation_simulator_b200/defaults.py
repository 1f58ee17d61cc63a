"""Default settings (values of defaults.py:7-42 of the reference)."""
from pathlib import Path
from sys import stderr, stdout

from .mut_types import MutType

_TTY = stdout.isatty() and stderr.isatty()


class Defaults:
    OUTBASE = Path(".")
    IGNORE_WARNINGS = False
    QUIET = False
    NO_COLOR = not _TTY
    NO_PROGRESS = not _TTY
    SPECIES_NAME = ASSEMBLY_NAME = SAMPLE_NAME = "Unknown"
    TITV = 1
    RATE = 0
    BLOCK = 1
    MINLEN, MAXLEN = 1, 2
    IV_MINLEN, IV_MAXLEN = 2, 3
    # extensions: one haploid sample; for a polyploid one, about the het:hom-alt ratio of 1.5-2 usually seen in one
    # human sample (a documented default, not a measured claim)
    PLOIDY = 1
    HOM_FRACTION = 0.35
    # --reads: a common short-read shape (2 x 150 bp, 500 bp inserts); documented choices, not measured claims
    READ_LENGTH = 150
    FRAGMENT_MEAN = 500
    FRAGMENT_SD = 50
    READ_ERROR_RATE = 0.001


Defaults.MUT_BLOCK = {t: Defaults.BLOCK for t in (MutType.SN, MutType.IN, MutType.DE, MutType.IV, MutType.DU, MutType.TL, MutType.TLI)}
