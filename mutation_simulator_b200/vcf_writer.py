"""VCF output: header on the host (vcf_writer.py:74-116), record lines from the GPU."""
from __future__ import annotations

from datetime import datetime

_FIXED_TAIL = (
    '##INFO=<ID=SVTYPE,Number=1,Type=String,Description="Type of structural variant">\n'
    '##INFO=<ID=END,Number=1,Type=Integer,Description="End position of the variant described in this record">\n'
    '##INFO=<ID=SVLEN,Number=.,Type=Integer,Description="Difference in length between REF and ALT alleles">\n'
    '##ALT=<ID=INS,Description="Insert">\n'
    '##ALT=<ID=DEL,Description="Deletion">\n'
    '##ALT=<ID=DUP,Description="Duplication">\n'
    '##ALT=<ID=INV,Description="Inversion">\n'
    '##ALT=<ID=DEL:ME,Description="Deletion of mobile element">\n'
    '##ALT=<ID=INS:ME,Description="Insertion of mobile element">\n'
    '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n')


class VcfWriterError(Exception):
    """Raised when the writer can not write to a file."""


class VcfRecord:
    """Field holder kept for API compatibility (vcf_writer.py:16-52)."""

    def __init__(self, svtype="", start=0, end=0, len=0, ref="", alt=""):
        self.svtype, self.start, self.end, self.len, self.ref, self.alt = svtype, start, end, len, ref, alt

    def __repr__(self):
        return f"{self.svtype} {self.start} {self.end} {self.len} {self.ref} {self.alt}"

    @property
    def info(self):
        return "." if self.svtype == "sn" else f"SVTYPE={self.svtype};END={self.end};SVLEN={self.len}"


def header_text(input_fasta, contigs, assembly_name, species_name, sample_name, now=None) -> str:
    """contigs: iterable of (name, length).  The date is un-padded YYYYMD like the reference's (SURVEY.md Q7)."""
    now = now or datetime.now()
    out = ["##fileformat=VCFv4.3\n", f"##filedate={now.year}{now.month}{now.day}\n", "##source=Mutation-Simulator\n",
           f"##reference={input_fasta}\n"]
    out += [f'##contig=<ID={n},length={ln},assembly={assembly_name},species="{species_name}">\n' for n, ln in contigs]
    out.append(_FIXED_TAIL)
    out.append(f"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t{sample_name}\n")
    return "".join(out)


class VcfWriter:
    def __init__(self, fname, bgzip: bool = False):
        """bgzip: the header and write_from_engine's body are written as BGZF members (write / write_body stay plain)."""
        self._bgzip = bgzip
        try:
            self._f = open(fname, "w+b")   # read-write: libmutsim_b200 maps the file for its parallel writers
        except OSError as e:
            raise VcfWriterError(f"Cannot write to VCF file {fname} {e}")

    def __del__(self):
        self.close()

    def close(self):
        if getattr(self, "_f", None) is not None and not self._f.closed:
            self._f.close()

    def write_header(self, input_fasta, fasta, assembly_name, species_name, sample_name):
        names = fasta.keys()
        head = header_text(input_fasta, [(fasta[n].name, len(fasta[n])) for n in names], assembly_name, species_name,
                           sample_name).encode("latin-1")
        if self._bgzip:
            from .bgzf import compress_host
            head = compress_host(head)
        self._f.write(head)

    def write_body(self, body):
        self._f.write(memoryview(body))

    def write_from_engine(self, engine, which: int):
        if self._bgzip:
            from .bgzf import write_from_engine
            return write_from_engine(self._f, engine, which)
        self._f.flush()
        off = self._f.tell()
        n = engine.download_to_fd(which, self._f.fileno(), off)
        self._f.seek(off + n)

    def write(self, record: VcfRecord, seq_name: str):
        if record.ref != record.alt:
            self._f.write(f"{seq_name}\t{record.start}\t.\t{record.ref}\t{record.alt}\t.\t.\t{record.info}\tGT\t1\n".encode("latin-1"))
