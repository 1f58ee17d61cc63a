"""FASTA output.  The GPU produces the complete file image (headers, wrapped lines,
separators: fasta_writer.py:40-65 of the reference is fused into the splice kernel);
this class owns the file handle with the reference's error contract and still offers
the per-base API for user code written against the reference."""
from __future__ import annotations


class FastaWriterError(Exception):
    """Raised when the writer can not write to a file."""


class FastaWriter:
    def __init__(self, fname, bgzip: bool = False):
        """bgzip: write_from_engine writes BGZF (the per-base API below always writes plain text)."""
        self._bgzip = bgzip
        try:
            self._f = open(fname, "w+b")   # read-write: libmutsim_b200 maps the file for its parallel writers
        except OSError as e:
            raise FastaWriterError(f"Cannot write to Fasta file {fname} {e}")
        self._written = 0
        self._bpl = 60

    def __del__(self):
        self.close()

    def close(self):
        if getattr(self, "_f", None) is not None and not self._f.closed:
            self._f.close()

    def write_image(self, image):
        """Write a complete device-built file image (bytes / memoryview / numpy uint8)."""
        self._f.write(memoryview(image))

    def write_from_engine(self, engine, which: int):
        """Stream a device buffer straight into the file (pinned double buffering inside libmutsim_b200)."""
        if self._bgzip:
            from .bgzf import write_from_engine
            return write_from_engine(self._f, engine, which)
        self._f.flush()
        off = self._f.tell()
        n = engine.download_to_fd(which, self._f.fileno(), off)
        self._f.seek(off + n)

    # reference-compatible streaming API
    def set_bpl(self, bpl: int):
        self._bpl = bpl

    def write_header(self, header: str):
        if self._written:
            self._f.write(b"\n")
        self._f.write(b">" + header.encode("latin-1") + b"\n")
        self._written = 0

    def write(self, base: str):
        self.write_multi(base)

    def write_multi(self, bases):
        data = "".join(bases).encode("latin-1") if not isinstance(bases, (bytes, bytearray)) else bytes(bases)
        i = 0
        while i < len(data):
            room = self._bpl - self._written
            chunk = data[i:i + room]
            self._f.write(chunk)
            self._written += len(chunk)
            i += len(chunk)
            if self._written == self._bpl:
                self._f.write(b"\n")
                self._written = 0
