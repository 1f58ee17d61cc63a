"""ctypes binding of libmutsim_b200.so (include/mutsim_b200.h).

There is no CPU fallback: if the shared library has not been built, or no CUDA
device is present, the calls below raise.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libmutsim_b200.so"


class MutSimError(RuntimeError):
    """A libmutsim_b200 call failed; ``code`` is the MS_ERR_* status."""

    def __init__(self, code: int, message: str):
        super().__init__(f"libmutsim_b200 error {code}: {message}")
        self.code = code
        self.message = message


class MsRange(C.Structure):
    _fields_ = [("contig", C.c_uint32), ("start", C.c_uint32), ("stop", C.c_uint32), ("k", C.c_uint32),
                ("limit", C.c_int64), ("cdf", C.c_double * 7), ("minlen", C.c_int32 * 7), ("maxlen", C.c_int32 * 7)]


class MsStats(C.Structure):
    _fields_ = [("n_candidates", C.c_int64), ("n_accepted", C.c_int64), ("n_records", C.c_int64),
                ("lit_bytes", C.c_int64), ("fasta_bytes", C.c_int64), ("vcf_bytes", C.c_int64),
                ("kernel_launches", C.c_int64), ("counts", C.c_int64 * 8), ("stage_ms", C.c_float * 16)]


MS_OK, MS_ERR_CUDA, MS_ERR_ARG, MS_ERR_STATE, MS_ERR_SAMPLE, MS_ERR_OVERLAP, MS_ERR_LIMIT, MS_ERR_INTERNAL = range(8)

_P, _I64, _I32, _U64, _U32 = C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_uint32

# name -> (restype, argtypes); every symbol include/mutsim_b200.h declares
PROTOTYPES = {
    "ms_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "ms_destroy": (C.c_int, [_P]),
    "ms_last_error": (C.c_char_p, [_P]),
    "ms_abi_version": (C.c_int, []),
    "ms_set_stream": (C.c_int, [_P, _P]),
    "ms_synchronize": (C.c_int, [_P]),
    "ms_genome_upload": (C.c_int, [_P, _P, _I64, _I32, _P, _P, _P, _P, _P, _P, _P]),
    "ms_genome_adopt": (C.c_int, [_P, _P, _I64, _I32, _P, _P, _P, _P, _P, _P, _P]),
    "ms_genome_synth": (C.c_int, [_P, _U64, _I32, _P, _P, _P, C.c_double, _I64, _P, _P, _P, _P]),
    "ms_hash_ranges": (C.c_int, [_P, C.c_int, _I32, _P, _P, _P]),
    "ms_genome_download": (C.c_int, [_P, _P, _I64]),
    "ms_genome_reserve": (C.c_int, [_P, _I64]),
    "ms_genome_export": (C.c_int, [_P, _P, _P]),
    "ms_peer_open": (C.c_int, [_P, _P, _I64, _P]),
    "ms_peer_pull": (C.c_int, [_P, C.c_int32, _P, _P, _P]),
    "ms_peer_close": (C.c_int, [_P]),
    "ms_genome_adopt_output": (C.c_int, [_P]),
    "ms_fasta_ingest_fd": (C.c_int, [_P, C.c_int, _I64, _P, _P]),
    "ms_fasta_ingest_ranges": (C.c_int, [_P, C.c_int, _I32, _P, _P, _P, _P]),
    "ms_fasta_index": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I64]),
    "ms_fasta_commit": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "ms_genome_read": (C.c_int, [_P, _I64, _I64, _P]),
    "ms_genome_subset": (C.c_int, [_P, _P, C.c_int32]),
    "ms_genome_declare": (C.c_int, [_P, _I64, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
    "ms_mutate_streamed": (C.c_int, [_P, C.c_uint64, _P, _P, _I64, _P, _I64, _P, _P, _I64]),
    "ms_contig_layout": (C.c_int, [_P, _P, _P, _P, _P]),
    "ms_contig_records": (C.c_int, [_P, _P]),
    "ms_sample_positions": (C.c_int, [_P, _U64, _I32, _P, _P, _P, _P, _I32, _P]),
    "ms_set_ranges": (C.c_int, [_P, _P, _I32, _P, _I32, C.c_double]),
    "ms_sample": (C.c_int, [_P, _U64]),
    "ms_load_records": (C.c_int, [_P, _P, _I64, _P, _I64]),
    "ms_load_vcf": (C.c_int, [_P, _P, _I64, _I32, C.POINTER(_I32), C.POINTER(_I64)]),
    "ms_apply": (C.c_int, [_P, C.POINTER(_I64), C.POINTER(_I64)]),
    "ms_apply_window": (C.c_int, [_P, _I32, _I32, _P]),
    "ms_download": (C.c_int, [_P, C.c_int, _P, _I64, C.POINTER(_I64)]),
    "ms_device_ptr": (C.c_int, [_P, C.c_int, C.POINTER(_P), C.POINTER(_I64)]),
    "ms_download_to_fd": (C.c_int, [_P, C.c_int, _I64, _I64, C.c_int, _I64]),
    "ms_contig_out_len": (C.c_int, [_P, _P]),
    "ms_it_breakpoints": (C.c_int, [_P, _U64, _I32, _P, _P, _P, _P, _P]),
    "ms_get_stats": (C.c_int, [_P, C.POINTER(MsStats)]),
    "ms_stage_name": (C.c_char_p, [C.c_int]),
    "ms_debug_candidates": (C.c_int, [_P, _I64, _P, _P, _P, _P, C.POINTER(_I64)]),
    "ms_bgzf_compress": (C.c_int, [_P, C.c_int, _I32, _P, _P, _P, _P, _P, C.POINTER(_I64)]),
    "ms_bgzf_compress_host": (C.c_int, [_P, _P, _I64, _P, _I64, C.POINTER(_I64)]),
}

_lib = None


def load() -> C.CDLL:
    """Load the CUDA library (built in-tree by mutation_simulator_b200.build)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise MutSimError(MS_ERR_STATE, f"{LIB_PATH} not found. Build it with "
                              "`python -m mutation_simulator_b200.build` (needs nvcc); there is no CPU fallback")
        lib = C.CDLL(str(LIB_PATH))
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
