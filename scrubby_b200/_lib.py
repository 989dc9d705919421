"""ctypes binding of libscrubby_gpu.so (include/scrubby_gpu.h).  No CPU fallback: if the
library cannot be built or loaded this module raises, it never substitutes another path."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

STATUS = {
    0: "SGPU_OK", 1: "SGPU_ERR_IO", 2: "SGPU_ERR_NIFFLER", 3: "SGPU_ERR_FASTQ_INVALID_START",
    4: "SGPU_ERR_FASTQ_INVALID_SEPARATOR", 5: "SGPU_ERR_FASTQ_UNEQUAL_LENGTHS",
    6: "SGPU_ERR_FASTQ_UNEXPECTED_END", 7: "SGPU_ERR_FASTQ_UNKNOWN_FORMAT", 8: "SGPU_ERR_RECORD_NAME_UTF8",
    9: "SGPU_ERR_FASTQ_HEADER", 10: "SGPU_ERR_PAF_INTEGER", 11: "SGPU_ERR_WOULD_PANIC",
    12: "SGPU_ERR_KRAKEN_REPORT_READS", 13: "SGPU_ERR_KRAKEN_REPORT_DIRECT", 14: "SGPU_ERR_KRAKEN_REPORT_PARENT",
    15: "SGPU_ERR_FASTA_UNSUPPORTED", 16: "SGPU_ERR_CUDA", 17: "SGPU_ERR_NOMEM", 18: "SGPU_ERR_INVALID_ARG",
    19: "SGPU_ERR_CAPACITY", 20: "SGPU_ERR_KEY_TOO_LONG", 21: "SGPU_ERR_HALO", 22: "SGPU_ERR_SAM_RECORD",
    23: "SGPU_ERR_BAM_RECORD", 24: "SGPU_ERR_PHASE_UNKNOWN", 25: "SGPU_ERR_NOT_SHARDABLE",
}
SGPU_ERR_CAPACITY = 19
SGPU_ERR_HALO = 21
SGPU_ERR_PHASE_UNKNOWN = 24
SGPU_ERR_NOT_SHARDABLE = 25
NEWLINES_UNKNOWN = (1 << 64) - 1


class Counts(C.Structure):
    _fields_ = [
        ("reads_in", C.c_uint64), ("reads_out", C.c_uint64), ("difference", C.c_uint64),
        ("error_record", C.c_uint64), ("crlf", C.c_uint32), ("empty_input", C.c_uint32),
        ("path", C.c_uint32), ("speculated", C.c_uint32), ("own_newlines", C.c_uint64), ("lead_newlines", C.c_uint64),
    ]


class IdSetImage(C.Structure):
    _fields_ = [
        ("d_table", C.c_void_p), ("table_bytes", C.c_uint64), ("d_arena", C.c_void_p),
        ("arena_bytes", C.c_uint64), ("capacity", C.c_uint64), ("count", C.c_uint64), ("has_empty", C.c_uint64),
    ]


# every symbol include/scrubby_gpu.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "sgpu_ctx_create", "sgpu_ctx_destroy", "sgpu_ctx_set_stream", "sgpu_ctx_set_mode", "sgpu_ctx_sync",
    "sgpu_strerror", "sgpu_last_cuda_error", "sgpu_abi_version", "sgpu_ctx_launch_count",
    "sgpu_ctx_set_profiling", "sgpu_ctx_fused_stats",
    "sgpu_idset_from_paf", "sgpu_idset_from_paf_dev", "sgpu_idset_from_sam", "sgpu_idset_from_sam_dev",
    "sgpu_idset_from_txt", "sgpu_idset_from_txt_dev",
    "sgpu_idset_from_reads", "sgpu_idset_from_reads_dev", "sgpu_idset_from_ids", "sgpu_idset_new",
    "sgpu_idset_len", "sgpu_idset_contains", "sgpu_idset_dump", "sgpu_idset_free", "sgpu_free",
    "sgpu_clean_fastq", "sgpu_clean_fastq_dev", "sgpu_clean_fastq_shard_dev", "sgpu_clean_fastq_shard", "sgpu_count_newlines_dev",
    "sgpu_diff", "sgpu_diff_dev", "sgpu_fastq_ids_shard_dev", "sgpu_idset_export", "sgpu_idset_import",
    "sgpu_idset_keys_dev", "sgpu_idset_from_bam", "sgpu_idset_partition_txt_dev", "sgpu_idset_assemble_dev",
    "sgpu_clean_fasta_shard_dev", "sgpu_clean_fasta_shard", "sgpu_fasta_ids_shard_dev",
    "sgpu_fastq_ids_route_shard_dev", "sgpu_fasta_ids_route_shard_dev", "sgpu_idset_probe_lines_dev",
]

_lib = None


def so_path() -> str:
    return _build.SO


def load():
    """Loads (building first if the .so is missing or stale and nvcc is present)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.SO
    if os.path.exists(_build.NVCC):
        path = _build.build()
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing and nvcc is not available: the CUDA extension is required "
            "(there is no CPU fallback); run `python -m scrubby_b200.build`")
    L = C.CDLL(path)
    vp, sz, u64, i32 = C.c_void_p, C.c_size_t, C.c_uint64, C.c_int
    P = C.POINTER
    L.sgpu_ctx_create.argtypes = [i32, P(vp)]
    L.sgpu_ctx_destroy.argtypes = [vp]
    L.sgpu_ctx_destroy.restype = None
    L.sgpu_ctx_set_stream.argtypes = [vp, vp]
    L.sgpu_ctx_set_mode.argtypes = [vp, i32]
    L.sgpu_ctx_sync.argtypes = [vp]
    L.sgpu_strerror.argtypes = [i32]
    L.sgpu_strerror.restype = C.c_char_p
    L.sgpu_last_cuda_error.restype = C.c_char_p
    L.sgpu_abi_version.restype = i32
    L.sgpu_ctx_launch_count.argtypes = [vp]
    L.sgpu_ctx_launch_count.restype = u64
    L.sgpu_ctx_set_profiling.argtypes = [vp, i32]
    L.sgpu_ctx_fused_stats.argtypes = [vp, P(C.c_double), P(u64), P(u64)]
    for name in ("sgpu_idset_from_paf", "sgpu_idset_from_paf_dev", "sgpu_idset_from_sam", "sgpu_idset_from_sam_dev",
                 "sgpu_idset_from_bam"):
        getattr(L, name).argtypes = [vp, vp, sz, u64, C.c_double, C.c_uint8, P(vp), P(u64)]
    for name in ("sgpu_idset_from_txt", "sgpu_idset_from_txt_dev"):
        getattr(L, name).argtypes = [vp, vp, sz, P(vp), P(u64)]
    for name in ("sgpu_idset_from_reads", "sgpu_idset_from_reads_dev"):
        getattr(L, name).argtypes = [vp, vp, sz, i32, P(C.c_char_p), P(sz), sz, P(vp), P(u64)]
    L.sgpu_idset_from_ids.argtypes = [vp, P(C.c_char_p), P(sz), sz, P(vp)]
    L.sgpu_idset_new.argtypes = [vp, P(vp)]
    L.sgpu_idset_len.argtypes = [vp]
    L.sgpu_idset_len.restype = u64
    L.sgpu_idset_contains.argtypes = [vp, vp, C.c_char_p, sz, P(i32)]
    L.sgpu_idset_dump.argtypes = [vp, vp, P(vp), P(sz)]
    L.sgpu_idset_free.argtypes = [vp]
    L.sgpu_idset_free.restype = None
    L.sgpu_free.argtypes = [vp]
    L.sgpu_free.restype = None
    for name in ("sgpu_clean_fastq", "sgpu_clean_fastq_dev"):
        getattr(L, name).argtypes = [vp, vp, vp, sz, i32, vp, sz, P(sz), vp, sz, P(sz), P(Counts)]
    L.sgpu_clean_fastq_shard_dev.argtypes = [vp, vp, vp, sz, sz, u64, i32, i32, i32, i32, vp, sz, P(sz), vp, sz,
                                             P(sz), P(Counts)]
    L.sgpu_clean_fastq_shard.argtypes = L.sgpu_clean_fastq_shard_dev.argtypes
    L.sgpu_count_newlines_dev.argtypes = [vp, vp, sz, P(u64)]
    L.sgpu_fastq_ids_shard_dev.argtypes = [vp, vp, vp, sz, sz, u64, i32, i32, vp, P(Counts)]
    L.sgpu_clean_fasta_shard_dev.argtypes = [vp, vp, vp, sz, sz, i32, i32, i32, i32, vp, sz, P(sz), vp, sz, P(sz),
                                             P(Counts), P(i32)]
    L.sgpu_clean_fasta_shard.argtypes = L.sgpu_clean_fasta_shard_dev.argtypes
    L.sgpu_fasta_ids_shard_dev.argtypes = [vp, vp, vp, sz, sz, i32, i32, vp, P(Counts)]
    L.sgpu_fastq_ids_route_shard_dev.argtypes = [vp, vp, sz, sz, u64, i32, i32, i32, vp, sz, P(sz), P(u64), P(u64),
                                                 P(Counts)]
    L.sgpu_fasta_ids_route_shard_dev.argtypes = [vp, vp, sz, sz, i32, i32, i32, vp, sz, P(sz), P(u64), P(u64), P(Counts)]
    L.sgpu_idset_probe_lines_dev.argtypes = [vp, vp, vp, sz, vp, P(Counts)]
    for name in ("sgpu_diff", "sgpu_diff_dev"):
        getattr(L, name).argtypes = [vp, vp, sz, vp, sz, P(Counts), P(vp)]
    L.sgpu_idset_export.argtypes = [vp, P(IdSetImage)]
    L.sgpu_idset_import.argtypes = [vp, P(IdSetImage), P(vp)]
    L.sgpu_idset_keys_dev.argtypes = [vp, vp, vp, sz, P(sz)]
    L.sgpu_idset_partition_txt_dev.argtypes = [vp, vp, sz, sz, i32, i32, C.c_uint32, vp, sz, vp, P(u64), P(u64)]
    L.sgpu_idset_assemble_dev.argtypes = [vp, i32, P(vp), P(vp), C.c_uint32, P(vp)]
    _lib = L
    return L
