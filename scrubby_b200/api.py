"""Thin Python harness over the C ABI (include/scrubby_gpu.h) for tests, bench.py and the
torch.distributed driver.  The drop-in host (CLI, report writer, taxon state machine) is the
C++ code under scrubby_b200/host/; this module only moves bytes and handles.

Every call goes to libscrubby_gpu.so -- there is no CPU path here.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

from . import _lib


class ScrubbyGpuError(RuntimeError):
    def __init__(self, status: int, index: int = 0, what: str = ""):
        L = _lib.load()
        msg = L.sgpu_strerror(status).decode()
        if status == 16:
            msg += ": " + L.sgpu_last_cuda_error().decode()
        super().__init__(f"{_lib.STATUS.get(status, status)} ({msg}) {what} at record/line {index}")
        self.status = status
        self.code = status
        self.index = index


def _check(status: int, index: int = 0, what: str = ""):
    if status != 0:
        raise ScrubbyGpuError(status, index, what)


def _host_ptr(buf):
    """(address, nbytes, keepalive) of bytes / bytearray / numpy / torch CPU uint8"""
    if isinstance(buf, (bytes, bytearray, memoryview)):
        b = bytes(buf) if not isinstance(buf, bytes) else buf
        arr = C.create_string_buffer(b, len(b)) if len(b) else C.create_string_buffer(1)
        return C.cast(arr, C.c_void_p), len(b), arr
    if hasattr(buf, "data_ptr"):  # torch tensor on the CPU
        assert buf.device.type == "cpu" and buf.is_contiguous()
        return C.c_void_p(buf.data_ptr()), buf.numel() * buf.element_size(), buf
    import numpy as np

    a = np.ascontiguousarray(buf, dtype=np.uint8)
    return C.c_void_p(a.ctypes.data), a.size, a


def _dev_ptr(t):
    assert t.is_cuda and t.is_contiguous(), "device tensor expected"
    return C.c_void_p(t.data_ptr()), t.numel() * t.element_size()


class Context:
    """sgpu_ctx: one per device / per host thread."""

    def __init__(self, device: int = 0, stream="torch"):
        """stream: "torch" (default) enqueues on torch's current stream of `device`, so work is ordered
        with the torch ops that produced the tensors; "own" uses a private non-blocking stream; a
        torch.cuda.Stream / raw cudaStream_t is used as given."""
        self.L = _lib.load()
        self.h = C.c_void_p()
        _check(self.L.sgpu_ctx_create(device, C.byref(self.h)), what="sgpu_ctx_create")
        self.device = device
        if stream == "torch":
            import torch

            self.set_stream(torch.cuda.current_stream(device))
        elif stream != "own" and stream is not None:
            self.set_stream(stream)

    def set_stream(self, stream):
        """stream: torch.cuda.Stream, raw cudaStream_t int, or None for an own stream.  torch's default
        stream has handle 0; it is passed as cudaStreamLegacy (0x1), which names the same stream."""
        if stream is None:
            _check(self.L.sgpu_ctx_set_stream(self.h, None))
            return
        raw = getattr(stream, "cuda_stream", stream)
        _check(self.L.sgpu_ctx_set_stream(self.h, C.c_void_p(raw if raw else 1)))

    def set_mode(self, mode: int):
        _check(self.L.sgpu_ctx_set_mode(self.h, mode))

    def sync(self):
        _check(self.L.sgpu_ctx_sync(self.h))

    def set_profiling(self, on: bool):
        _check(self.L.sgpu_ctx_set_profiling(self.h, int(on)))

    def fused_stats(self):
        """(device ms, launches, algorithmic bytes) of the fused-kernel launches since the last call"""
        ms, n, b = C.c_double(), C.c_uint64(), C.c_uint64()
        _check(self.L.sgpu_ctx_fused_stats(self.h, C.byref(ms), C.byref(n), C.byref(b)))
        return ms.value, int(n.value), int(b.value)

    @property
    def launches(self) -> int:
        return int(self.L.sgpu_ctx_launch_count(self.h))

    def close(self):
        if self.h:
            self.L.sgpu_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class IdSet:
    """sgpu_idset: the HashSet<String> of read ids, resident in HBM."""

    def __init__(self, ctx: Context, handle):
        self.ctx = ctx
        self.h = handle if isinstance(handle, C.c_void_p) else C.c_void_p(handle)

    # -- constructors mirroring the reference's evidence parsers ---------------------------
    @classmethod
    def empty(cls, ctx):
        h = C.c_void_p()
        _check(ctx.L.sgpu_idset_new(ctx.h, C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def from_ids(cls, ctx, ids):
        bs = [i.encode() if isinstance(i, str) else bytes(i) for i in ids]
        arr = (C.c_char_p * max(1, len(bs)))(*bs)
        lens = (C.c_size_t * max(1, len(bs)))(*[len(b) for b in bs])
        h = C.c_void_p()
        _check(ctx.L.sgpu_idset_from_ids(ctx.h, arr, lens, len(bs), C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def from_paf(cls, ctx, buf, min_len=0, min_cov=0.0, min_mapq=0):
        """ReadAlignment::from_paf, alignment.rs:84-114"""
        h, err = C.c_void_p(), C.c_uint64()
        if hasattr(buf, "is_cuda") and buf.is_cuda:
            p, n = _dev_ptr(buf)
            rc = ctx.L.sgpu_idset_from_paf_dev(ctx.h, p, n, min_len, min_cov, min_mapq, C.byref(h), C.byref(err))
        else:
            p, n, keep = _host_ptr(buf)
            rc = ctx.L.sgpu_idset_from_paf(ctx.h, p, n, min_len, min_cov, min_mapq, C.byref(h), C.byref(err))
        _check(rc, err.value, "from_paf")
        return cls(ctx, h)

    @classmethod
    def from_sam(cls, ctx, buf, min_len=0, min_cov=0.0, min_mapq=0):
        """ReadAlignment::from_bam, alignment.rs:117-146, for text SAM"""
        h, err = C.c_void_p(), C.c_uint64()
        if hasattr(buf, "is_cuda") and buf.is_cuda:
            p, n = _dev_ptr(buf)
            rc = ctx.L.sgpu_idset_from_sam_dev(ctx.h, p, n, min_len, min_cov, min_mapq, C.byref(h), C.byref(err))
        else:
            p, n, keep = _host_ptr(buf)
            rc = ctx.L.sgpu_idset_from_sam(ctx.h, p, n, min_len, min_cov, min_mapq, C.byref(h), C.byref(err))
        _check(rc, err.value, "from_sam")
        return cls(ctx, h)

    @classmethod
    def from_bam(cls, ctx, buf, min_len=0, min_cov=0.0, min_mapq=0):
        """ReadAlignment::from_bam, alignment.rs:117-146, for binary BAM: `buf` = the BGZF-decompressed stream (host)"""
        h, err = C.c_void_p(), C.c_uint64()
        p, n, keep = _host_ptr(buf)
        rc = ctx.L.sgpu_idset_from_bam(ctx.h, p, n, min_len, min_cov, min_mapq, C.byref(h), C.byref(err))
        _check(rc, err.value, "from_bam")
        return cls(ctx, h)

    @classmethod
    def from_txt(cls, ctx, buf):
        """ReadAlignment::from_txt, alignment.rs:60-82"""
        h, err = C.c_void_p(), C.c_uint64()
        if hasattr(buf, "is_cuda") and buf.is_cuda:
            p, n = _dev_ptr(buf)
            rc = ctx.L.sgpu_idset_from_txt_dev(ctx.h, p, n, C.byref(h), C.byref(err))
        else:
            p, n, keep = _host_ptr(buf)
            rc = ctx.L.sgpu_idset_from_txt(ctx.h, p, n, C.byref(h), C.byref(err))
        _check(rc, err.value, "from_txt")
        return cls(ctx, h)

    @classmethod
    def from_reads(cls, ctx, buf, style: int, taxids):
        """get_taxid_reads_kraken (style 0) / get_taxid_reads_metabuli (style 1), classifier.rs:270-328"""
        bs = [t.encode() if isinstance(t, str) else bytes(t) for t in taxids]
        arr = (C.c_char_p * max(1, len(bs)))(*bs)
        lens = (C.c_size_t * max(1, len(bs)))(*[len(b) for b in bs])
        h, err = C.c_void_p(), C.c_uint64()
        if hasattr(buf, "is_cuda") and buf.is_cuda:
            p, n = _dev_ptr(buf)
            rc = ctx.L.sgpu_idset_from_reads_dev(ctx.h, p, n, style, arr, lens, len(bs), C.byref(h), C.byref(err))
        else:
            p, n, keep = _host_ptr(buf)
            rc = ctx.L.sgpu_idset_from_reads(ctx.h, p, n, style, arr, lens, len(bs), C.byref(h), C.byref(err))
        _check(rc, err.value, "from_reads")
        return cls(ctx, h)

    # -- HashSet surface ----------------------------------------------------------------------
    def __len__(self):
        return int(self.ctx.L.sgpu_idset_len(self.h))

    def __contains__(self, key):
        b = key.encode() if isinstance(key, str) else bytes(key)
        found = C.c_int()
        _check(self.ctx.L.sgpu_idset_contains(self.ctx.h, self.h, b, len(b), C.byref(found)))
        return bool(found.value)

    def sorted_ids(self) -> list[bytes]:
        out, n = C.c_void_p(), C.c_size_t()
        _check(self.ctx.L.sgpu_idset_dump(self.ctx.h, self.h, C.byref(out), C.byref(n)))
        raw = C.string_at(out, n.value)
        self.ctx.L.sgpu_free(out)
        return raw.split(b"\n")[:-1] if raw else []

    def keys_dev(self):
        """the keys as an unsorted "id\\n" list in a device uint8 tensor (sgpu_idset_keys_dev)"""
        import torch

        n = C.c_size_t()
        rc = self.ctx.L.sgpu_idset_keys_dev(self.ctx.h, self.h, None, 0, C.byref(n))
        if rc not in (0, _lib.SGPU_ERR_CAPACITY):
            _check(rc, 0, "idset_keys_dev")
        out = torch.empty(n.value, dtype=torch.uint8, device=torch.device("cuda", self.ctx.device))
        if n.value:
            _check(self.ctx.L.sgpu_idset_keys_dev(self.ctx.h, self.h, C.c_void_p(out.data_ptr()), n.value, C.byref(n)),
                   0, "idset_keys_dev")
        return out

    def image(self) -> _lib.IdSetImage:
        img = _lib.IdSetImage()
        _check(self.ctx.L.sgpu_idset_export(self.h, C.byref(img)))
        return img

    @classmethod
    def from_image(cls, ctx, img):
        h = C.c_void_p()
        _check(ctx.L.sgpu_idset_import(ctx.h, C.byref(img), C.byref(h)))
        return cls(ctx, h)

    def free(self):
        if self.h:
            self.ctx.L.sgpu_idset_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


@dataclass
class CleanResult:
    written: bytes
    other: bytes
    reads_in: int
    reads_out: int
    crlf: bool
    empty_input: bool
    path: int
    error: int = 0
    error_record: int = 0


def clean_fastq(ctx: Context, ids: IdSet, buf, reverse: bool = False, want_other: bool = True,
                raise_on_error: bool = True) -> CleanResult:
    """FastqCleaner::clean_reads (cleaner.rs:731-760) on HOST bytes, copies included."""
    import numpy as np

    p, n, keep = _host_ptr(buf)
    cap = 2 * n + 64
    o1 = np.empty(cap, dtype=np.uint8)
    o2 = np.empty(cap if want_other else 1, dtype=np.uint8)
    n1, n2, c = C.c_size_t(), C.c_size_t(), _lib.Counts()
    rc = ctx.L.sgpu_clean_fastq(ctx.h, ids.h, p, n, int(reverse), o1.ctypes.data, cap, C.byref(n1),
                                o2.ctypes.data if want_other else None, cap if want_other else 0, C.byref(n2),
                                C.byref(c))
    if rc and (raise_on_error or rc >= 16):
        raise ScrubbyGpuError(rc, c.error_record, "clean_fastq")
    return CleanResult(o1[: n1.value].tobytes(), o2[: n2.value].tobytes() if want_other else b"", c.reads_in,
                       c.reads_out, bool(c.crlf), bool(c.empty_input), c.path, rc, c.error_record)


@dataclass
class DevCleanResult:
    n_written: int
    n_other: int
    reads_in: int
    reads_out: int
    crlf: bool
    empty_input: bool
    path: int
    status: int = 0          # 0, or SGPU_ERR_PHASE_UNKNOWN from a speculative shard call (nothing was produced)
    speculated: bool = False
    own_newlines: int = 0    # speculative shards: newlines of the owned range / before the first produced record
    lead_newlines: int = 0


def clean_fastq_dev(ctx: Context, ids: IdSet, d_in, n_in: int, d_out, d_other=None, reverse: bool = False
                    ) -> DevCleanResult:
    """same on device tensors (uint8, 16-byte aligned); outputs land in d_out / d_other"""
    n1, n2, c = C.c_size_t(), C.c_size_t(), _lib.Counts()
    rc = ctx.L.sgpu_clean_fastq_dev(
        ctx.h, ids.h, C.c_void_p(d_in.data_ptr()), n_in, int(reverse), C.c_void_p(d_out.data_ptr()), d_out.numel(),
        C.byref(n1), C.c_void_p(d_other.data_ptr()) if d_other is not None else None,
        d_other.numel() if d_other is not None else 0, C.byref(n2), C.byref(c))
    _check(rc, c.error_record, "clean_fastq_dev")
    return DevCleanResult(n1.value, n2.value, c.reads_in, c.reads_out, bool(c.crlf), bool(c.empty_input), c.path)


def clean_fastq_shard_dev(ctx: Context, ids: IdSet, d_in, n_in: int, own_len: int, newlines_before, is_first: bool,
                          is_last: bool, crlf, d_out, d_other=None, reverse: bool = False) -> DevCleanResult:
    """sgpu_clean_fastq_shard_dev.  newlines_before=None / crlf=None: not exchanged yet -- the shard speculates its line
    phase (one pass, no newline count before it); the result then carries own_newlines / lead_newlines for the caller's
    check, or status == SGPU_ERR_PHASE_UNKNOWN when the exact protocol has to take over."""
    n1, n2, c = C.c_size_t(), C.c_size_t(), _lib.Counts()
    nb = _lib.NEWLINES_UNKNOWN if (newlines_before is None and not is_first) else int(newlines_before or 0)
    rc = ctx.L.sgpu_clean_fastq_shard_dev(
        ctx.h, ids.h, C.c_void_p(d_in.data_ptr()), n_in, own_len, nb, int(is_first), int(is_last),
        -1 if crlf is None else int(crlf), int(reverse), C.c_void_p(d_out.data_ptr()), d_out.numel(), C.byref(n1),
        C.c_void_p(d_other.data_ptr()) if d_other is not None else None,
        d_other.numel() if d_other is not None else 0, C.byref(n2), C.byref(c))
    if rc != _lib.SGPU_ERR_PHASE_UNKNOWN:
        _check(rc, c.error_record, "clean_fastq_shard_dev")
    return DevCleanResult(n1.value, n2.value, c.reads_in, c.reads_out, bool(c.crlf), bool(c.empty_input), c.path, rc,
                          bool(c.speculated), c.own_newlines, c.lead_newlines)


def clean_fastq_shard_host(ctx: Context, ids: IdSet, h_in, n_in: int, own_len: int, newlines_before, is_first: bool,
                           is_last: bool, crlf, h_out, h_other=None, reverse: bool = False) -> DevCleanResult:
    """sgpu_clean_fastq_shard: the shard contract of clean_fastq_shard_dev on caller-owned HOST tensors (pinned for full
    PCIe rate); the chunked H2D / kernel / D2H pipeline runs inside the call"""
    n1, n2, c = C.c_size_t(), C.c_size_t(), _lib.Counts()
    nb = _lib.NEWLINES_UNKNOWN if (newlines_before is None and not is_first) else int(newlines_before or 0)
    rc = ctx.L.sgpu_clean_fastq_shard(
        ctx.h, ids.h, C.c_void_p(h_in.data_ptr()), n_in, own_len, nb, int(is_first), int(is_last),
        -1 if crlf is None else int(crlf), int(reverse), C.c_void_p(h_out.data_ptr()), h_out.numel(), C.byref(n1),
        C.c_void_p(h_other.data_ptr()) if h_other is not None else None,
        h_other.numel() if h_other is not None else 0, C.byref(n2), C.byref(c))
    if rc != _lib.SGPU_ERR_PHASE_UNKNOWN:
        _check(rc, c.error_record, "clean_fastq_shard")
    return DevCleanResult(n1.value, n2.value, c.reads_in, c.reads_out, bool(c.crlf), bool(c.empty_input), c.path, rc,
                          bool(c.speculated), c.own_newlines, c.lead_newlines)


@dataclass
class FastaShardResult:
    n_written: int
    n_other: int
    reads_in: int
    reads_out: int
    crlf: bool          # the line ending this shard wrote with
    empty_input: bool
    le_own: int         # the decision of the shard's own first deciding record: -1 none, 0 LF, 1 CRLF
    path: int = 3
    error: int = 0      # a parse error (raise_on_error=False): its class; the records before it were produced
    error_record: int = 0


def _fasta_shard(fn, what, ctx, ids, buf, n_in, own_len, is_first, is_last, le_before, out, other, reverse,
                 raise_on_error):
    n1, n2, c, le = C.c_size_t(), C.c_size_t(), _lib.Counts(), C.c_int()
    rc = fn(ctx.h, ids.h, C.c_void_p(buf.data_ptr()), n_in, own_len, int(is_first), int(is_last), int(le_before),
            int(reverse), C.c_void_p(out.data_ptr()), out.numel(), C.byref(n1),
            C.c_void_p(other.data_ptr()) if other is not None else None, other.numel() if other is not None else 0,
            C.byref(n2), C.byref(c), C.byref(le))
    if rc and (raise_on_error or rc >= 16):
        raise ScrubbyGpuError(rc, c.error_record, what)
    return FastaShardResult(n1.value, n2.value, c.reads_in, c.reads_out, bool(c.crlf), bool(c.empty_input), le.value,
                            c.path, rc, c.error_record)


def clean_fasta_shard_dev(ctx: Context, ids: IdSet, d_in, n_in: int, own_len: int, is_first: bool, is_last: bool,
                          le_before: int, d_out, d_other=None, reverse: bool = False,
                          raise_on_error: bool = True) -> FastaShardResult:
    """sgpu_clean_fasta_shard_dev: the FASTA records that start in the owned range of a device buffer (uint8, 16-byte
    aligned).  le_before: -1 undecided, 0 / 1 LF / CRLF decided by an earlier shard."""
    return _fasta_shard(ctx.L.sgpu_clean_fasta_shard_dev, "clean_fasta_shard_dev", ctx, ids, d_in, n_in, own_len,
                        is_first, is_last, le_before, d_out, d_other, reverse, raise_on_error)


def clean_fasta_shard_host(ctx: Context, ids: IdSet, h_in, n_in: int, own_len: int, is_first: bool, is_last: bool,
                           le_before: int, h_out, h_other=None, reverse: bool = False,
                           raise_on_error: bool = True) -> FastaShardResult:
    """sgpu_clean_fasta_shard: the same contract on caller-owned HOST tensors (pinned for full PCIe rate); the chunked
    H2D / kernel / D2H pipeline runs inside the call"""
    return _fasta_shard(ctx.L.sgpu_clean_fasta_shard, "clean_fasta_shard", ctx, ids, h_in, n_in, own_len, is_first,
                        is_last, le_before, h_out, h_other, reverse, raise_on_error)


def fasta_ids_shard_dev(ctx: Context, probe, d_buf, n_buf: int, own_len: int, is_first: bool, is_last: bool,
                        into: IdSet):
    """one shard of ReadDifference::get_difference's loops over a FASTA file: ids of the owned records absent from
    `probe` (None: all) go into `into`; returns (records, picked records)"""
    c = _lib.Counts()
    rc = ctx.L.sgpu_fasta_ids_shard_dev(ctx.h, probe.h if probe is not None else None, C.c_void_p(d_buf.data_ptr()),
                                        n_buf, own_len, int(is_first), int(is_last), into.h if into is not None else None,
                                        C.byref(c))
    _check(rc, c.error_record, "fasta_ids_shard_dev")
    return c.reads_in, c.difference


def idset_partition_txt_dev(ctx: Context, d_buf, n: int, own_len: int, starts_line: bool, is_last: bool, log2_vpages: int,
                            d_recs, d_vstart):
    """sgpu_idset_partition_txt_dev (sharded set build, step 1): this rank's id-list shard -> slot images grouped by
    virtual page in d_recs (uint8 tensor, 16 bytes per record) / d_vstart (int64 tensor of 2^log2_vpages + 2).
    Returns the number of records, or None when the evidence cannot take the sharded build."""
    n_recs, err = C.c_uint64(), C.c_uint64()
    rc = ctx.L.sgpu_idset_partition_txt_dev(ctx.h, C.c_void_p(d_buf.data_ptr()), n, own_len, int(starts_line), int(is_last),
                                            log2_vpages, C.c_void_p(d_recs.data_ptr()), d_recs.numel() // 16,
                                            C.c_void_p(d_vstart.data_ptr()), C.byref(n_recs), C.byref(err))
    if rc in (_lib.SGPU_ERR_NOT_SHARDABLE, _lib.SGPU_ERR_CAPACITY):
        return None
    _check(rc, err.value, "idset_partition_txt_dev")
    return int(n_recs.value)


def idset_assemble_dev(ctx: Context, recs, vstarts, log2_vpages: int):
    """sgpu_idset_assemble_dev (step 2): the whole table from every rank's list (device tensors valid on this device:
    pulled copies or mapped peer memory).  Returns an IdSet, or None (fall back to the replicated build)."""
    n = len(recs)
    a = (C.c_void_p * n)(*[t.data_ptr() for t in recs])
    b = (C.c_void_p * n)(*[t.data_ptr() for t in vstarts])
    h = C.c_void_p()
    rc = ctx.L.sgpu_idset_assemble_dev(ctx.h, n, a, b, log2_vpages, C.byref(h))
    if rc == _lib.SGPU_ERR_NOT_SHARDABLE:
        return None
    _check(rc, 0, "idset_assemble_dev")
    return IdSet(ctx, h)


def count_newlines_dev(ctx: Context, d_buf, n: int) -> int:
    out = C.c_uint64()
    _check(ctx.L.sgpu_count_newlines_dev(ctx.h, C.c_void_p(d_buf.data_ptr()), n, C.byref(out)))
    return int(out.value)


def fastq_ids_shard_dev(ctx: Context, probe, d_buf, n_buf: int, own_len: int, newlines_before: int, is_first: bool,
                        is_last: bool, into: IdSet):
    """one shard of ReadDifference::get_difference's loops (utils.rs:259-283): ids of the records that start in the
    owned range and are absent from `probe` (None: all) go into `into`; returns (records, picked records)"""
    c = _lib.Counts()
    rc = ctx.L.sgpu_fastq_ids_shard_dev(ctx.h, probe.h if probe is not None else None, C.c_void_p(d_buf.data_ptr()),
                                        n_buf, own_len, newlines_before, int(is_first), int(is_last),
                                        into.h if into is not None else None, C.byref(c))
    _check(rc, c.error_record, "fastq_ids_shard_dev")
    return c.reads_in, c.difference


def diff(ctx: Context, pairs, raise_on_error: bool = True):
    """ReadDifference::get_difference (utils.rs:250-285) over [(input, output), ...] host or device buffers
    -> (reads_in, reads_out, difference, IdSet of absent ids)"""
    c = _lib.Counts()
    h = C.c_void_p()
    for fin, fout in pairs:
        if hasattr(fin, "is_cuda") and fin.is_cuda:
            p1, n1 = _dev_ptr(fin)
            p2, n2 = _dev_ptr(fout)
            rc = ctx.L.sgpu_diff_dev(ctx.h, p1, n1, p2, n2, C.byref(c), C.byref(h))
        else:
            p1, n1, k1 = _host_ptr(fin)
            p2, n2, k2 = _host_ptr(fout)
            rc = ctx.L.sgpu_diff(ctx.h, p1, n1, p2, n2, C.byref(c), C.byref(h))
        if rc:
            if h:
                ctx.L.sgpu_idset_free(h)
            if raise_on_error:
                raise ScrubbyGpuError(rc, c.error_record, "diff")
            return rc, c.error_record
    ids = IdSet(ctx, h) if h else IdSet.empty(ctx)
    return c.reads_in, c.reads_out, c.difference, ids


def clean_fastq_host(ctx: Context, ids: IdSet, h_in, n_in: int, h_out, h_other=None, reverse: bool = False
                     ) -> DevCleanResult:
    """sgpu_clean_fastq on caller-owned HOST tensors (pinned for full PCIe rate): the H2D copy of the
    input and the D2H copy of the outputs happen inside the call.  This is bench.py's e2e path."""
    n1, n2, c = C.c_size_t(), C.c_size_t(), _lib.Counts()
    rc = ctx.L.sgpu_clean_fastq(
        ctx.h, ids.h, C.c_void_p(h_in.data_ptr()), n_in, int(reverse), C.c_void_p(h_out.data_ptr()), h_out.numel(),
        C.byref(n1), C.c_void_p(h_other.data_ptr()) if h_other is not None else None,
        h_other.numel() if h_other is not None else 0, C.byref(n2), C.byref(c))
    _check(rc, c.error_record, "clean_fastq")
    return DevCleanResult(n1.value, n2.value, c.reads_in, c.reads_out, bool(c.crlf), bool(c.empty_input), c.path)
