// capi.cu -- extern "C" entry points of libscrubby_gpu.so (see include/scrubby_gpu.h): argument checks, the format
// decision, the chunked and one-shot host-buffer paths.  The work itself is done by the shard cores declared in
// fastq_records.cuh; a whole file is the shard (n, n, first = 1, last = 1) of either format.
#include <vector>

#include "fastq_records.cuh"

namespace sgpu {
const char *last_cuda_error_text();

enum class Fmt { fastq, fasta, empty, unknown };

// needletail picks the parser from the first byte; niffler needs 5 bytes (utils.rs:359-383).  `whole`: the 5-byte rule
// applies to the buffer (a file, or a shard the caller treats as one).  Byte 0 is read only when the decision needs
// it; a device buffer's comes back with a one-byte copy (the stream is synchronised).
static sgpu_status input_format(sgpu_ctx *c, const uint8_t *buf, bool on_device, size_t n, bool whole, Fmt *f) {
    *f = Fmt::empty;
    if (n == 0 || (whole && n < 5)) return SGPU_OK;
    const uint8_t *b0 = buf;
    if (on_device) {
        SGPU_CUDA(cudaMemcpyAsync(c->h_pinned, buf, 1, cudaMemcpyDeviceToHost, c->stream));
        SGPU_CUDA(cudaStreamSynchronize(c->stream));
        b0 = (const uint8_t *)c->h_pinned;
    }
    const uint8_t b = *b0;
    *f = b == '>' ? Fmt::fasta : b == '@' ? Fmt::fastq : Fmt::unknown;
    return SGPU_OK;
}

// a whole file whose format is known: '>' hands it to needletail's FASTA reader, FASTQ is the shard (n, n, 0, 1, 1,
// crlf -1)
static sgpu_status clean_file(sgpu_ctx *c, const sgpu_idset *set, const Shard &s, Fmt f, int reverse, const Outs &out,
                              sgpu_counts *counts) {
    clear_outputs(out, counts);
    switch (f) {
    case Fmt::fasta: {
        int le_own;
        return clean_fasta_shard(c, set, s, -1, reverse, out, counts, &le_own);
    }
    case Fmt::empty: counts->empty_input = 1; return SGPU_OK;
    case Fmt::unknown: return SGPU_ERR_FASTQ_UNKNOWN_FORMAT;
    default: return clean_fastq_shard(c, set, s, 0, -1, reverse, out, counts, false);
    }
}

// the ids of a FASTQ shard, or of a whole FASTA file (sgpu_diff_dev, sgpu_fastq_ids_shard_dev); a first shard that
// starts with '>' but is not the whole file is refused with SGPU_ERR_FASTA_UNSUPPORTED
static sgpu_status ids_locked(sgpu_ctx *c, const Shard &s, uint64_t newlines_before, const sgpu_idset *probe,
                              int want_absent, const SpanSink &sink, uint64_t *n_records, uint64_t *n_picked,
                              uint64_t *err_record, sgpu_counts *spec_out = nullptr) {
    *n_records = *n_picked = 0;
    if (s.is_first) {
        Fmt f;
        SGPU_TRY(input_format(c, s.p, true, s.n, true, &f));
        if (f == Fmt::empty) return SGPU_OK;
        if (f == Fmt::unknown) return SGPU_ERR_FASTQ_UNKNOWN_FORMAT;
        if (f == Fmt::fasta)
            return s.is_last && s.own_len == s.n
                       ? fasta_ids_shard(c, s, probe, want_absent, sink, n_records, n_picked, err_record)
                       : SGPU_ERR_FASTA_UNSUPPORTED;
    }
    return fastq_ids_shard(c, s, newlines_before, probe, want_absent, sink, n_records, n_picked, err_record, spec_out);
}

void ctx_release(sgpu_ctx *c) {
    if (c->refs.fetch_sub(1) != 1) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    if (c->s_in) cudaStreamDestroy(c->s_in);
    if (c->s_out) cudaStreamDestroy(c->s_out);
    if (c->h_pinned) cudaFreeHost(c->h_pinned);
    for (int i = 0; i < 5; i++)
        if (c->pipe_buf[i]) cudaFree(c->pipe_buf[i]);
    for (auto &e : c->prof_events) {
        cudaEventDestroy(e.first);
        cudaEventDestroy(e.second);
    }
    delete c;
}

}  // namespace sgpu

using namespace sgpu;

extern "C" {

int sgpu_abi_version(void) { return SGPU_ABI_VERSION; }

const char *sgpu_last_cuda_error(void) { return last_cuda_error_text(); }

const char *sgpu_strerror(int s) {
    switch (s) {
    case SGPU_OK: return "ok";
    case SGPU_ERR_IO: return "I/O error: stream did not contain valid UTF-8";
    case SGPU_ERR_NIFFLER: return "compression sniffing failed";
    case SGPU_ERR_FASTQ_INVALID_START: return "FASTQ record does not start with '@'";
    case SGPU_ERR_FASTQ_INVALID_SEPARATOR: return "FASTQ separator line does not start with '+'";
    case SGPU_ERR_FASTQ_UNEQUAL_LENGTHS: return "FASTQ sequence and quality lengths differ";
    case SGPU_ERR_FASTQ_UNEXPECTED_END: return "FASTQ ended in the middle of a record";
    case SGPU_ERR_FASTQ_UNKNOWN_FORMAT: return "input is neither FASTQ nor FASTA";
    case SGPU_ERR_RECORD_NAME_UTF8: return "failed to parse record name from BAM";
    case SGPU_ERR_FASTQ_HEADER: return "failed to extract a valid header of read";
    case SGPU_ERR_PAF_INTEGER: return "failed to parse a valid integer from PAF";
    case SGPU_ERR_WOULD_PANIC: return "record has too few columns (the reference panics here)";
    case SGPU_ERR_KRAKEN_REPORT_READS: return "failed to convert the read field in the report from `Kraken2`";
    case SGPU_ERR_KRAKEN_REPORT_DIRECT: return "failed to convert the direct read field in the report from `Kraken2`";
    case SGPU_ERR_KRAKEN_REPORT_PARENT: return "failed to provide a parent taxon while parsing report from `Kraken2`";
    case SGPU_ERR_FASTA_UNSUPPORTED: return "FASTA input given to a FASTQ shard entry point (use the FASTA shard entry points)";
    case SGPU_ERR_CUDA: return "CUDA error (see sgpu_last_cuda_error)";
    case SGPU_ERR_NOMEM: return "out of memory";
    case SGPU_ERR_INVALID_ARG: return "invalid argument";
    case SGPU_ERR_CAPACITY: return "output buffer too small";
    case SGPU_ERR_KEY_TOO_LONG: return "read id of 16 MiB or more";
    case SGPU_ERR_HALO: return "shard halo too small: last owned record does not end inside the buffer";
    case SGPU_ERR_SAM_RECORD: return "failed to parse a SAM record";
    case SGPU_ERR_BAM_RECORD: return "failed to read a BAM header or record";
    case SGPU_ERR_NOT_SHARDABLE: return "evidence cannot take the sharded set build (long ids, or too many keys): replicate it";
    case SGPU_ERR_PHASE_UNKNOWN: return "shard needs the exact newlines_before / crlf (speculation not applicable)";
    default: return "unknown status";
    }
}

sgpu_status sgpu_ctx_create(int device, sgpu_ctx **out) {
    if (!out) return SGPU_ERR_INVALID_ARG;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) {
        set_cuda_error(e != cudaSuccess ? e : cudaErrorNoDevice, __FILE__, __LINE__);
        return SGPU_ERR_CUDA;  // no CPU fallback by design
    }
    SGPU_CUDA(cudaSetDevice(device));
    if (const char *g = getenv("SGPU_L2_FETCH")) {  // tuning: L2 fetch granularity in bytes (32 / 64 / 128)
        size_t before = 0, after = 0;
        cudaDeviceGetLimit(&before, cudaLimitMaxL2FetchGranularity);
        cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(g));
        cudaDeviceGetLimit(&after, cudaLimitMaxL2FetchGranularity);
        fprintf(stderr, "[sgpu] L2 fetch granularity %zu -> %zu\n", before, after);
        cudaGetLastError();
    }
    sgpu_ctx *c = new (std::nothrow) sgpu_ctx();
    if (!c) return SGPU_ERR_NOMEM;
    c->device = device;
    cudaDeviceProp prop;
    SGPU_CUDA(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    SGPU_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    c->own_stream = true;
    SGPU_CUDA(cudaHostAlloc((void **)&c->h_pinned, 64 * 8, cudaHostAllocDefault));
    // keep freed scratch in the pool: steady-state steps do not touch the driver allocator
    cudaMemPool_t pool;
    SGPU_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t thr = ~0ull;
    SGPU_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
    *out = c;
    return SGPU_OK;
}

void sgpu_ctx_destroy(sgpu_ctx *c) {
    if (c) ctx_release(c);
}

sgpu_status sgpu_ctx_set_stream(sgpu_ctx *c, void *stream) {
    if (!c) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    SGPU_CUDA(cudaStreamSynchronize(c->stream));
    if (c->own_stream) {
        cudaStreamDestroy(c->stream);
        c->own_stream = false;
    }
    if (stream) {
        c->stream = (cudaStream_t)stream;
    } else {
        SGPU_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        c->own_stream = true;
    }
    return SGPU_OK;
}

sgpu_status sgpu_ctx_set_mode(sgpu_ctx *c, int mode) {
    if (!c || (mode != 0 && mode != 1)) return SGPU_ERR_INVALID_ARG;
    c->mode = mode;
    return SGPU_OK;
}

sgpu_status sgpu_ctx_sync(sgpu_ctx *c) {
    if (!c) return SGPU_ERR_INVALID_ARG;
    SGPU_CUDA(cudaSetDevice(c->device));
    SGPU_CUDA(cudaStreamSynchronize(c->stream));
    return SGPU_OK;
}

uint64_t sgpu_ctx_launch_count(const sgpu_ctx *c) { return c ? c->launches : 0; }

sgpu_status sgpu_ctx_set_profiling(sgpu_ctx *c, int on) {
    if (!c) return SGPU_ERR_INVALID_ARG;
    c->profiling = on != 0;
    return SGPU_OK;
}

sgpu_status sgpu_ctx_fused_stats(sgpu_ctx *c, double *ms, uint64_t *launches, uint64_t *alg_bytes) {
    if (!c || !ms || !launches || !alg_bytes) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    SGPU_CUDA(cudaStreamSynchronize(c->stream));
    double total = 0;
    for (size_t i = 0; i < c->prof_used; i++) {
        float t = 0;
        SGPU_CUDA(cudaEventElapsedTime(&t, c->prof_events[i].first, c->prof_events[i].second));
        total += t;
    }
    *ms = total;
    *launches = c->prof_used;
    *alg_bytes = c->prof_alg_bytes;
    c->prof_used = 0;
    c->prof_alg_bytes = 0;
    return SGPU_OK;
}

sgpu_status sgpu_count_newlines_dev(sgpu_ctx *c, const uint8_t *d_buf, size_t n, uint64_t *count) {
    if (!c || !count || (n && !d_buf)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    return count_newlines(c, d_buf, n, count);
}

// argument checks shared by the FASTQ shard entry points
static bool fastq_shard_args_ok(size_t n_in, size_t own_len, uint64_t newlines_before, int is_first, int is_last,
                                int crlf) {
    return own_len <= n_in && (!is_last || own_len == n_in) && (!is_first || newlines_before == 0) && crlf >= -1 &&
           crlf <= 1 && (is_first || crlf >= 0 || newlines_before == SGPU_NEWLINES_UNKNOWN);
}

sgpu_status sgpu_clean_fastq_dev(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *d_in, size_t n_in, int reverse,
                                 uint8_t *d_out_w, size_t cap_w, size_t *n_w, uint8_t *d_out_o, size_t cap_o,
                                 size_t *n_o, sgpu_counts *counts) {
    if (!c || !set || !n_w || !counts || (n_in && !d_in) || (cap_w && !d_out_w)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    const Outs out{d_out_w, cap_w, n_w, d_out_o, cap_o, n_o};
    clear_outputs(out, counts);
    if (n_in && ((uintptr_t)d_in & 15)) return SGPU_ERR_INVALID_ARG;
    Fmt f;
    SGPU_TRY(input_format(c, d_in, true, n_in, true, &f));
    return clean_file(c, set, Shard{d_in, n_in, n_in, 1, 1}, f, reverse, out, counts);
}

sgpu_status sgpu_clean_fastq_shard_dev(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *d_in, size_t n_in,
                                       size_t own_len, uint64_t newlines_before, int is_first, int is_last, int crlf,
                                       int reverse, uint8_t *d_out_w, size_t cap_w, size_t *n_w, uint8_t *d_out_o,
                                       size_t cap_o, size_t *n_o, sgpu_counts *counts) {
    if (!c || !set || !n_w || !counts || (n_in && !d_in) ||
        !fastq_shard_args_ok(n_in, own_len, newlines_before, is_first, is_last, crlf))
        return SGPU_ERR_INVALID_ARG;
    if (n_in && ((uintptr_t)d_in & 15)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    return clean_fastq_shard(c, set, Shard{d_in, n_in, own_len, is_first, is_last}, newlines_before, crlf, reverse,
                             Outs{d_out_w, cap_w, n_w, d_out_o, cap_o, n_o}, counts, crlf < 0);
}

}  // extern "C"

// Host buffers, large input: the file (or one shard of it) goes through the GPU in chunks (shards of one device) so
// that the host->device copy of chunk k+1.., the kernels of chunk k and the device->host copy of chunk k-1 overlap on
// three streams -- the end-to-end time approaches the PCIe time of the larger direction instead of the sum.
// Results are identical to the one-shot path (the same shard logic the multi-GPU driver uses; the record that
// straddles a cut belongs to the chunk where it starts).  The staging, upload and download loop is shared by the
// formats; `Fmt` holds what differs: the shard call of one chunk and the state the next chunk starts from
// (FastqChunks: the running newline count; FastaChunks: the line-ending decision).
// The buffer is a shard: own bytes [0, own_len) + halo; a whole file is the shard (n_in, n_in, first, last).
// *done = 0: not applicable here (small input, halo too small for a record ...), take the one-shot path.
template <class Chunks>
static sgpu_status pipeline_host(sgpu_ctx *c, const Shard &s, const Outs &out, sgpu_counts *counts, int *done,
                                 Chunks &fmt) {
    *done = 0;
    const size_t n_in = s.n, own_len = s.own_len;
    uint8_t *out_o = out.o;
    // (environment knobs so that tests can drive the chunk logic with small inputs)
    const size_t CHUNK = getenv("SGPU_PIPE_CHUNK") ? (size_t)atoll(getenv("SGPU_PIPE_CHUNK")) & ~(size_t)15
                                                   : (size_t)128 << 20;
    const size_t HALO = getenv("SGPU_PIPE_HALO") ? (size_t)atoll(getenv("SGPU_PIPE_HALO")) : (size_t)8 << 20;
    if (CHUNK < 4096 || own_len < 2 * CHUNK) return SGPU_OK;
    if (!c->s_in) {
        SGPU_CUDA(cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking));
        SGPU_CUDA(cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking));
    }
    cudaStream_t st = c->stream;
    const size_t K = ceil_div(own_len, CHUNK);  // kernel chunks: the owned range
    const size_t U = ceil_div(n_in, CHUNK);     // upload pieces: the whole buffer (own range + halo)
    const size_t tail_halo = n_in - own_len;
    const size_t obuf = Chunks::OUT_FACTOR * (CHUNK + std::max(HALO, tail_halo)) + 64;
    // context-owned staging (the context is locked): 0 the file, 1-2 kept chunks, 3-4 removed chunks
    auto staging = [&](int i, size_t bytes, uint8_t **p) -> sgpu_status {
        if (c->pipe_cap[i] < bytes) {
            SGPU_CUDA(cudaStreamSynchronize(st));
            if (c->pipe_buf[i]) SGPU_CUDA(cudaFree(c->pipe_buf[i]));
            c->pipe_buf[i] = nullptr;
            c->pipe_cap[i] = 0;
            const size_t want = bytes + (bytes >> 4);  // a little slack: mate files differ by a few bytes
            cudaError_t e = cudaMalloc((void **)&c->pipe_buf[i], want);
            if (e != cudaSuccess) {
                set_cuda_error(e, __FILE__, __LINE__);
                return e == cudaErrorMemoryAllocation ? SGPU_ERR_NOMEM : SGPU_ERR_CUDA;
            }
            c->pipe_cap[i] = want;
        }
        *p = c->pipe_buf[i];
        return SGPU_OK;
    };
    struct Ptr {
        uint8_t *p = nullptr;
    } d_in, d_w[2], d_o[2];
    SGPU_TRY(staging(0, n_in + 16, &d_in.p));
    for (int r = 0; r < 2; r++) {
        SGPU_TRY(staging(1 + r, obuf, &d_w[r].p));
        if (out_o) SGPU_TRY(staging(3 + r, obuf, &d_o[r].p));
    }
    SGPU_CUDA(cudaStreamSynchronize(st));  // earlier work on `st` that used the staging is done
    std::vector<cudaEvent_t> ev_in(U);
    cudaEvent_t ev_k[2], ev_out[2];
    for (size_t k = 0; k < U; k++) SGPU_CUDA(cudaEventCreateWithFlags(&ev_in[k], cudaEventDisableTiming));
    for (int r = 0; r < 2; r++) {
        SGPU_CUDA(cudaEventCreateWithFlags(&ev_k[r], cudaEventDisableTiming));
        SGPU_CUDA(cudaEventCreateWithFlags(&ev_out[r], cudaEventDisableTiming));
    }
    auto upload = [&](size_t k) -> cudaError_t {
        const size_t a = k * CHUNK, len = std::min(CHUNK, n_in - a);
        cudaError_t e = cudaMemcpyAsync(d_in.p + a, s.p + a, len, cudaMemcpyHostToDevice, c->s_in);
        if (e != cudaSuccess) return e;
        return cudaEventRecord(ev_in[k], c->s_in);
    };
    sgpu_status rc = SGPU_OK;
    size_t off_w = 0, off_o = 0;
    bool bail = false, unknown = false;
    sgpu_counts total;
    memset(&total, 0, sizeof(total));
    total.path = 1;
    cudaError_t ce = cudaSuccess;
    size_t up_next = 0;
    for (; up_next < std::min<size_t>(U, 3) && ce == cudaSuccess; up_next++) ce = upload(up_next);
    for (size_t k = 0; k < K && ce == cudaSuccess && rc == SGPU_OK && !bail; k++) {
        const int r = (int)(k & 1);
        const size_t a = k * CHUNK;
        size_t own = std::min(CHUNK, own_len - a);
        bool last_chunk = k + 1 == K;
        if (!last_chunk && s.is_last && a + own + HALO >= n_in) {
            // the chunk's buffer reaches EOF: it owns the rest, as only the last chunk may apply the end-of-file rules
            // (a record that runs to EOF would otherwise be a halo problem and send the whole call to the one-shot path)
            own = own_len - a;
            last_chunk = true;
        }
        const size_t buf_len = last_chunk ? n_in - a : std::min(n_in - a, own + HALO);
        // keep the copy engine three pieces ahead, and at least as far as this chunk's halo reaches
        while (up_next < U && ce == cudaSuccess && (up_next < k + 4 || up_next * CHUNK < a + buf_len)) ce = upload(up_next++);
        if (ce != cudaSuccess) break;
        // the chunk and its halo (inside the next pieces) are on the device; the output buffer is free again
        for (size_t j = k; j < U && j * CHUNK < a + buf_len; j++) cudaStreamWaitEvent(st, ev_in[j], 0);
        if (k >= 2) cudaStreamWaitEvent(st, ev_out[r], 0);
        size_t nw = 0, no = 0;
        sgpu_counts ck;
        rc = fmt.run(c, k, a, Shard{d_in.p + a, buf_len, own, s.is_first && k == 0, last_chunk && s.is_last},
                     Outs{d_w[r].p, obuf, &nw, out_o ? d_o[r].p : nullptr, obuf, &no}, &ck);
        if (fmt.unknown(rc, ck)) {
            rc = SGPU_OK;  // speculation not applicable: the caller comes back with the exact phase
            unknown = true;
            break;
        }
        if (rc == SGPU_ERR_HALO) {  // a record longer than the halo: the one-shot path handles any length
            rc = SGPU_OK;
            bail = true;
            break;
        }
        if (rc == SGPU_ERR_CAPACITY || rc == SGPU_ERR_CUDA || rc == SGPU_ERR_NOMEM) break;
        const sgpu_status parse_rc = rc;  // a parse error: like the one-shot path (and the reference, which
        rc = SGPU_OK;                     // leaves the records before the error on disk) the output so far stays
        if (parse_rc != SGPU_OK) total.error_record = ck.error_record + total.reads_in;  // earlier chunks come first
        if (off_w + nw > out.cap_w || (out_o && off_o + no > out.cap_o)) {
            rc = SGPU_ERR_CAPACITY;
            break;
        }
        cudaEventRecord(ev_k[r], st);
        cudaStreamWaitEvent(c->s_out, ev_k[r], 0);
        if (nw) ce = cudaMemcpyAsync(out.w + off_w, d_w[r].p, nw, cudaMemcpyDeviceToHost, c->s_out);
        if (out_o && no && ce == cudaSuccess)
            ce = cudaMemcpyAsync(out_o + off_o, d_o[r].p, no, cudaMemcpyDeviceToHost, c->s_out);
        cudaEventRecord(ev_out[r], c->s_out);
        off_w += nw;
        off_o += no;
        total.reads_in += ck.reads_in;
        total.reads_out += ck.reads_out;
        total.crlf = ck.crlf ? 1 : total.crlf;
        if (ck.path != 1) total.path = ck.path;
        if (parse_rc != SGPU_OK) {
            rc = parse_rc;
            break;
        }
        rc = fmt.advance(c, k, d_in.p + a, own, last_chunk, ck);
        if (last_chunk) break;
    }
    cudaStreamSynchronize(c->s_in);
    cudaStreamSynchronize(c->s_out);
    cudaStreamSynchronize(st);
    for (size_t k = 0; k < U; k++) cudaEventDestroy(ev_in[k]);
    for (int r = 0; r < 2; r++) {
        cudaEventDestroy(ev_k[r]);
        cudaEventDestroy(ev_out[r]);
    }
    if (ce != cudaSuccess) {
        set_cuda_error(ce, __FILE__, __LINE__);
        return SGPU_ERR_CUDA;
    }
    if (unknown) {
        *done = 1;
        clear_outputs(out, counts);
        return SGPU_ERR_PHASE_UNKNOWN;
    }
    if (bail) return SGPU_OK;  // *done stays 0
    *done = 1;
    *counts = total;
    fmt.finish(counts);
    *out.n_w = off_w;
    if (out.n_o) *out.n_o = out_o ? off_o : 0;
    return rc;
}

// FASTQ: the line phase of chunk k+1 comes from the running newline count.  newlines_before == SGPU_NEWLINES_UNKNOWN:
// chunk 0 speculates the line phase, the later chunks continue from it, counts->{own_newlines, lead_newlines} let the
// caller verify it.
struct FastqChunks {
    static constexpr size_t OUT_FACTOR = 1;
    const sgpu_idset *set;
    int crlf_in, reverse;
    bool spec;
    int crlf;
    uint64_t nb;  // running count: exact, or relative to the speculated phase
    uint64_t own_nl_total = 0, lead_nl = 0;

    sgpu_status run(sgpu_ctx *c, size_t k, size_t a, const Shard &d, const Outs &o, sgpu_counts *ck) {
        const bool spec0 = spec && k == 0;
        const sgpu_status rc = clean_fastq_shard(c, set, d, spec0 ? SGPU_NEWLINES_UNKNOWN : nb, spec0 ? -1 : crlf, reverse,
                                                 o, ck, true);
        if (getenv("SGPU_DEBUG"))
            fprintf(stderr, "[sgpu] pipe chunk %zu a=%zu own=%zu buf=%zu nlb=%llu -> rc=%d nw=%zu no=%zu in=%llu out=%llu path=%u own_nl=%llu lead_nl=%llu\n",
                    k, a, d.own_len, d.n, (unsigned long long)nb, (int)rc, *o.n_w, *o.n_o,
                    (unsigned long long)ck->reads_in, (unsigned long long)ck->reads_out, ck->path,
                    (unsigned long long)ck->own_newlines, (unsigned long long)ck->lead_newlines);
        return rc;
    }
    bool unknown(sgpu_status rc, const sgpu_counts &ck) const {
        return rc == SGPU_ERR_PHASE_UNKNOWN || (spec && rc == SGPU_OK && ck.path != 1);
    }
    sgpu_status advance(sgpu_ctx *c, size_t k, const uint8_t *d, size_t own, bool last_chunk, const sgpu_counts &ck) {
        // this chunk's newlines: a by-product of the single-pass kernel, else one counting pass
        sgpu_status rc = SGPU_OK;
        uint64_t cnt = ck.own_newlines;
        if (ck.path != 1 && (!last_chunk || crlf_in < 0)) rc = count_newlines(c, d, own, &cnt);
        if (spec && k == 0) {
            lead_nl = ck.lead_newlines;
            nb = (4 - (lead_nl & 3)) & 3;  // the phase the speculation stands for
        }
        nb += cnt;
        own_nl_total += cnt;
        return rc;
    }
    void finish(sgpu_counts *counts) const {
        counts->own_newlines = own_nl_total;
        counts->lead_newlines = lead_nl;
        counts->speculated = spec ? 1 : 0;
    }
};

static sgpu_status clean_host_pipelined(sgpu_ctx *c, const sgpu_idset *set, const Shard &s, uint64_t newlines_before,
                                        int crlf_in, int reverse, const Outs &out, sgpu_counts *counts, int *done) {
    *done = 0;
    if (c->mode != 0) return SGPU_OK;
    if (s.is_first) {
        Fmt f;
        SGPU_TRY(input_format(c, s.p, false, s.n, true, &f));
        if (f != Fmt::fastq) return SGPU_OK;  // FASTA / unknown format / too small: not this format's pipeline
    }
    const bool spec = !s.is_first && newlines_before == SGPU_NEWLINES_UNKNOWN;
    int crlf = crlf_in > 0;
    if (s.is_first) {  // needletail decides the line ending on the first record's first line
        const uint8_t *nl = (const uint8_t *)memchr(s.p, '\n', s.n);
        crlf = nl && nl > s.p && nl[-1] == '\r';
    }
    FastqChunks f{set, crlf_in, reverse, spec, crlf, spec ? 0 : newlines_before};
    return pipeline_host(c, s, out, counts, done, f);
}

// FASTA: chunk k+1 starts from chunk k's line-ending state, le_before(k) when that was decided, else le_own(k) -- exact,
// nothing is speculated.  A chunk's output is at most twice its records' bytes (">a\n" -> ">a\r\n\r\n").
struct FastaChunks {
    static constexpr size_t OUT_FACTOR = 2;
    const sgpu_idset *set;
    int reverse;
    int le;            // le_before of the next chunk
    int le_own = -1;   // the shard's own decision: the first chunk's that has one
    int le_chunk = -1;

    sgpu_status run(sgpu_ctx *c, size_t, size_t, const Shard &d, const Outs &o, sgpu_counts *ck) {
        const sgpu_status rc = clean_fasta_shard(c, set, d, le, reverse, o, ck, &le_chunk);
        if (le_own < 0) le_own = le_chunk;  // (also from a chunk that stops on a parse error: decided before the error)
        return rc;
    }
    bool unknown(sgpu_status, const sgpu_counts &) const { return false; }
    sgpu_status advance(sgpu_ctx *, size_t, const uint8_t *, size_t, bool, const sgpu_counts &) {
        if (le < 0) le = le_chunk;
        return SGPU_OK;
    }
    void finish(sgpu_counts *) const {}
};

static sgpu_status fasta_host_pipelined(sgpu_ctx *c, const sgpu_idset *set, const Shard &s, int le_before, int reverse,
                                        const Outs &out, sgpu_counts *counts, int *le_own, int *done) {
    FastaChunks f{set, reverse, le_before};
    const sgpu_status rc = pipeline_host(c, s, out, counts, done, f);
    *le_own = f.le_own;
    return rc;
}

// the one-shot host path: the whole buffer on the device, `call(d, d_out)` on it -- d is the shard `s` with its bytes
// on the device, d_out the device outputs --, outputs back.
// write_fastq's output is the input re-serialised: larger only when line endings are rewritten (FASTQ: LF records
// after a CRLF first record) or FASTA header-only records gain an empty sequence line.  Device buffers are sized for
// the common case first.
template <class Call>
static sgpu_status oneshot_host(sgpu_ctx *c, const Shard &s, const Outs &out, Call call) {
    cudaStream_t st = c->stream;
    DevBuf<uint8_t> d_in, d_w, d_o;
    SGPU_TRY(d_in.alloc(s.n + 16, st));
    if (s.n) SGPU_CUDA(cudaMemcpyAsync(d_in.p, s.p, s.n, cudaMemcpyHostToDevice, st));
    sgpu_status rc = SGPU_OK;
    for (int attempt = 0; attempt < 2; attempt++) {
        const size_t want = attempt ? ~(size_t)0 : s.n + s.n / 16 + 4096;
        const size_t dcap_w = std::min(out.cap_w, want), dcap_o = std::min(out.cap_o, want);
        SGPU_TRY(d_w.alloc(dcap_w + 16, st));
        if (out.o) SGPU_TRY(d_o.alloc(dcap_o + 16, st));
        rc = call(Shard{d_in.p, s.n, s.own_len, s.is_first, s.is_last},
                  Outs{d_w.p, dcap_w, out.n_w, out.o ? d_o.p : nullptr, dcap_o, out.n_o});
        if (rc != SGPU_ERR_CAPACITY || (dcap_w == out.cap_w && (!out.o || dcap_o == out.cap_o))) break;
    }
    if (rc == SGPU_ERR_CAPACITY || rc == SGPU_ERR_CUDA || rc == SGPU_ERR_NOMEM || rc == SGPU_ERR_PHASE_UNKNOWN) return rc;
    if (*out.n_w) SGPU_CUDA(cudaMemcpyAsync(out.w, d_w.p, *out.n_w, cudaMemcpyDeviceToHost, st));
    if (out.o && out.n_o && *out.n_o) SGPU_CUDA(cudaMemcpyAsync(out.o, d_o.p, *out.n_o, cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(cudaStreamSynchronize(st));
    return rc;
}

extern "C" {

sgpu_status sgpu_clean_fastq(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *in, size_t n_in, int reverse,
                             uint8_t *out_w, size_t cap_w, size_t *n_w, uint8_t *out_o, size_t cap_o, size_t *n_o,
                             sgpu_counts *counts) {
    if (!c || !set || !n_w || !counts || (n_in && !in) || (cap_w && !out_w)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    const Shard s{in, n_in, n_in, 1, 1};
    const Outs out{out_w, cap_w, n_w, out_o, cap_o, n_o};
    Fmt f;
    SGPU_TRY(input_format(c, in, false, n_in, true, &f));
    {
        int done = 0, le_own;
        sgpu_status prc = f == Fmt::fasta ? fasta_host_pipelined(c, set, s, -1, reverse, out, counts, &le_own, &done)
                                          : clean_host_pipelined(c, set, s, 0, -1, reverse, out, counts, &done);
        if (done || prc != SGPU_OK) return prc;
    }
    return oneshot_host(c, s, out, [&](const Shard &d, const Outs &d_out) {
        return clean_file(c, set, d, f, reverse, d_out, counts);
    });
}

sgpu_status sgpu_clean_fastq_shard(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *in, size_t n_in, size_t own_len,
                                   uint64_t newlines_before, int is_first, int is_last, int crlf, int reverse,
                                   uint8_t *out_w, size_t cap_w, size_t *n_w, uint8_t *out_o, size_t cap_o, size_t *n_o,
                                   sgpu_counts *counts) {
    if (!c || !set || !n_w || !counts || (n_in && !in) || (cap_w && !out_w) ||
        !fastq_shard_args_ok(n_in, own_len, newlines_before, is_first, is_last, crlf))
        return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    const Shard s{in, n_in, own_len, is_first, is_last};
    const Outs out{out_w, cap_w, n_w, out_o, cap_o, n_o};
    {
        int done = 0;
        sgpu_status prc = clean_host_pipelined(c, set, s, newlines_before, crlf, reverse, out, counts, &done);
        if (done || prc != SGPU_OK) return prc;
    }
    return oneshot_host(c, s, out, [&](const Shard &d, const Outs &d_out) {
        return clean_fastq_shard(c, set, d, newlines_before, crlf, reverse, d_out, counts, crlf < 0);
    });
}

// argument checks shared by the FASTA shard entry points
static bool fasta_shard_args_ok(size_t n_in, size_t own_len, int is_last, int le_before, int is_first) {
    return own_len <= n_in && (!is_last || own_len == n_in) && le_before >= -1 && le_before <= 1 &&
           (!is_first || le_before == -1);
}

// the FASTA shard's first byte and the empty-input rule (context locked).  *empty: a first-and-last shard of fewer
// than 5 bytes (utils.rs:359-375); SGPU_ERR_INVALID_ARG: a first shard that does not start with '>'
static sgpu_status fasta_shard_head(sgpu_ctx *c, const Shard &s, bool on_device, bool *empty) {
    *empty = false;
    if (!s.is_first) return SGPU_OK;
    Fmt f;
    SGPU_TRY(input_format(c, s.p, on_device, s.n, s.is_last, &f));
    *empty = f == Fmt::empty && s.is_last;
    return *empty || f == Fmt::fasta ? SGPU_OK : SGPU_ERR_INVALID_ARG;
}

}  // extern "C"

// the ids entry points of both formats (context locked): the shard's ids go to `sink`; counts->reads_in += records,
// counts->difference += picked records, error_record on a failure (FASTQ: the single-pass kernel's speculation counts)
static sgpu_status fastq_ids_entry(sgpu_ctx *c, const Shard &s, uint64_t newlines_before, const sgpu_idset *probe,
                                   const SpanSink &sink, sgpu_counts *counts) {
    uint64_t n_rec = 0, n_pick = 0, err = 0;
    sgpu_counts spec;
    memset(&spec, 0, sizeof(spec));
    sgpu_status rc = ids_locked(c, s, newlines_before, probe, probe != nullptr, sink, &n_rec, &n_pick, &err, &spec);
    if (rc == SGPU_OK) {
        counts->reads_in += n_rec;
        counts->difference += n_pick;
        counts->speculated = spec.speculated;
        counts->own_newlines = spec.own_newlines;
        counts->lead_newlines = spec.lead_newlines;
    } else {
        counts->error_record = err;
    }
    cudaStreamSynchronize(c->stream);
    return rc;
}

static sgpu_status fasta_ids_entry(sgpu_ctx *c, const Shard &s, const sgpu_idset *probe, const SpanSink &sink,
                                   sgpu_counts *counts) {
    bool empty;
    SGPU_TRY(fasta_shard_head(c, s, true, &empty));
    if (empty) return SGPU_OK;
    uint64_t n_rec = 0, n_pick = 0, err = 0;
    sgpu_status rc = fasta_ids_shard(c, s, probe, probe != nullptr, sink, &n_rec, &n_pick, &err);
    if (rc == SGPU_OK) {
        counts->reads_in += n_rec;
        counts->difference += n_pick;
    } else {
        counts->error_record = err;
    }
    cudaStreamSynchronize(c->stream);
    return rc;
}

// the route sink of the route entry points: outputs zeroed before anything runs
static bool route_args_ok(int n_parts, uint8_t *d_lines, size_t cap, size_t *n_lines, uint64_t *part_bytes,
                          uint64_t *part_lines) {
    if (!n_lines || !part_bytes || !part_lines || n_parts < 1 || n_parts > 64 || (cap && !d_lines)) return false;
    *n_lines = 0;
    memset(part_bytes, 0, (size_t)n_parts * sizeof(uint64_t));
    memset(part_lines, 0, (size_t)n_parts * sizeof(uint64_t));
    return true;
}

extern "C" {

sgpu_status sgpu_clean_fasta_shard_dev(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *d_in, size_t n_in,
                                       size_t own_len, int is_first, int is_last, int le_before, int reverse,
                                       uint8_t *d_out_w, size_t cap_w, size_t *n_w, uint8_t *d_out_o, size_t cap_o,
                                       size_t *n_o, sgpu_counts *counts, int *le_own) {
    if (!c || !set || !n_w || !counts || !le_own || (n_in && !d_in) || (cap_w && !d_out_w) ||
        !fasta_shard_args_ok(n_in, own_len, is_last, le_before, is_first))
        return SGPU_ERR_INVALID_ARG;
    if (n_in && ((uintptr_t)d_in & 15)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    const Shard s{d_in, n_in, own_len, is_first, is_last};
    const Outs out{d_out_w, cap_w, n_w, d_out_o, cap_o, n_o};
    clear_outputs(out, counts);
    *le_own = -1;
    bool empty;
    SGPU_TRY(fasta_shard_head(c, s, true, &empty));
    if (empty) {
        counts->empty_input = 1;
        return SGPU_OK;
    }
    return clean_fasta_shard(c, set, s, le_before, reverse, out, counts, le_own);
}

sgpu_status sgpu_clean_fasta_shard(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *in, size_t n_in, size_t own_len,
                                   int is_first, int is_last, int le_before, int reverse, uint8_t *out_w, size_t cap_w,
                                   size_t *n_w, uint8_t *out_o, size_t cap_o, size_t *n_o, sgpu_counts *counts,
                                   int *le_own) {
    if (!c || !set || !n_w || !counts || !le_own || (n_in && !in) || (cap_w && !out_w) ||
        !fasta_shard_args_ok(n_in, own_len, is_last, le_before, is_first))
        return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    const Shard s{in, n_in, own_len, is_first, is_last};
    const Outs out{out_w, cap_w, n_w, out_o, cap_o, n_o};
    clear_outputs(out, counts);
    *le_own = -1;
    bool empty;
    SGPU_TRY(fasta_shard_head(c, s, false, &empty));
    if (empty) {
        counts->empty_input = 1;
        return SGPU_OK;
    }
    {
        int done = 0;
        sgpu_status prc = fasta_host_pipelined(c, set, s, le_before, reverse, out, counts, le_own, &done);
        if (done || prc != SGPU_OK) return prc;
    }
    return oneshot_host(c, s, out, [&](const Shard &d, const Outs &d_out) {
        return clean_fasta_shard(c, set, d, le_before, reverse, d_out, counts, le_own);
    });
}

sgpu_status sgpu_fasta_ids_shard_dev(sgpu_ctx *c, const sgpu_idset *probe, const uint8_t *d_buf, size_t n_buf,
                                     size_t own_len, int is_first, int is_last, sgpu_idset *into, sgpu_counts *counts) {
    if (!c || !counts || (n_buf && !d_buf) || !fasta_shard_args_ok(n_buf, own_len, is_last, -1, is_first))
        return SGPU_ERR_INVALID_ARG;
    if (n_buf && ((uintptr_t)d_buf & 15)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    return fasta_ids_entry(c, Shard{d_buf, n_buf, own_len, is_first, is_last}, probe, SpanSink{into, nullptr}, counts);
}

sgpu_status sgpu_diff_dev(sgpu_ctx *c, const uint8_t *d_in, size_t n_in, const uint8_t *d_out, size_t n_out,
                          sgpu_counts *counts, sgpu_idset **diff_ids) {
    if (!c || !counts || !diff_ids || (n_in && !d_in) || (n_out && !d_out)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    if (!*diff_ids) SGPU_TRY(idset_create(c, diff_ids));
    sgpu_idset *o_ids = nullptr;  // utils.rs:257 reads2_ids
    SGPU_TRY(idset_create(c, &o_ids));
    uint64_t n_rec = 0, n_pick = 0, err = 0;
    sgpu_status rc = ids_locked(c, Shard{d_out, n_out, n_out, 1, 1}, 0, nullptr, 0, SpanSink{o_ids, nullptr}, &n_rec, &n_pick, &err);  // :259-267
    if (rc == SGPU_OK) {
        counts->reads_out += n_rec;
        rc = ids_locked(c, Shard{d_in, n_in, n_in, 1, 1}, 0, o_ids, 1, SpanSink{*diff_ids, nullptr}, &n_rec, &n_pick, &err);  // :269-283
        if (rc == SGPU_OK) {
            counts->reads_in += n_rec;
            counts->difference += n_pick;
        }
    }
    if (rc != SGPU_OK) counts->error_record = err;
    cudaStreamSynchronize(c->stream);
    sgpu_idset_free(o_ids);
    return rc;
}

sgpu_status sgpu_fastq_ids_shard_dev(sgpu_ctx *c, const sgpu_idset *probe, const uint8_t *d_buf, size_t n_buf,
                                     size_t own_len, uint64_t newlines_before, int is_first, int is_last,
                                     sgpu_idset *into, sgpu_counts *counts) {
    if (!c || !counts || (n_buf && !d_buf) || !fastq_shard_args_ok(n_buf, own_len, newlines_before, is_first, is_last, 0))
        return SGPU_ERR_INVALID_ARG;
    if (n_buf && ((uintptr_t)d_buf & 15)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    return fastq_ids_entry(c, Shard{d_buf, n_buf, own_len, is_first, is_last}, newlines_before, probe,
                           SpanSink{into, nullptr}, counts);
}

sgpu_status sgpu_diff(sgpu_ctx *c, const uint8_t *in, size_t n_in, const uint8_t *out, size_t n_out,
                      sgpu_counts *counts, sgpu_idset **diff_ids) {
    if (!c || !counts || !diff_ids || (n_in && !in) || (n_out && !out)) return SGPU_ERR_INVALID_ARG;
    DevBuf<uint8_t> d_in, d_out;
    {
        std::lock_guard<std::mutex> lk(c->mu);
        SGPU_CUDA(cudaSetDevice(c->device));
        cudaStream_t st = c->stream;
        SGPU_TRY(d_in.alloc(n_in + 16, st));
        SGPU_TRY(d_out.alloc(n_out + 16, st));
        if (n_in) SGPU_CUDA(cudaMemcpyAsync(d_in.p, in, n_in, cudaMemcpyHostToDevice, st));
        if (n_out) SGPU_CUDA(cudaMemcpyAsync(d_out.p, out, n_out, cudaMemcpyHostToDevice, st));
    }
    sgpu_status rc = sgpu_diff_dev(c, d_in.p, n_in, d_out.p, n_out, counts, diff_ids);
    cudaStreamSynchronize(c->stream);
    return rc;
}

sgpu_status sgpu_fastq_ids_route_shard_dev(sgpu_ctx *c, const uint8_t *d_buf, size_t n_buf, size_t own_len,
                                           uint64_t newlines_before, int is_first, int is_last, int n_parts,
                                           uint8_t *d_lines, size_t cap, size_t *n_lines, uint64_t *part_bytes,
                                           uint64_t *part_lines, sgpu_counts *counts) {
    if (!c || !counts || (n_buf && !d_buf) || !fastq_shard_args_ok(n_buf, own_len, newlines_before, is_first, is_last, 0) ||
        !route_args_ok(n_parts, d_lines, cap, n_lines, part_bytes, part_lines))
        return SGPU_ERR_INVALID_ARG;
    if (n_buf && ((uintptr_t)d_buf & 15)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    RouteOut r{(uint32_t)n_parts, d_lines, cap, 0, part_bytes, part_lines};
    const sgpu_status rc = fastq_ids_entry(c, Shard{d_buf, n_buf, own_len, is_first, is_last}, newlines_before, nullptr,
                                           SpanSink{nullptr, &r}, counts);
    *n_lines = r.n_lines;
    return rc;
}

sgpu_status sgpu_fasta_ids_route_shard_dev(sgpu_ctx *c, const uint8_t *d_buf, size_t n_buf, size_t own_len, int is_first,
                                           int is_last, int n_parts, uint8_t *d_lines, size_t cap, size_t *n_lines,
                                           uint64_t *part_bytes, uint64_t *part_lines, sgpu_counts *counts) {
    if (!c || !counts || (n_buf && !d_buf) || !fasta_shard_args_ok(n_buf, own_len, is_last, -1, is_first) ||
        !route_args_ok(n_parts, d_lines, cap, n_lines, part_bytes, part_lines))
        return SGPU_ERR_INVALID_ARG;
    if (n_buf && ((uintptr_t)d_buf & 15)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    RouteOut r{(uint32_t)n_parts, d_lines, cap, 0, part_bytes, part_lines};
    const sgpu_status rc = fasta_ids_entry(c, Shard{d_buf, n_buf, own_len, is_first, is_last}, nullptr,
                                           SpanSink{nullptr, &r}, counts);
    *n_lines = r.n_lines;
    return rc;
}

}  // extern "C"
