// capi.cu -- extern "C" entry points of libscrubby_gpu.so (see include/scrubby_gpu.h).
#include <vector>

#include "fastq_records.cuh"

namespace sgpu {
const char *last_cuda_error_text();
// fastq_fused.cu: single-pass kernel; returns SGPU_OK with *used = 0 when the input is not canonical
sgpu_status clean_fused(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *d_in, size_t n_in, int reverse,
                        uint8_t *d_out_w, size_t cap_w, size_t *n_w, uint8_t *d_out_o, size_t cap_o, size_t *n_o,
                        sgpu_counts *counts, int *used);
sgpu_status ids_fused(sgpu_ctx *c, const sgpu_idset *probe, const uint8_t *d_in, size_t n_in, size_t own_len,
                      uint64_t newlines_before, int is_first, int is_last, uint64_t *span_off, uint32_t *span_len,
                      uint64_t cap, uint64_t *n_spans, uint64_t *span_base, uint64_t *n_records, int *used,
                      sgpu_counts *spec_out);
sgpu_status clean_fused_shard(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *d_in, size_t n_in, size_t own_len,
                              uint64_t newlines_before, int is_first, int is_last, int reverse, uint8_t *d_out_w,
                              size_t cap_w, size_t *n_w, uint8_t *d_out_o, size_t cap_o, size_t *n_o,
                              sgpu_counts *counts, int *used, bool want_nl);

// ids of every record of a FASTQ buffer (diff): span + validity
__global__ void __launch_bounds__(128)
    fastq_ids_kernel(RecParams P, IdSetView probe, int want_absent, uint64_t *key_off, uint32_t *key_len, uint8_t *sel,
                     unsigned long long *err_word, unsigned long long *counters) {
    uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool rec = false, pick = false;
    if (k <= P.k_full) {
        RecMeta m = {0, 0, 0, 0};
        uint64_t start, p1, p3;
        size_t id_off = 0, id_len = 0;
        uint64_t off = 0;
        uint32_t len = 0;
        if (locate_record(P, k, &start, &p1, &p3, &m, &id_off, &id_len, err_word)) {
            rec = true;
            off = start + 1 + id_off;
            len = (uint32_t)id_len;
            if (want_absent)
                pick = !(id_len <= IDSET_MAX_KEY && idset_contains(probe, P.in + off, len));
            else
                pick = true;
        }
        key_off[k] = off;
        key_len[k] = len;
        sel[k] = pick ? 1 : 0;
    }
    unsigned br = __ballot_sync(0xffffffffu, rec), bp = __ballot_sync(0xffffffffu, pick);
    if ((threadIdx.x & 31) == 0) {
        if (br) atomicAdd(&counters[0], (unsigned long long)__popc(br));
        if (bp) atomicAdd(&counters[1], (unsigned long long)__popc(bp));
    }
}

// needletail picks the parser from the first byte; niffler needs 5 bytes (utils.rs:359-383)
static sgpu_status sniff(sgpu_ctx *c, const uint8_t *d_in, size_t n_in, bool *empty) {
    *empty = n_in < 5;
    if (*empty) return SGPU_OK;
    SGPU_CUDA(cudaMemcpyAsync(c->h_pinned, d_in, 1, cudaMemcpyDeviceToHost, c->stream));
    SGPU_CUDA(cudaStreamSynchronize(c->stream));
    uint8_t b = *(uint8_t *)c->h_pinned;
    if (b == '>') return SGPU_ERR_FASTA_UNSUPPORTED;
    if (b != '@') return SGPU_ERR_FASTQ_UNKNOWN_FORMAT;
    return SGPU_OK;
}

// one FASTQ buffer (or one shard of it: the records that start in [0, own_len], see sgpu_clean_fastq_shard_dev)
// -> ids (all, or only those absent from `probe`) inserted into `into`
static sgpu_status fastq_ids_into(sgpu_ctx *c, const uint8_t *d_buf, size_t n, size_t own_len, uint64_t newlines_before,
                                  int is_first, int is_last, const sgpu_idset *probe, int want_absent, sgpu_idset *into,
                                  uint64_t *n_records, uint64_t *n_picked, uint64_t *err_record,
                                  sgpu_counts *spec_out = nullptr) {
    *n_records = *n_picked = 0;
    const bool spec = !is_first && newlines_before == SGPU_NEWLINES_UNKNOWN;
    if (is_first) {
        bool empty;
        const sgpu_status src = sniff(c, d_buf, n, &empty);
        if (src == SGPU_ERR_FASTA_UNSUPPORTED && is_last && own_len == n)  // a whole FASTA file
            return fasta_ids_shard(c, d_buf, n, n, 1, 1, probe, want_absent, into, n_records, n_picked, err_record);
        if (src != SGPU_OK) return src;
        if (empty) return SGPU_OK;
    } else if (n == 0 || own_len == 0) {
        return SGPU_OK;
    }
    cudaStream_t st = c->stream;
    if (c->mode == 0 && ((uintptr_t)d_buf & 15) == 0) {
        // canonical input: one pass of the fused kernel in ids mode -> (offset, length) spans of the wanted ids
        DevBuf<uint64_t> s_off;
        DevBuf<uint32_t> s_len;
        const uint64_t cap = n / 100 + 4096;  // the fused kernel handles >= ~102 bytes per record
        SGPU_TRY(s_off.alloc(cap, st));
        SGPU_TRY(s_len.alloc(cap, st));
        uint64_t n_spans = 0, n_rec = 0, base = 0;
        int used = 0;
        SGPU_TRY(ids_fused(c, want_absent ? probe : nullptr, d_buf, n, own_len, newlines_before, is_first, is_last,
                           s_off.p, s_len.p, cap, &n_spans, &base, &n_rec, &used, spec_out));
        if (used) {
            *n_records = n_rec;
            *n_picked = n_spans;
            if (into && n_spans)
                SGPU_TRY(idset_insert_spans(c, into, d_buf + base, s_off.p, s_len.p, nullptr, (size_t)n_spans));
            return SGPU_OK;
        }
    }
    if (spec) return SGPU_ERR_PHASE_UNKNOWN;
    DevBuf<uint64_t> nlpos, key_off, scratch;
    DevBuf<uint32_t> key_len;
    DevBuf<uint8_t> sel;
    uint64_t n_nl;
    SGPU_TRY(index_newlines(c, d_buf, n, nlpos, &n_nl));
    RecParams P;
    P.in = d_buf;
    P.n_in = n;
    P.own_len = own_len;
    P.nlpos = nlpos.p;
    P.is_last = is_last;
    P.reverse = 0;
    P.crlf = 0;
    P.set = view_of(nullptr);
    if (!setup_records(P, n_nl, newlines_before, is_first)) {
        // no record boundary in the whole buffer: a record longer than the halo (or a truncated file)
        return is_last ? SGPU_ERR_FASTQ_UNEXPECTED_END : SGPU_ERR_HALO;
    }
    uint64_t n_thr = P.k_full + 1;
    SGPU_TRY(key_off.alloc(n_thr, st));
    SGPU_TRY(key_len.alloc(n_thr, st));
    SGPU_TRY(sel.alloc(n_thr, st));
    SGPU_TRY(scratch.alloc(4, st));
    uint64_t init[4] = {~0ull, 0, 0, 0};
    memcpy(c->h_pinned + 32, init, sizeof(init));
    SGPU_CUDA(cudaMemcpyAsync(scratch.p, c->h_pinned + 32, sizeof(init), cudaMemcpyHostToDevice, st));
    fastq_ids_kernel<<<(unsigned)ceil_div(n_thr, 128), 128, 0, st>>>(P, view_of(probe), want_absent, key_off.p,
                                                                      key_len.p, sel.p, (unsigned long long *)scratch.p,
                                                                      (unsigned long long *)(scratch.p + 1));
    SGPU_LAUNCH(c);
    uint64_t h[3];
    SGPU_TRY(read_u64s(c, scratch.p, h, 3));
    if (h[0] != ~0ull) {
        if (err_record) *err_record = h[0] >> 8;
        return (sgpu_status)(h[0] & 0xFF);
    }
    *n_records = h[1];
    *n_picked = h[2];
    if (into) SGPU_TRY(idset_insert_spans(c, into, d_buf, key_off.p, key_len.p, sel.p, n_thr));
    return SGPU_OK;
}

static sgpu_status clean_dev_locked(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *d_in, size_t n_in, int reverse,
                                    uint8_t *d_out_w, size_t cap_w, size_t *n_w, uint8_t *d_out_o, size_t cap_o,
                                    size_t *n_o, sgpu_counts *counts) {
    memset(counts, 0, sizeof(*counts));
    *n_w = 0;
    if (n_o) *n_o = 0;
    if (n_in && ((uintptr_t)d_in & 15)) return SGPU_ERR_INVALID_ARG;
    bool empty;
    {
        const sgpu_status src = sniff(c, d_in, n_in, &empty);
        if (src == SGPU_ERR_FASTA_UNSUPPORTED) {  // '>': needletail's FASTA reader takes over
            int le_own;
            return clean_fasta_shard(c, set, d_in, n_in, n_in, 1, 1, -1, reverse, d_out_w, cap_w, n_w, d_out_o, cap_o, n_o,
                                     counts, &le_own);
        }
        if (src != SGPU_OK) return src;
    }
    if (empty) {
        counts->empty_input = 1;
        return SGPU_OK;
    }
    if (c->mode == 0) {
        int used = 0;
        SGPU_TRY(clean_fused(c, set, d_in, n_in, reverse, d_out_w, cap_w, n_w, d_out_o, cap_o, n_o, counts, &used));
        if (used) return SGPU_OK;
        memset(counts, 0, sizeof(*counts));
    }
    return clean_general(c, set, d_in, n_in, n_in, 0, 1, 1, -1, reverse, d_out_w, cap_w, n_w, d_out_o, cap_o, n_o,
                         counts);
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

sgpu_status sgpu_clean_fastq_dev(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *d_in, size_t n_in, int reverse,
                                 uint8_t *d_out_w, size_t cap_w, size_t *n_w, uint8_t *d_out_o, size_t cap_o,
                                 size_t *n_o, sgpu_counts *counts) {
    if (!c || !set || !n_w || !counts || (n_in && !d_in) || (cap_w && !d_out_w)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    return clean_dev_locked(c, set, d_in, n_in, reverse, d_out_w, cap_w, n_w, d_out_o, cap_o, n_o, counts);
}

static sgpu_status clean_shard_locked(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *d_in, size_t n_in,
                                      size_t own_len, uint64_t newlines_before, int is_first, int is_last, int crlf,
                                      int reverse, uint8_t *d_out_w, size_t cap_w, size_t *n_w, uint8_t *d_out_o,
                                      size_t cap_o, size_t *n_o, sgpu_counts *counts, bool want_nl);

sgpu_status sgpu_clean_fastq_shard_dev(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *d_in, size_t n_in,
                                       size_t own_len, uint64_t newlines_before, int is_first, int is_last, int crlf,
                                       int reverse, uint8_t *d_out_w, size_t cap_w, size_t *n_w, uint8_t *d_out_o,
                                       size_t cap_o, size_t *n_o, sgpu_counts *counts) {
    if (!c || !set || !n_w || !counts || (n_in && !d_in) || own_len > n_in || (is_last && own_len != n_in) ||
        (is_first && newlines_before != 0) || crlf < -1 || crlf > 1 || (!is_first && crlf < 0 && newlines_before != SGPU_NEWLINES_UNKNOWN))
        return SGPU_ERR_INVALID_ARG;
    if (n_in && ((uintptr_t)d_in & 15)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    return clean_shard_locked(c, set, d_in, n_in, own_len, newlines_before, is_first, is_last, crlf, reverse, d_out_w,
                              cap_w, n_w, d_out_o, cap_o, n_o, counts, crlf < 0);
}

// shard body shared by sgpu_clean_fastq_shard_dev and the pipelined host path (context locked, device set).
// want_nl: when the single-pass kernel produces the result, counts->own_newlines is filled from its per-tile counts
static sgpu_status clean_shard_locked(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *d_in, size_t n_in,
                                      size_t own_len, uint64_t newlines_before, int is_first, int is_last, int crlf,
                                      int reverse, uint8_t *d_out_w, size_t cap_w, size_t *n_w, uint8_t *d_out_o,
                                      size_t cap_o, size_t *n_o, sgpu_counts *counts, bool want_nl) {
    memset(counts, 0, sizeof(*counts));
    *n_w = 0;
    if (n_o) *n_o = 0;
    // crlf == -1: not exchanged yet.  The single-pass kernel only takes LF input, so whatever it produces is right for a
    // file whose first record is LF (the caller checks shard 0's counts->crlf); the first shard decides it itself.
    const bool spec = !is_first && (newlines_before == SGPU_NEWLINES_UNKNOWN || crlf < 0);
    if (spec && newlines_before != SGPU_NEWLINES_UNKNOWN) return SGPU_ERR_INVALID_ARG;
    if (c->mode == 0 && crlf <= 0 && n_in >= 5) {
        int used = 0;
        SGPU_TRY(clean_fused_shard(c, set, d_in, n_in, own_len, newlines_before, is_first, is_last, reverse, d_out_w,
                                   cap_w, n_w, d_out_o, cap_o, n_o, counts, &used, want_nl));
        if (used) return SGPU_OK;
        memset(counts, 0, sizeof(*counts));
        *n_w = 0;
        if (n_o) *n_o = 0;
    }
    if (spec) return SGPU_ERR_PHASE_UNKNOWN;  // the exact protocol (newline counts exchanged first) takes over
    return clean_general(c, set, d_in, n_in, own_len, newlines_before, is_first, is_last, is_first && crlf < 0 ? -1 : (crlf ? 1 : 0),
                         reverse, d_out_w, cap_w, n_w, d_out_o, cap_o, n_o, counts);
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
template <class Fmt>
static sgpu_status pipeline_host(sgpu_ctx *c, const uint8_t *in, size_t n_in, size_t own_len, int is_last, uint8_t *out_w,
                                 size_t cap_w, size_t *n_w, uint8_t *out_o, size_t cap_o, size_t *n_o,
                                 sgpu_counts *counts, int *done, Fmt &fmt) {
    *done = 0;
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
    const size_t obuf = Fmt::OUT_FACTOR * (CHUNK + std::max(HALO, tail_halo)) + 64;
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
        cudaError_t e = cudaMemcpyAsync(d_in.p + a, in + a, len, cudaMemcpyHostToDevice, c->s_in);
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
        if (!last_chunk && is_last && a + own + HALO >= n_in) {
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
        rc = fmt.run(c, k, a, d_in.p + a, buf_len, own, last_chunk && is_last, d_w[r].p, out_o ? d_o[r].p : nullptr, obuf,
                     &nw, &no, &ck);
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
        if (off_w + nw > cap_w || (out_o && off_o + no > cap_o)) {
            rc = SGPU_ERR_CAPACITY;
            break;
        }
        cudaEventRecord(ev_k[r], st);
        cudaStreamWaitEvent(c->s_out, ev_k[r], 0);
        if (nw) ce = cudaMemcpyAsync(out_w + off_w, d_w[r].p, nw, cudaMemcpyDeviceToHost, c->s_out);
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
        memset(counts, 0, sizeof(*counts));
        *n_w = 0;
        if (n_o) *n_o = 0;
        return SGPU_ERR_PHASE_UNKNOWN;
    }
    if (bail) return SGPU_OK;  // *done stays 0
    *done = 1;
    *counts = total;
    fmt.finish(counts);
    *n_w = off_w;
    if (n_o) *n_o = out_o ? off_o : 0;
    return rc;
}

// FASTQ: the line phase of chunk k+1 comes from the running newline count.  newlines_before == SGPU_NEWLINES_UNKNOWN:
// chunk 0 speculates the line phase, the later chunks continue from it, counts->{own_newlines, lead_newlines} let the
// caller verify it.
struct FastqChunks {
    static constexpr size_t OUT_FACTOR = 1;
    const sgpu_idset *set;
    int is_first, crlf_in, reverse;
    bool spec;
    int crlf;
    uint64_t nb;  // running count: exact, or relative to the speculated phase
    uint64_t own_nl_total = 0, lead_nl = 0;

    sgpu_status run(sgpu_ctx *c, size_t k, size_t a, const uint8_t *d, size_t buf_len, size_t own, bool last, uint8_t *dw,
                    uint8_t *dov, size_t obuf, size_t *nw, size_t *no, sgpu_counts *ck) {
        const bool spec0 = spec && k == 0;
        const sgpu_status rc = clean_shard_locked(c, set, d, buf_len, own, spec0 ? SGPU_NEWLINES_UNKNOWN : nb,
                                                  is_first && k == 0, last, spec0 ? -1 : crlf, reverse, dw, obuf, nw, dov,
                                                  obuf, no, ck, true);
        if (getenv("SGPU_DEBUG"))
            fprintf(stderr, "[sgpu] pipe chunk %zu a=%zu own=%zu buf=%zu nlb=%llu -> rc=%d nw=%zu no=%zu in=%llu out=%llu path=%u own_nl=%llu lead_nl=%llu\n",
                    k, a, own, buf_len, (unsigned long long)nb, (int)rc, *nw, *no,
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

static sgpu_status clean_host_pipelined(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *in, size_t n_in, size_t own_len,
                                        uint64_t newlines_before, int is_first, int is_last, int crlf_in, int reverse,
                                        uint8_t *out_w, size_t cap_w, size_t *n_w, uint8_t *out_o, size_t cap_o,
                                        size_t *n_o, sgpu_counts *counts, int *done) {
    *done = 0;
    if (c->mode != 0) return SGPU_OK;
    if (is_first && n_in && in[0] != '@') return SGPU_OK;  // FASTA / unknown format: not this format's pipeline
    const bool spec = !is_first && newlines_before == SGPU_NEWLINES_UNKNOWN;
    int crlf = crlf_in > 0;
    if (is_first) {  // needletail decides the line ending on the first record's first line
        const uint8_t *nl = (const uint8_t *)memchr(in, '\n', n_in);
        crlf = nl && nl > in && nl[-1] == '\r';
    }
    FastqChunks f{set, is_first, crlf_in, reverse, spec, crlf, spec ? 0 : newlines_before};
    return pipeline_host(c, in, n_in, own_len, is_last, out_w, cap_w, n_w, out_o, cap_o, n_o, counts, done, f);
}

// FASTA: chunk k+1 starts from chunk k's line-ending state, le_before(k) when that was decided, else le_own(k) -- exact,
// nothing is speculated.  A chunk's output is at most twice its records' bytes (">a\n" -> ">a\r\n\r\n").
struct FastaChunks {
    static constexpr size_t OUT_FACTOR = 2;
    const sgpu_idset *set;
    int is_first, reverse;
    int le;            // le_before of the next chunk
    int le_own = -1;   // the shard's own decision: the first chunk's that has one
    int le_chunk = -1;

    sgpu_status run(sgpu_ctx *c, size_t k, size_t, const uint8_t *d, size_t buf_len, size_t own, bool last, uint8_t *dw,
                    uint8_t *dov, size_t obuf, size_t *nw, size_t *no, sgpu_counts *ck) {
        memset(ck, 0, sizeof(*ck));
        *nw = *no = 0;
        const sgpu_status rc = clean_fasta_shard(c, set, d, buf_len, own, is_first && k == 0, last, le, reverse, dw, obuf, nw,
                                                 dov, obuf, no, ck, &le_chunk);
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

static sgpu_status fasta_host_pipelined(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *in, size_t n_in, size_t own_len,
                                        int is_first, int is_last, int le_before, int reverse, uint8_t *out_w, size_t cap_w,
                                        size_t *n_w, uint8_t *out_o, size_t cap_o, size_t *n_o, sgpu_counts *counts,
                                        int *le_own, int *done) {
    FastaChunks f{set, is_first, reverse, le_before};
    const sgpu_status rc =
        pipeline_host(c, in, n_in, own_len, is_last, out_w, cap_w, n_w, out_o, cap_o, n_o, counts, done, f);
    *le_own = f.le_own;
    return rc;
}

// the one-shot host path: the whole buffer on the device, `call(d_in, d_w, cap_w, d_o, cap_o)` on it, outputs back.
// write_fastq's output is the input re-serialised: larger only when line endings are rewritten (FASTQ: LF records
// after a CRLF first record) or FASTA header-only records gain an empty sequence line.  Device buffers are sized for
// the common case first.
template <class Call>
static sgpu_status oneshot_host(sgpu_ctx *c, const uint8_t *in, size_t n_in, uint8_t *out_w, size_t cap_w, size_t *n_w,
                                uint8_t *out_o, size_t cap_o, size_t *n_o, Call call) {
    cudaStream_t st = c->stream;
    DevBuf<uint8_t> d_in, d_w, d_o;
    SGPU_TRY(d_in.alloc(n_in + 16, st));
    if (n_in) SGPU_CUDA(cudaMemcpyAsync(d_in.p, in, n_in, cudaMemcpyHostToDevice, st));
    sgpu_status rc = SGPU_OK;
    for (int attempt = 0; attempt < 2; attempt++) {
        const size_t want = attempt ? ~(size_t)0 : n_in + n_in / 16 + 4096;
        const size_t dcap_w = std::min(cap_w, want), dcap_o = std::min(cap_o, want);
        SGPU_TRY(d_w.alloc(dcap_w + 16, st));
        if (out_o) SGPU_TRY(d_o.alloc(dcap_o + 16, st));
        rc = call(d_in.p, d_w.p, dcap_w, out_o ? d_o.p : nullptr, dcap_o);
        if (rc != SGPU_ERR_CAPACITY || (dcap_w == cap_w && (!out_o || dcap_o == cap_o))) break;
    }
    if (rc == SGPU_ERR_CAPACITY || rc == SGPU_ERR_CUDA || rc == SGPU_ERR_NOMEM || rc == SGPU_ERR_PHASE_UNKNOWN) return rc;
    if (*n_w) SGPU_CUDA(cudaMemcpyAsync(out_w, d_w.p, *n_w, cudaMemcpyDeviceToHost, st));
    if (out_o && n_o && *n_o) SGPU_CUDA(cudaMemcpyAsync(out_o, d_o.p, *n_o, cudaMemcpyDeviceToHost, st));
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
    {
        int done = 0, le_own;
        sgpu_status prc = n_in >= 5 && in[0] == '>'
                              ? fasta_host_pipelined(c, set, in, n_in, n_in, 1, 1, -1, reverse, out_w, cap_w, n_w, out_o,
                                                     cap_o, n_o, counts, &le_own, &done)
                              : clean_host_pipelined(c, set, in, n_in, n_in, 0, 1, 1, -1, reverse, out_w, cap_w, n_w, out_o,
                                                     cap_o, n_o, counts, &done);
        if (done || prc != SGPU_OK) return prc;
    }
    return oneshot_host(c, in, n_in, out_w, cap_w, n_w, out_o, cap_o, n_o,
                        [&](const uint8_t *d_in, uint8_t *d_w, size_t dcap_w, uint8_t *d_o, size_t dcap_o) {
                            return clean_dev_locked(c, set, d_in, n_in, reverse, d_w, dcap_w, n_w, d_o, dcap_o, n_o, counts);
                        });
}

sgpu_status sgpu_clean_fastq_shard(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *in, size_t n_in, size_t own_len,
                                   uint64_t newlines_before, int is_first, int is_last, int crlf, int reverse,
                                   uint8_t *out_w, size_t cap_w, size_t *n_w, uint8_t *out_o, size_t cap_o, size_t *n_o,
                                   sgpu_counts *counts) {
    if (!c || !set || !n_w || !counts || (n_in && !in) || (cap_w && !out_w) || own_len > n_in ||
        (is_last && own_len != n_in) || (is_first && newlines_before != 0) || crlf < -1 || crlf > 1 ||
        (!is_first && crlf < 0 && newlines_before != SGPU_NEWLINES_UNKNOWN))
        return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    {
        int done = 0;
        sgpu_status prc = clean_host_pipelined(c, set, in, n_in, own_len, newlines_before, is_first, is_last, crlf, reverse,
                                               out_w, cap_w, n_w, out_o, cap_o, n_o, counts, &done);
        if (done || prc != SGPU_OK) return prc;
    }
    return oneshot_host(c, in, n_in, out_w, cap_w, n_w, out_o, cap_o, n_o,
                        [&](const uint8_t *d_in, uint8_t *d_w, size_t dcap_w, uint8_t *d_o, size_t dcap_o) {
                            return clean_shard_locked(c, set, d_in, n_in, own_len, newlines_before, is_first, is_last, crlf,
                                                      reverse, d_w, dcap_w, n_w, d_o, dcap_o, n_o, counts, crlf < 0);
                        });
}

// argument checks shared by the FASTA shard entry points
static bool fasta_shard_args_ok(size_t n_in, size_t own_len, int is_last, int le_before, int is_first) {
    return own_len <= n_in && (!is_last || own_len == n_in) && le_before >= -1 && le_before <= 1 &&
           (!is_first || le_before == -1);
}

// the FASTA shard's first byte and the empty-input rule (context locked).  *empty: a first-and-last shard of fewer
// than 5 bytes (utils.rs:359-375); SGPU_ERR_INVALID_ARG: a first shard that does not start with '>'
static sgpu_status fasta_shard_head(sgpu_ctx *c, const uint8_t *buf, bool on_device, size_t n_in, int is_first,
                                    int is_last, bool *empty) {
    *empty = is_first && is_last && n_in < 5;
    if (*empty || !is_first) return SGPU_OK;
    if (n_in == 0) return SGPU_ERR_INVALID_ARG;
    if (!on_device) return buf[0] == '>' ? SGPU_OK : SGPU_ERR_INVALID_ARG;
    SGPU_CUDA(cudaMemcpyAsync(c->h_pinned, buf, 1, cudaMemcpyDeviceToHost, c->stream));
    SGPU_CUDA(cudaStreamSynchronize(c->stream));
    return *(uint8_t *)c->h_pinned == '>' ? SGPU_OK : SGPU_ERR_INVALID_ARG;
}

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
    memset(counts, 0, sizeof(*counts));
    *n_w = 0;
    if (n_o) *n_o = 0;
    *le_own = -1;
    bool empty;
    SGPU_TRY(fasta_shard_head(c, d_in, true, n_in, is_first, is_last, &empty));
    if (empty) {
        counts->empty_input = 1;
        return SGPU_OK;
    }
    return clean_fasta_shard(c, set, d_in, n_in, own_len, is_first, is_last, le_before, reverse, d_out_w, cap_w, n_w, d_out_o,
                             cap_o, n_o, counts, le_own);
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
    memset(counts, 0, sizeof(*counts));
    *n_w = 0;
    if (n_o) *n_o = 0;
    *le_own = -1;
    bool empty;
    SGPU_TRY(fasta_shard_head(c, in, false, n_in, is_first, is_last, &empty));
    if (empty) {
        counts->empty_input = 1;
        return SGPU_OK;
    }
    {
        int done = 0;
        sgpu_status prc = fasta_host_pipelined(c, set, in, n_in, own_len, is_first, is_last, le_before, reverse, out_w, cap_w,
                                               n_w, out_o, cap_o, n_o, counts, le_own, &done);
        if (done || prc != SGPU_OK) return prc;
    }
    return oneshot_host(c, in, n_in, out_w, cap_w, n_w, out_o, cap_o, n_o,
                        [&](const uint8_t *d_in, uint8_t *d_w, size_t dcap_w, uint8_t *d_o, size_t dcap_o) {
                            memset(counts, 0, sizeof(*counts));
                            return clean_fasta_shard(c, set, d_in, n_in, own_len, is_first, is_last, le_before, reverse, d_w,
                                                     dcap_w, n_w, d_o, dcap_o, n_o, counts, le_own);
                        });
}

sgpu_status sgpu_fasta_ids_shard_dev(sgpu_ctx *c, const sgpu_idset *probe, const uint8_t *d_buf, size_t n_buf,
                                     size_t own_len, int is_first, int is_last, sgpu_idset *into, sgpu_counts *counts) {
    if (!c || !counts || (n_buf && !d_buf) || !fasta_shard_args_ok(n_buf, own_len, is_last, -1, is_first))
        return SGPU_ERR_INVALID_ARG;
    if (n_buf && ((uintptr_t)d_buf & 15)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    bool empty;
    SGPU_TRY(fasta_shard_head(c, d_buf, true, n_buf, is_first, is_last, &empty));
    if (empty) return SGPU_OK;
    uint64_t n_rec = 0, n_pick = 0, err = 0;
    sgpu_status rc = fasta_ids_shard(c, d_buf, n_buf, own_len, is_first, is_last, probe, probe != nullptr, into, &n_rec,
                                     &n_pick, &err);
    if (rc == SGPU_OK) {
        counts->reads_in += n_rec;
        counts->difference += n_pick;
    } else {
        counts->error_record = err;
    }
    cudaStreamSynchronize(c->stream);
    return rc;
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
    sgpu_status rc = fastq_ids_into(c, d_out, n_out, n_out, 0, 1, 1, nullptr, 0, o_ids, &n_rec, &n_pick, &err);  // :259-267
    if (rc == SGPU_OK) {
        counts->reads_out += n_rec;
        rc = fastq_ids_into(c, d_in, n_in, n_in, 0, 1, 1, o_ids, 1, *diff_ids, &n_rec, &n_pick, &err);  // :269-283
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
    if (!c || !counts || (n_buf && !d_buf) || own_len > n_buf || (is_last && own_len != n_buf) ||
        (is_first && newlines_before != 0))
        return SGPU_ERR_INVALID_ARG;
    if (n_buf && ((uintptr_t)d_buf & 15)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    uint64_t n_rec = 0, n_pick = 0, err = 0;
    sgpu_counts spec;
    memset(&spec, 0, sizeof(spec));
    sgpu_status rc = fastq_ids_into(c, d_buf, n_buf, own_len, newlines_before, is_first, is_last, probe, probe != nullptr,
                                    into, &n_rec, &n_pick, &err, &spec);
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

}  // extern "C"
