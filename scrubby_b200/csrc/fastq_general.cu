// fastq_general.cu -- the FASTQ shard core (clean_fastq_shard, fastq_ids_shard) and its GENERAL (always exact) path.
//
// Replaces FastqCleaner::clean_reads (cleaner.rs:731-760), needletail 0.5.1's fastq
// Reader::next/validate/check_end + write_fastq, get_id (utils.rs:91-103), and the loops of
// ReadDifference::get_difference (utils.rs:259-283).
//
// Both operations work on a shard; a whole file is the shard (n, n, newlines_before 0, first, last, crlf -1).
// The fused single-pass kernel (fastq_fused.cu) runs first and takes canonical input; everything else
// goes through the general path, whose record table (fastq_records) clean and ids share:
//   1. '\n' index (scan.cu)                       -> nlpos[]
//   2. fastq_record_kernel: thread per record     -> validation, trimmed spans, id, probe,
//                                                    normalised output length
//      (ids: fastq_ids_kernel -> id spans of the wanted records)
//   3. exclusive scans of the written / other lengths
//   4. fastq_copy_kernel: warp per record         -> '@' id E seq E '+' E qual E
// It handles CRLF, "+id" separator lines, a missing final newline, blank tails, non-ASCII
// headers, every parse error class, and shards cut at arbitrary byte offsets.
#include "fastq_records.cuh"

namespace sgpu {

__global__ void __launch_bounds__(128)
    fastq_record_kernel(RecParams P, RecMeta *meta, uint32_t *len_w, uint32_t *len_o, unsigned long long *err_word) {
    uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k > P.k_full) return;
    uint32_t lw = 0, lo = 0;
    RecMeta m = {0, 0, 0, 0};
    uint64_t start, p1, p3;
    size_t id_off = 0, id_len = 0;
    if (locate_record(P, k, &start, &p1, &p3, &m, &id_off, &id_len, err_word)) {
        bool hit = id_len <= IDSET_MAX_KEY && idset_contains(P.set, P.in + start + 1 + id_off, (uint32_t)id_len);
        bool written = P.reverse ? hit : !hit;
        uint32_t e = P.crlf ? 2u : 1u;
        uint32_t out_len = 2u + m.id_n + m.seq_n + m.qual_n + 4u * e;
        m.flags = 1u | (written ? 2u : 0u);
        if (written) lw = out_len; else lo = out_len;
    }
    meta[k] = m;
    len_w[k] = lw;
    len_o[k] = lo;
}

// records at or after the first error are not produced (the reference stops there)
__global__ void fastq_mask_kernel(RecMeta *meta, uint32_t *len_w, uint32_t *len_o, uint64_t from, uint64_t n) {
    uint64_t k = from + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    meta[k].flags = 0;
    len_w[k] = 0;
    len_o[k] = 0;
}

__global__ void fastq_count_kernel(const RecMeta *meta, uint64_t n, unsigned long long *counters) {
    uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t f = k < n ? meta[k].flags : 0;
    // one pair of atomics per block (per warp they queue up on two addresses: 0.2 ms per 5 M records)
    const int bi = __syncthreads_count(f & 1u), bo = __syncthreads_count(f & 2u);
    if (threadIdx.x == 0) {
        if (bi) atomicAdd(&counters[0], (unsigned long long)bi);
        if (bo) atomicAdd(&counters[1], (unsigned long long)bo);
    }
}

__global__ void __launch_bounds__(256)
    fastq_copy_kernel(RecParams P, const RecMeta *meta, const uint64_t *off_w, const uint64_t *off_o, uint8_t *out_w,
                      uint8_t *out_o, uint64_t n_rec) {
    uint64_t k = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (k >= n_rec) return;
    RecMeta m = meta[k];
    if (!(m.flags & 1u)) return;
    uint8_t *dst;
    if (m.flags & 2u) {
        dst = out_w + off_w[k];
    } else {
        if (!out_o) return;
        dst = out_o + off_o[k];
    }
    uint64_t b = P.b0 + 4 * k;
    uint64_t start = (b == 0) ? 0 : P.nlpos[b - 1] + 1;
    uint64_t p1 = P.nlpos[b], p3 = P.nlpos[b + 2];
    const uint8_t *in = P.in;
    const uint32_t e = P.crlf ? 2u : 1u;
    // '@' id E
    if (lane == 0) dst[0] = '@';
    warp_copy(dst + 1, in + start + 1, m.id_n, lane);
    uint8_t *q = dst + 1 + m.id_n;
    if (lane == 0) {
        if (P.crlf) q[0] = '\r';
        q[e - 1] = '\n';
    }
    q += e;
    // seq E '+' E
    warp_copy(q, in + p1 + 1, m.seq_n, lane);
    q += m.seq_n;
    if (lane == 0) {
        uint32_t w = 0;
        if (P.crlf) q[w++] = '\r';
        q[w++] = '\n';
        q[w++] = '+';
        if (P.crlf) q[w++] = '\r';
        q[w++] = '\n';
    }
    q += 2 * e + 1;
    // qual E
    warp_copy(q, in + p3 + 1, m.qual_n, lane);
    q += m.qual_n;
    if (lane == 0) {
        if (P.crlf) q[0] = '\r';
        q[e - 1] = '\n';
    }
}

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

// the record table of a FASTQ shard (the '\n' index and RecParams over it) and its scratch words ([0] the error word,
// the rest zero); shared by clean and ids.  P.crlf is left to the caller.  *any = false: the shard owns no record
// boundary (nothing is allocated after the index)
struct FqTable {
    DevBuf<uint64_t> nlpos, scratch;
    RecParams P;
};

static sgpu_status fastq_records(sgpu_ctx *c, const Shard &s, uint64_t newlines_before, const sgpu_idset *set,
                                 int reverse, FqTable &T, bool *any) {
    uint64_t n_nl = 0;
    SGPU_TRY(index_newlines(c, s.p, s.n, T.nlpos, &n_nl));
    RecParams &P = T.P;
    P.in = s.p;
    P.n_in = s.n;
    P.own_len = s.own_len;
    P.nlpos = T.nlpos.p;
    P.is_last = s.is_last;
    P.reverse = reverse;
    P.crlf = 0;
    P.set = view_of(set);
    *any = setup_records(P, n_nl, newlines_before, s.is_first);
    if (!*any) return SGPU_OK;
    SGPU_TRY(T.scratch.alloc(8, c->stream));
    const uint64_t init[8] = {~0ull, 0, 0, 0, 0, 0, 0, 0};
    return write_u64s(c, T.scratch.p, init, 8);
}

// the general path: device pointers in, device outputs filled, counts on the host
static sgpu_status clean_general(sgpu_ctx *c, const sgpu_idset *set, const Shard &s, uint64_t newlines_before,
                                 int crlf_in, int reverse, const Outs &out, sgpu_counts *counts) {
    cudaStream_t st = c->stream;
    counts->path = 2;
    FqTable T;
    bool any;
    SGPU_TRY(fastq_records(c, s, newlines_before, set, reverse, T, &any));
    RecParams &P = T.P;
    int crlf = crlf_in;
    if (s.is_first && crlf_in < 0) {
        // find_line_ending on the first record: is its first '\n' preceded by '\r'?
        crlf = 0;
        if (P.n_nl >= 1) {
            uint64_t p0;
            SGPU_TRY(read_u64s(c, T.nlpos.p, &p0, 1));
            if (p0 > 0) {
                uint8_t ch;
                SGPU_CUDA(cudaMemcpyAsync(c->h_pinned, s.p + p0 - 1, 1, cudaMemcpyDeviceToHost, st));
                SGPU_CUDA(cudaStreamSynchronize(st));
                ch = *(uint8_t *)c->h_pinned;
                crlf = ch == '\r';
            }
        }
    }
    P.crlf = crlf;
    counts->crlf = (uint32_t)crlf;
    if (!any) return SGPU_OK;  // a non-first shard without a single record boundary: it owns no record start
    uint64_t n_thr = P.k_full + 1;  // + the tail candidate

    DevBuf<RecMeta> meta;
    DevBuf<uint32_t> len_w, len_o;
    DevBuf<uint64_t> off_w, off_o;
    uint64_t *scratch = T.scratch.p;  // [0] err word, [1] total_w, [2] total_o, [3] reads_in, [4] reads_out
    SGPU_TRY(meta.alloc(n_thr, st));
    SGPU_TRY(len_w.alloc(n_thr, st));
    SGPU_TRY(len_o.alloc(n_thr, st));
    SGPU_TRY(off_w.alloc(n_thr, st));

    fastq_record_kernel<<<(unsigned)ceil_div(n_thr, 128), 128, 0, st>>>(P, meta.p, len_w.p, len_o.p,
                                                                         (unsigned long long *)scratch);
    SGPU_LAUNCH(c);
    uint64_t err_word;
    SGPU_TRY(read_u64s(c, scratch, &err_word, 1));
    sgpu_status rc = SGPU_OK;
    if (err_word != ~0ull) {
        rc = (sgpu_status)(err_word & 0xFF);
        counts->error_record = err_word >> 8;
        if (rc == SGPU_ERR_HALO) return rc;
        uint64_t from = err_word >> 8;
        fastq_mask_kernel<<<(unsigned)ceil_div(n_thr - from, 256), 256, 0, st>>>(meta.p, len_w.p, len_o.p, from,
                                                                                 n_thr);
        SGPU_LAUNCH(c);
    }
    fastq_count_kernel<<<(unsigned)ceil_div(n_thr, 256), 256, 0, st>>>(meta.p, n_thr,
                                                                        (unsigned long long *)(scratch + 3));
    SGPU_LAUNCH(c);
    SGPU_TRY(exclusive_scan_u32_to_u64(c, len_w.p, off_w.p, n_thr, scratch + 1));
    if (out.o) {
        SGPU_TRY(off_o.alloc(n_thr, st));
        SGPU_TRY(exclusive_scan_u32_to_u64(c, len_o.p, off_o.p, n_thr, scratch + 2));
    }
    uint64_t h[5];
    SGPU_TRY(read_u64s(c, scratch, h, 5));
    *out.n_w = (size_t)h[1];
    if (out.n_o) *out.n_o = out.o ? (size_t)h[2] : 0;
    counts->reads_in = h[3];
    counts->reads_out = h[4];
    if (h[1] > out.cap_w || (out.o && h[2] > out.cap_o)) return SGPU_ERR_CAPACITY;
    fastq_copy_kernel<<<(unsigned)ceil_div(n_thr * 32, 256), 256, 0, st>>>(P, meta.p, off_w.p, off_o.p, out.w, out.o,
                                                                           n_thr);
    SGPU_LAUNCH(c);
    SGPU_CUDA(cudaGetLastError());
    SGPU_CUDA(cudaStreamSynchronize(st));  // scratch buffers are released after this call returns
    return rc;
}

sgpu_status clean_fastq_shard(sgpu_ctx *c, const sgpu_idset *set, const Shard &s, uint64_t newlines_before, int crlf,
                              int reverse, const Outs &out, sgpu_counts *counts, bool want_nl) {
    clear_outputs(out, counts);
    // crlf == -1: not exchanged yet.  The single-pass kernel only takes LF input, so whatever it produces is right for a
    // file whose first record is LF (the caller checks shard 0's counts->crlf); the first shard decides it itself.
    const bool spec = !s.is_first && (newlines_before == SGPU_NEWLINES_UNKNOWN || crlf < 0);
    if (spec && newlines_before != SGPU_NEWLINES_UNKNOWN) return SGPU_ERR_INVALID_ARG;
    if (c->mode == 0 && crlf <= 0 && s.n >= 5) {
        int used = 0;
        SGPU_TRY(fused_shard(c, set, s, newlines_before, reverse, out, nullptr, counts, &used, want_nl));
        if (used) return SGPU_OK;
        clear_outputs(out, counts);
    }
    if (spec) return SGPU_ERR_PHASE_UNKNOWN;  // the exact protocol (newline counts exchanged first) takes over
    return clean_general(c, set, s, newlines_before, s.is_first && crlf < 0 ? -1 : (crlf ? 1 : 0), reverse, out, counts);
}

sgpu_status fastq_ids_shard(sgpu_ctx *c, const Shard &s, uint64_t newlines_before, const sgpu_idset *probe,
                            int want_absent, const SpanSink &sink, uint64_t *n_records, uint64_t *n_picked,
                            uint64_t *err_record, sgpu_counts *spec_out) {
    *n_records = *n_picked = 0;
    if (!s.is_first && (s.n == 0 || s.own_len == 0)) return SGPU_OK;
    const bool spec = !s.is_first && newlines_before == SGPU_NEWLINES_UNKNOWN;
    cudaStream_t st = c->stream;
    if (c->mode == 0 && ((uintptr_t)s.p & 15) == 0) {
        // canonical input: one pass of the fused kernel in ids mode -> (offset, length) spans of the wanted ids
        DevBuf<uint64_t> s_off;
        DevBuf<uint32_t> s_len;
        const uint64_t cap = s.n / 100 + 4096;  // the fused kernel handles >= ~102 bytes per record
        SGPU_TRY(s_off.alloc(cap, st));
        SGPU_TRY(s_len.alloc(cap, st));
        IdsOut ids{s_off.p, s_len.p, cap, 0, 0};
        sgpu_counts ck;
        memset(&ck, 0, sizeof(ck));
        int used = 0;
        SGPU_TRY(fused_shard(c, want_absent ? probe : nullptr, s, newlines_before, 0, Outs{}, &ids, &ck, &used, false));
        if (spec_out) *spec_out = ck;
        if (used) {
            *n_records = ck.reads_in;
            *n_picked = ids.n_spans;
            if (ids.n_spans)  // (listed in tile completion order)
                SGPU_TRY(sink_spans(c, sink, s.p + ids.base, s_off.p, s_len.p, nullptr, (size_t)ids.n_spans, false,
                                    s.n - ids.base));
            return SGPU_OK;
        }
    }
    if (spec) return SGPU_ERR_PHASE_UNKNOWN;
    FqTable T;
    bool any;
    SGPU_TRY(fastq_records(c, s, newlines_before, nullptr, 0, T, &any));
    // no record boundary in the whole buffer: a record longer than the halo (or a truncated file)
    if (!any) return s.is_last ? SGPU_ERR_FASTQ_UNEXPECTED_END : SGPU_ERR_HALO;
    DevBuf<uint64_t> key_off;
    DevBuf<uint32_t> key_len;
    DevBuf<uint8_t> sel;
    const uint64_t n_thr = T.P.k_full + 1;
    SGPU_TRY(key_off.alloc(n_thr, st));
    SGPU_TRY(key_len.alloc(n_thr, st));
    SGPU_TRY(sel.alloc(n_thr, st));
    fastq_ids_kernel<<<(unsigned)ceil_div(n_thr, 128), 128, 0, st>>>(T.P, view_of(probe), want_absent, key_off.p,
                                                                      key_len.p, sel.p,
                                                                      (unsigned long long *)T.scratch.p,
                                                                      (unsigned long long *)(T.scratch.p + 1));
    SGPU_LAUNCH(c);
    uint64_t h[3];
    SGPU_TRY(read_u64s(c, T.scratch.p, h, 3));
    if (h[0] != ~0ull) {
        if (err_record) *err_record = h[0] >> 8;
        return (sgpu_status)(h[0] & 0xFF);
    }
    *n_records = h[1];
    *n_picked = h[2];
    SGPU_TRY(sink_spans(c, sink, s.p, key_off.p, key_len.p, sel.p, n_thr));
    return SGPU_OK;
}

}  // namespace sgpu
