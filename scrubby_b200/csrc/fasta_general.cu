// fasta_general.cu -- FASTA input (SURVEY 8f row 4): needletail switches to its FASTA reader when the first byte is
// '>' (utils.rs:377-383 parse_fastx_file), and FastqCleaner::clean_reads (cleaner.rs:731-760) / ReadDifference
// (utils.rs:250-285) then run unchanged on those records.
//
// needletail 0.5.1 fasta::Reader::next / find / _find restated (un-vendored dependency; parity unpinned; the same
// rules are listed in include/scrubby_gpu.h):
//   record  : from its '>' to the newline in front of the next "\n>" (or the end of the input);
//   seq_pos : the record's newline positions, except a newline on the LAST byte of the input, which is appended at end
//             of input only when an earlier one exists; without a trailing newline the end of the input is appended;
//   id      = trim_cr(buf[start+1 .. first)), raw_seq = trim_cr(buf[first+1 .. last)) when there are >= 2 positions, else
//             empty; inner line breaks of a multi-line sequence are kept verbatim (write_fasta gets raw_seq);
//   a record without a position is UnexpectedEnd; the line ending comes from the first record whose [start, last)
//   holds a newline, records written before that use LF;
//   output  : '>' id E raw_seq E.
//
// Pipeline (a whole file, or one shard of it: the contract is written down in include/scrubby_gpu.h):
//   newline index (scan.cu) -> mark the newlines followed by '>' (and count the owned ones) -> scan -> record table ->
//   thread per owned record (spans, get_id, probe) -> line-ending decision -> lengths -> scans -> warp per record copy.
// A whole file is the shard (own_len = n, is_first = 1, is_last = 1, le_before = -1).
#include "fastq_records.cuh"

namespace sgpu {

struct FaParams {
    const uint8_t *in;
    uint64_t n_in;
    const uint64_t *nlpos;
    uint64_t n_nl;
    const uint64_t *rec_nl;  // record k starts right after newline rec_nl[k] (record 0 of a first shard: at byte 0)
    uint64_t n_rec;          // records the shard owns
    uint64_t n_tab;          // entries of rec_nl: the owned records + the next record start, when the buffer holds it
    int at0;                 // record 0 starts at byte 0 (first shard); rec_nl[0] is then unused
};

struct FaMeta {
    uint64_t seq;  // offset of raw_seq
    uint32_t id_n, seq_n;
    uint32_t flags;  // bit0 valid, bit1 written, bit2 the record's [start, last) holds a newline, bit3 that one follows a CR
    uint32_t pad;
};

// record starts: a '>' that follows a newline; the shard owns those with the newline before own_len
__global__ void fa_mark_kernel(const uint8_t *in, uint64_t n_in, const uint64_t *nlpos, uint64_t n_nl, uint64_t own_len,
                               uint32_t *mark, unsigned long long *n_owned) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t m = 0;
    uint64_t p = 0;
    if (j < n_nl) {
        p = nlpos[j];
        m = (p + 1 < n_in && in[p + 1] == '>') ? 1u : 0u;
        mark[j] = m;
    }
    const int owned = __syncthreads_count(m && p < own_len);
    if (threadIdx.x == 0 && owned) atomicAdd(n_owned, (unsigned long long)owned);
}

__global__ void fa_scatter_kernel(const uint32_t *mark, const uint64_t *rank, uint64_t n_nl, uint64_t *rec_nl) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_nl) return;
    if (mark[j]) rec_nl[rank[j] + 1] = j;
}

__device__ __forceinline__ uint64_t fa_start(const FaParams &P, uint64_t k) {
    return (k == 0 && P.at0) ? 0 : P.nlpos[P.rec_nl[k]] + 1;
}

// start byte, first / last position of record k; false when the record has no position (UnexpectedEnd)
__device__ __forceinline__ bool fa_locate(const FaParams &P, uint64_t k, uint64_t *start, uint64_t *first, uint64_t *last,
                                          uint32_t *npos) {
    const uint64_t f = (k == 0 && P.at0) ? 0 : P.rec_nl[k] + 1;  // index of the first newline at or after the start
    *start = fa_start(P, k);
    if (k + 1 < P.n_tab) {  // the newline in front of the next '>' closes the record
        const uint64_t l = P.rec_nl[k + 1];
        *first = P.nlpos[f];
        *last = P.nlpos[l];
        *npos = (uint32_t)(l - f + 1 > 2 ? 2 : l - f + 1);
        return true;
    }
    // the last record of the input (only the last shard gets here): newlines f .. n_nl-1; one on the input's last byte
    // only counts after another one
    uint64_t cnt = P.n_nl > f ? P.n_nl - f : 0;
    const bool trailing = cnt && P.nlpos[P.n_nl - 1] + 1 == P.n_in;
    if (trailing && cnt == 1) cnt = 0;
    if (cnt == 0) return false;
    *first = P.nlpos[f];
    if (trailing) {
        *last = P.nlpos[P.n_nl - 1];
        *npos = cnt > 2 ? 2u : (uint32_t)cnt;
    } else {
        *last = P.n_in;  // no trailing newline: the end of the input closes the last line
        *npos = 2;
    }
    return true;
}

// one thread per record: spans, get_id, probe.  ids mode (key_off != nullptr): the id span of every record that is
// absent from the set (all records when want_absent == 0) is offered for insertion
__global__ void __launch_bounds__(128)
    fa_record_kernel(FaParams P, IdSetView set, int reverse, int want_absent, FaMeta *meta, uint64_t *key_off,
                     uint32_t *key_len, uint8_t *sel, unsigned long long *err_word, unsigned long long *first_le) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= P.n_rec) return;
    FaMeta m = {0, 0, 0, 0, 0};
    uint64_t koff = 0;
    uint32_t klen = 0;
    uint8_t pick = 0;
    uint64_t start, first, last;
    uint32_t npos;
    if (!fa_locate(P, k, &start, &first, &last, &npos)) {
        report_error(err_word, k, SGPU_ERR_FASTQ_UNEXPECTED_END);
    } else {
        const uint8_t *in = P.in;
        m.id_n = trim_cr_len(in + start + 1, first - (start + 1));
        m.seq = first + 1;
        m.seq_n = npos > 1 ? trim_cr_len(in + first + 1, last - (first + 1)) : 0u;
        size_t id_off = 0, id_len = 0;
        const int code = get_id_span(in + start + 1, m.id_n, &id_off, &id_len);
        if (code) {
            report_error(err_word, k, code);
        } else {
            const bool hit = id_len <= IDSET_MAX_KEY && idset_contains(set, in + start + 1 + id_off, (uint32_t)id_len);
            const bool written = reverse ? hit : !hit;
            m.flags = 1u | (written ? 2u : 0u);
            if (first < last) {  // find_line_ending over [start, last): this record can decide the line ending
                m.flags |= 4u | ((first > start && in[first - 1] == '\r') ? 8u : 0u);
                atomicMin(first_le, (unsigned long long)k);
            }
            koff = start + 1 + id_off;
            klen = (uint32_t)id_len;
            pick = want_absent ? (hit ? 0 : 1) : 1;
        }
    }
    meta[k] = m;
    if (key_off) {
        key_off[k] = koff;
        key_len[k] = klen;
        sel[k] = pick;
    }
}

// output length of every record; records at or after the first error are not produced (the reference stops there)
__global__ void fa_len_kernel(FaMeta *meta, uint64_t n_rec, uint64_t err_from, uint64_t le_from, int crlf, uint32_t *len_w,
                              uint32_t *len_o, unsigned long long *counters) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t lw = 0, lo = 0, f = 0;
    if (k < n_rec) {
        FaMeta m = meta[k];
        if (k >= err_from) m.flags = 0;
        f = m.flags;
        if (f & 1u) {
            const uint32_t e = (crlf && k >= le_from) ? 2u : 1u;
            const uint32_t out_len = 1u + m.id_n + m.seq_n + 2u * e;
            if (f & 2u) lw = out_len; else lo = out_len;
        }
        meta[k].flags = f;
        len_w[k] = lw;
        len_o[k] = lo;
    }
    const int bi = __syncthreads_count(f & 1u), bo = __syncthreads_count(f & 2u);
    if (threadIdx.x == 0) {
        if (bi) atomicAdd(&counters[0], (unsigned long long)bi);
        if (bo) atomicAdd(&counters[1], (unsigned long long)bo);
    }
}

__global__ void __launch_bounds__(256)
    fa_copy_kernel(FaParams P, const FaMeta *meta, const uint64_t *off_w, const uint64_t *off_o, uint64_t le_from, int crlf,
                   uint8_t *out_w, uint8_t *out_o) {
    const uint64_t k = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (k >= P.n_rec) return;
    const FaMeta m = meta[k];
    if (!(m.flags & 1u)) return;
    uint8_t *dst;
    if (m.flags & 2u) {
        dst = out_w + off_w[k];
    } else {
        if (!out_o) return;
        dst = out_o + off_o[k];
    }
    const uint64_t start = fa_start(P, k);
    const uint32_t e = (crlf && k >= le_from) ? 2u : 1u;
    if (lane == 0) dst[0] = '>';
    warp_copy(dst + 1, P.in + start + 1, m.id_n, lane);
    uint8_t *q = dst + 1 + m.id_n;
    if (lane == 0) {
        if (e == 2) q[0] = '\r';
        q[e - 1] = '\n';
    }
    q += e;
    warp_copy(q, P.in + m.seq, m.seq_n, lane);
    q += m.seq_n;
    if (lane == 0) {
        if (e == 2) q[0] = '\r';
        q[e - 1] = '\n';
    }
}

__global__ void fa_count_sel_kernel(const uint8_t *sel, uint64_t n, unsigned long long *counter) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int b = __syncthreads_count(k < n && sel[k]);
    if (threadIdx.x == 0 && b) atomicAdd(counter, (unsigned long long)b);
}

// the record table of a FASTA shard + the per-record pass; shared by clean and ids
struct FaTables {
    DevBuf<uint64_t> nlpos, rank, rec_nl, key_off, scratch;
    DevBuf<uint32_t> mark, key_len;
    DevBuf<uint8_t> sel;
    DevBuf<FaMeta> meta;
    FaParams P;
    uint64_t err_word = ~0ull, le_from = ~0ull;
};

// SGPU_ERR_HALO: a shard that is not the last one does not hold the start of the record after its last owned one.
// T.P.n_rec == 0: the shard owns no record (nothing was launched after the table)
static sgpu_status fasta_records(sgpu_ctx *c, const Shard &s, const sgpu_idset *set, int reverse, int want_absent,
                                 bool want_keys, FaTables &T) {
    cudaStream_t st = c->stream;
    // [0] err word, [1] first record that decides the line ending, [2] starts, [3..4] counters, [5..6] totals, [7] owned starts
    SGPU_TRY(T.scratch.alloc(8, st));
    const uint64_t init[8] = {~0ull, ~0ull, 0, 0, 0, 0, 0, 0};
    SGPU_TRY(write_u64s(c, T.scratch.p, init, 8));
    uint64_t n_nl = 0;
    SGPU_TRY(index_newlines(c, s.p, s.n, T.nlpos, &n_nl));
    uint64_t h[6] = {0, 0, 0, 0, 0, 0};  // scratch [2..7]
    if (n_nl) {
        SGPU_TRY(T.mark.alloc(n_nl, st));
        SGPU_TRY(T.rank.alloc(n_nl, st));
        fa_mark_kernel<<<(unsigned)ceil_div(n_nl, (uint64_t)256), 256, 0, st>>>(s.p, s.n, T.nlpos.p, n_nl, s.own_len,
                                                                                T.mark.p,
                                                                                (unsigned long long *)(T.scratch.p + 7));
        SGPU_LAUNCH(c);
        SGPU_TRY(exclusive_scan_u32_to_u64(c, T.mark.p, T.rank.p, n_nl, T.scratch.p + 2));
        SGPU_TRY(read_u64s(c, T.scratch.p + 2, h, 6));
    }
    const uint64_t n_starts = h[0], n_owned = h[5];
    const uint64_t n_rec = (s.is_first ? 1 : 0) + n_owned;
    const uint64_t n_tab = (s.is_first ? 1 : 0) + n_starts;
    T.P = FaParams{s.p, (uint64_t)s.n, T.nlpos.p, n_nl, nullptr, n_rec, n_tab, s.is_first ? 1 : 0};
    if (n_rec == 0) return SGPU_OK;
    if (!s.is_last && n_tab == n_rec) return SGPU_ERR_HALO;  // the end of the last owned record is not in the buffer
    SGPU_TRY(T.rec_nl.alloc(n_starts + 1, st));
    if (n_starts) {
        fa_scatter_kernel<<<(unsigned)ceil_div(n_nl, (uint64_t)256), 256, 0, st>>>(T.mark.p, T.rank.p, n_nl, T.rec_nl.p);
        SGPU_LAUNCH(c);
    }
    T.P.rec_nl = T.rec_nl.p + (s.is_first ? 0 : 1);  // table entry 0 stands for byte 0
    SGPU_TRY(T.meta.alloc(n_rec, st));
    if (want_keys) {
        SGPU_TRY(T.key_off.alloc(n_rec, st));
        SGPU_TRY(T.key_len.alloc(n_rec, st));
        SGPU_TRY(T.sel.alloc(n_rec, st));
    }
    fa_record_kernel<<<(unsigned)ceil_div(n_rec, (uint64_t)128), 128, 0, st>>>(
        T.P, view_of(set), reverse, want_absent, T.meta.p, want_keys ? T.key_off.p : nullptr,
        want_keys ? T.key_len.p : nullptr, want_keys ? T.sel.p : nullptr, (unsigned long long *)T.scratch.p,
        (unsigned long long *)(T.scratch.p + 1));
    SGPU_LAUNCH(c);
    uint64_t e[2];
    SGPU_TRY(read_u64s(c, T.scratch.p, e, 2));
    T.err_word = e[0];
    T.le_from = e[1];
    return SGPU_OK;
}

// FastqCleaner::clean_reads over the FASTA records a shard owns.  Device pointers in, device outputs filled, counts on
// the host.  le_before: -1 undecided, 0 / 1 LF / CRLF decided by an earlier shard; *le_own: what this shard's first
// deciding record (before an error) says, -1 when it has none.
sgpu_status clean_fasta_shard(sgpu_ctx *c, const sgpu_idset *set, const Shard &s, int le_before, int reverse,
                              const Outs &out, sgpu_counts *counts, int *le_own) {
    cudaStream_t st = c->stream;
    clear_outputs(out, counts);
    counts->path = 3;
    *le_own = -1;
    FaTables T;
    SGPU_TRY(fasta_records(c, s, set, reverse, 0, false, T));
    const uint64_t n_rec = T.P.n_rec;
    if (n_rec == 0) {
        counts->crlf = le_before > 0;
        return SGPU_OK;
    }
    sgpu_status rc = SGPU_OK;
    uint64_t err_from = ~0ull;
    if (T.err_word != ~0ull) {
        rc = (sgpu_status)(T.err_word & 0xFF);
        err_from = T.err_word >> 8;
        counts->error_record = err_from;
    }
    // the line ending: decided by the first record (before any error) whose bytes hold a newline
    int crlf = 0;
    uint64_t le_from = T.le_from;
    if (le_from != ~0ull && le_from < err_from) {
        FaMeta m;
        SGPU_CUDA(cudaMemcpyAsync(c->h_pinned + 32, T.meta.p + le_from, sizeof(FaMeta), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(cudaStreamSynchronize(st));
        memcpy(&m, c->h_pinned + 32, sizeof(m));
        crlf = (m.flags & 8u) ? 1 : 0;
        *le_own = crlf;
    } else {
        le_from = ~0ull;
    }
    if (le_before >= 0) {  // an earlier shard decided: every record of this one uses it
        crlf = le_before;
        le_from = 0;
    }
    counts->crlf = (uint32_t)crlf;
    DevBuf<uint32_t> len_w, len_o;
    DevBuf<uint64_t> off_w, off_o;
    SGPU_TRY(len_w.alloc(n_rec, st));
    SGPU_TRY(len_o.alloc(n_rec, st));
    SGPU_TRY(off_w.alloc(n_rec, st));
    fa_len_kernel<<<(unsigned)ceil_div(n_rec, (uint64_t)256), 256, 0, st>>>(T.meta.p, n_rec, err_from, le_from, crlf, len_w.p,
                                                                             len_o.p, (unsigned long long *)(T.scratch.p + 3));
    SGPU_LAUNCH(c);
    SGPU_TRY(exclusive_scan_u32_to_u64(c, len_w.p, off_w.p, n_rec, T.scratch.p + 5));
    if (out.o) {
        SGPU_TRY(off_o.alloc(n_rec, st));
        SGPU_TRY(exclusive_scan_u32_to_u64(c, len_o.p, off_o.p, n_rec, T.scratch.p + 6));
    }
    uint64_t h[4];
    SGPU_TRY(read_u64s(c, T.scratch.p + 3, h, 4));
    counts->reads_in = h[0];
    counts->reads_out = h[1];
    *out.n_w = (size_t)h[2];
    if (out.n_o) *out.n_o = out.o ? (size_t)h[3] : 0;
    if (h[2] > out.cap_w || (out.o && h[3] > out.cap_o)) return SGPU_ERR_CAPACITY;
    fa_copy_kernel<<<(unsigned)ceil_div(n_rec * 32, (uint64_t)256), 256, 0, st>>>(T.P, T.meta.p, off_w.p, off_o.p, le_from, crlf,
                                                                                  out.w, out.o);
    SGPU_LAUNCH(c);
    SGPU_CUDA(cudaGetLastError());
    SGPU_CUDA(cudaStreamSynchronize(st));  // scratch buffers are released after this call returns
    return rc;
}

// one loop of ReadDifference::get_difference (utils.rs:259-267 / 269-283) over the FASTA records a shard owns
sgpu_status fasta_ids_shard(sgpu_ctx *c, const Shard &s, const sgpu_idset *probe, int want_absent, const SpanSink &sink,
                            uint64_t *n_records, uint64_t *n_picked, uint64_t *err_record) {
    *n_records = *n_picked = 0;
    FaTables T;
    SGPU_TRY(fasta_records(c, s, want_absent ? probe : nullptr, 0, want_absent, true, T));
    const uint64_t n_rec = T.P.n_rec;
    if (n_rec == 0) return SGPU_OK;
    if (T.err_word != ~0ull) {
        if (err_record) *err_record = T.err_word >> 8;
        return (sgpu_status)(T.err_word & 0xFF);
    }
    // every record is valid here; picked = the selected spans
    cudaStream_t st = c->stream;
    fa_count_sel_kernel<<<(unsigned)ceil_div(n_rec, (uint64_t)256), 256, 0, st>>>(T.sel.p, n_rec,
                                                                                 (unsigned long long *)(T.scratch.p + 3));
    SGPU_LAUNCH(c);
    uint64_t picked = 0;
    SGPU_TRY(read_u64s(c, T.scratch.p + 3, &picked, 1));
    *n_records = n_rec;
    *n_picked = picked;
    if (picked) SGPU_TRY(sink_spans(c, sink, s.p, T.key_off.p, T.key_len.p, T.sel.p, (size_t)n_rec));
    SGPU_CUDA(cudaStreamSynchronize(st));
    return SGPU_OK;
}

}  // namespace sgpu
