// fastq_records.cuh -- record location / validation shared by the general clean path and diff, and the internal
// interface of the FASTQ and FASTA shard cores.
// Restates needletail 0.5.1 fastq Reader::next / find / validate / check_end over a '\n' index.
#pragma once
#include "idset.cuh"

namespace sgpu {

struct RecMeta {
    uint32_t id_n, seq_n, qual_n;
    uint32_t flags;  // bit0: valid & owned, bit1: written
};

struct RecParams {
    const uint8_t *in;
    uint64_t n_in, own_len;
    const uint64_t *nlpos;
    uint64_t n_nl;
    uint64_t b0;      // newline index where local record 0 begins (its first '\n' is nlpos[b0])
    uint64_t k_full;  // records with all four newlines inside the buffer
    int starts_at_zero, is_last, crlf, reverse;
    IdSetView set;
};

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t trim_cr_len(const uint8_t *s, uint64_t n) {
    return (uint32_t)((n && s[n - 1] == '\r') ? n - 1 : n);
}

// Candidate record k (k == k_full is the tail with fewer than four newlines).
// Returns 1 and fills start/p1/p3, m->{id_n,seq_n,qual_n}, id span when a valid owned record
// exists; 0 when there is none; errors are reported through err_word.
__device__ __forceinline__ int locate_record(const RecParams &P, uint64_t k, uint64_t *start_o, uint64_t *p1_o,
                                             uint64_t *p3_o, RecMeta *m, size_t *id_off, size_t *id_len,
                                             unsigned long long *err_word) {
    uint64_t b = P.b0 + 4 * k;
    uint64_t start = (b == 0) ? 0 : P.nlpos[b - 1] + 1;
    const uint8_t *in = P.in;
    // a record that starts exactly at own_len (the next shard's first byte) is owned HERE: the next shard
    // cannot know that its byte 0 follows a newline
    if (P.is_last ? start >= P.own_len : start > P.own_len) return 0;
    uint64_t p1 = 0, p2 = 0, p3 = 0, end = 0;
    bool have = false;
    if (k < P.k_full) {
        p1 = P.nlpos[b];
        p2 = P.nlpos[b + 1];
        p3 = P.nlpos[b + 2];
        end = P.nlpos[b + 3];
        have = true;
    } else {
        // the tail: fewer than four newlines remain (needletail check_end)
        uint64_t mrem = P.n_nl - b;
        if (!P.is_last) {
            report_error(err_word, k, SGPU_ERR_HALO);
        } else if (mrem == 3) {
            p1 = P.nlpos[b];
            p2 = P.nlpos[b + 1];
            p3 = P.nlpos[b + 2];
            end = P.n_in;  // SearchPosition::Quality: last record without a trailing newline
            have = true;
        } else {
            // a tail of blank lines (after trim_cr) is tolerated, anything else is UnexpectedEnd
            uint64_t s = start;
            bool blank = true;
            for (uint64_t j = 0; j <= mrem && blank; j++) {
                uint64_t e = j < mrem ? P.nlpos[b + j] : P.n_in;
                if (e > s && trim_cr_len(in + s, e - s) != 0) blank = false;
                s = e + 1;
            }
            if (!blank) report_error(err_word, k, SGPU_ERR_FASTQ_UNEXPECTED_END);
        }
    }
    if (!have) return 0;
    int code = 0;
    if (in[start] != '@') {
        code = SGPU_ERR_FASTQ_INVALID_START;
    } else if (in[p2 + 1] != '+') {
        code = SGPU_ERR_FASTQ_INVALID_SEPARATOR;
    } else {
        m->id_n = trim_cr_len(in + start + 1, p1 - (start + 1));
        m->seq_n = trim_cr_len(in + p1 + 1, p2 - (p1 + 1));
        m->qual_n = trim_cr_len(in + p3 + 1, end - (p3 + 1));
        if (m->seq_n != m->qual_n) code = SGPU_ERR_FASTQ_UNEQUAL_LENGTHS;
    }
    if (!code) code = get_id_span(in + start + 1, m->id_n, id_off, id_len);
    if (code) {
        report_error(err_word, k, code);
        return 0;
    }
    *start_o = start;
    *p1_o = p1;
    *p3_o = p3;
    return 1;
}
#endif

// fills b0 / k_full / starts_at_zero for a buffer; returns false if the shard owns no record boundary
static inline bool setup_records(RecParams &P, uint64_t n_nl, uint64_t newlines_before, int is_first) {
    P.n_nl = n_nl;
    P.starts_at_zero = is_first;
    if (is_first) {
        P.b0 = 0;
    } else {
        // the newline that ends the previous record has global index == 3 (mod 4)
        uint64_t i0 = (3 - (newlines_before & 3)) & 3;
        P.b0 = i0 + 1;
    }
    if (n_nl < P.b0) {
        P.k_full = 0;
        return false;
    }
    P.k_full = (n_nl - P.b0) / 4;
    return true;
}

// one shard of a file: its own bytes [0, own_len) followed by a halo (the contracts are those of the shard entry points
// in include/scrubby_gpu.h); a whole file is the shard {p, n, n, 1, 1}
struct Shard {
    const uint8_t *p;
    size_t n, own_len;
    int is_first, is_last;
};

// the two outputs of a clean call: the written records and the others (o == nullptr: not produced), their capacities,
// and where the produced sizes go (n_o may be nullptr)
struct Outs {
    uint8_t *w;
    size_t cap_w;
    size_t *n_w;
    uint8_t *o;
    size_t cap_o;
    size_t *n_o;
};

// nothing produced (yet): counts and produced sizes zeroed
static inline void clear_outputs(const Outs &out, sgpu_counts *counts) {
    memset(counts, 0, sizeof(*counts));
    *out.n_w = 0;
    if (out.n_o) *out.n_o = 0;
}

// Where an ids pass sends the id spans it selected: inserted into a set, or routed as "id\n" lines grouped by owner
// partition (the hash-partitioned diff).
struct RouteOut {
    uint32_t n_parts;     // 1..64
    uint8_t *lines;       // device
    size_t cap;
    size_t n_lines;       // out: bytes written (bytes needed with SGPU_ERR_CAPACITY)
    uint64_t *part_bytes;  // out: host arrays of n_parts
    uint64_t *part_lines;
};
struct SpanSink {
    sgpu_idset *into;  // insert into this set (nullptr: count only) ...
    RouteOut *route;   // ... unless this is set: route
};

// idset_route.cu: spans d_src[off[i] .. off[i]+len[i]) with sel[i] != 0 (sel nullptr: all) to the sink.  `in_order`:
// the spans are listed in file order; otherwise (the single-pass kernel's list) routing sorts them by offset first,
// so that lines keep file order inside a partition (`range`: the offsets lie in [0, range)).
sgpu_status sink_spans(sgpu_ctx *c, const SpanSink &k, const uint8_t *d_src, const uint64_t *d_off, const uint32_t *d_len,
                       const uint8_t *d_sel, size_t n, bool in_order = true, uint64_t range = 0);

// fastq_general.cu: FastqCleaner::clean_reads and one loop of ReadDifference::get_difference over the FASTQ records a
// shard owns (the contracts are sgpu_clean_fastq_shard_dev's and sgpu_fastq_ids_shard_dev's; a whole file is the shard
// (n, n, newlines_before 0, first, last, crlf -1)).  The single-pass kernel runs when it takes the input, else the
// general path.  want_nl: when the single-pass kernel produces the result, counts->own_newlines is filled from its
// per-tile counts.  spec_out (may be nullptr): the single-pass kernel's counts (speculated, own / lead newlines); the
// general path adds nothing to it.  A non-first shard without a record boundary: clean produces zero records, ids returns
// SGPU_ERR_FASTQ_UNEXPECTED_END (last shard) or SGPU_ERR_HALO
sgpu_status clean_fastq_shard(sgpu_ctx *c, const sgpu_idset *set, const Shard &s, uint64_t newlines_before, int crlf,
                              int reverse, const Outs &out, sgpu_counts *counts, bool want_nl);
sgpu_status fastq_ids_shard(sgpu_ctx *c, const Shard &s, uint64_t newlines_before, const sgpu_idset *probe,
                            int want_absent, const SpanSink &sink, uint64_t *n_records, uint64_t *n_picked,
                            uint64_t *err_record, sgpu_counts *spec_out);

// fastq_fused.cu: the single-pass kernel over one FASTQ shard; *used = 0 when the input is not canonical (the caller
// then takes the general path).  ids mode (ids != nullptr, `out` unused): nothing is written; the id tokens of the
// records absent from `set` (nullptr: every record) are listed as (offset, length) spans
struct IdsOut {
    uint64_t *off;
    uint32_t *len;
    uint64_t cap;
    uint64_t n_spans;  // out
    uint64_t base;     // out: the spans' offsets are relative to the shard's byte `base`
};
sgpu_status fused_shard(sgpu_ctx *c, const sgpu_idset *set, const Shard &s, uint64_t newlines_before, int reverse,
                        const Outs &out, IdsOut *ids, sgpu_counts *counts, int *used, bool want_nl);

// fasta_general.cu: the same two operations over the FASTA records a shard owns (needletail's FASTA reader; a whole
// file is the shard (n, n, first, last)); the shard contract is sgpu_clean_fasta_shard_dev's
sgpu_status clean_fasta_shard(sgpu_ctx *c, const sgpu_idset *set, const Shard &s, int le_before, int reverse,
                              const Outs &out, sgpu_counts *counts, int *le_own);
sgpu_status fasta_ids_shard(sgpu_ctx *c, const Shard &s, const sgpu_idset *probe, int want_absent, const SpanSink &sink,
                            uint64_t *n_records, uint64_t *n_picked, uint64_t *err_record);

}  // namespace sgpu
