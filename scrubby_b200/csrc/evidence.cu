// evidence.cu -- alignment / classifier evidence -> read-id set.
//
// PAF, TXT id lists and Kraken2 / Metabuli per-read lines take one of two kernels with the same per-line rules:
//   lines_tile_kernel     one CTA per 16 KiB tile, no newline index (the normal case);
//   lines_indexed_kernel  one thread per line over a newline index: inputs with a tile too dense for the tile kernel,
//                         and sgpu_ctx_set_mode(1).
// Both decide a line with the same scanners; the tile kernel's ASCII fast path shares their decision helpers:
//   paf_line_scan   replaces ReadAlignment::from_paf (alignment.rs:84-114), PafRecord::from_str (:244-263) and
//       query_aligned_length / query_coverage (:265-275, alignment_passes).  Every passing record offers its qname and
//       the set makes the per-read aggregation (the duplicate loop at cleaner.rs:669-678): a logical OR of per-record
//       predicates (SURVEY F9), NOT a sum of aligned lengths.
//   evidence_line   replaces ReadAlignment::from_txt (alignment.rs:60-82) and get_taxid_reads_kraken / _metabuli
//       (classifier.rs:270-290, 308-328) with KrakenReadRecord / MetabuliReadRecord::from_str (:401-419, :497-517,
//       reads_key); taxid membership is a bitmap lookup for canonical decimal taxids and a byte compare against the
//       (normally empty) list of non-canonical taxid strings.
// Lines follow std::io::BufRead::lines: split on '\n', one '\r' stripped before it, UTF-8 checked.
#include <string>
#include <vector>

#include <chrono>
#include "idset.cuh"

namespace sgpu {

struct LineParams {
    const uint8_t *in;
    uint64_t n;
    const uint64_t *nlpos;
    uint64_t n_nl;
};

// raw line i = [s, e) (without '\n'); returns false if there is no such line
__device__ __forceinline__ bool line_span(const LineParams &P, uint64_t i, uint64_t *s, uint64_t *e) {
    uint64_t st = i ? P.nlpos[i - 1] + 1 : 0;
    uint64_t en;
    if (i < P.n_nl) {
        en = P.nlpos[i];
    } else {
        if (st >= P.n) return false;  // the buffer ended with '\n' (or is empty)
        en = P.n;
    }
    *s = st;
    *e = en;
    return true;
}

struct PafParams {
    uint64_t min_len;
    double min_cov;
    uint32_t min_mapq;
};

// the per-record predicate of PAF, SAM and BAM (alignment.rs:102-104, :265-275): aligned length or query coverage,
// and mapping quality.  The u32 lengths of SAM and BAM convert to double exactly.
__device__ __forceinline__ bool alignment_passes(const PafParams &F, uint64_t alen, uint64_t qlen, uint64_t mapq) {
    const double cov = qlen == 0 ? 0.0 : __ull2double_rn(alen) / __ull2double_rn(qlen);
    return (alen >= F.min_len || cov >= F.min_cov) && mapq >= F.min_mapq;
}

// ------------------------------------------------------------------ SAM (text) records
// Replaces ReadAlignment::from_bam (alignment.rs:117-146) + BamRecord::from / qalen_from_cigar /
// query_coverage (:154-211) for text SAM; the restated sam_parse1 rules are listed in include/scrubby_gpu.h.
__device__ __forceinline__ bool sam_int(const uint8_t *s, uint64_t n, bool allow_sign, long long *out) {
    uint64_t i = 0;
    bool neg = false;
    if (n && allow_sign && (s[0] == '-' || s[0] == '+')) {
        neg = s[0] == '-';
        i = 1;
    }
    if (i >= n || n - i > 18) return false;
    long long v = 0;
    for (; i < n; i++) {
        if (s[i] < '0' || s[i] > '9') return false;
        v = v * 10 + (s[i] - '0');
    }
    *out = neg ? -v : v;
    return true;
}
__device__ __forceinline__ bool sam_flag(const uint8_t *s, uint64_t n, uint32_t *out) {
    uint32_t base = 10, v = 0;
    uint64_t i = 0;
    if (n >= 2 && s[0] == '0' && (s[1] == 'x' || s[1] == 'X')) {
        base = 16;
        i = 2;
    } else if (n >= 2 && s[0] == '0') {
        base = 8;
        i = 1;
    }
    if (i >= n) return false;
    for (; i < n; i++) {
        uint32_t d;
        const uint8_t ch = s[i];
        if (ch >= '0' && ch <= '9') d = ch - '0';
        else if (ch >= 'a' && ch <= 'f') d = ch - 'a' + 10;
        else if (ch >= 'A' && ch <= 'F') d = ch - 'A' + 10;
        else return false;
        if (d >= base) return false;
        v = v * base + d;
        if (v > 65535u) return false;
    }
    *out = v;
    return true;
}
__device__ __forceinline__ bool sam_cigar(const uint8_t *s, uint64_t n, uint32_t *n_ops, uint32_t *qlen, uint32_t *qalen) {
    *n_ops = *qlen = *qalen = 0;
    if (n == 1 && s[0] == '*') return true;
    if (n == 0) return false;
    uint64_t i = 0;
    while (i < n) {
        uint64_t cnt = 0;
        const uint64_t d0 = i;
        while (i < n && s[i] >= '0' && s[i] <= '9') {
            cnt = cnt * 10 + (s[i] - '0');
            if (cnt >= (1ull << 28)) return false;
            i++;
        }
        if (i == d0 || i >= n) return false;
        const uint8_t op = s[i++];
        const bool q = op == 'M' || op == 'I' || op == 'S' || op == '=' || op == 'X';
        if (!(q || op == 'D' || op == 'N' || op == 'H' || op == 'P' || op == 'B')) return false;
        (*n_ops)++;
        if (op == 'M' || op == 'I') *qalen += (uint32_t)cnt;
        if (q) *qlen += (uint32_t)cnt;
    }
    return true;
}

// the reference names the header declares: SN: of every "@SQ" line (htslib's bam_name2id looks RNAME up among them)
__global__ void __launch_bounds__(128)
    sam_sq_kernel(LineParams P, uint64_t n_lines, uint64_t *key_off, uint32_t *key_len, uint8_t *sel) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_lines) return;
    uint64_t s, e, koff = 0;
    uint32_t klen = 0;
    uint8_t ok = 0;
    if (line_span(P, i, &s, &e)) {
        const uint8_t *in = P.in;
        if (i < P.n_nl && e > s && in[e - 1] == '\r') e--;
        if (e - s >= 4 && in[s] == '@' && in[s + 1] == 'S' && in[s + 2] == 'Q' && in[s + 3] == '\t') {
            uint64_t a = s + 4;
            while (a < e && !ok) {
                uint64_t b = a;
                while (b < e && in[b] != '\t') b++;
                if (b - a >= 3 && in[a] == 'S' && in[a + 1] == 'N' && in[a + 2] == ':') {
                    koff = a + 3;
                    klen = (uint32_t)(b - a - 3);
                    ok = 1;
                }
                a = b + 1;
            }
        }
    }
    key_off[i] = koff;
    key_len[i] = klen;
    sel[i] = ok;
}

__global__ void __launch_bounds__(128)
    sam_parse_kernel(LineParams P, PafParams F, IdSetView refs, int have_sq, uint64_t n_lines, uint64_t *key_off,
                     uint32_t *key_len, uint8_t *sel, unsigned long long *err_word) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_lines) return;
    uint64_t s, e;
    uint8_t ok = 0;
    uint64_t koff = 0;
    uint32_t klen = 0;
    if (line_span(P, i, &s, &e)) {
        const uint8_t *in = P.in;
        if (i < P.n_nl && e > s && in[e - 1] == '\r') e--;
        if (!(e > s && in[s] == '@')) {  // header lines are skipped
            // the first eleven tab-separated fields
            uint64_t fs[11], fe[11];
            int f = 0;
            uint64_t st = s;
            for (uint64_t pos = s; pos <= e && f < 11; pos++) {
                if (pos == e || in[pos] == '\t') {
                    fs[f] = st;
                    fe[f] = pos;
                    f++;
                    st = pos + 1;
                }
            }
            int code = 0;
            uint32_t flag = 0, n_ops = 0, cq = 0, qalen = 0;
            long long p = 0, mapq = 0, t = 0;
            if (f < 11) {
                code = SGPU_ERR_SAM_RECORD;
            } else {
#define FLEN(k) (fe[k] - fs[k])
                // RNAME other than "*" with no @SQ line at all: htslib's "no SQ lines present in the header" parse error
                const bool rname_star = FLEN(2) == 1 && in[fs[2]] == '*';
                const bool good = FLEN(0) && sam_flag(in + fs[1], FLEN(1), &flag) && FLEN(2) && (rname_star || have_sq) &&
                                  sam_int(in + fs[3], FLEN(3), true, &p) && sam_int(in + fs[4], FLEN(4), false, &mapq) &&
                                  mapq <= 255 && sam_cigar(in + fs[5], FLEN(5), &n_ops, &cq, &qalen) && FLEN(6) &&
                                  sam_int(in + fs[7], FLEN(7), true, &t) && sam_int(in + fs[8], FLEN(8), true, &t) &&
                                  FLEN(9) && FLEN(10);
                if (!good) {
                    code = SGPU_ERR_SAM_RECORD;
                } else {
                    const bool seq_star = FLEN(9) == 1 && in[fs[9]] == '*';
                    const uint32_t qlen = seq_star ? 0u : (uint32_t)FLEN(9);
                    const bool qual_star = FLEN(10) == 1 && in[fs[10]] == '*';
                    if ((n_ops && !seq_star && cq != qlen) || (!qual_star && FLEN(10) != (seq_star ? 0 : FLEN(9)))) {
                        code = SGPU_ERR_SAM_RECORD;
                    } else if (!utf8_valid(in + fs[0], FLEN(0))) {
                        code = SGPU_ERR_RECORD_NAME_UTF8;
                    } else {
                        // an undeclared RNAME: "unrecognized reference name; treated as unmapped" (tid -1 -> BAM_FUNMAP)
                        const bool declared = !rname_star && (FLEN(2) == 0 ? false : (FLEN(2) <= IDSET_MAX_KEY &&
                                                              idset_contains(refs, in + fs[2], (uint32_t)FLEN(2))));
                        const bool unmapped = (flag & 4u) || rname_star || !declared || p < 1;
                        if (!unmapped) {
                            ok = alignment_passes(F, qalen, qlen, (uint32_t)mapq) ? 1 : 0;
                            koff = fs[0];
                            klen = (uint32_t)FLEN(0);
                        }
                    }
                }
#undef FLEN
            }
            if (code) report_error(err_word, i, code);
        }
    }
    key_off[i] = koff;
    key_len[i] = klen;
    sel[i] = ok;
}

// ---------------------------------------------------------------- binary BAM records
// ReadAlignment::from_bam (alignment.rs:117-146) + BamRecord::from (:180-197) over the BGZF-decompressed BAM stream:
// one thread per record (the host has walked the block_size chain: rec_off[i] is where record i's block_size sits
// and every block lies inside the buffer with block_size >= 32).  The rules restated from the BAM specification and
// htslib's bam_read1 / bam_tag2cigar are listed in include/scrubby_gpu.h.
__device__ __forceinline__ uint32_t ld_le32(const uint8_t *p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
// the CG:B,I / B,i array among the auxiliary fields [a, e): element count (and *arr), or -1
__device__ inline long long bam_find_cg(const uint8_t *a, const uint8_t *e, const uint8_t **arr) {
    while (e - a >= 3) {
        const uint8_t t0 = a[0], t1 = a[1], ty = a[2];
        a += 3;
        size_t sz = 0;
        if (ty == 'A' || ty == 'c' || ty == 'C') sz = 1;
        else if (ty == 's' || ty == 'S') sz = 2;
        else if (ty == 'i' || ty == 'I' || ty == 'f') sz = 4;
        else if (ty == 'd') sz = 8;
        else if (ty == 'Z' || ty == 'H') {
            const uint8_t *z = a;
            while (z < e && *z) z++;
            if (z == e) return -1;
            sz = (size_t)(z - a) + 1;
        } else if (ty == 'B') {
            if (e - a < 5) return -1;
            const uint8_t sub = a[0];
            const uint32_t cnt = ld_le32(a + 1);
            const size_t es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2
                              : (sub == 'i' || sub == 'I' || sub == 'f') ? 4 : 0;
            if (!es || (unsigned long long)cnt * es > (unsigned long long)(e - a - 5)) return -1;
            if (t0 == 'C' && t1 == 'G') {
                if (sub != 'I' && sub != 'i') return -1;
                *arr = a + 5;
                return (long long)cnt;
            }
            sz = 5 + (size_t)cnt * es;
        } else {
            return -1;
        }
        if (t0 == 'C' && t1 == 'G') return -1;  // a CG tag of another type is not a CIGAR
        if ((size_t)(e - a) < sz) return -1;
        a += sz;
    }
    return -1;
}

__global__ void __launch_bounds__(128)
    bam_parse_kernel(const uint8_t *in, const uint64_t *rec_off, uint64_t n_rec, PafParams F, uint64_t *key_off,
                     uint32_t *key_len, uint8_t *sel, unsigned long long *err_word) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rec) return;
    const uint8_t *b = in + rec_off[i] + 4;
    const uint32_t bs = ld_le32(b - 4);
    const int32_t ref_id = (int32_t)ld_le32(b), rpos = (int32_t)ld_le32(b + 4);
    const uint32_t l_name = b[8], mapq = b[9];
    const uint32_t n_cig = (uint32_t)b[12] | ((uint32_t)b[13] << 8), flag = (uint32_t)b[14] | ((uint32_t)b[15] << 8);
    const int32_t l_seq = (int32_t)ld_le32(b + 16);
    uint8_t ok = 0;
    uint64_t koff = 0;
    uint32_t klen = 0;
    if (l_name < 1 || l_seq < 0 ||
        32ull + l_name + 4ull * n_cig + (((unsigned long long)l_seq + 1) >> 1) + (unsigned long long)l_seq > bs) {
        report_error(err_word, i, SGPU_ERR_BAM_RECORD);
    } else if (!(flag & 4u)) {  // unmapped records are skipped before anything else is looked at
        const uint8_t *name = b + 32;
        const uint32_t qn = name[l_name - 1] == 0 ? l_name - 1 : l_name;
        if (!utf8_valid(name, qn)) {
            report_error(err_word, i, SGPU_ERR_RECORD_NAME_UTF8);
        } else {
            const uint8_t *cig = name + l_name;
            unsigned long long n_ops = n_cig;
            if (n_cig && ref_id >= 0 && rpos >= 0 && (ld_le32(cig) & 15u) == 4u && (ld_le32(cig) >> 4) == (uint32_t)l_seq) {
                // the long-CIGAR placeholder: the real CIGAR is the CG:B,I tag (htslib bam_tag2cigar)
                const uint8_t *aux = cig + 4ull * n_cig + (((unsigned long long)l_seq + 1) >> 1) + (unsigned long long)l_seq;
                const uint8_t *arr = nullptr;
                const long long k = bam_find_cg(aux, b + bs, &arr);
                if (k >= (long long)n_cig && k < (1ll << 29)) {
                    cig = arr;
                    n_ops = (unsigned long long)k;
                }
            }
            uint32_t qalen = 0;  // u32: wraps like the reference's release build (alignment.rs:161-169)
            for (unsigned long long q = 0; q < n_ops; q++) {
                const uint32_t v = ld_le32(cig + 4 * q);
                if ((v & 15u) <= 1u) qalen += v >> 4;  // M and I
            }
            const uint32_t qlen = (uint32_t)l_seq;
            ok = alignment_passes(F, qalen, qlen, mapq) ? 1 : 0;
            koff = (uint64_t)(name - in);
            klen = qn;
        }
    }
    key_off[i] = koff;
    key_len[i] = klen;
    sel[i] = ok;
}

struct TaxSet {
    const uint32_t *bitmap;  // canonical decimal taxids
    uint64_t bits;
    const uint8_t *exotic;   // non-canonical taxid strings, flat
    const uint32_t *exotic_off;  // n_exotic + 1 offsets
    uint32_t n_exotic;
};

__device__ __forceinline__ bool taxid_member(const TaxSet &T, const uint8_t *s, uint32_t n) {
    // canonical decimal: digits only, no sign, no leading zero (except "0") -> bitmap
    bool canon = n >= 1 && n <= 10 && !(n > 1 && s[0] == '0');
    uint64_t v = 0;
    for (uint32_t k = 0; k < n && canon; k++) {
        uint32_t d = (uint32_t)s[k] - '0';
        canon = d <= 9;
        v = v * 10 + d;
    }
    if (canon && v < T.bits) return (T.bitmap[v >> 5] >> (v & 31)) & 1u;
    for (uint32_t x = 0; x < T.n_exotic; x++) {
        uint32_t a = T.exotic_off[x], b = T.exotic_off[x + 1];
        if (b - a == n && bytes_equal(T.exotic + a, s, n)) return true;
    }
    return false;
}

// str::trim on the read id f1 and the taxid f2 (Unicode White_Space if the line has a non-ASCII byte, ASCII otherwise),
// then the taxid's membership: true if the line selects its read, whose id is [*k_begin, *k_begin + *k_len) of f1
__device__ __forceinline__ bool reads_key(const uint8_t *f1, uint64_t n1, const uint8_t *f2, uint64_t n2, bool high,
                                          const TaxSet &T, uint64_t *k_begin, uint32_t *k_len) {
    size_t b1 = 0, e1 = n1, b2 = 0, e2 = n2;
    if (high) {
        utf8_trim(f1, n1, &b1, &e1);
        utf8_trim(f2, n2, &b2, &e2);
    } else {
        while (b1 < e1 && is_ws_ascii(f1[b1])) b1++;
        while (e1 > b1 && is_ws_ascii(f1[e1 - 1])) e1--;
        while (b2 < e2 && is_ws_ascii(f2[b2])) b2++;
        while (e2 > b2 && is_ws_ascii(f2[e2 - 1])) e2--;
    }
    if (!taxid_member(T, f2 + b2, (uint32_t)(e2 - b2))) return false;
    *k_begin = b1;
    *k_len = (uint32_t)(e1 - b1);
    return true;
}

// ------------------------------------------------------------------ tile kernel
// A PAF record, a TXT id or a Kraken2 / Metabuli line is decided on its own and the set does not care about insertion
// order (PAF included: every passing record offers its qname and the set makes the per-read OR), so no global line
// index is needed.  One CTA per 16 KiB tile: 16-byte loads -> '\n' masks -> the tile's newline positions in shared
// memory -> one thread per line that STARTS in the tile (it reads on past the tile's end if the line does) -> selected
// (offset, length) spans compacted into a candidate list with one global atomic per CTA.  A tile denser than LT_LMAX
// lines or LT_SMAX separators sends the buffer to lines_indexed_kernel, which decides each line with the same scanners.
constexpr int LT_NT = 256, LT_FC = 4, LT_TILE = LT_NT * LT_FC * 16, LT_LMAX = 2048, LT_HALO = 1024, LT_SMAX = 5120;

struct TileOut {
    uint64_t *cand_off;
    uint32_t *cand_len;
    uint64_t cap;
    unsigned long long *n_cand;   // candidates found (may exceed cap: the caller retries with more room)
    unsigned long long *err_word; // (line start offset << 8) | code, smallest wins
    unsigned long long *dense;    // a tile with more than LT_LMAX lines: use the indexed path
    unsigned long long *stats;    // [0] bytes of candidates longer than 15, [1] an empty candidate, [2] one of >= 16 MiB:
                                  // what idset_measure_kernel would find, so the set build can skip that pass
    // a SHARD of an evidence file (sharded set build): only the lines that START before own_end are this shard's; the
    // buffer carries a halo behind own_end, and a line of the shard that does not end inside it is SGPU_ERR_HALO
    uint64_t own_begin, own_end;  // 0, ~0: the whole buffer
    int not_last;                 // the buffer does not end at the end of the file
};

// The scanners decide one line [s, e_raw) of the buffer (e_raw = position of its '\n', or n for an unterminated last
// line) with BufRead::lines semantics (UTF-8 check, "\r\n" stripped).  They return 1 and the key span if the line offers
// a key, 0 if not, and set *err to the line's status code (0: none); the caller reports it in its own unit.

// TXT (mode 1) and Kraken2 / Metabuli (mode 0) lines.  One pass over the line's aligned 4-byte words finds the high-bit
// bytes (UTF-8 screening) and the tabs.
__device__ __forceinline__ int evidence_line(const uint8_t *in, uint64_t s, uint64_t e_raw, bool has_nl, int mode,
                                             const TaxSet &T, int need_fields, uint64_t *koff, uint32_t *klen, int *err) {
    uint64_t e = e_raw;
    uint32_t acc = 0;
    int f = 0;  // fields closed so far
    uint64_t fs = s, f1s = 0, f1e = 0, f2s = 0, f2e = 0;
    *err = 0;
    {
        const uintptr_t base = (uintptr_t)in;
        uint64_t w0 = (base + s) & ~(uintptr_t)3;         // address of the first word
        const uint64_t w1 = (base + e + 3) & ~(uintptr_t)3;  // one past the last word
        for (uint64_t a = w0; a < w1; a += 4) {
            uint32_t w = *reinterpret_cast<const uint32_t *>(a);
            // bytes outside [s, e) read as zero (neither tab nor high)
            const int64_t lo = (int64_t)(base + s) - (int64_t)a, hi = (int64_t)(base + e) - (int64_t)a;
            if (lo > 0) w &= 0xFFFFFFFFu << (8 * lo);
            if (hi < 4) w &= hi <= 0 ? 0u : (0xFFFFFFFFu >> (8 * (4 - hi)));
            acc |= w;
            if (mode == 0 && f < need_fields) {
                uint32_t t = eq_mask4(w, 0x09090909u);
                while (t) {
                    const uint64_t pos = (a - base) + (uint64_t)(__ffs(t) - 1);
                    t &= t - 1;
                    if (f == 1) { f1s = fs; f1e = pos; }
                    if (f == 2) { f2s = fs; f2e = pos; }
                    f++;
                    fs = pos + 1;
                    if (f >= need_fields) break;
                }
            }
        }
    }
    // BufRead::lines: UTF-8 check, strip "\n" / "\r\n"
    const bool high = (acc & 0x80808080u) != 0;
    if (high && !utf8_valid(in + s, e - s)) {
        *err = SGPU_ERR_IO;
        return 0;
    }
    if (has_nl && e > s && in[e - 1] == '\r') e--;
    if (mode == 1) {  // TXT: the line is the id, verbatim (alignment.rs:72-75)
        *koff = s;
        *klen = (uint32_t)(e - s);
        return 1;
    }
    if (f < need_fields) {  // the end of the line closes the last field (a stripped '\r' is not part of it)
        if (f == 1) { f1s = fs; f1e = e; }
        if (f == 2) { f2s = fs; f2e = e; }
        f++;
    }
    if (f < need_fields) {
        *err = SGPU_ERR_WOULD_PANIC;  // classifier.rs:412-415 / :508-513
        return 0;
    }
    // a field that ended at the raw end of a "\r\n" line: the '\r' was stripped by lines()
    if (f1e > e) f1e = e;
    if (f2e > e) f2e = e;
    if (!reads_key(in + f1s, f1e - f1s, in + f2s, f2e - f2s, high, T, koff, klen)) return 0;
    *koff += f1s;
    return 1;
}

// <uN as FromStr>::from_str for the common case (at most 18 digits cannot overflow a u64); same result as
// parse_uint
__device__ __forceinline__ bool parse_uint_short(const uint8_t *p, uint32_t n, uint64_t maxv, uint64_t *out) {
    if (n == 0 || n > 18 || p[0] == '+' || p[0] == '-') return parse_uint(p, n, maxv, out);
    uint64_t v = 0;
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t d = (uint32_t)p[i] - '0';
        if (d > 9) return false;
        v = v * 10 + d;
    }
    if (v > maxv) return false;
    *out = v;
    return true;
}

// PAF records (the tile kernel's fast path does not take non-ASCII tiles, lines that leave the halo, lines with fewer
// than 12 fields): the fields in column order, the first bad integer is the error
__device__ __noinline__ int paf_line_scan(const uint8_t *in, uint64_t s, uint64_t e_raw, bool has_nl, const PafParams &F,
                                          uint64_t *koff, uint32_t *klen, int *err) {
    uint64_t e = e_raw;
    // only a line with a high-bit byte can fail the UTF-8 check: screen it in aligned 4-byte words first
    uint32_t acc = 0;
    uint64_t k = s;
    while (k < e && ((uintptr_t)(in + k) & 3)) acc |= in[k++];
    for (; k + 4 <= e; k += 4) acc |= *reinterpret_cast<const uint32_t *>(in + k);
    while (k < e) acc |= in[k++];
    if ((acc & 0x80808080u) && !utf8_valid(in + s, e - s)) {
        *err = SGPU_ERR_IO;
        return 0;
    }
    if (has_nl && e > s && in[e - 1] == '\r') e--;
    int f = 0, code = 0;
    uint64_t fs = s, qlen = 0, qstart = 0, qend = 0, mapq = 0, k_end = s;
    for (uint64_t pos = s; pos <= e && f < 12; pos++) {
        if (pos == e || in[pos] == '\t') {
            uint64_t v = 0;
            const bool is_int = (f >= 1 && f <= 3) || (f >= 6 && f <= 11);
            if (is_int && !parse_uint(in + fs, pos - fs, f == 11 ? 255ull : ~0ull, &v)) {
                code = SGPU_ERR_PAF_INTEGER;
                break;
            }
            if (f == 0) k_end = pos;
            else if (f == 1) qlen = v;
            else if (f == 2) qstart = v;
            else if (f == 3) qend = v;
            else if (f == 11) mapq = v;
            f++;
            fs = pos + 1;
        }
    }
    if (!code && f < 12) code = SGPU_ERR_WOULD_PANIC;  // fields[f] out of bounds (alignment.rs:248-259)
    *err = code;
    // usize subtraction wraps in release builds
    if (code || !alignment_passes(F, qend - qstart, qlen, mapq)) return 0;
    *koff = s;
    *klen = (uint32_t)(k_end - s);
    return 1;
}

// 16-bit masks of the '\n' and '\t' bytes of a 16-byte chunk
__device__ __forceinline__ void sep_masks16(uint4 v, bool want_tabs, uint32_t *m_nl, uint32_t *m_tab) {
    *m_nl = nl_mask16(v);
    const uint32_t c = 0x09090909u;
    *m_tab = want_tabs ? eq_mask16(v, c) : 0u;
}

// The tile kernel proper.  P1 turns every 16-byte chunk of the tile (+ halo) into '\n' / '\t' masks and
// scatters the separator positions, in order, into one list (bit 15 = newline) plus the list index of every
// newline; a line's fields are then consecutive list entries -- no per-line scanning.  Tiles with a
// non-ASCII byte and lines that run past the halo take the scanners (evidence_line, paf_line_scan) instead.
__global__ void __launch_bounds__(LT_NT)
    lines_tile_kernel(const uint8_t *in, uint64_t n, TaxSet T, int need_fields, int mode, PafParams F, TileOut O) {
    constexpr int NWARP = LT_NT / 32;
    constexpr int ROWS = LT_FC + 1;  // LT_FC rounds over the tile + one over the halo (warps 0 and 1)
    __shared__ __align__(16) uint8_t tile[LT_TILE + LT_HALO];
    __shared__ uint16_t seps[LT_SMAX];   // separator positions (tile offsets), bit 15: it is a newline
    __shared__ uint16_t nl_idx[LT_LMAX]; // list index of the i-th newline
    __shared__ uint32_t warp_tot[NWARP], warp_cand[NWARP], halo_tot[2];
    __shared__ unsigned long long cand_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t g0 = (uint64_t)blockIdx.x * LT_TILE;
    const uint32_t tile_len = (uint32_t)((n - g0) < (uint64_t)LT_TILE ? (n - g0) : (uint64_t)LT_TILE);
    // bytes of the halo that exist (whole 16-byte chunks only)
    const uint32_t halo_len =
        tile_len < (uint32_t)LT_TILE ? 0u
                                     : (uint32_t)(((n - g0 - LT_TILE) < (uint64_t)LT_HALO ? (n - g0 - LT_TILE) : (uint64_t)LT_HALO) & ~15ull);
    const bool want_tabs = mode != 1;  // mode 0: Kraken2 / Metabuli lines, 1: TXT ids, 2: PAF records
    // ---- P1: masks.  Warp w owns tile chunks [w*128, w*128+128): lane l takes chunk k*32 + l in round k;
    //      round LT_FC is the halo (64 chunks: warps 0 and 1)
    uint32_t mn[ROWS], mt[ROWS];
    uint32_t hi_or = 0;
    uint64_t pk = 0;  // per round: separators (low 8 bits... 6 used) | newlines << 8, 16 bits per round
#pragma unroll
    for (int k = 0; k < ROWS; k++) {
        uint32_t pos, limit;
        bool mine;
        if (k < LT_FC) {
            pos = ((uint32_t)warp * (LT_FC * 32) + (uint32_t)lane + k * 32) * 16;
            limit = tile_len;
            mine = true;
        } else {
            pos = (uint32_t)LT_TILE + ((uint32_t)warp * 32 + (uint32_t)lane) * 16;
            limit = (uint32_t)LT_TILE + halo_len;
            mine = warp < 2;
        }
        uint32_t a = 0, b = 0;
        if (mine && pos + 16 <= limit) {
            const uint4 v = ld_nc_u4(in + g0 + pos);
            *reinterpret_cast<uint4 *>(tile + pos) = v;
            sep_masks16(v, want_tabs, &a, &b);
            hi_or |= v.x | v.y | v.z | v.w;
        } else if (mine && pos < limit) {  // the buffer's last, partial chunk
            for (uint32_t q = 0; pos + q < limit; q++) {
                const uint8_t ch = in[g0 + pos + q];
                tile[pos + q] = ch;
                a |= (ch == '\n' ? 1u : 0u) << q;
                b |= (want_tabs && ch == '\t' ? 1u : 0u) << q;
                hi_or |= ch;
            }
        }
        mn[k] = a;
        mt[k] = b;
        if (k < LT_FC) pk |= ((uint64_t)__popc(a | b) | ((uint64_t)__popc(a) << 8)) << (16 * k);
    }
    const bool high_w = __any_sync(0xffffffffu, (hi_or & 0x80808080u) != 0);
    // ---- ranks: inclusive warp scan of the packed per-round counts (a round of 32 chunks has <= 512
    //      separators: the 8-bit fields may carry into each other, so scan the two kinds separately)
    uint64_t pk_s = 0, pk_n = 0;
#pragma unroll
    for (int k = 0; k < LT_FC; k++) {
        pk_s |= (uint64_t)__popc(mn[k] | mt[k]) << (16 * k);
        pk_n |= (uint64_t)__popc(mn[k]) << (16 * k);
    }
    (void)pk;
    uint64_t inc_s = pk_s, inc_n = pk_n;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint64_t x = __shfl_up_sync(0xffffffffu, inc_s, d), y = __shfl_up_sync(0xffffffffu, inc_n, d);
        if (lane >= d) {
            inc_s += x;
            inc_n += y;
        }
    }
    const uint64_t rt_s = __shfl_sync(0xffffffffu, inc_s, 31), rt_n = __shfl_sync(0xffffffffu, inc_n, 31);
    const uint64_t ex_s = inc_s - pk_s, ex_n = inc_n - pk_n;
    uint32_t base_s[LT_FC], base_n[LT_FC], wtot_s = 0, wtot_n = 0;
#pragma unroll
    for (int k = 0; k < LT_FC; k++) {
        base_s[k] = wtot_s + (uint32_t)((ex_s >> (16 * k)) & 0xFFFF);
        base_n[k] = wtot_n + (uint32_t)((ex_n >> (16 * k)) & 0xFFFF);
        wtot_s += (uint32_t)((rt_s >> (16 * k)) & 0xFFFF);
        wtot_n += (uint32_t)((rt_n >> (16 * k)) & 0xFFFF);
    }
    // the halo round (warps 0, 1): ranks within the halo
    uint32_t h_s = 0, h_ex = 0;
    {
        const uint32_t c = (uint32_t)__popc(mn[LT_FC] | mt[LT_FC]);
        uint32_t ic = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t x = __shfl_up_sync(0xffffffffu, ic, d);
            if (lane >= d) ic += x;
        }
        h_ex = ic - c;
        h_s = __shfl_sync(0xffffffffu, ic, 31);
    }
    if (lane == 0) {
        warp_tot[warp] = wtot_s | (wtot_n << 16) | (high_w ? 0x80000000u : 0u);
        if (warp < 2) halo_tot[warp] = h_s;
    }
    __syncthreads();
    uint32_t n_sep = 0, n_nl = 0, wb_s = 0, wb_n = 0, high_seen = 0;
#pragma unroll
    for (int w = 0; w < NWARP; w++) {
        const uint32_t x = warp_tot[w];
        if (w == warp) {
            wb_s = n_sep;
            wb_n = n_nl;
        }
        n_sep += x & 0xFFFF;
        n_nl += (x >> 16) & 0x7FFF;
        high_seen |= x >> 31;
    }
    const uint32_t n_halo = halo_tot[0] + halo_tot[1];
    if (n_sep + n_halo > (uint32_t)LT_SMAX || n_nl > (uint32_t)LT_LMAX) {  // (uniform) pathological density
        if (tid == 0) atomicExch(O.dense, 1ull);
        return;
    }
    // ---- scatter, in order
#pragma unroll
    for (int k = 0; k < ROWS; k++) {
        uint32_t mm = mn[k] | mt[k];
        if (mm == 0) continue;
        uint32_t pos, r, rn = 0;
        if (k < LT_FC) {
            pos = ((uint32_t)warp * (LT_FC * 32) + (uint32_t)lane + k * 32) * 16;
            r = wb_s + base_s[k];
            rn = wb_n + base_n[k];
        } else {
            pos = (uint32_t)LT_TILE + ((uint32_t)warp * 32 + (uint32_t)lane) * 16;
            r = n_sep + (warp == 1 ? halo_tot[0] : 0u) + h_ex;
        }
        while (mm) {
            const uint32_t bit = (uint32_t)(__ffs(mm) - 1);
            mm &= mm - 1;
            const bool is_nl = (mn[k] >> bit) & 1u;
            seps[r] = (uint16_t)((pos + bit) | (is_nl ? 0x8000u : 0u));
            if (is_nl && k < LT_FC) nl_idx[rn++] = (uint16_t)r;
            r++;
        }
    }
    __syncthreads();
    const uint32_t n_all = n_sep + n_halo;  // list entries (the halo's come last)
    const bool high = high_seen != 0;
    // ---- one thread per line that starts in the tile
    const bool first_ok = g0 == 0 || in[g0 - 1] == '\n';  // the tile's first byte starts a line
    const uint32_t n_lines = n_nl + (first_ok ? 1u : 0u);  // candidates (the last may start at tile_len: skipped)
    for (uint32_t qb = 0; qb < n_lines; qb += LT_NT) {  // (uniform trip count)
        const uint32_t q = qb + (uint32_t)tid;
        int sel = 0;
        uint64_t koff = 0;
        uint32_t klen = 0;
        if (q < n_lines) {
            const int pi = (int)q - (first_ok ? 1 : 0);  // which newline precedes the line, -1: it starts the tile
            const int i0 = pi >= 0 ? (int)nl_idx[pi] : -1;  // its list index
            const uint32_t s = pi >= 0 ? ((uint32_t)seps[i0] & 0x7FFFu) + 1u : 0u;
            if (s < tile_len && g0 + s >= O.own_begin && g0 + s < O.own_end) {
                // the line's own newline: the next newline entry of the list
                bool fast = !high;
                uint32_t e_nl = 0;  // tile offset of the line's '\n'
                if (mode == 1) {
                    // TXT: the next list entry is the line's newline
                    if ((uint32_t)(i0 + 1) < n_all) e_nl = (uint32_t)seps[i0 + 1] & 0x7FFFu;
                    else fast = false;
                    if (fast) {
                        uint32_t e = e_nl;
                        if (e > s && tile[e - 1] == '\r') e--;
                        koff = g0 + s;
                        klen = e - s;
                        sel = 1;
                    }
                } else if (mode == 2) {
                    // PAF: the twelve fields are the list entries i0+1 .. i0+12 (the twelfth closes at a tab
                    // or at the line's newline); an earlier newline = fewer than 12 columns: the scanner
                    // reports what the reference would (bad integer before the missing column, else panic).
                    // Every passing line offers its qname: the set makes the per-read OR (alignment.rs:102-107)
                    if (fast && (uint32_t)i0 + 12u < n_all) {
                        uint32_t any_nl = 0;
                        for (uint32_t x = 1; x <= 11; x++) any_nl |= seps[i0 + x];
                        if (any_nl & 0x8000u) fast = false;
                    } else {
                        fast = false;
                    }
                    if (fast) {
                        // PafRecord::from_str (alignment.rs:244-263): columns in order, the first bad integer
                        // is the error; then the predicate (:265-275, :102-104)
                        uint32_t fs = s, name_end = s;
                        uint64_t qlen = 0, qstart = 0, qend = 0, mapq = 0;
                        int code = 0;
#pragma unroll
                        for (int x = 0; x < 12; x++) {
                            const uint32_t pe = (uint32_t)seps[i0 + 1 + x] & 0x7FFFu;
                            uint32_t fe = pe;
                            // lines() strips the '\r' of "\r\n": it can only sit at the end of the twelfth field
                            if (x == 11 && (seps[i0 + 12] & 0x8000u) && fe > fs && tile[fe - 1] == '\r') fe--;
                            if (x == 0) {
                                name_end = pe;
                            } else if (x <= 3 || x >= 6) {
                                uint64_t v = 0;
                                if (!code && !parse_uint_short(tile + fs, fe - fs, x == 11 ? 255ull : ~0ull, &v))
                                    code = SGPU_ERR_PAF_INTEGER;
                                if (x == 1) qlen = v;
                                else if (x == 2) qstart = v;
                                else if (x == 3) qend = v;
                                else if (x == 11) mapq = v;
                            }
                            fs = pe + 1u;
                        }
                        if (code) {
                            report_error(O.err_word, g0 + s, code);
                        } else if (alignment_passes(F, qend - qstart, qlen, mapq)) {  // (usize subtraction wraps)
                            sel = 1;
                            koff = g0 + s;
                            klen = name_end - s;
                        }
                    }
                } else if (fast) {
                    // fields 1 and 2 end at tabs 2 and 3; the line must have need_fields - 1 tabs
                    const uint32_t need_tabs = (uint32_t)need_fields - 1u;
                    if ((uint32_t)i0 + need_tabs < n_all) {
                        uint32_t any_nl = 0;
                        for (uint32_t x = 1; x <= need_tabs; x++) any_nl |= seps[i0 + x];
                        if (any_nl & 0x8000u) {
                            report_error(O.err_word, g0 + s, SGPU_ERR_WOULD_PANIC);  // classifier.rs:412-415 / :508-513
                        } else {
                            const uint32_t f1s = ((uint32_t)seps[i0 + 1]) + 1u, f1e = seps[i0 + 2];
                            const uint32_t f2s = f1e + 1u, f2e = seps[i0 + 3];
                            if (reads_key(tile + f1s, f1e - f1s, tile + f2s, f2e - f2s, false, T, &koff, &klen)) {
                                sel = 1;
                                koff += g0 + f1s;
                            }
                        }
                    } else {
                        fast = false;  // the list ends inside the line: it runs past the halo (or the buffer ends)
                    }
                }
                if (!fast) {
                    // scanning routine over the buffer: non-ASCII tile, or a line that leaves the halo
                    uint64_t e = g0 + s;
                    while (e < n && in[e] != '\n') e++;
                    int code = 0;
                    if (e == n && O.not_last) code = SGPU_ERR_HALO;  // the halo is too short
                    else if (mode == 2) sel = paf_line_scan(in, g0 + s, e, e < n, F, &koff, &klen, &code);
                    else sel = evidence_line(in, g0 + s, e, e < n, mode, T, need_fields, &koff, &klen, &code);
                    if (code) report_error(O.err_word, g0 + s, code);
                }
            }
        }
        // ---- compaction: order does not matter, one global atomic per CTA and round
        const unsigned b = __ballot_sync(0xffffffffu, sel != 0);
        if (lane == 0) warp_cand[warp] = (uint32_t)__popc(b);
        __syncthreads();
        uint32_t before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < NWARP; w++) {
            const uint32_t x = warp_cand[w];
            if (w < warp) before += x;
            total += x;
        }
        if (tid == 0 && total) cand_base = atomicAdd(O.n_cand, (unsigned long long)total);
        {   // candidate statistics for the set build
            unsigned long long lb = (sel && klen > IDSET_INLINE_MAX && klen <= IDSET_MAX_KEY) ? arena_padded(klen) : 0ull;
            for (int d = 16; d; d >>= 1) lb += __shfl_xor_sync(0xffffffffu, lb, d);
            if (lane == 0 && lb) atomicAdd(O.stats, lb);
            if (sel && klen == 0) O.stats[1] = 1ull;
            if (sel && klen > IDSET_MAX_KEY) O.stats[2] = 1ull;
        }
        __syncthreads();
        if (sel) {
            const uint64_t slot = cand_base + before + (uint32_t)__popc(b & ((1u << lane) - 1u));
            if (slot < O.cap) {
                O.cand_off[slot] = koff;
                O.cand_len[slot] = klen;
            }
        }
        __syncthreads();  // cand_base / warp_cand are reused
    }
}

// The same formats one thread per line over the newline index, with the tile kernel's scanners; every line writes its
// key span and selection, and an error is reported at the line's index.
__global__ void __launch_bounds__(128)
    lines_indexed_kernel(LineParams P, TaxSet T, int need_fields, int mode, PafParams F, uint64_t n_lines,
                         uint64_t *key_off, uint32_t *key_len, uint8_t *sel, unsigned long long *err_word) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_lines) return;
    uint64_t s, e, koff = 0;
    uint32_t klen = 0;
    int ok = 0, code = 0;
    if (line_span(P, i, &s, &e)) {
        if (mode == 2) ok = paf_line_scan(P.in, s, e, i < P.n_nl, F, &koff, &klen, &code);
        else ok = evidence_line(P.in, s, e, i < P.n_nl, mode, T, need_fields, &koff, &klen, &code);
        if (code) report_error(err_word, i, code);
    }
    key_off[i] = koff;
    key_len[i] = klen;
    sel[i] = (uint8_t)ok;
}

enum EvidenceKind { EV_PAF, EV_TXT, EV_READS, EV_SAM };

static sgpu_status evidence_to_set(sgpu_ctx *c, EvidenceKind kind, const uint8_t *d_buf, size_t n, PafParams F,
                                   const TaxSet *T, int need_fields, sgpu_idset **out, uint64_t *err_line) {
    cudaStream_t st = c->stream;
    sgpu_idset *set = nullptr;
    SGPU_TRY(idset_create(c, &set));
    if (n == 0) {  // is_file_empty (alignment.rs:64,93): nothing to insert
        *out = set;
        return SGPU_OK;
    }
    if ((uintptr_t)d_buf & 15) {  // both kernels and the newline index load the buffer in aligned 16-byte words
        sgpu_idset_free(set);
        return SGPU_ERR_INVALID_ARG;
    }
    sgpu_status rc = SGPU_OK;
    bool done = false;
    const int mode = kind == EV_TXT ? 1 : kind == EV_PAF ? 2 : 0;  // (the format argument of both kernels)
    const TaxSet none{nullptr, 0, nullptr, nullptr, 0};
    // The stream may still be busy with what produced d_buf (an NCCL all-gather of the evidence shards, an upload): wait
    // here, BEFORE the scratch and the table are taken from the stream-ordered pool.  The first host round trip of the
    // build is microseconds away anyway, and allocating while the previous set's frees are still queued behind that work
    // makes the pool grow instead of reusing them -- with peer access enabled (NCCL) growing costs milliseconds
    // (measured at 2 GPUs: set build 10.3 ms -> 5.0 ms per step).
    SGPU_CUDA(cudaStreamSynchronize(st));
    if (c->mode == 0 && kind != EV_SAM) {
        // ---- order-free evidence: the tile kernel, no newline index
        do {
            DevBuf<uint64_t> cand_off, ctr;
            DevBuf<uint32_t> cand_len;
            uint64_t cap = (kind == EV_TXT ? n / 8 : n / 32) + 4096;  // (more candidates than room: one retry with the count)
            for (int attempt = 0; attempt < 2 && rc == SGPU_OK; attempt++) {
                if ((rc = cand_off.alloc(cap, st)) != SGPU_OK) break;
                if ((rc = cand_len.alloc(cap, st)) != SGPU_OK) break;
                if ((rc = ctr.alloc(6, st)) != SGPU_OK) break;
                const uint64_t init[6] = {0, ~0ull, 0, 0, 0, 0};
                memcpy(c->h_pinned + 40, init, sizeof(init));
                cudaMemcpyAsync(ctr.p, c->h_pinned + 40, sizeof(init), cudaMemcpyHostToDevice, st);
                TileOut O{cand_off.p, cand_len.p, cap, (unsigned long long *)ctr.p, (unsigned long long *)ctr.p + 1,
                          (unsigned long long *)ctr.p + 2, (unsigned long long *)ctr.p + 3, 0ull, ~0ull, 0};
                lines_tile_kernel<<<(unsigned)ceil_div(n, (size_t)LT_TILE), LT_NT, 0, st>>>(
                    d_buf, (uint64_t)n, T ? *T : none, need_fields, mode, F, O);
                SGPU_LAUNCH(c);
                uint64_t h[6];
                if ((rc = read_u64s(c, ctr.p, h, 6)) != SGPU_OK) break;
                if (h[2]) break;  // pathological line density: the indexed path below
                if (h[1] != ~0ull) {
                    rc = (sgpu_status)(h[1] & 0xFF);
                    if (err_line) {  // the line number of the offending line = newlines before its start
                        uint64_t off = h[1] >> 8, before = 0;
                        // count over the 16-byte aligned prefix, the remaining bytes on the host side are
                        // not available: count_newlines handles any length
                        if (off && count_newlines(c, d_buf, (size_t)off, &before) != SGPU_OK) before = 0;
                        *err_line = before;
                    }
                    done = true;
                    break;
                }
                if (h[0] > cap) {  // more candidates than room: once more with the exact count
                    cap = h[0];
                    continue;
                }
                if (h[0]) {  // every candidate is selected: the kernel has already measured them
                    const SpanStats known{h[0], h[3], h[4] != 0, h[5] != 0};
                    rc = idset_insert_spans(c, set, d_buf, cand_off.p, cand_len.p, nullptr, (size_t)h[0], &known);
                }
                done = true;
                break;
            }
        } while (0);
    }
    sgpu_idset *sam_refs = nullptr;
    if (!done && rc == SGPU_OK) do {
        DevBuf<uint64_t> nlpos, key_off, errw;
        DevBuf<uint32_t> key_len;
        DevBuf<uint8_t> sel;
        uint64_t n_nl = 0;
        if ((rc = index_newlines(c, d_buf, n, nlpos, &n_nl)) != SGPU_OK) break;
        uint64_t n_lines = n_nl + 1;  // the last thread handles an unterminated final line (if any)
        LineParams P{d_buf, (uint64_t)n, nlpos.p, n_nl};
        if ((rc = key_off.alloc(n_lines, st)) != SGPU_OK) break;
        if ((rc = key_len.alloc(n_lines, st)) != SGPU_OK) break;
        if ((rc = sel.alloc(n_lines, st)) != SGPU_OK) break;
        if ((rc = errw.alloc(1, st)) != SGPU_OK) break;
        cudaMemsetAsync(errw.p, 0xFF, 8, st);
        unsigned grid = (unsigned)ceil_div(n_lines, 128);
        if (kind == EV_SAM) {
            // the header's @SQ names first (a small exact set of their own), then the records
            sam_sq_kernel<<<grid, 128, 0, st>>>(P, n_lines, key_off.p, key_len.p, sel.p);
            SGPU_LAUNCH(c);
            if ((rc = idset_create(c, &sam_refs)) != SGPU_OK) break;
            if ((rc = idset_insert_spans(c, sam_refs, d_buf, key_off.p, key_len.p, sel.p, n_lines)) != SGPU_OK) break;
            sam_parse_kernel<<<grid, 128, 0, st>>>(P, F, view_of(sam_refs), sgpu_idset_len(sam_refs) != 0, n_lines, key_off.p,
                                                   key_len.p, sel.p, (unsigned long long *)errw.p);
            SGPU_LAUNCH(c);
        } else {
            lines_indexed_kernel<<<grid, 128, 0, st>>>(P, T ? *T : none, need_fields, mode, F, n_lines, key_off.p,
                                                       key_len.p, sel.p, (unsigned long long *)errw.p);
            SGPU_LAUNCH(c);
        }
        uint64_t ew;
        if ((rc = read_u64s(c, errw.p, &ew, 1)) != SGPU_OK) break;
        if (ew != ~0ull) {
            rc = (sgpu_status)(ew & 0xFF);
            if (err_line) *err_line = ew >> 8;
            break;
        }
        rc = idset_insert_spans(c, set, d_buf, key_off.p, key_len.p, sel.p, n_lines);
        // txt: a blank line is the empty id; the tail thread of a '\n'-terminated buffer offers
        // nothing because its sel is 0
    } while (0);
    if (sam_refs) {
        cudaStreamSynchronize(st);  // the record pass reads the reference names
        sgpu_idset_free(sam_refs);
    }
    if (rc != SGPU_OK) {
        sgpu_idset_free(set);
        return rc;
    }
    *out = set;
    return SGPU_OK;
}

// H2D staging for the host-pointer entry points
static sgpu_status stage_in(sgpu_ctx *c, const uint8_t *h, size_t n, DevBuf<uint8_t> &d) {
    SGPU_TRY(d.alloc(n + 16, c->stream));
    if (n) SGPU_CUDA(cudaMemcpyAsync(d.p, h, n, cudaMemcpyHostToDevice, c->stream));
    return SGPU_OK;
}

// host stage: HashSet<String> of taxids (classifier.rs:124-252 output) -> bitmap + exotic list
static sgpu_status build_taxset(sgpu_ctx *c, const char *const *taxids, const size_t *lens, size_t n,
                                DevBuf<uint32_t> &d_bitmap, DevBuf<uint8_t> &d_exotic, DevBuf<uint32_t> &d_exoff,
                                TaxSet *T) {
    const uint64_t BIT_LIMIT = 1ull << 31;
    uint64_t maxv = 0;
    std::vector<uint64_t> vals;
    std::vector<uint8_t> exotic;
    std::vector<uint32_t> exoff{0};
    for (size_t i = 0; i < n; i++) {
        const char *s = taxids[i];
        size_t l = lens[i];
        bool canon = l >= 1 && l <= 10 && !(l > 1 && s[0] == '0');
        uint64_t v = 0;
        for (size_t k = 0; k < l && canon; k++) {
            canon = s[k] >= '0' && s[k] <= '9';
            v = v * 10 + (uint64_t)(s[k] - '0');
        }
        if (canon && v < BIT_LIMIT) {
            vals.push_back(v);
            if (v > maxv) maxv = v;
        } else {
            exotic.insert(exotic.end(), s, s + l);
            exoff.push_back((uint32_t)exotic.size());
        }
    }
    uint64_t bits = vals.empty() ? 0 : maxv + 1;
    size_t words = (size_t)((bits + 31) / 32);
    std::vector<uint32_t> bm(words ? words : 1, 0);
    for (uint64_t v : vals) bm[v >> 5] |= 1u << (v & 31);
    cudaStream_t st = c->stream;
    SGPU_TRY(d_bitmap.alloc(bm.size(), st));
    SGPU_TRY(d_exotic.alloc(exotic.size() + 1, st));
    SGPU_TRY(d_exoff.alloc(exoff.size(), st));
    SGPU_CUDA(cudaMemcpyAsync(d_bitmap.p, bm.data(), bm.size() * 4, cudaMemcpyHostToDevice, st));
    if (!exotic.empty())
        SGPU_CUDA(cudaMemcpyAsync(d_exotic.p, exotic.data(), exotic.size(), cudaMemcpyHostToDevice, st));
    SGPU_CUDA(cudaMemcpyAsync(d_exoff.p, exoff.data(), exoff.size() * 4, cudaMemcpyHostToDevice, st));
    SGPU_CUDA(cudaStreamSynchronize(st));  // host vectors die at scope exit
    T->bitmap = d_bitmap.p;
    T->bits = bits;
    T->exotic = d_exotic.p;
    T->exotic_off = d_exoff.p;
    T->n_exotic = (uint32_t)(exoff.size() - 1);
    return SGPU_OK;
}

}  // namespace sgpu

using namespace sgpu;

extern "C" {

sgpu_status sgpu_idset_from_paf_dev(sgpu_ctx *c, const uint8_t *d_buf, size_t n, uint64_t min_len, double min_cov,
                                    uint8_t min_mapq, sgpu_idset **out, uint64_t *err_line) {
    if (!c || !out || (n && !d_buf)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    PafParams F{min_len, min_cov, min_mapq};
    return evidence_to_set(c, EV_PAF, d_buf, n, F, nullptr, 0, out, err_line);
}

sgpu_status sgpu_idset_from_paf(sgpu_ctx *c, const uint8_t *buf, size_t n, uint64_t min_len, double min_cov,
                                uint8_t min_mapq, sgpu_idset **out, uint64_t *err_line) {
    if (!c || !out || (n && !buf)) return SGPU_ERR_INVALID_ARG;
    DevBuf<uint8_t> d;
    {
        std::lock_guard<std::mutex> lk(c->mu);
        SGPU_CUDA(cudaSetDevice(c->device));
        SGPU_TRY(stage_in(c, buf, n, d));
    }
    sgpu_status rc = sgpu_idset_from_paf_dev(c, d.p, n, min_len, min_cov, min_mapq, out, err_line);
    cudaStreamSynchronize(c->stream);
    return rc;
}

sgpu_status sgpu_idset_from_sam_dev(sgpu_ctx *c, const uint8_t *d_buf, size_t n, uint64_t min_len, double min_cov,
                                    uint8_t min_mapq, sgpu_idset **out, uint64_t *err_line) {
    if (!c || !out || (n && !d_buf)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    PafParams F{min_len, min_cov, min_mapq};
    return evidence_to_set(c, EV_SAM, d_buf, n, F, nullptr, 0, out, err_line);
}

sgpu_status sgpu_idset_from_sam(sgpu_ctx *c, const uint8_t *buf, size_t n, uint64_t min_len, double min_cov,
                                uint8_t min_mapq, sgpu_idset **out, uint64_t *err_line) {
    if (!c || !out || (n && !buf)) return SGPU_ERR_INVALID_ARG;
    DevBuf<uint8_t> d;
    {
        std::lock_guard<std::mutex> lk(c->mu);
        SGPU_CUDA(cudaSetDevice(c->device));
        SGPU_TRY(stage_in(c, buf, n, d));
    }
    sgpu_status rc = sgpu_idset_from_sam_dev(c, d.p, n, min_len, min_cov, min_mapq, out, err_line);
    cudaStreamSynchronize(c->stream);
    return rc;
}

// binary BAM: `buf` is the BGZF-decompressed stream in HOST memory.  The block_size chain is sequential, so the host
// walks it (one 4-byte read per record) while the bytes are on their way to the device; the records are then parsed by
// one thread each.  An error found by the walk (truncated / undersized record k) only counts when no record before k
// fails on the device: the reference stops at the FIRST failing record.
sgpu_status sgpu_idset_from_bam(sgpu_ctx *c, const uint8_t *buf, size_t n, uint64_t min_len, double min_cov,
                                uint8_t min_mapq, sgpu_idset **out, uint64_t *err_record) {
    if (!c || !out || (n && !buf)) return SGPU_ERR_INVALID_ARG;
    if (err_record) *err_record = 0;
    auto le32 = [&](size_t p) {
        return (uint32_t)buf[p] | ((uint32_t)buf[p + 1] << 8) | ((uint32_t)buf[p + 2] << 16) | ((uint32_t)buf[p + 3] << 24);
    };
    // header: magic, l_text, text, n_ref, (l_name, name, l_ref) per reference
    if (n < 12 || memcmp(buf, "BAM\1", 4) != 0) return SGPU_ERR_BAM_RECORD;
    size_t pos = 8;
    const uint32_t l_text = le32(4);
    if (l_text > n - pos || n - pos - l_text < 4) return SGPU_ERR_BAM_RECORD;
    pos += l_text;
    const uint32_t n_ref = le32(pos);
    pos += 4;
    for (uint32_t r = 0; r < n_ref; r++) {
        if (n - pos < 4) return SGPU_ERR_BAM_RECORD;
        const uint32_t l_name = le32(pos);
        pos += 4;
        if (l_name > n - pos || n - pos - l_name < 4) return SGPU_ERR_BAM_RECORD;
        pos += (size_t)l_name + 4;
    }
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const bool dbg = getenv("SGPU_DEBUG") != nullptr;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto ms_since = [&](std::chrono::steady_clock::time_point t0) {
        return std::chrono::duration<double, std::milli>(now() - t0).count();
    };
    const auto t_start = now();
    DevBuf<uint8_t> d;
    SGPU_TRY(stage_in(c, buf, n, d));  // (asynchronous for pinned buffers: overlaps the walk below)
    const double ms_stage = ms_since(t_start);
    std::vector<uint64_t> offs;
    offs.reserve((n - pos) / 256 + 16);
    bool walk_error = false;
    while (pos < n) {
        if (n - pos < 4) {
            walk_error = true;
            break;
        }
        const uint32_t bs = le32(pos);
        if (bs < 32 || bs > n - pos - 4) {
            walk_error = true;
            break;
        }
        offs.push_back((uint64_t)pos);
        pos += 4 + (size_t)bs;
        // the chain is a dependent load per record (a cache miss each: 37 ns per record measured); records of one
        // file have similar sizes, so the line where the 16th record from here probably starts is fetched now
        const size_t ahead = pos + 16 * (4 + (size_t)bs);
        if (ahead + 64 < n) {
            __builtin_prefetch(buf + ahead);
            __builtin_prefetch(buf + ahead + 64);
        }
    }
    const double ms_walk = ms_since(t_start);
    sgpu_idset *set = nullptr;
    SGPU_TRY(idset_create(c, &set));
    sgpu_status rc = SGPU_OK;
    const uint64_t n_rec = offs.size();
    double ms_parse = 0;
    if (n_rec) do {
        DevBuf<uint64_t> d_off, key_off, errw;
        DevBuf<uint32_t> key_len;
        DevBuf<uint8_t> sel;
        if ((rc = d_off.alloc(n_rec, st)) != SGPU_OK) break;
        if ((rc = key_off.alloc(n_rec, st)) != SGPU_OK) break;
        if ((rc = key_len.alloc(n_rec, st)) != SGPU_OK) break;
        if ((rc = sel.alloc(n_rec, st)) != SGPU_OK) break;
        if ((rc = errw.alloc(1, st)) != SGPU_OK) break;
        if (cudaMemcpyAsync(d_off.p, offs.data(), n_rec * 8, cudaMemcpyHostToDevice, st) != cudaSuccess) {
            rc = SGPU_ERR_CUDA;
            break;
        }
        cudaMemsetAsync(errw.p, 0xFF, 8, st);
        bam_parse_kernel<<<(unsigned)ceil_div(n_rec, (uint64_t)128), 128, 0, st>>>(
            d.p, d_off.p, n_rec, PafParams{min_len, min_cov, min_mapq}, key_off.p, key_len.p, sel.p,
            (unsigned long long *)errw.p);
        SGPU_LAUNCH(c);
        uint64_t ew;
        if ((rc = read_u64s(c, errw.p, &ew, 1)) != SGPU_OK) break;  // (synchronises: `offs` may go out of scope)
        ms_parse = ms_since(t_start);
        if (ew != ~0ull) {
            rc = (sgpu_status)(ew & 0xFF);
            if (err_record) *err_record = ew >> 8;
            break;
        }
        if (!walk_error) rc = idset_insert_spans(c, set, d.p, key_off.p, key_len.p, sel.p, (size_t)n_rec);
    } while (0);
    if (rc == SGPU_OK && walk_error) {
        rc = SGPU_ERR_BAM_RECORD;
        if (err_record) *err_record = n_rec;
    }
    cudaStreamSynchronize(st);
    if (dbg)
        fprintf(stderr, "[sgpu] from_bam: %llu records; cumulative ms: copy issued %.2f, chain walked %.2f, parsed %.2f, set built %.2f\n",
                (unsigned long long)n_rec, ms_stage, ms_walk, ms_parse, ms_since(t_start));
    if (rc != SGPU_OK) {
        sgpu_idset_free(set);
        return rc;
    }
    *out = set;
    return SGPU_OK;
}

sgpu_status sgpu_idset_from_txt_dev(sgpu_ctx *c, const uint8_t *d_buf, size_t n, sgpu_idset **out,
                                    uint64_t *err_line) {
    if (!c || !out || (n && !d_buf)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    return evidence_to_set(c, EV_TXT, d_buf, n, PafParams{0, 0.0, 0}, nullptr, 0, out, err_line);
}

sgpu_status sgpu_idset_from_txt(sgpu_ctx *c, const uint8_t *buf, size_t n, sgpu_idset **out, uint64_t *err_line) {
    if (!c || !out || (n && !buf)) return SGPU_ERR_INVALID_ARG;
    DevBuf<uint8_t> d;
    {
        std::lock_guard<std::mutex> lk(c->mu);
        SGPU_CUDA(cudaSetDevice(c->device));
        SGPU_TRY(stage_in(c, buf, n, d));
    }
    sgpu_status rc = sgpu_idset_from_txt_dev(c, d.p, n, out, err_line);
    cudaStreamSynchronize(c->stream);
    return rc;
}

// position of the first '\n' of buf[0..n), or ~0: one warp
__global__ void first_newline_kernel(const uint8_t *buf, uint64_t n, unsigned long long *out) {
    const int lane = threadIdx.x;
    for (uint64_t base = 0; base < n; base += 512) {
        const uint64_t pos = base + (uint64_t)lane * 16;
        uint32_t m = 0;
        if (pos < n) {
            m = nl_mask16(ld_nc_u4(buf + pos));
            if (n - pos < 16) m &= (1u << (n - pos)) - 1u;
        }
        const unsigned b = __ballot_sync(0xffffffffu, m != 0);
        if (b) {
            const int first = __ffs(b) - 1;
            if (lane == first) *out = pos + (uint64_t)(__ffs(m) - 1);
            return;
        }
    }
}

sgpu_status sgpu_idset_partition_txt_dev(sgpu_ctx *c, const uint8_t *d_buf, size_t n, size_t own_len, int starts_line,
                                         int is_last, uint32_t log2_vpages, void *d_recs, size_t cap_recs,
                                         uint64_t *d_vstart, uint64_t *n_recs, uint64_t *err_line) {
    if (!c || !d_recs || !d_vstart || !n_recs || (n && !d_buf) || own_len > n || (is_last && own_len != n) ||
        log2_vpages < 1 || log2_vpages > 30 || ((uintptr_t)d_buf & 15))
        return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    SGPU_CUDA(cudaStreamSynchronize(st));  // (scratch comes from the stream-ordered pool: see evidence_to_set)
    if (err_line) *err_line = 0;
    *n_recs = 0;
    // the first line this shard owns: a partial first line is the previous shard's
    uint64_t own_begin = 0;
    if (!starts_line) {
        DevBuf<unsigned long long> pos;
        SGPU_TRY(pos.alloc(1, st));
        SGPU_CUDA(cudaMemsetAsync(pos.p, 0xFF, 8, st));
        first_newline_kernel<<<1, 32, 0, st>>>(d_buf, own_len, pos.p);
        SGPU_LAUNCH(c);
        uint64_t p;
        SGPU_TRY(read_u64s(c, pos.p, &p, 1));
        own_begin = p == ~0ull ? (uint64_t)own_len : p + 1;
    }
    DevBuf<uint64_t> cand_off, ctr;
    DevBuf<uint32_t> cand_len;
    uint64_t cap = n / 8 + 4096, h[6] = {0, 0, 0, 0, 0, 0};
    const TaxSet none{nullptr, 0, nullptr, nullptr, 0};
    for (int attempt = 0; attempt < 2; attempt++) {
        SGPU_TRY(cand_off.alloc(cap, st));
        SGPU_TRY(cand_len.alloc(cap, st));
        SGPU_TRY(ctr.alloc(6, st));
        const uint64_t init[6] = {0, ~0ull, 0, 0, 0, 0};
        memcpy(c->h_pinned + 40, init, sizeof(init));
        SGPU_CUDA(cudaMemcpyAsync(ctr.p, c->h_pinned + 40, sizeof(init), cudaMemcpyHostToDevice, st));
        TileOut O{cand_off.p, cand_len.p, cap, (unsigned long long *)ctr.p, (unsigned long long *)ctr.p + 1,
                  (unsigned long long *)ctr.p + 2, (unsigned long long *)ctr.p + 3, own_begin, (uint64_t)own_len, is_last ? 0 : 1};
        if (is_last) O.own_end = ~0ull;
        if (n) {
            lines_tile_kernel<<<(unsigned)ceil_div(n, (size_t)LT_TILE), LT_NT, 0, st>>>(d_buf, (uint64_t)n, none, 0, 1,
                                                                                       PafParams{0, 0.0, 0}, O);
            SGPU_LAUNCH(c);
        }
        SGPU_TRY(read_u64s(c, ctr.p, h, 6));
        if (h[0] <= cap) break;
        cap = h[0];
    }
    // anything out of the ordinary (a parse error, pathological line density, a line past the halo): the replicated build
    // reports it exactly as the unsharded call would
    if (h[2] || h[1] != ~0ull) return SGPU_ERR_NOT_SHARDABLE;
    const uint64_t flags = ((h[3] || h[5]) ? 1ull : 0ull) | (h[4] ? 2ull : 0ull);
    SGPU_TRY(idset_partition(c, d_buf, cand_off.p, cand_len.p, (size_t)h[0], log2_vpages, (ulonglong2 *)d_recs, cap_recs, d_vstart,
                             flags));
    *n_recs = (flags & 1) ? 0 : h[0];
    return SGPU_OK;
}

sgpu_status sgpu_idset_assemble_dev(sgpu_ctx *c, int n_parts, const void *const *d_recs, const uint64_t *const *d_vstart,
                                    uint32_t log2_vpages, sgpu_idset **out) {
    if (!c || !out || !d_recs || !d_vstart) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    SGPU_CUDA(cudaStreamSynchronize(c->stream));
    sgpu_idset *set = nullptr;
    SGPU_TRY(idset_create(c, &set));
    const sgpu_status rc = idset_assemble(c, n_parts, (const ulonglong2 *const *)d_recs, d_vstart, log2_vpages, set);
    if (rc != SGPU_OK) {
        sgpu_idset_free(set);
        return rc;
    }
    *out = set;
    return SGPU_OK;
}

sgpu_status sgpu_idset_from_reads_dev(sgpu_ctx *c, const uint8_t *d_buf, size_t n, int style,
                                      const char *const *taxids, const size_t *taxid_lens, size_t n_taxids,
                                      sgpu_idset **out, uint64_t *err_line) {
    if (!c || !out || (n && !d_buf) || (n_taxids && (!taxids || !taxid_lens)) || (style != 0 && style != 1))
        return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    DevBuf<uint32_t> bm, exoff;
    DevBuf<uint8_t> ex;
    TaxSet T;
    SGPU_TRY(build_taxset(c, taxids, taxid_lens, n_taxids, bm, ex, exoff, &T));
    return evidence_to_set(c, EV_READS, d_buf, n, PafParams{0, 0.0, 0}, &T, style == 0 ? 5 : 7, out, err_line);
}

sgpu_status sgpu_idset_from_reads(sgpu_ctx *c, const uint8_t *buf, size_t n, int style, const char *const *taxids,
                                  const size_t *taxid_lens, size_t n_taxids, sgpu_idset **out, uint64_t *err_line) {
    if (!c || !out || (n && !buf)) return SGPU_ERR_INVALID_ARG;
    DevBuf<uint8_t> d;
    {
        std::lock_guard<std::mutex> lk(c->mu);
        SGPU_CUDA(cudaSetDevice(c->device));
        SGPU_TRY(stage_in(c, buf, n, d));
    }
    sgpu_status rc = sgpu_idset_from_reads_dev(c, d.p, n, style, taxids, taxid_lens, n_taxids, out, err_line);
    cudaStreamSynchronize(c->stream);
    return rc;
}

}  // extern "C"
