// common.cuh -- shared host/device helpers for libscrubby_gpu (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "../../include/scrubby_gpu.h"

namespace sgpu {

// ---------------------------------------------------------------- host side
void set_cuda_error(cudaError_t e, const char *file, int line);

#define SGPU_CUDA(call)                                        \
    do {                                                       \
        cudaError_t _e = (call);                               \
        if (_e != cudaSuccess) {                               \
            ::sgpu::set_cuda_error(_e, __FILE__, __LINE__);    \
            return SGPU_ERR_CUDA;                              \
        }                                                      \
    } while (0)

#define SGPU_TRY(call)                     \
    do {                                   \
        sgpu_status _s = (call);           \
        if (_s != SGPU_OK) return _s;      \
    } while (0)

static inline size_t ceil_div(size_t a, size_t b) { return (a + b - 1) / b; }
static inline uint64_t next_pow2(uint64_t v) {
    uint64_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

struct Ctx;

// Stream-ordered scratch buffer (cudaMallocAsync on the context's stream), freed on scope exit.
template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    cudaStream_t st = nullptr;
    DevBuf() {}
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    sgpu_status alloc(size_t count, cudaStream_t s) {
        release();
        st = s;
        n = count;
        size_t bytes = (count ? count : 1) * sizeof(T);
        cudaError_t e = cudaMallocAsync((void **)&p, bytes, s);
        if (e != cudaSuccess) {
            p = nullptr;
            set_cuda_error(e, __FILE__, __LINE__);
            return e == cudaErrorMemoryAllocation ? SGPU_ERR_NOMEM : SGPU_ERR_CUDA;
        }
        return SGPU_OK;
    }
    void release() {
        if (p) cudaFreeAsync(p, st);
        p = nullptr;
        n = 0;
    }
    T *take() {
        T *q = p;
        p = nullptr;
        return q;
    }
};

}  // namespace sgpu

struct sgpu_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int mode = 0;
    int sm_count = 148;
    uint64_t launches = 0;
    std::atomic<int> refs{1};  // the handle itself + every live idset built on it
    std::mutex mu;
    // pinned staging for small D2H results
    uint64_t *h_pinned = nullptr;  // 64 x u64
    // copy streams of the pipelined host-buffer path (created on first use)
    cudaStream_t s_in = nullptr, s_out = nullptr;
    // grow-only staging of that path (input file, two kept and two removed chunk buffers): taking GBs from the
    // stream-ordered pool on every call costs an occasional 0.3-0.6 s remap; released with the context
    uint8_t *pipe_buf[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t pipe_cap[5] = {0, 0, 0, 0, 0};
    // optional timing of the dominant (fused) kernel with CUDA events on the launching stream
    bool profiling = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
    size_t prof_used = 0;
    uint64_t prof_alg_bytes = 0;
};

struct Slot {
    unsigned long long lo, hi;
};

#ifndef SGPU_IDSET_BUCKET
#define SGPU_IDSET_BUCKET 8  // slots per bucket (idset.cuh)
#endif

struct sgpu_idset {
    sgpu_ctx *ctx = nullptr;  // owner of the stream the buffers were allocated on
    int device = 0;
    Slot *d_table = nullptr;
    uint64_t n_buckets = 0;  // 128-byte buckets of eight slots: a whole number of 256-bucket pages (0 = no table yet)
    uint64_t slots() const { return n_buckets * SGPU_IDSET_BUCKET; }
    uint8_t *d_arena = nullptr;
    uint64_t arena_used = 0, arena_cap = 0;
    uint64_t count = 0;      // distinct non-empty ids
    bool has_empty = false;  // "" is a member
};

namespace sgpu {

#define SGPU_LAUNCH(ctx) ((ctx)->launches++)

// ---------------------------------------------------------------- device side
#ifdef __CUDACC__

__device__ __forceinline__ uint4 ld_nc_u4(const void *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// bit i of the result (i in 0..3) is set iff byte i of w equals c.  Exact (no borrow artefacts).
__device__ __forceinline__ uint32_t eq_mask4(uint32_t w, uint32_t c4) {
    uint32_t x = w ^ c4;                                        // zero bytes where equal
    uint32_t t = ((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x;         // bit7 set iff byte non-zero
    t = ~t & 0x80808080u;                                       // bit7 set iff byte zero
    return ((t >> 7) & 1u) | ((t >> 14) & 2u) | ((t >> 21) & 4u) | ((t >> 28) & 8u);
}

// 0x80 in every byte of w that equals the byte of c4 (exact for every byte value)
__device__ __forceinline__ uint32_t eq_flags4(uint32_t w, uint32_t c4) {
    const uint32_t x = w ^ c4;
    return ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
}
// 16-bit mask (bit i <-> byte i) of the bytes of a 16-byte chunk that equal the byte of c4: four words of
// 0x80 flags gathered with dp4a (the flag byte times its bit weight, summed per word pair)
__device__ __forceinline__ uint32_t eq_mask16(uint4 v, uint32_t c4) {
    const uint32_t lo = __dp4a(eq_flags4(v.x, c4), 0x08040201u, __dp4a(eq_flags4(v.y, c4), 0x80402010u, 0u));
    const uint32_t hi = __dp4a(eq_flags4(v.z, c4), 0x08040201u, __dp4a(eq_flags4(v.w, c4), 0x80402010u, 0u));
    return (lo >> 7) | (hi << 1);
}
// 16-bit mask of bytes equal to '\n' in a 16-byte chunk (bit i <-> byte i)
__device__ __forceinline__ uint32_t nl_mask16(uint4 v) { return eq_mask16(v, 0x0a0a0a0au); }

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 32;
    x *= 0xd6e8feb86659fd93ULL;
    x ^= x >> 32;
    x *= 0xd6e8feb86659fd93ULL;
    x ^= x >> 32;
    return x;
}

// Unicode White_Space (Rust char::is_whitespace)
__device__ __forceinline__ bool is_ws_cp(uint32_t cp) {
    if (cp >= 0x09 && cp <= 0x0D) return true;
    if (cp == 0x20 || cp == 0x85 || cp == 0xA0 || cp == 0x1680) return true;
    if (cp >= 0x2000 && cp <= 0x200A) return true;
    return cp == 0x2028 || cp == 0x2029 || cp == 0x202F || cp == 0x205F || cp == 0x3000;
}
__device__ __forceinline__ bool is_ws_ascii(uint8_t c) { return (c >= 0x09 && c <= 0x0D) || c == 0x20; }

// Rust std::str::from_utf8 acceptance
__device__ inline bool utf8_valid(const uint8_t *s, size_t n) {
    size_t i = 0;
    while (i < n) {
        uint8_t c = s[i];
        if (c < 0x80) {
            i++;
        } else if (c >= 0xC2 && c <= 0xDF) {
            if (i + 1 >= n || (s[i + 1] & 0xC0) != 0x80) return false;
            i += 2;
        } else if (c >= 0xE0 && c <= 0xEF) {
            if (i + 2 >= n) return false;
            uint8_t c1 = s[i + 1], c2 = s[i + 2];
            uint8_t lo = c == 0xE0 ? 0xA0 : 0x80, hi = c == 0xED ? 0x9F : 0xBF;
            if (c1 < lo || c1 > hi || (c2 & 0xC0) != 0x80) return false;
            i += 3;
        } else if (c >= 0xF0 && c <= 0xF4) {
            if (i + 3 >= n) return false;
            uint8_t c1 = s[i + 1], c2 = s[i + 2], c3 = s[i + 3];
            uint8_t lo = c == 0xF0 ? 0x90 : 0x80, hi = c == 0xF4 ? 0x8F : 0xBF;
            if (c1 < lo || c1 > hi || (c2 & 0xC0) != 0x80 || (c3 & 0xC0) != 0x80) return false;
            i += 4;
        } else {
            return false;
        }
    }
    return true;
}

__device__ __forceinline__ size_t utf8_decode(const uint8_t *s, size_t i, uint32_t *cp) {
    uint8_t c = s[i];
    if (c < 0x80) { *cp = c; return 1; }
    if (c < 0xE0) { *cp = ((uint32_t)(c & 0x1F) << 6) | (s[i + 1] & 0x3F); return 2; }
    if (c < 0xF0) {
        *cp = ((uint32_t)(c & 0x0F) << 12) | ((uint32_t)(s[i + 1] & 0x3F) << 6) | (s[i + 2] & 0x3F);
        return 3;
    }
    *cp = ((uint32_t)(c & 0x07) << 18) | ((uint32_t)(s[i + 1] & 0x3F) << 12) |
          ((uint32_t)(s[i + 2] & 0x3F) << 6) | (s[i + 3] & 0x3F);
    return 4;
}

// str::trim over VALID utf-8: [*b, *e) is the trimmed range
__device__ inline void utf8_trim(const uint8_t *s, size_t n, size_t *b, size_t *e) {
    size_t i = 0;
    while (i < n) {
        uint32_t cp;
        size_t l = utf8_decode(s, i, &cp);
        if (!is_ws_cp(cp)) break;
        i += l;
    }
    size_t j = n;
    while (j > i) {
        size_t k = j - 1;
        while (k > i && (s[k] & 0xC0) == 0x80) k--;
        uint32_t cp;
        utf8_decode(s, k, &cp);
        if (!is_ws_cp(cp)) break;
        j = k;
    }
    *b = i;
    *e = j;
}

// utils.rs:91-103 get_id over the header bytes (without '@', trailing CR trimmed).
// Returns 0, SGPU_ERR_RECORD_NAME_UTF8 or SGPU_ERR_FASTQ_HEADER.
__device__ inline int get_id_span(const uint8_t *h, size_t n, size_t *off, size_t *len) {
    // ASCII fast path (identical to the Unicode rules when no byte has its high bit set)
    bool high = false;
    for (size_t k = 0; k < n; k++) high |= h[k] >= 0x80;
    size_t i = 0, j;
    if (!high) {
        while (i < n && is_ws_ascii(h[i])) i++;
        if (i >= n) return SGPU_ERR_FASTQ_HEADER;
        j = i;
        while (j < n && !is_ws_ascii(h[j])) j++;
        *off = i;
        *len = j - i;
        return 0;
    }
    // slow path: full validation + Unicode whitespace
    if (!utf8_valid(h, n)) return SGPU_ERR_RECORD_NAME_UTF8;
    i = 0;
    while (i < n) {
        uint32_t cp;
        size_t l = utf8_decode(h, i, &cp);
        if (!is_ws_cp(cp)) break;
        i += l;
    }
    if (i >= n) return SGPU_ERR_FASTQ_HEADER;
    j = i;
    while (j < n) {
        uint32_t cp;
        size_t l = utf8_decode(h, j, &cp);
        if (is_ws_cp(cp)) break;
        j += l;
    }
    *off = i;
    *len = j - i;
    return 0;
}

// <uN as FromStr>::from_str: optional '+', ASCII digits, overflow is an error
__device__ inline bool parse_uint(const uint8_t *s, size_t n, uint64_t maxv, uint64_t *out) {
    if (n == 0) return false;
    if (s[0] == '+' || s[0] == '-') {
        if (n == 1 || s[0] == '-') return false;
        s++;
        n--;
    }
    uint64_t v = 0;
    for (size_t i = 0; i < n; i++) {
        uint32_t d = (uint32_t)s[i] - '0';
        if (d > 9) return false;
        if (v > (0xFFFFFFFFFFFFFFFFULL - d) / 10) return false;
        v = v * 10 + d;
        if (v > maxv) return false;
    }
    *out = v;
    return true;
}

// first error wins: (index << 8 | code), smaller is earlier
__device__ __forceinline__ void report_error(unsigned long long *err_word, uint64_t index, int code) {
    atomicMin(err_word, (unsigned long long)((index << 8) | (uint64_t)code));
}

// cooperative copy by one warp; src/dst arbitrary alignment, 4-byte coalesced stores
__device__ __forceinline__ void warp_copy(uint8_t *dst, const uint8_t *src, size_t n, int lane) {
    size_t head = (4 - ((uintptr_t)dst & 3)) & 3;
    if (head > n) head = n;
    if ((size_t)lane < head) dst[lane] = src[lane];
    dst += head;
    src += head;
    n -= head;
    size_t nw = n >> 2;
    const unsigned sh = ((unsigned)((uintptr_t)src & 3)) * 8;
    const uint32_t *s32 = (const uint32_t *)((uintptr_t)src & ~(uintptr_t)3);
    uint32_t *d32 = (uint32_t *)dst;
    for (size_t i = lane; i < nw; i += 32) {
        uint32_t lo = s32[i];
        uint32_t hi = sh ? s32[i + 1] : 0u;
        d32[i] = __funnelshift_r(lo, hi, sh);
    }
    size_t tail = n & 3;
    if ((size_t)lane < tail) dst[(nw << 2) + lane] = src[(nw << 2) + lane];
}

#endif  // __CUDACC__

// ---------------------------------------------------------------- internal API (host)
// scan.cu
sgpu_status exclusive_scan_u32_to_u64(sgpu_ctx *c, const uint32_t *d_in, uint64_t *d_out, size_t n,
                                      uint64_t *d_total);
sgpu_status exclusive_scan_u64(sgpu_ctx *c, const uint64_t *d_in, uint64_t *d_out, size_t n,
                               uint64_t *d_total);
// lines.cu: positions of every '\n' in d_buf[0..n)
sgpu_status index_newlines(sgpu_ctx *c, const uint8_t *d_buf, size_t n, DevBuf<uint64_t> &nlpos,
                           uint64_t *n_newlines);
sgpu_status count_newlines(sgpu_ctx *c, const uint8_t *d_buf, size_t n, uint64_t *count);
// d2h of a few u64 through the pinned staging buffer, synchronises the stream
sgpu_status read_u64s(sgpu_ctx *c, const void *d_src, uint64_t *h_dst, size_t count);
// h2d of a few u64 (scratch initialisation) through the upper half of the pinned staging buffer, stream-ordered
sgpu_status write_u64s(sgpu_ctx *c, void *d_dst, const uint64_t *h_src, size_t count);

// capi.cu: drops one reference; the last one tears the context down
void ctx_release(sgpu_ctx *c);

// idset.cu
sgpu_status idset_create(sgpu_ctx *c, sgpu_idset **out);
// insert the selected keys: key i is d_src[off[i] .. off[i]+len[i]) when sel[i] != 0
// `known`: what a pass over the candidates would find (the producer has already counted), or nullptr
struct SpanStats {
    uint64_t n_sel, long_bytes;
    bool has_empty, too_long;
};
sgpu_status idset_insert_spans(sgpu_ctx *c, sgpu_idset *s, const uint8_t *d_src, const uint64_t *d_off,
                               const uint32_t *d_len, const uint8_t *d_sel, size_t n, const SpanStats *known = nullptr);

// idset_build.cu: the sharded build (slot images grouped by virtual page per rank, assembled from all ranks' lists)
sgpu_status idset_partition(sgpu_ctx *c, const uint8_t *d_src, const uint64_t *d_off, const uint32_t *d_len, size_t n,
                            uint32_t log2_v, ulonglong2 *d_recs, size_t cap_recs, uint64_t *d_vstart, uint64_t flags);
sgpu_status idset_assemble(sgpu_ctx *c, int n_parts, const ulonglong2 *const *recs, const uint64_t *const *vstart,
                           uint32_t log2_v, sgpu_idset *s);

// fastq.cu
struct FastqIndex;  // per-record metadata produced by the general path

}  // namespace sgpu
