// fastq_fused.cu -- single-pass fused parse -> probe -> compact kernel for CANONICAL FASTQ.
//
// Replaces the whole of FastqCleaner::clean_reads (cleaner.rs:731-760) -- needletail framing,
// get_id (utils.rs:91-103), `read_ids.contains` and `record.write` -- with ONE kernel that
// reads every input byte once and writes every output byte once.
//
// Canonical input = LF line endings, bare "+" separator lines, a final newline, ASCII
// bytes, well-formed records.  For such input the reference's output is a byte partition
// of the input (SURVEY 8a row a2), so the work is an order-preserving stream compaction of
// records.  Anything else (CRLF, "+id" separators, missing final newline, non-ASCII bytes,
// parse errors, pathological line density) raises the device `fallback` flag and the caller
// re-runs the always-exact general path (fastq_general.cu); nothing is approximated.
//
// Structure (v3.3): persistent CTAs of 256 threads, five resident per SM, each looping over
// dynamically ticketed 36 KiB tiles (tickets are taken in order, so every tile a look-back waits on is
// owned by a running CTA).  One shared-memory tile buffer per CTA; the latency
// of a tile's dependent steps (load, set probes, look-back) is hidden by the other resident CTAs.
// The byte-level phases (P1, P4) run on all warps; the record-level phases run with one thread per
// newline / per record, so only as many warps as there are records execute them.
//   load : one thread issues a TMA bulk copy (cp.async.bulk + mbarrier) of the tile + 16 B pre-halo
//          + post-halo into shared memory; tiles are pulled into L2 one generation of CTAs ahead;
//   P1   : 16-byte vector loads -> exact '\n' bit masks (SWAR + dp4a gather), packed warp scan of
//          the counts, newline positions scattered in order;
//   phase: line number mod 4 SPECULATED from the first "\n+\n" in the tile and published at once
//          (a tile without one does a real decoupled look-back over 2-bit phases);
//   P2   : one thread per newline: CR / "+\n" checks by role, record starts;
//   P3   : one thread per record start: '@', id token -> slot image straight from a 16-byte
//          window, exact probe of the id set, seq/qual length check, warp scans of kept bytes;
//          runs of consecutive records with the same fate are found with ballots and cut into
//          copy items (source, length, stream offset);
//   scan : decoupled look-back by one warp over (kept bytes, state of the record that straddles
//          the tile edge), 32 descriptors per round, combined as a 3-state transducer; it starts
//          before the tile's own records are done (it only needs the tiles before);
//   P4   : a warp per copy item: 16-byte destination-aligned stores, the source re-aligned from two
//          16-byte shared loads with funnel shifts (the shift is uniform per item), edge bytes by
//          one byte store per lane.
// The speculated phases and the cross-tile seq/qual length sums are verified exactly by a tiny
// follow-up kernel over per-tile metadata; any mismatch is a fallback, never a wrong answer.
// Records may straddle any number of tiles (ONT reads); only the id token must lie within the
// post-halo of the tile where the record starts.
//
// Shards (multi-GPU, SURVEY 8e): the buffer starts `lead` (< 16) bytes before the first owned
// record start and holds a halo after `own_len`; records that start after own_len are seen but
// belong to the next shard (state "none": written to neither stream).
#include <stdlib.h>

#include "fastq_records.cuh"

namespace sgpu {

#ifndef SGPU_FUSED_CTAS
#define SGPU_FUSED_CTAS 5
#endif
#ifndef SGPU_FUSED_PIECE
#define SGPU_FUSED_PIECE 2048
#endif
#ifndef SGPU_FUSED_HALO
#define SGPU_FUSED_HALO 256
#endif
constexpr int NT = 256;                 // threads per CTA
constexpr int NW = NT / 32;             // warps per CTA
constexpr int NTHREADS = NT;
// Throughput = tile bytes resident in shared memory / time a tile stays there (load .. copy-out, ~15 us of
// which ~6 us are the in-order wait and the load): the tile is as large as five CTAs per SM allow.
#ifndef SGPU_FUSED_FC
#define SGPU_FUSED_FC 9
#endif
constexpr int FC = SGPU_FUSED_FC;       // 16-byte chunks per thread
constexpr int TILE = NT * FC * 16;      // 36 KiB
constexpr int PRE = 16;                 // pre-halo (previous 16 bytes)
constexpr int HALO = SGPU_FUSED_HALO;   // post-halo: id token of the last record start, "+\n" after the last newline
constexpr int BUF = PRE + TILE + HALO;  // bytes of the tile buffer
#ifndef SGPU_FUSED_RMAX_PER_KIB
#define SGPU_FUSED_RMAX_PER_KIB 10
#endif
constexpr int RMAX = TILE / 1024 * SGPU_FUSED_RMAX_PER_KIB;  // record starts per tile (>= 102 bytes per record on average)
constexpr int LMAX = 4 * RMAX + 8;      // newline list capacity per tile
constexpr int PIECE = SGPU_FUSED_PIECE; // copy items are at most this long
constexpr int IMAX = RMAX + 2 * (TILE / PIECE) + 8;  // copy items per tile
#ifndef SGPU_FUSED_DSTRIDE
#define SGPU_FUSED_DSTRIDE 4
#endif
#ifndef SGPU_FUSED_POLL_NS
#define SGPU_FUSED_POLL_NS 500
#endif
#ifndef SGPU_FUSED_LOAD_PIECE
#define SGPU_FUSED_LOAD_PIECE 16384
#endif
#ifndef SGPU_FUSED_LB_K
#define SGPU_FUSED_LB_K 1
#endif
// 64-bit words between the look-back #2 descriptors of two tiles: one 32-byte sector each, so that the
// hundreds of polling warps do not all hit the same few L2 lines (measured: 1.18 -> 1.06 ms per 1.65 GB)
constexpr int DSTRIDE = SGPU_FUSED_DSTRIDE;
constexpr int LOAD_PIECE = SGPU_FUSED_LOAD_PIECE;  // bytes per bulk copy of a tile load
constexpr int CTAS_PER_SM = SGPU_FUSED_CTAS;  // resident CTAs the kernel is sized for (registers, shared memory)
static_assert(TILE + HALO < 65536 && TILE / PIECE <= 32 && HALO % 16 == 0, "tile offsets are 16-bit; head pieces fit a warp");

constexpr uint64_t ST_AGG = 1ull << 62, ST_INC = 2ull << 62, ST_MASK = 3ull << 62;
// run / carry states
constexpr uint32_t F_OTHER = 0, F_KEPT = 1, F_NONE = 2, F_INVALID = 3;
// copy item tags
constexpr uint32_t TAG_KEPT = 0u << 30, TAG_OTHER = 1u << 30, TAG_HEAD = 2u << 30;

struct FusedResult {
    unsigned long long fallback;    // != 0: input is not canonical, use the general path
    unsigned long long kept_total;  // bytes written to out_w
    unsigned long long reads_in, reads_out;
    unsigned long long ticket;      // dynamic tile counter
    unsigned long long reason;      // first fallback reason (diagnostics)
    unsigned long long owned_end;   // end of the last owned record (shards); ~0 when no foreign record was seen
    unsigned long long n_spans;     // ids mode: id tokens emitted
    unsigned long long overflow;    // != 0: an output buffer was too small (nothing is written past its capacity)
    unsigned long long own_newlines;  // shards: '\n' bytes in the owned range (fused_own_newlines_kernel)
};

struct FusedParams {
    const uint8_t *in;
    uint64_t n_in;
    uint64_t n_tiles;
    uint64_t own_len;  // records that start after own_len belong to the next shard (ignored when is_last)
    uint32_t lead;     // bytes before the first record start (< 16; they belong to the previous shard)
    int is_last;       // the buffer ends at the end of the file
    uint8_t *out_w, *out_o;
    uint64_t cap_w, cap_o;  // capacities of the two outputs: a copy item that would end past one raises `overflow`
    int reverse;
    IdSetView set;
    unsigned long long *desc1, *desc2;  // per tile look-back descriptors (zero initialised)
    long long *sum_total, *sum_head;    // per tile signed newline-position sums (length check)
    uint32_t *nl_count;                 // per tile newline count (phase verification)
    uint8_t *has_term, *phase_used;     // per tile: has a record end; line phase (mod 4) the tile assumed
    uint64_t pf_dist;  // L2 prefetch distance in tiles (0 = off)
    // ids mode (ReadDifference::get_difference, utils.rs:250-285): nothing is copied; the id token of every
    // record that is NOT in `set` (all records when the set is empty) is appended to a span list, any order
    int ids_mode;
    uint64_t *span_off;  // offset of the token in `in`
    uint32_t *span_len;
    uint64_t span_cap;
    FusedResult *res;
};

// ------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
#ifdef SGPU_LD_EF  // experiment: the input is read once -- evict-first in L2
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
                 : "memory");
#else
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
#endif
}
__device__ __forceinline__ void bulk_prefetch_l2(const void *src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(1000000u)  // suspend-time hint (ns): sleep in hardware, do not spin
        : "memory");
    return ok != 0;
}

// The look-back descriptors carry their whole payload in one 64-bit word, so relaxed
// (non-fencing) gpu-scope accesses are sufficient: nothing else is ordered against them.
__device__ __forceinline__ unsigned long long ld_relaxed(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed(unsigned long long *p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_global_v4(void *p, uint4 v) {
#ifdef SGPU_ST_CS  // experiment: streaming (evict-first) output stores
    asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
#else
    asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
#endif
}
__device__ __forceinline__ void st_global_u8(void *p, uint32_t v) {
    asm volatile("st.global.u8 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint4 lds_v4(uint32_t saddr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
    return v;
}

// ------------------------------------------------------------------ byte classification
// flag byte (0x80 per matching byte) of the bytes of w equal to '\n'.  Exact for every byte value:
// low 7 bits zero after the xor  <=>  the add does not carry into bit 7; bit 7 of w itself must be clear.
__device__ __forceinline__ uint32_t nl_flags(uint32_t w) {
    const uint32_t b = ((w ^ 0x0a0a0a0au) & 0x7f7f7f7fu) + 0x7f7f7f7fu;
    return ~(b | w) & 0x80808080u;
}
// four words of 0x80 flags -> 16-bit mask in byte order (bit i <-> byte i): dp4a sums flag * weight
__device__ __forceinline__ uint32_t gather16(uint32_t f0, uint32_t f1, uint32_t f2, uint32_t f3) {
    const uint32_t lo = __dp4a(f0, 0x08040201u, __dp4a(f1, 0x80402010u, 0u));  // 128 * (bits 0..7)
    const uint32_t hi = __dp4a(f2, 0x08040201u, __dp4a(f3, 0x80402010u, 0u));  // 128 * (bits 8..15)
    return (lo >> 7) | (hi << 1);
}
__device__ __forceinline__ uint32_t nl_mask16_v2(uint4 v) {
    return gather16(nl_flags(v.x), nl_flags(v.y), nl_flags(v.z), nl_flags(v.w));
}
// 0x80 per byte <= 0x20 (ASCII input: every byte < 0x80, so the add cannot carry between bytes)
__device__ __forceinline__ uint32_t le20_flags(uint32_t w) { return ~(w + 0x5f5f5f5fu) & 0x80808080u; }

// ------------------------------------------------------------------ shared memory
struct __align__(8) Item {
    uint16_t src, len;  // source offset in the tile, bytes (1..PIECE)
    uint32_t rel;       // tag | offset relative to the stream's base for this tile
};

struct __align__(128) CtaSmem {
    uint64_t full;         // mbarrier: tile load complete
    uint64_t first_tile;   // the CTA's first ticket
    uint64_t next_tile;    // the ticket after the tile in flight
    uint64_t kept_before;  // look-back #2 result
    uint32_t carry;        // state of the record carried into the tile
    uint64_t span_base;    // ids mode: where this tile's spans go
    uint32_t c0;           // newlines before the tile, mod 4 (only when the speculation found no "\n+\n")
    uint32_t n_items;
    uint32_t last_flag;    // fate of the last record that starts in the tile
    uint32_t head_len;     // bytes of the carried-in record (== tile_len when no record starts in the tile)
    uint32_t rest_total;   // kept bytes of the records that start in the tile
    uint32_t none_pos;     // first record start of the tile that belongs to the next shard
    uint32_t none_cnt;
    uint32_t warp_tot[NW];  // newlines of the warp's region (bit 31: a 16-byte chunk with more than two)
    uint32_t scan_tot[NW];
    __align__(16) uint16_t nlp[LMAX];  // newline positions of the tile, in order
    Item items[IMAX];
    __align__(16) uint8_t buf[BUF];
};

__device__ __forceinline__ void set_fallback(FusedResult *res, int reason) {
    if (atomicExch(&res->fallback, 1ull) == 0ull) {
        res->reason = (unsigned long long)reason;
        // the result will be discarded: no CTA takes another tile (the tiles in flight finish: everything they
        // wait for was ticketed before them)
        atomicAdd(&res->ticket, 1ull << 40);
    }
}

// ------------------------------------------------------------------ look-back #1 (rare): line phase
// exclusive prefix of the newline counts mod 4, by one warp, for tiles without a "\n+\n"
__device__ __forceinline__ uint32_t lookback_phase_warp(unsigned long long *desc, uint64_t t, uint32_t mine, int lane) {
    if (lane == 0) st_relaxed(desc + t, ST_AGG | (mine & 3));
    uint32_t acc = 0;
    int64_t base = (int64_t)t - 1;
    while (true) {
        const int64_t idx = base - lane;
        unsigned long long d = ST_INC;  // virtual tiles before the buffer: inclusive prefix 0
        if (idx >= 0) {
            while (((d = ld_relaxed(desc + idx)) & ST_MASK) == 0) __nanosleep(64);
        }
        const unsigned b = __ballot_sync(0xffffffffu, (d & ST_MASK) == ST_INC);
        const int first = b ? __ffs(b) - 1 : 32;
        acc += __reduce_add_sync(0xffffffffu, lane <= first ? (uint32_t)(d & 3) : 0u);
        if (b) break;
        base -= 32;
    }
    if (lane == 0) st_relaxed(desc + t, ST_INC | ((acc + mine) & 3));
    return acc & 3;
}

// ------------------------------------------------------------------ look-back #2: kept bytes + carried state
// aggregate:  [61] has_start  [60:59] state of the last record  [58:30] head_len  [29:0] rest_kept
// inclusive:  [60:59] state carried out of the tile              [58:0] kept bytes up to and including the tile
// A tile is a transducer on the carried state c: it keeps (c == KEPT ? head_len : 0) + rest bytes and
// carries out (has_start ? last : c).  A run of tiles composes into {P: bytes kept iff c == KEPT, K: bytes
// kept regardless, has, out}; composition is associative.  A warp looks at 32 descriptors at a time (one per
// lane): with ballots every lane finds the state carried into its tile, two warp reductions give the
// window's composite.  The look-back only needs the tiles BEFORE t, so it runs while the CTA's other warps
// are still busy with the records of tile t.
struct Comp {
    uint32_t P, K, has, out;
};
__device__ __forceinline__ Comp comp_identity() { return Comp{0u, 0u, 0u, 0u}; }
__device__ __forceinline__ Comp compose(const Comp A /*earlier*/, const Comp B /*later*/) {
    Comp R;
    if (!A.has) {
        R.P = A.P + B.P;
        R.K = B.K;
        R.has = B.has;
        R.out = B.out;
    } else {
        R.P = A.P;
        R.K = A.K + B.K + (A.out == F_KEPT ? B.P : 0u);
        R.has = 1u;
        R.out = B.has ? B.out : A.out;
    }
    return R;
}

// (kept bytes before tile t, state carried into it) from the descriptors of the tiles before t
#ifdef SGPU_FUSED_LB_NOINLINE
__device__ __noinline__ void lookback_pred_warp(const unsigned long long *desc, uint64_t t, int lane,
#else
__device__ __forceinline__ void lookback_pred_warp(const unsigned long long *desc, uint64_t t, int lane,
#endif
                                                   uint64_t *kept_before, uint32_t *carry) {
    Comp acc_all = comp_identity();  // composite of every window visited so far (nearer windows are later)
    uint64_t inc_total = 0;
    int64_t base = (int64_t)t - 1;  // nearest tile of the window; lane l looks at tile base - l
    const uint64_t virt = ST_INC | ((uint64_t)F_NONE << 59);  // before the buffer: nothing kept, nothing carried
    // LBK windows are fetched per round trip: the nearest inclusive descriptor is typically ~200 tiles back
    // (every resident CTA is between its load and its own look-back), one L2 latency per window adds up
    constexpr int LBK = SGPU_FUSED_LB_K;
    bool done = false;
    while (!done) {
        unsigned long long xs[LBK];
#pragma unroll
        for (int k = 0; k < LBK; k++) {
            const int64_t idx = base - 32 * k - lane;
            xs[k] = idx >= 0 ? ld_relaxed(desc + idx * DSTRIDE) : virt;
        }
#pragma unroll
        for (int k = 0; k < LBK; k++) {
        if (done) break;  // (warp-uniform)
        const int64_t idx = base - 32 * k - lane;
        unsigned long long x = xs[k];
        int L;
        // every descriptor up to the nearest inclusive one must be there
        while (true) {
            const uint32_t st = (uint32_t)(x >> 62);
            const unsigned binc = __ballot_sync(0xffffffffu, st == 2u);
            const unsigned bzero = __ballot_sync(0xffffffffu, st == 0u);
            L = binc ? __ffs(binc) - 1 : 32;
            const unsigned upto = L < 31 ? (2u << L) - 1u : 0xffffffffu;  // lanes <= L
            if ((bzero & upto) == 0) break;
            // a predecessor is still parsing (microseconds away): poll slowly, the issue slots belong to the
            // warps that work
            __nanosleep(SGPU_FUSED_POLL_NS);
            if (st == 0u && lane <= L) x = ld_relaxed(desc + idx * DSTRIDE);
        }
        const bool agg = lane < L, isL = lane == L;
        const uint32_t fl = (uint32_t)(x >> 59) & 3u;
        const bool has = isL || (agg && ((x >> 61) & 1ull));
        const uint32_t hl = agg ? (uint32_t)(x >> 30) & 0x1FFFFFFFu : 0u;
        const uint32_t rs = agg ? (uint32_t)x & 0x3FFFFFFFu : 0u;
        const unsigned has_m = __ballot_sync(0xffffffffu, has);
        const unsigned kept_m = __ballot_sync(0xffffffffu, has && fl == F_KEPT);
        // the state carried into my tile = state of the nearest earlier tile with a record start:
        // the lowest set bit of has_m strictly above my lane
        const unsigned hm = has_m & (0xFFFFFFFEu << lane);
        const bool found = hm != 0u;
        const bool in_kept = found && ((kept_m >> (__ffs(hm) - 1)) & 1u);
        const uint32_t sumK = __reduce_add_sync(0xffffffffu, rs + (in_kept ? hl : 0u));
        const uint32_t sumP = __reduce_add_sync(0xffffffffu, found ? 0u : hl);
        Comp W;
        W.P = sumP;
        W.K = sumK;
        W.has = has_m != 0u;
        W.out = __shfl_sync(0xffffffffu, fl, has_m ? __ffs(has_m) - 1 : 0);
        acc_all = compose(W, acc_all);
        if (L < 32) {
            inc_total = __shfl_sync(0xffffffffu, x, L) & ((1ull << 59) - 1);
            done = true;
        }
        }
        base -= 32 * LBK;
    }
    // acc_all starts with the inclusive descriptor (has == 1, P == 0)
    *kept_before = inc_total + acc_all.K;
    *carry = acc_all.out;
}
__device__ __forceinline__ unsigned long long agg_desc(bool has_start, uint32_t last_flag, uint32_t head_len,
                                                       uint32_t rest) {
    return ST_AGG | (has_start ? (1ull << 61) : 0ull) | ((uint64_t)last_flag << 59) | ((uint64_t)head_len << 30) | rest;
}
__device__ __forceinline__ unsigned long long inc_desc(bool has_start, uint32_t last_flag, uint32_t head_len,
                                                       uint32_t rest, uint64_t kept_before, uint32_t carry) {
    const uint64_t incl = kept_before + (carry == F_KEPT ? head_len : 0u) + rest;
    return ST_INC | ((uint64_t)(has_start ? last_flag : carry) << 59) | incl;
}

// ------------------------------------------------------------------ tile load (one thread)
__device__ __forceinline__ void issue_load(const FusedParams &P, CtaSmem *S, uint64_t t) {
    // bytes [t*TILE - PRE, t*TILE + TILE + HALO) clipped to the buffer, rounded up to 16
    const uint64_t g0 = t * (uint64_t)TILE;
    const uint64_t src0 = t ? g0 - PRE : 0;
    uint64_t end = g0 + TILE + HALO;
    if (end > P.n_in) end = P.n_in;
    const uint32_t bytes = (uint32_t)(((end - src0) + 15) & ~15ull);
    // (the reads of the buffer through the generic proxy are ordered before this point by the CTA barrier
    // the caller has just passed; like the usual consumer-release -> TMA producer hand-over, no proxy fence)
    mbar_expect_tx(&S->full, bytes);
    // several smaller bulk copies: they are fetched concurrently
    uint8_t *dst = S->buf + (t ? 0 : PRE);
    const uint8_t *src = P.in + src0;
    for (uint32_t o = 0; o < bytes; o += LOAD_PIECE) {
        const uint32_t nb = bytes - o < (uint32_t)LOAD_PIECE ? bytes - o : (uint32_t)LOAD_PIECE;
        bulk_g2s(dst + o, src + o, nb, &S->full);
    }
}
__device__ __forceinline__ void prefetch_tile(const FusedParams &P, uint64_t t) {
    if (t >= P.n_tiles) return;
    const uint64_t p0 = t * (uint64_t)TILE;
    uint64_t pe = p0 + TILE;
    if (pe > P.n_in) pe = P.n_in;
    const uint32_t pb = (uint32_t)((pe - p0) & ~15ull);
    if (pb) bulk_prefetch_l2(P.in + p0, pb);
}

// ------------------------------------------------------------------ per-record helpers (P3)
// id token of the record that starts at tile[sp] ('@'): fast path = 16-byte window at the token start ->
// length and inline slot image in registers.  mode 1: (lo, hi) is the image; mode 2: take the general scan.
struct RecPrep {
    uint32_t mode;
    uint64_t lo, hi;
};
__device__ __forceinline__ RecPrep record_prepare(uint32_t tile_s, uint32_t sp, uint32_t avail) {
    RecPrep R;
    R.mode = 2;
    R.lo = R.hi = 0;
    const uint32_t i = sp + 1;
    if (i + 16 > avail) return R;
    const uint32_t sa = tile_s + i;
    const uint32_t wa = sa & ~3u, sh = (sa & 3u) * 8u;
    const uint32_t x0 = lds_u32(wa), x1 = lds_u32(wa + 4), x2 = lds_u32(wa + 8), x3 = lds_u32(wa + 12),
                   x4 = lds_u32(wa + 16);
    const uint32_t w0 = __funnelshift_r(x0, x1, sh), w1 = __funnelshift_r(x1, x2, sh),
                   w2 = __funnelshift_r(x2, x3, sh), w3 = __funnelshift_r(x3, x4, sh);
    const uint32_t stop = gather16(le20_flags(w0), le20_flags(w1), le20_flags(w2), le20_flags(w3));
    const uint32_t len = stop ? (uint32_t)(__ffs(stop) - 1) : 16u;
    // the stop byte must be real whitespace, the token non-empty and short enough to be inline
    const uint32_t cw = len < 4 ? w0 : len < 8 ? w1 : len < 12 ? w2 : w3;
    const uint32_t cb = (cw >> (8 * (len & 3))) & 0xFFu;
    if (!(len >= 1 && len <= IDSET_INLINE_MAX && (cb == 0x20u || (cb - 9u) < 5u))) return R;
    // image = (token << 8 | len) cut to len + 1 bytes
    uint32_t s0 = (w0 << 8) | len, s1 = __funnelshift_l(w0, w1, 8), s2 = __funnelshift_l(w1, w2, 8),
             s3 = __funnelshift_l(w2, w3, 8);
    const uint32_t nb = len + 1;  // 2..16
    const uint32_t full = nb >> 2, part = (nb & 3u) * 8u;
    const uint32_t pm = (1u << part) - 1u;  // part == 0 -> 0
    s0 = full > 0 ? s0 : s0 & pm;
    s1 = full > 1 ? s1 : (full == 1 ? s1 & pm : 0u);
    s2 = full > 2 ? s2 : (full == 2 ? s2 & pm : 0u);
    s3 = full > 3 ? s3 : (full == 3 ? s3 & pm : 0u);
    R.lo = (uint64_t)s0 | ((uint64_t)s1 << 32);
    R.hi = (uint64_t)s2 | ((uint64_t)s3 << 32);
    R.mode = 1;
    return R;
}
// Ids of 16..64 bytes (Illumina / ONT read names) without byte loops: the token's end from 16-byte windows, the hash
// word-wise from shared memory (hash_words == hash_bytes), four independent slot loads per round, and a fingerprint
// hit verified word-wise against the 16-byte aligned arena entry -- only HITS touch the arena.  It runs inside the
// (not inlined) scanning routines below: its registers stay out of the kernel's budget, the inline-id path is the
// tuned one.
// Returns (token length << 1) | member, or LONG_NA: not applicable (leading blank, longer than 64 bytes, a stop byte
// that is not white space, too close to the end of the buffer) -- the scanning routine decides.
constexpr uint32_t LONG_NA = 0xFFFFFFFFu;
__device__ __forceinline__ uint32_t record_probe_long(const IdSetView &set, uint32_t tile_s, uint32_t sp, uint32_t avail) {
    const uint32_t a = sp + 1;
    if (a + 84 > avail) return LONG_NA;
    const uint32_t sa = tile_s + a;
    const uint32_t wa = sa & ~3u, sh = (sa & 3u) * 8u;
    auto word = [&](uint32_t k) { return __funnelshift_r(lds_u32(wa + 4 * k), lds_u32(wa + 4 * k + 4), sh); };
    uint32_t len = 0, cb = 0;
    bool found = false;
#pragma unroll 1
    for (uint32_t w = 0; w < 5 && !found; w++) {
        const uint32_t w0 = word(4 * w), w1 = word(4 * w + 1), w2 = word(4 * w + 2), w3 = word(4 * w + 3);
        const uint32_t stop = gather16(le20_flags(w0), le20_flags(w1), le20_flags(w2), le20_flags(w3));
        if (stop) {
            const uint32_t k = (uint32_t)(__ffs(stop) - 1);
            len = 16 * w + k;
            const uint32_t cw = k < 4 ? w0 : k < 8 ? w1 : k < 12 ? w2 : w3;
            cb = (cw >> (8 * (k & 3))) & 0xFFu;
            found = true;
        }
    }
    if (!found || len <= IDSET_INLINE_MAX || len > 64 || !(cb == 0x20u || (cb - 9u) < 5u)) return LONG_NA;
    if (set.table == nullptr) return len << 1;
    const uint64_t lo = 0x80ull | (hash_words(word, len) & ~0xFFull);
    uint64_t b = home_bucket(mix64(lo), set.n_pages);
    int q = 0;
    while (true) {
        const Slot *bp = set.table + b * IDSET_BUCKET + q;
        Slot s[4];
#pragma unroll
        for (int k = 0; k < 4; k++) s[k] = load_slot(bp + k);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if ((s[k].lo | s[k].hi) == 0) return len << 1;
            if (s[k].lo == lo && (s[k].hi & 0xFFFFFFull) == len && arena_equal_words(set.arena + (s[k].hi >> 24), word, len))
                return (len << 1) | 1u;
        }
        q += 4;
        if (q >= (int)IDSET_BUCKET) {
            q = 0;
            b = next_bucket(b);
        }
    }
}

// general token scan + probe: skip leading blanks, run to the next blank / newline
// LONG: the set holds ids of 16 bytes and more (it has a key arena): the vectorised long-id probe goes first.  A set of
// inline ids only cannot hold a long id, and the kernel variant for it keeps these routines (and the registers the
// calls cost around them) as light as they were.
template <bool LONG>
__device__ __forceinline__ bool record_probe_scan(const IdSetView &set, const uint8_t *tile, uint32_t sp, uint32_t avail,
                                                  uint32_t *why, uint32_t *tok_a, uint32_t *tok_len) {
    if (LONG) {
        const uint32_t lr = record_probe_long(set, smem_u32(tile), sp, avail);
        if (lr != LONG_NA) {
            *tok_a = sp + 1;
            *tok_len = lr >> 1;
            return (lr & 1u) != 0;
        }
    }
    uint32_t a = sp + 1;
    while (a < avail && is_ws_ascii(tile[a]) && tile[a] != '\n') a++;
    uint32_t q = a;
    while (q < avail && !is_ws_ascii(tile[q])) q++;
    if (q >= avail || q == a) {  // token past the halo, or empty id (error 9)
        *why = *why ? *why : 7u;
        return false;
    }
    *tok_a = a;
    *tok_len = q - a;
    return idset_contains(set, tile + a, q - a);
}
template <bool LONG>
__device__ __noinline__ bool record_probe_slow(const IdSetView &set, const uint8_t *tile, uint32_t sp, uint32_t avail,
                                               uint32_t *why) {
    uint32_t ta, tl;
    return record_probe_scan<LONG>(set, tile, sp, avail, why, &ta, &tl);
}
// ids mode: the token's span as well
template <bool LONG>
__device__ __noinline__ bool record_probe_slow_span(const IdSetView &set, const uint8_t *tile, uint32_t sp,
                                                    uint32_t avail, uint32_t *why, uint32_t *tok_a, uint32_t *tok_len) {
    return record_probe_scan<LONG>(set, tile, sp, avail, why, tok_a, tok_len);
}
// the first HALF of the home bucket of an inline key: four independent 16-byte loads of one 128-byte line.  The
// occupied slots of a bucket are a prefix of it, so the second half is only looked at when the first is full of
// other keys (the line is in L1 by then: ld.global.nc allocates)
#ifndef SGPU_FUSED_HALF
#define SGPU_FUSED_HALF 4
#endif
constexpr int HALF = SGPU_FUSED_HALF < (int)IDSET_BUCKET ? SGPU_FUSED_HALF : (int)IDSET_BUCKET;
struct Bucket {
    Slot s[HALF];
};
__device__ __forceinline__ Bucket load_bucket(const IdSetView &set, uint64_t lo, uint64_t hi) {
    const Slot *bp = set.table + home_bucket(inline_hash(lo, hi), set.n_pages) * IDSET_BUCKET;
    Bucket B;
#ifndef SGPU_NO_LD256  // two 256-bit loads (sm_100: LDG.E.256) instead of four 128-bit ones: half the L1 wavefronts per
                       // lookup (measured: 1.827 -> 1.810 ms per 3.3 GB against a 50 M-id set)
    static_assert(HALF == 4, "two slots per 256-bit load");
#pragma unroll
    for (int q = 0; q < HALF; q += 2) {
        unsigned long long a, b, c, d;
        asm volatile("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(bp + q));
        B.s[q].lo = a;
        B.s[q].hi = b;
        B.s[q + 1].lo = c;
        B.s[q + 1].hi = d;
    }
#else
#pragma unroll
    for (int q = 0; q < HALF; q++) B.s[q] = load_slot(bp + q);
#endif
    return B;
}
// exact membership given the first half of the home bucket.  Beyond it the probe sequence is followed four slots at
// a time -- four INDEPENDENT loads per round trip, never a chain of dependent single-slot loads
__device__ __forceinline__ bool probe_bucket(const IdSetView &set, const Bucket &B, uint64_t lo, uint64_t hi) {
    bool hit = false, open = false;
#pragma unroll
    for (int q = 0; q < HALF; q++) {
        hit |= B.s[q].lo == lo && B.s[q].hi == hi;
        open |= (B.s[q].lo | B.s[q].hi) == 0;
    }
    if (hit || open) return hit;
    uint64_t b = home_bucket(inline_hash(lo, hi), set.n_pages);
    int q = HALF;
    while (true) {
        if (q >= (int)IDSET_BUCKET) {
            q = 0;
            b = next_bucket(b);
        }
        const Slot *bp = set.table + b * IDSET_BUCKET + q;
        Slot s[4];
#pragma unroll
        for (int k = 0; k < 4; k++) s[k] = load_slot(bp + k);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            hit |= s[k].lo == lo && s[k].hi == hi;
            open |= (s[k].lo | s[k].hi) == 0;
        }
        if (hit || open) return hit;
        q += 4;
    }
}

// ------------------------------------------------------------------ P3: runs -> copy items (one warp)
// Lanes hold consecutive records: flag, source start sp, end e, kept bytes before the record Kx.  A run is a
// maximal group of consecutive lanes with flag == WANT (its bytes are contiguous in the tile AND in the
// stream); the lane that ends a run cuts it into items of at most PIECE bytes.
template <uint32_t WANT>
__device__ __forceinline__ void emit_runs(CtaSmem *S, uint32_t flag, uint32_t sp, uint32_t e, uint32_t Kx,
                                          uint32_t head_len, int lane) {
    const unsigned km = __ballot_sync(0xffffffffu, flag == WANT);
    if (km == 0) return;  // warp-uniform
    const unsigned below = ~km & ((1u << lane) - 1u);
    const int start_lane = below ? 32 - __clz(below) : 0;
    const uint32_t s_src = __shfl_sync(0xffffffffu, sp, start_lane);
    const uint32_t s_K = __shfl_sync(0xffffffffu, Kx, start_lane);
    const bool mine = (km >> lane) & 1u;
    const bool nxt = lane < 31 ? ((km >> (lane + 1)) & 1u) != 0 : false;
    if (mine && !nxt) {
        const uint32_t run_len = e - s_src;
        const uint32_t rel = WANT == F_KEPT ? s_K : s_src - head_len - s_K;
        const uint32_t np = (run_len + PIECE - 1) / PIECE;
        const uint32_t slot = atomicAdd(&S->n_items, np);
        for (uint32_t q = 0; q < np; q++) {
            const uint32_t o = q * PIECE;
            const uint32_t l = run_len - o < (uint32_t)PIECE ? run_len - o : (uint32_t)PIECE;
            if (slot + q < (uint32_t)IMAX) {
                Item it;
                it.src = (uint16_t)(s_src + o);
                it.len = (uint16_t)l;
                it.rel = (WANT == F_KEPT ? TAG_KEPT : TAG_OTHER) | (rel + o);
                S->items[slot + q] = it;
            }
        }
    }
}

// ------------------------------------------------------------------ P4: one copy item (one warp)
// 16-byte chunks of the destination, each built from two aligned 16-byte shared loads; WS = word part of
// the source misalignment (uniform over the item), bsh = byte part * 8
template <int WS>
__device__ __forceinline__ void copy_body(uint32_t sa0, uint32_t bsh, uint8_t *d0, uint32_t nfull, int lane) {
    const uint32_t al = sa0 & ~15u;
    for (uint32_t i = lane; i < nfull; i += 32) {
        const uint4 A = lds_v4(al + (i << 4)), B = lds_v4(al + (i << 4) + 16);
        const uint32_t x[8] = {A.x, A.y, A.z, A.w, B.x, B.y, B.z, B.w};
        uint4 o;
        o.x = __funnelshift_r(x[WS], x[WS + 1], bsh);
        o.y = __funnelshift_r(x[WS + 1], x[WS + 2], bsh);
        o.z = __funnelshift_r(x[WS + 2], x[WS + 3], bsh);
        o.w = __funnelshift_r(x[WS + 3], x[WS + 4], bsh);
        st_global_v4(d0 + ((size_t)i << 4), o);
    }
}
__device__ __forceinline__ void copy_piece(uint32_t src_s, uint32_t len, uint8_t *dst, int lane) {
    const uint32_t a = (uint32_t)(uintptr_t)dst & 15u;
    uint32_t hn = (16u - a) & 15u;  // bytes before the first aligned chunk
    if (hn > len) hn = len;
    const uint32_t body = len - hn;
    const uint32_t nfull = body >> 4, tn = body & 15u;
    const uint32_t sa0 = src_s + hn;
    const uint32_t bsh = (sa0 & 3u) * 8u;
    switch ((sa0 >> 2) & 3u) {  // warp-uniform
        case 0: copy_body<0>(sa0, bsh, dst + hn, nfull, lane); break;
        case 1: copy_body<1>(sa0, bsh, dst + hn, nfull, lane); break;
        case 2: copy_body<2>(sa0, bsh, dst + hn, nfull, lane); break;
        default: copy_body<3>(sa0, bsh, dst + hn, nfull, lane); break;
    }
    // edge bytes: lanes 0..14 the head, lanes 16..30 the tail
    if ((uint32_t)lane < hn) {
        st_global_u8(dst + lane, lds_u8(src_s + lane));
    } else if (lane >= 16 && (uint32_t)(lane - 16) < tn) {
        const uint32_t off = hn + (nfull << 4) + (uint32_t)(lane - 16);
        st_global_u8(dst + off, lds_u8(src_s + off));
    }
}

// ------------------------------------------------------------------ phase timing (diagnostics, -DSGPU_FUSED_TIMING)
#ifdef SGPU_FUSED_TIMING
__device__ unsigned long long g_phase_cycles[16];
__device__ unsigned long long *g_trace;  // per tile: ticket, loaded, agg, inc, done (globaltimer ns), smid
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long v;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
    return v;
}
__device__ __forceinline__ uint32_t smid() {
    uint32_t v;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(v));
    return v;
}
#define TRACE(t, slot)                                                  \
    do {                                                                \
        if (g_trace) g_trace[(t) * 8 + (slot)] = gtime();               \
    } while (0)
#else
#define TRACE(t, slot) \
    do {               \
    } while (0)
#endif
#ifdef SGPU_FUSED_TIMING
#define PHASE_MARK(i)                                  \
    do {                                               \
        if (tid == 0) {                                \
            const long long now_ = clock64();          \
            ph_acc[i] += (unsigned long long)(now_ - ph_last); \
            ph_last = now_;                            \
        }                                              \
    } while (0)
#else
#define PHASE_MARK(i) \
    do {              \
    } while (0)
#endif

// ------------------------------------------------------------------ the kernel
// named barriers: 0 = the whole CTA; 1 = the records' scan (B4); 2 = totals handed to the look-back warp
__device__ __forceinline__ void bar_sync(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(NT) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(NT) : "memory"); }

// CR / "+\n" checks of one newline by its role (the newlines of whole records are checked by the record's thread)
// (a sequence line whose "+\n" lies beyond the last byte of a buffer that does not end the file -- p + 2 >= avail only
// happens at the end of the buffer -- belongs to a record that starts in the halo, the next shard's)
// A buffer that ends within two bytes of a sequence line's newline used to send the whole shard to the general path
// (one chunk in 165 of a 2x150 file): only the file's last buffer (is_last) has to hold the separator line.
__device__ __forceinline__ uint32_t check_newline(const FusedParams &P, const uint8_t *tile, uint32_t p, uint32_t role,
                                                  uint32_t avail) {
    uint32_t fb = 0;
    if (tile[(int)p - 1] == '\r') fb = 3;  // CRLF: not canonical
    if (role == 1) {                       // end of the sequence line: "+\n" must follow
        if (p + 2 >= avail) {
            if (P.is_last) fb = 4;
        } else if (tile[p + 1] != '+' || tile[p + 2] != '\n') {
            fb = 4;
        }
    }
    return fb;
}

template <bool IDS, bool LONG>
__global__ void __launch_bounds__(NTHREADS, CTAS_PER_SM) fastq_fused_kernel(FusedParams P) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    CtaSmem *S = reinterpret_cast<CtaSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint8_t *buf = S->buf;
    const uint8_t *tile = buf + PRE;  // tile[-16 .. avail)
    const uint32_t tile_s = smem_u32(tile);
    if (tid == 0) {
        mbar_init(&S->full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const unsigned long long t0 = atomicAdd(&P.res->ticket, 1ull);
        S->first_tile = t0;
        if (t0 < P.n_tiles) {
            TRACE(t0, 0);
            issue_load(P, S, t0);
        }
    }
    __syncthreads();
    uint64_t t = S->first_tile;
    unsigned long long my_reads_in = 0, my_reads_out = 0;  // thread 0 only
#ifdef SGPU_FUSED_TIMING
    unsigned long long ph_acc[12] = {0};
    long long ph_last = clock64();
#endif
    for (uint32_t it = 0; t < P.n_tiles; it++) {
        // the tile some CTA will take one generation from now: pull it into L2
        if (tid == 0 && P.pf_dist) prefetch_tile(P, t + P.pf_dist);
        if (lane == 0) {
            while (!mbar_try_wait(&S->full, it & 1)) {
            }
        }
        __syncwarp();
        PHASE_MARK(0);  // load wait
        if (tid == 0) {
            TRACE(t, 1);
#ifdef SGPU_FUSED_TIMING
            if (g_trace) g_trace[t * 8 + 5] = smid();
#endif
        }
        const uint64_t g0 = t * (uint64_t)TILE;
        const uint32_t tile_len = (uint32_t)((P.n_in - g0) < (uint64_t)TILE ? (P.n_in - g0) : (uint64_t)TILE);
        const uint32_t avail =
            (uint32_t)((P.n_in - g0) < (uint64_t)(TILE + HALO) ? (P.n_in - g0) : (uint64_t)(TILE + HALO));
        const uint32_t lead_t = t == 0 ? P.lead : 0u;
        uint32_t fb = 0;  // this thread's fallback reason (0 = none)
        if (t == 0 || tile_len < (uint32_t)TILE) {  // (CTA-uniform) first / last tile of the buffer
            // every thread observes the completed load, then the edges are patched
            while (!mbar_try_wait(&S->full, it & 1)) {
            }
            if (t == 0 && tid < PRE) buf[tid] = '\n';  // no predecessor: the pre-halo reads as a newline
            // bytes past the end of the buffer are stale: zero them (never a newline, ASCII)
            for (uint32_t o = tile_len + tid; o < (uint32_t)TILE; o += NT) buf[PRE + o] = 0;
            __syncthreads();
        }

        // ---- P1: newline masks and counts.  Warp w owns chunks [w*FC*32, (w+1)*FC*32); lane l takes
        //      chunk k*32 + l of them in round k (conflict-free 16-byte shared loads)
        uint32_t m[FC];
        uint32_t hi_or = 0;
        const uint32_t cbase = (uint32_t)warp * (FC * 32) + (uint32_t)lane;
#pragma unroll
        for (int k = 0; k < FC; k++) {
            const uint4 v = lds_v4(tile_s + (cbase + k * 32) * 16);
            m[k] = nl_mask16_v2(v);
            hi_or |= (v.x | v.y | v.z | v.w);
        }
        if (lead_t && tid == 0) m[0] &= ~((1u << lead_t) - 1u);  // the previous shard's bytes
        if (hi_or & 0x80808080u) fb = 1;                         // reason 1: non-ASCII byte, Unicode rules needed
        // inclusive warp scan of the per-round counts: three 10-bit fields per word (a round has <= 512 newlines)
        constexpr int PW = (FC + 2) / 3;
        uint32_t pk[PW], inc[PW];
        uint32_t many = 0;  // a chunk with more than two newlines: lines shorter than the fast path handles
#pragma unroll
        for (int q = 0; q < PW; q++) pk[q] = 0;
#pragma unroll
        for (int k = 0; k < FC; k++) {
            const uint32_t c = (uint32_t)__popc(m[k]);
            many |= (c + 1u) >> 2;  // != 0 iff c >= 3
            pk[k / 3] |= c << (10 * (k % 3));
        }
#pragma unroll
        for (int q = 0; q < PW; q++) inc[q] = pk[q];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
#pragma unroll
            for (int q = 0; q < PW; q++) {
                const uint32_t x = __shfl_up_sync(0xffffffffu, inc[q], d);
                if (lane >= d) inc[q] += x;
            }
        }
        uint32_t row_base[FC];
        uint32_t wtot = 0;
#pragma unroll
        for (int q = 0; q < PW; q++) {
            const uint32_t rt = __shfl_sync(0xffffffffu, inc[q], 31);
            const uint32_t ex = inc[q] - pk[q];  // exclusive within the round
#pragma unroll
            for (int k = 3 * q; k < 3 * q + 3 && k < FC; k++) {
                row_base[k] = wtot + ((ex >> (10 * (k % 3))) & 1023u);
                wtot += (rt >> (10 * (k % 3))) & 1023u;
            }
        }
        const bool many_w = __any_sync(0xffffffffu, many != 0u);
        if (lane == 0) S->warp_tot[warp] = wtot | (many_w ? 0x80000000u : 0u);
        if (tid == 0) {
            S->n_items = 0;
            S->none_pos = 0xFFFFFFFFu;
            S->none_cnt = 0;
        }
        PHASE_MARK(1);    // P1 own work
        __syncthreads();  // B1
        PHASE_MARK(2);    // B1 wait
        // newlines before the warp's region / in the tile: lane w holds warp w's count
        uint32_t n_nl, wbase;
        bool dense;
        {
            const uint32_t x = lane < NW ? S->warp_tot[lane] : 0u;
            const uint32_t cnt = x & 0x7FFFFFFFu;
            uint32_t ic = cnt;
#pragma unroll
            for (int d = 1; d < NW; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, ic, d);
                if (lane >= d) ic += y;
            }
            n_nl = __shfl_sync(0xffffffffu, ic, NW - 1);
            wbase = __shfl_sync(0xffffffffu, ic - cnt, warp);
            dense = __any_sync(0xffffffffu, (x >> 31) != 0u) || n_nl > (uint32_t)LMAX;
        }
        // ---- the newline positions, in order (at most two per 16-byte chunk here: "\n+\n")
        if (!dense) {
#pragma unroll
            for (int k = 0; k < FC; k++) {
                uint32_t mm = m[k];
                if (mm) {
                    const uint32_t r = wbase + row_base[k];
                    const uint32_t pos = (cbase + k * 32) * 16;
                    S->nlp[r] = (uint16_t)(pos + (uint32_t)(__ffs(mm) - 1));
                    mm &= mm - 1;
                    if (mm) S->nlp[r + 1] = (uint16_t)(pos + (uint32_t)(__ffs(mm) - 1));
                }
            }
        } else {
            fb = 2;
        }
        __syncthreads();  // B2
        PHASE_MARK(3);    // scatter + B2
        // ---- line phase: the first newline followed by "+\n" ends a sequence line (role 1).  Every warp
        //      evaluates the same 32 candidates, so the outcome is CTA-uniform without a barrier.
        uint32_t c0 = 0;
        if (t == 0) {
            if (tid == 0) st_relaxed(P.desc1 + t, ST_INC | (n_nl & 3));
        } else {
            bool hit = false;
            if (!dense && (uint32_t)lane < n_nl) {
                const uint32_t p = S->nlp[lane];
                hit = p + 2 < avail && tile[p + 1] == '+' && tile[p + 2] == '\n';
            }
            const unsigned b = __ballot_sync(0xffffffffu, hit);
            if (b) {
                c0 = (1u - (uint32_t)(__ffs(b) - 1)) & 3u;  // role(first) = (c0 + first) & 3 == 1
                if (tid == 0) st_relaxed(P.desc1 + t, ST_INC | ((c0 + n_nl) & 3));
            } else {
                if (warp == 0) {
                    c0 = lookback_phase_warp(P.desc1, t, n_nl, lane);
                    if (lane == 0) S->c0 = c0;
                }
                __syncthreads();
                c0 = S->c0;
            }
        }
        // the first byte of the tile starts a record iff 4k newlines precede it and the previous byte is one;
        // tile 0 starts with a record by construction (at `lead`)
        const bool pos0_start = t == 0 || ((c0 == 0) && tile[-1] == '\n');
        const uint32_t r3 = (3u - c0) & 3u;  // index of the first newline that ends a record
        // number of record starts inside the tile
        const uint32_t n_term = (c0 + n_nl) >> 2;
        uint32_t n_starts = n_term + (pos0_start ? 1u : 0u);
        if (n_term > 0 && !dense) {
            // the last terminating newline may sit on the tile's final byte: its record belongs to the next tile
            if ((uint32_t)S->nlp[r3 + 4u * (n_term - 1)] + 1u >= tile_len) n_starts--;
        }
        if (n_starts > (uint32_t)RMAX) fb = 5;
        if (dense || n_starts > (uint32_t)RMAX) n_starts = 0;  // (a fallback reason is raised)
        // the carried-in record's bytes
        const uint32_t head_len =
            n_starts ? (pos0_start ? lead_t : (uint32_t)S->nlp[r3] + 1u) : tile_len;
        // the look-back only needs the tiles before this one: when the last warp has no record to look after,
        // it runs the look-back while the others work on the records (CTA-uniform)
        const bool early = !IDS && n_starts <= (uint32_t)(NT - 32);

        uint32_t rest_total = 0, kept_recs = 0;
        if (early && warp == NW - 1) {
            if (lane == 0) S->scan_tot[warp] = 0;
            bar_arrive(1);  // B4: nothing to contribute
            // the carried-in head as copy items (its fate is known after the look-back); the `lead` bytes of
            // tile 0 belong to the previous shard
            const uint32_t nph = t == 0 ? 0u : (head_len + PIECE - 1) / PIECE;
            if (nph) {
                uint32_t slot = 0;
                if (lane == 0) slot = atomicAdd(&S->n_items, nph);
                slot = __shfl_sync(0xffffffffu, slot, 0);
                if ((uint32_t)lane < nph && slot + lane < (uint32_t)IMAX) {
                    const uint32_t o = (uint32_t)lane * PIECE;
                    Item itm;
                    itm.src = (uint16_t)o;
                    itm.len = (uint16_t)(head_len - o < (uint32_t)PIECE ? head_len - o : (uint32_t)PIECE);
                    itm.rel = TAG_HEAD | o;
                    S->items[slot + lane] = itm;
                }
            }
            uint64_t kept_before;
            uint32_t carry;
#ifdef SGPU_ABL_NOLB  // ablation (timing only, output is garbage): no in-order commit
            kept_before = g0 / 2;
            carry = F_OTHER;
#else
            lookback_pred_warp(P.desc2, t, lane, &kept_before, &carry);
#endif
            bar_sync(2);  // the workers' totals are in shared memory (and the aggregate is published)
            if (lane == 0) {
                TRACE(t, 3);
                st_relaxed(P.desc2 + t * DSTRIDE,
                           inc_desc(n_starts > 0, S->last_flag, head_len, S->rest_total, kept_before, carry));
                S->kept_before = kept_before;
                S->carry = carry;
            }
        } else {
            // ---- P3: one thread per record start: checks of the record's lines, '@', id token -> exact probe,
            //      kept bytes scanned per warp, runs cut into copy items.  NT records per round (almost
            //      always one round)
            const uint32_t n_rounds = n_starts > (uint32_t)NT ? (n_starts + NT - 1) / NT : 1u;
            for (uint32_t round = 0; round < n_rounds; round++) {
                const uint32_t jb = round * NT;
                const uint32_t j = jb + (uint32_t)tid;
                const bool warp_active = jb + (uint32_t)warp * 32u < n_starts;
                uint32_t flag = F_INVALID, sp = 0, e = 0, v = 0, inc = 0;
                uint32_t tok_a = 0, tok_len = 0;  // ids mode: the id token (tile offset, bytes)
                bool pick = false;
                if (warp_active) {
                    if (j < n_starts) {
                        // index of the newline before the record (-1: the record starts the tile)
                        const int s_idx = pos0_start ? 4 * (int)j - 1 : (int)r3 + 4 * (int)j;
                        sp = s_idx >= 0 ? (uint32_t)S->nlp[s_idx] + 1u : lead_t;
                        const bool whole = s_idx + 4 < (int)n_nl;  // its four newlines are inside the tile
                        uint32_t why = tile[sp] == '@' ? 0u : 6u;  // 6 '@', 7 id token, 8 seq/qual lengths
                        e = tile_len;
                        if (whole) {
                            const uint32_t p1 = S->nlp[s_idx + 1], p2 = S->nlp[s_idx + 2], p3 = S->nlp[s_idx + 3],
                                           p4 = S->nlp[s_idx + 4];
                            if (j + 1 < n_starts) e = p4 + 1;
                            if (tile[p1 - 1] == '\r' || tile[p2 - 1] == '\r' || tile[p4 - 1] == '\r') fb = 3;
                            if (p3 != p2 + 2 || tile[p2 + 1] != '+') fb = 4;
                            if (p2 - p1 != p4 - p3) why = why ? why : 8u;
                        }
                        const bool owned = P.is_last || (g0 + sp <= P.own_len);
                        if (!owned) {
                            flag = F_NONE;
                            atomicMin(&S->none_pos, sp);
                            atomicAdd(&S->none_cnt, 1u);
                        } else {
                            const RecPrep R = record_prepare(tile_s, sp, avail);
                            const bool inl = R.mode == 1 && !why && P.set.table != nullptr;
                            Bucket first;
#pragma unroll
                            for (int q = 0; q < HALF; q++) first.s[q].lo = first.s[q].hi = 0;
#ifndef SGPU_ABL_NOPROBE
                            if (inl) first = load_bucket(P.set, R.lo, R.hi);
#endif
                            bool hit = false;
                            if (!why) {
#ifdef SGPU_ABL_NOPROBE  // ablation (timing only): no memory access for the lookup
                                if (R.mode == 1) hit = __popcll(R.lo ^ R.hi) & 1;
#else
                                if (R.mode == 1) hit = inl && probe_bucket(P.set, first, R.lo, R.hi);
#endif
                                else if (IDS) hit = record_probe_slow_span<LONG>(P.set, tile, sp, avail, &why, &tok_a, &tok_len);
                                else hit = record_probe_slow<LONG>(P.set, tile, sp, avail, &why);
                                if (IDS && R.mode == 1) {
                                    tok_a = sp + 1;
                                    tok_len = (uint32_t)(R.lo & 0xFFu);
                                }
                            }
                            flag = (P.reverse ? hit : !hit) ? F_KEPT : F_OTHER;
                            if (why) {
                                fb = why;
                                flag = F_OTHER;
                            }
                            if (IDS) {
                                pick = !why && !hit;
                                flag = F_OTHER;
                            }
                        }
                        if (j == n_starts - 1) S->last_flag = flag;
                    }
                    v = flag == F_KEPT ? ((e - sp) | (1u << 16)) : 0u;  // kept bytes | kept records << 16
                    if (IDS) v = pick ? 1u : 0u;                  // ids mode: picked records
                    inc = v;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        const uint32_t x = __shfl_up_sync(0xffffffffu, inc, d);
                        if (lane >= d) inc += x;
                    }
                }
                if (lane == 31) S->scan_tot[warp] = inc;
                PHASE_MARK(5);  // P3 own work (probe included)
                bar_sync(1);    // B4
                PHASE_MARK(6);  // B4 wait
                uint32_t base = 0, tot = 0;
                {
                    const uint32_t x = lane < NW ? S->scan_tot[lane] : 0u;
                    uint32_t ic = x;
#pragma unroll
                    for (int d = 1; d < NW; d <<= 1) {
                        const uint32_t y = __shfl_up_sync(0xffffffffu, ic, d);
                        if (lane >= d) ic += y;
                    }
                    tot = __shfl_sync(0xffffffffu, ic, NW - 1);
                    base = __shfl_sync(0xffffffffu, ic - x, warp);
                }
                const uint32_t Kx = rest_total + ((base + inc - v) & 0xFFFFu);  // kept bytes of the records before
                if (IDS) {
                    // one reservation per tile in the span list, then every picked record writes its token
                    if (tid == 0) S->span_base = atomicAdd(&P.res->n_spans, (unsigned long long)(tot & 0xFFFFu));
                    __syncthreads();
                    if (pick) {
                        const uint64_t idx = S->span_base + ((base + inc - v) & 0xFFFFu);
                        if (idx < P.span_cap) {
                            P.span_off[idx] = g0 + tok_a;
                            P.span_len[idx] = tok_len;
                        } else {
                            fb = 13;  // more records than the list was sized for: the general path
                        }
                    }
                    tot = 0;
                }
                rest_total += tot & 0xFFFFu;
                kept_recs += tot >> 16;
                if (round + 1 == n_rounds && tid == 0) {
                    // the aggregate: every later tile may be waiting for it
                    const uint32_t last_flag = n_starts ? S->last_flag : F_OTHER;
                    TRACE(t, 2);
                    st_relaxed(P.desc2 + t * DSTRIDE, agg_desc(n_starts > 0, last_flag, head_len, rest_total));
                    S->rest_total = rest_total;
                    if (!n_starts) S->last_flag = F_OTHER;
                }
                if (round + 1 == n_rounds && early) bar_arrive(2);  // totals handed to the look-back warp
                if (warp_active) {
                    emit_runs<F_KEPT>(S, flag, sp, e, Kx, head_len, lane);
                    if (P.out_o) emit_runs<F_OTHER>(S, flag, sp, e, Kx, head_len, lane);
                }
                if (round + 1 < n_rounds) __syncthreads();  // scan_tot is reused
            }
            if (tid == 0) {
                my_reads_in += n_starts - S->none_cnt;
                my_reads_out += kept_recs;
                if (S->none_pos != 0xFFFFFFFFu) atomicMin(&P.res->owned_end, (unsigned long long)(g0 + S->none_pos));
            }
            if (tid == NT - 64) {
                // per-tile metadata for the verification kernel, and the checks of the newlines that do not
                // belong to a whole record of this tile.  Signed newline-position sums: -p1 +p2 +p3 -p4 per
                // record must vanish
                long long head = 0, total = 0;
                if (!dense) {
                    if (n_term == 0) {
                        for (uint32_t r = 0; r < n_nl; r++) {
                            const uint32_t role = (c0 + r) & 3, p = S->nlp[r];
                            const long long pp = (long long)(g0 + p);
                            total += (role == 0 || role == 3) ? -pp : pp;
                            const uint32_t f = check_newline(P, tile, p, role, avail);
                            if (f) fb = f;
                        }
                    } else {
                        for (uint32_t r = 0; r <= r3; r++) {
                            const uint32_t role = (c0 + r) & 3, p = S->nlp[r];
                            const long long pp = (long long)(g0 + p);
                            head += (role == 0 || role == 3) ? -pp : pp;
                            const uint32_t f = check_newline(P, tile, p, role, avail);
                            if (f) fb = f;
                        }
                        total = head;
                        for (uint32_t r = r3 + 4u * (n_term - 1) + 1u; r < n_nl; r++) {
                            const uint32_t role = (c0 + r) & 3, p = S->nlp[r];
                            const long long pp = (long long)(g0 + p);
                            total += (role == 0 || role == 3) ? -pp : pp;
                            const uint32_t f = check_newline(P, tile, p, role, avail);
                            if (f) fb = f;
                        }
                    }
                }
                P.sum_total[t] = total;
                P.sum_head[t] = head;
                P.has_term[t] = n_term > 0 ? 1 : 0;
                P.nl_count[t] = n_nl;
                P.phase_used[t] = (uint8_t)c0;
                // end-of-file condition of canonical input (the line count is checked by the follow-up kernel)
                if (P.is_last && t + 1 == P.n_tiles && tile[tile_len - 1] != '\n') set_fallback(P.res, 9);
            }
            if (!early && !IDS && warp == NW - 1) {
                // (rare) the last warp had records of its own: head items and look-back only now
                const uint32_t nph = t == 0 ? 0u : (head_len + PIECE - 1) / PIECE;
                if (nph) {
                    uint32_t slot = 0;
                    if (lane == 0) slot = atomicAdd(&S->n_items, nph);
                    slot = __shfl_sync(0xffffffffu, slot, 0);
                    if ((uint32_t)lane < nph && slot + lane < (uint32_t)IMAX) {
                        const uint32_t o = (uint32_t)lane * PIECE;
                        Item itm;
                        itm.src = (uint16_t)o;
                        itm.len = (uint16_t)(head_len - o < (uint32_t)PIECE ? head_len - o : (uint32_t)PIECE);
                        itm.rel = TAG_HEAD | o;
                        S->items[slot + lane] = itm;
                    }
                }
                uint64_t kept_before;
                uint32_t carry;
#ifdef SGPU_ABL_NOLB
                kept_before = g0 / 2;
                carry = F_OTHER;
#else
                lookback_pred_warp(P.desc2, t, lane, &kept_before, &carry);
#endif
                if (lane == 0) {
                    TRACE(t, 3);
                    st_relaxed(P.desc2 + t * DSTRIDE, inc_desc(n_starts > 0, n_starts ? S->last_flag : F_OTHER, head_len,
                                                     rest_total, kept_before, carry));
                    S->kept_before = kept_before;
                    S->carry = carry;
                }
            }
        }
        if (fb) set_fallback(P.res, (int)fb);
        PHASE_MARK(7);    // emit
        __syncthreads();  // B5: kept_before / carry / every copy item are there
        PHASE_MARK(8);    // B5 wait (look-back)

        // ---- P4: a warp per copy item.  The next ticket is taken only now: a ticket held while this tile
        //      still waits on its look-back would stall every later tile behind this CTA
        unsigned long long nt = 0;
        if (tid == 0) nt = atomicAdd(&P.res->ticket, 1ull);
        {
            const uint64_t kept_before = S->kept_before;
            const uint32_t carry = S->carry;
            uint32_t n_items = S->n_items;
            if (n_items > (uint32_t)IMAX) n_items = IMAX;
            const uint32_t head_kept = carry == F_KEPT ? head_len : 0u;
            uint8_t *const base_w = P.out_w + kept_before;  // the head goes here when it is kept
            // bytes of the other stream before this tile = owned bytes before it - kept bytes before it
            uint8_t *const base_o = P.out_o ? P.out_o + (t == 0 ? 0 : (g0 - P.lead) - kept_before) : nullptr;
            const uint32_t head_other = carry == F_OTHER ? head_len : 0u;
            // the outputs are sized by the caller (a depleted file is smaller than its input): room left in each
            // stream from this tile's base, so that no item is ever written past a buffer
            const uint64_t off_w = kept_before, off_o = t == 0 ? 0 : (g0 - P.lead) - kept_before;
            const uint32_t room_w = P.cap_w > off_w ? (uint32_t)(P.cap_w - off_w < 0xFFFFFFFFull ? P.cap_w - off_w : 0xFFFFFFFFull) : 0u;
            const uint32_t room_o = P.cap_o > off_o ? (uint32_t)(P.cap_o - off_o < 0xFFFFFFFFull ? P.cap_o - off_o : 0xFFFFFFFFull) : 0u;
            for (uint32_t i = warp; i < n_items; i += NW) {
                const Item itm = S->items[i];
                const uint32_t tag = itm.rel & (3u << 30), rel = itm.rel & 0x3FFFFFFFu;
                uint32_t off;
                bool to_w = true;
                if (tag == TAG_KEPT) {
                    off = head_kept + rel;
                } else if (tag == TAG_OTHER) {
                    off = head_other + rel;
                    to_w = false;
                } else {
                    off = rel;
                    if (carry == F_OTHER && base_o) to_w = false;
                    else if (carry != F_KEPT) continue;
                }
                if (off + itm.len > (to_w ? room_w : room_o)) {
                    if (lane == 0) P.res->overflow = 1;
                    continue;
                }
                uint8_t *const dst = (to_w ? base_w : base_o) + off;
#ifndef SGPU_ABL_NOCOPY  // ablation (timing only): nothing is written
                copy_piece(tile_s + itm.src, itm.len, dst, lane);
#endif
            }
            if (t + 1 == P.n_tiles && tid == 0) P.res->kept_total = kept_before + head_kept + S->rest_total;
        }
        PHASE_MARK(9);  // copy own work
        if (tid == 0) {
            TRACE(t, 4);
            if (nt < P.n_tiles) TRACE(nt, 0);
        }
        if (tid == 0) S->next_tile = nt;
        __syncthreads();  // B6: every read of the tile buffer and the lists is done
        PHASE_MARK(10);   // ticket + B6 wait
        const uint64_t next_t = S->next_tile;
        if (tid == 0 && next_t < P.n_tiles) issue_load(P, S, next_t);
        t = next_t;
    }
#ifdef SGPU_FUSED_TIMING
    if (tid == 0)
        for (int i = 0; i < 12; i++) atomicAdd(&g_phase_cycles[i], ph_acc[i]);
#endif
    if (tid == 0) {
        if (my_reads_out) atomicAdd(&P.res->reads_out, my_reads_out);
        if (my_reads_in) atomicAdd(&P.res->reads_in, my_reads_in);
    }
}

// exact verification of what the tiles assumed: (1) the speculated line phase of every tile against the
// true prefix of newline counts, (2) the signed newline-position sums vanish at every record end
// (seq and qual lengths agree for records that straddle tiles), (3) the file's line count is a multiple of 4
__global__ void fused_verify_kernel(const uint64_t *sum_prefix, const long long *sum_head, const uint8_t *has_term,
                                    const uint64_t *nl_prefix, const uint32_t *nl_count, const uint8_t *phase_used,
                                    uint64_t n_tiles, int is_last, FusedResult *res) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    if ((uint32_t)(nl_prefix[t] & 3) != (uint32_t)phase_used[t]) set_fallback(res, 11);
    if (has_term[t] && (long long)sum_prefix[t] + sum_head[t] != 0) set_fallback(res, 10);
    if (t + 1 == n_tiles && is_last) {
        const uint64_t lines = nl_prefix[t] + nl_count[t];
        if (lines & 3) set_fallback(res, 9);
    }
}

// '\n' bytes in [lead, own_len) of the range the fused kernel ran over, from its per-tile counts (whole tiles below
// own_len: the exclusive prefix) plus the bytes of the one tile own_len cuts.  One CTA.
__global__ void fused_own_newlines_kernel(const uint8_t *in, uint32_t lead, uint64_t own_len, const uint64_t *nl_prefix,
                                          const uint32_t *nl_count, uint64_t n_tiles, FusedResult *res) {
    const uint64_t tb = own_len / (uint64_t)TILE;
    uint64_t a = own_len;
    if (tb < n_tiles) a = tb * (uint64_t)TILE;  // (16-byte aligned)
    uint32_t cnt = 0;
    for (uint64_t pos = a + (uint64_t)threadIdx.x * 16; pos < own_len; pos += (uint64_t)blockDim.x * 16) {
        uint32_t m = nl_mask16_v2(ld_nc_u4(in + pos));  // (the buffer is readable up to a multiple of 16 past n_in)
        if (own_len - pos < 16) m &= (1u << (own_len - pos)) - 1u;
        if (pos < lead) m &= ~((1u << (lead - pos)) - 1u);
        cnt += __popc(m);
    }
    __shared__ unsigned int s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    if (cnt) atomicAdd(&s_cnt, cnt);
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint64_t whole = tb < n_tiles ? nl_prefix[tb] : nl_prefix[n_tiles - 1] + nl_count[n_tiles - 1];
        res->own_newlines = whole + s_cnt;
    }
}

// Runs the fused kernel over d_in[0..n_in).  The first owned record starts at `lead` (< 16); records that
// start after own_len (when !is_last) are left to the next shard.  *used = 0 when the input turned out
// not to be canonical (the caller then takes the general path).
// ids mode (IdsOut != nullptr): nothing is written; the id tokens of the records absent from `set` are listed
// want_own_nl: also count the '\n' bytes of [lead, own_len) into counts->own_newlines (speculative shards)
static sgpu_status clean_fused_range(sgpu_ctx *c, const sgpu_idset *set, const uint8_t *d_in, size_t n_in, uint32_t lead,
                                     size_t own_len, int is_last, int reverse, const Outs &out, sgpu_counts *counts,
                                     int *used, IdsOut *ids, bool want_own_nl) {
    *used = 0;
    if (n_in == 0 || lead >= 16) return SGPU_OK;
    // (the outputs may be smaller than the input: the kernel never writes past cap_w / cap_o and reports it)
    cudaStream_t st = c->stream;
    static bool attr_done[64] = {false};
    const size_t smem = sizeof(CtaSmem);
    if (!attr_done[c->device & 63]) {
        const void *variants[4] = {(const void *)fastq_fused_kernel<false, false>, (const void *)fastq_fused_kernel<false, true>,
                                   (const void *)fastq_fused_kernel<true, false>, (const void *)fastq_fused_kernel<true, true>};
        for (const void *k : variants) {
            SGPU_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            SGPU_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        }
        attr_done[c->device & 63] = true;
    }
    uint64_t n_tiles = ceil_div(n_in, (size_t)TILE);
    DevBuf<unsigned long long> desc;
    DevBuf<long long> sums;
    DevBuf<uint64_t> prefix;
    DevBuf<uint32_t> nl_count;
    DevBuf<uint8_t> bytes;
    DevBuf<FusedResult> res;
    SGPU_TRY(desc.alloc((1 + DSTRIDE) * n_tiles, st));
    SGPU_TRY(sums.alloc(2 * n_tiles, st));
    SGPU_TRY(prefix.alloc(2 * n_tiles, st));
    SGPU_TRY(nl_count.alloc(n_tiles, st));
    SGPU_TRY(bytes.alloc(2 * n_tiles, st));
    SGPU_TRY(res.alloc(1, st));
    SGPU_CUDA(cudaMemsetAsync(desc.p, 0, (1 + DSTRIDE) * n_tiles * 8, st));
    FusedResult init;
    memset(&init, 0, sizeof(init));
    init.owned_end = ~0ull;
    static_assert(sizeof(FusedResult) % 8 == 0 && sizeof(FusedResult) <= 32 * 8, "pinned staging too small");
    SGPU_TRY(write_u64s(c, res.p, (const uint64_t *)&init, sizeof(FusedResult) / 8));
    FusedParams P;
    P.in = d_in;
    P.n_in = n_in;
    P.n_tiles = n_tiles;
    P.own_len = own_len;
    P.lead = lead;
    P.is_last = is_last;
    P.out_w = out.w;
    P.out_o = out.o;
    P.cap_w = out.cap_w;
    P.cap_o = out.o ? out.cap_o : 0;
    P.reverse = reverse;
    P.set = view_of(set);
    P.desc1 = desc.p;
    P.desc2 = desc.p + n_tiles;
    P.sum_total = sums.p;
    P.sum_head = sums.p + n_tiles;
    P.nl_count = nl_count.p;
    P.has_term = bytes.p;
    P.phase_used = bytes.p + n_tiles;
    P.res = res.p;
    P.ids_mode = ids ? 1 : 0;
    P.span_off = ids ? ids->off : nullptr;
    P.span_len = ids ? ids->len : nullptr;
    P.span_cap = ids ? ids->cap : 0;
    static int occ[64] = {0};
    if (!occ[c->device & 63]) {
        int o = 0;
        SGPU_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, fastq_fused_kernel<false, false>, NTHREADS, smem));
        occ[c->device & 63] = o > 0 ? o : 1;
        if (getenv("SGPU_DEBUG"))
            fprintf(stderr, "[sgpu] fused kernel: tile %d B, %zu B shared memory per CTA, %d CTAs per SM\n", TILE, smem, o);
    }
    uint64_t grid = (uint64_t)c->sm_count * occ[c->device & 63];  // persistent: every CTA is resident
    if (grid > n_tiles) grid = n_tiles;
    // tiles are pulled into L2 one generation of CTAs ahead (SGPU_FUSED_PF scales the distance, 0 = off)
    static const double pf_factor = getenv("SGPU_FUSED_PF") ? atof(getenv("SGPU_FUSED_PF")) : 0.5;
    P.pf_dist = (uint64_t)((double)grid * pf_factor);
    if (c->profiling) {
        if (c->prof_used == c->prof_events.size()) {
            cudaEvent_t a, b;
            SGPU_CUDA(cudaEventCreate(&a));
            SGPU_CUDA(cudaEventCreate(&b));
            c->prof_events.emplace_back(a, b);
        }
        SGPU_CUDA(cudaEventRecord(c->prof_events[c->prof_used].first, st));
    }
#ifdef SGPU_FUSED_TIMING
    unsigned long long *d_trace = nullptr;
    if (getenv("SGPU_FUSED_TRACE")) {
        cudaMalloc((void **)&d_trace, n_tiles * 64);
        cudaMemset(d_trace, 0, n_tiles * 64);
    }
    cudaMemcpyToSymbol(g_trace, &d_trace, sizeof(d_trace));
#endif
    // a set with a key arena holds ids of 16 bytes and more: the variant with the vectorised long-id probe
    const bool long_ids = set && set->arena_used > 0;
    if (ids) {
        if (long_ids) fastq_fused_kernel<true, true><<<(unsigned)grid, NTHREADS, smem, st>>>(P);
        else fastq_fused_kernel<true, false><<<(unsigned)grid, NTHREADS, smem, st>>>(P);
    } else {
        if (long_ids) fastq_fused_kernel<false, true><<<(unsigned)grid, NTHREADS, smem, st>>>(P);
        else fastq_fused_kernel<false, false><<<(unsigned)grid, NTHREADS, smem, st>>>(P);
    }
    SGPU_LAUNCH(c);
    if (c->profiling) SGPU_CUDA(cudaEventRecord(c->prof_events[c->prof_used++].second, st));
    SGPU_TRY(exclusive_scan_u64(c, (const uint64_t *)P.sum_total, prefix.p, n_tiles, nullptr));
    SGPU_TRY(exclusive_scan_u32_to_u64(c, nl_count.p, prefix.p + n_tiles, n_tiles, nullptr));
    fused_verify_kernel<<<(unsigned)ceil_div(n_tiles, 256), 256, 0, st>>>(prefix.p, P.sum_head, P.has_term,
                                                                         prefix.p + n_tiles, nl_count.p, P.phase_used,
                                                                         n_tiles, is_last, res.p);
    SGPU_LAUNCH(c);
    if (want_own_nl) {
        fused_own_newlines_kernel<<<1, 1024, 0, st>>>(d_in, lead, own_len, prefix.p + n_tiles, nl_count.p, n_tiles, res.p);
        SGPU_LAUNCH(c);
    }
    SGPU_CUDA(cudaGetLastError());
    FusedResult h;
    SGPU_TRY(read_u64s(c, res.p, (uint64_t *)&h, sizeof(FusedResult) / 8));
#ifdef SGPU_FUSED_TIMING
    {
        unsigned long long ph[16], zero[16] = {0};
        cudaMemcpyFromSymbol(ph, g_phase_cycles, sizeof(ph));
        cudaMemcpyToSymbol(g_phase_cycles, zero, sizeof(zero));
        static const char *names[11] = {"load wait", "P1", "B1 wait", "scatter+B2", "phase+P2+B3", "P3 own", "B4 wait",
                                        "emit", "B5 wait (look-back)", "copy", "ticket+B6"};
        unsigned long long tot = 0;
        for (int i = 0; i < 11; i++) tot += ph[i];
        fprintf(stderr, "[sgpu] fused phases, thread 0, cycles per tile (%llu tiles):", (unsigned long long)n_tiles);
        for (int i = 0; i < 11; i++) fprintf(stderr, " %s=%.0f", names[i], (double)ph[i] / (double)n_tiles);
        fprintf(stderr, " total=%.0f\n", (double)tot / (double)n_tiles);
        if (d_trace) {
            std::vector<unsigned long long> tr(n_tiles * 8);
            cudaMemcpy(tr.data(), d_trace, n_tiles * 64, cudaMemcpyDeviceToHost);
            cudaFree(d_trace);
            FILE *f = fopen(getenv("SGPU_FUSED_TRACE"), "wb");
            if (f) {
                fwrite(tr.data(), 8, tr.size(), f);
                fclose(f);
            }
        }
    }
#endif
    // a shard must have seen the start of a foreign record: only then is its last owned record complete
    if (!h.fallback && !is_last && h.owned_end == ~0ull) {
        h.fallback = 1;
        h.reason = 12;
    }
    if (h.fallback) {  // *used stays 0: the general path decides (and reports errors)
        if (getenv("SGPU_DEBUG")) fprintf(stderr, "[sgpu] fused kernel fell back, reason %llu\n", h.reason);
        return SGPU_OK;
    }
    if (h.overflow) return SGPU_ERR_CAPACITY;
    *used = 1;
    counts->own_newlines = want_own_nl ? h.own_newlines : 0;
    if (ids) {
        ids->n_spans = h.n_spans;
        counts->reads_in = h.reads_in;
        counts->path = 1;
        return SGPU_OK;
    }
    const uint64_t owned_end = is_last ? n_in : h.owned_end;
    const uint64_t other_total = owned_end - lead - h.kept_total;
    if (c->profiling) c->prof_alg_bytes += n_in + h.kept_total + (out.o ? other_total : 0);
    *out.n_w = (size_t)h.kept_total;
    if (out.n_o) *out.n_o = out.o ? (size_t)other_total : 0;
    counts->reads_in = h.reads_in;
    counts->reads_out = h.reads_out;
    counts->crlf = 0;
    counts->path = 1;
    return SGPU_OK;
}

// positions of the first four '\n' bytes of buf[0..n) (~0 where there is none): one warp, 512 bytes per step (shards:
// the first record boundary lies within the first record's length of the cut)
__global__ void first_newlines_kernel(const uint8_t *buf, uint64_t n, unsigned long long *out) {
    const int lane = threadIdx.x;
    uint32_t seen = 0;
    for (uint64_t base = 0; base < n && seen < 4; base += 512) {
        const uint64_t pos = base + (uint64_t)lane * 16;
        uint32_t m = 0;
        if (pos < n) {
            m = nl_mask16_v2(ld_nc_u4(buf + pos));
            if (n - pos < 16) m &= (1u << (n - pos)) - 1u;
        }
        uint32_t inc = __popc(m);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t x = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += x;
        }
        uint32_t idx = seen + inc - __popc(m);  // index of this lane's first newline
        for (uint32_t mm = m; mm && idx < 4; mm &= mm - 1, idx++) out[idx] = pos + (uint64_t)(__ffs(mm) - 1);
        seen += __shfl_sync(0xffffffffu, inc, 31);
    }
    // out[4 + i] = 1 when newline i is followed by "+\n" (the end of a sequence line of canonical FASTQ)
    __syncwarp();
    if (lane < 4) {
        const unsigned long long p = *((volatile unsigned long long *)out + lane);
        out[4 + lane] = (p != ~0ull && p + 2 < n && buf[p + 1] == '+' && buf[p + 2] == '\n') ? 1ull : 0ull;
    }
}

// one shard (see sgpu_clean_fastq_shard_dev): locate the first owned record start, then run the fused kernel
// from the 16-byte aligned address below it.  A whole file is the shard (n, n, 0, 1, 1): the range is the buffer.
// newlines_before == SGPU_NEWLINES_UNKNOWN: the line phase is SPECULATED from the first "\n+\n" among the shard's first
// four newlines (it ends a sequence line, so the newline two places before / behind it ends a record); the caller
// verifies (true newlines_before + counts->lead_newlines) % 4 == 0 once the shards' own_newlines are exchanged.
sgpu_status fused_shard(sgpu_ctx *c, const sgpu_idset *set, const Shard &s, uint64_t newlines_before, int reverse,
                        const Outs &out, IdsOut *ids, sgpu_counts *counts, int *used, bool want_nl) {
    *used = 0;
    const bool spec = newlines_before == SGPU_NEWLINES_UNKNOWN;
    want_nl = want_nl || spec;
    uint64_t s0 = 0, lead_nl = 0;
    if (!s.is_first) {
        DevBuf<unsigned long long> pos;
        SGPU_TRY(pos.alloc(8, c->stream));
        SGPU_CUDA(cudaMemsetAsync(pos.p, 0xFF, 64, c->stream));
        first_newlines_kernel<<<1, 32, 0, c->stream>>>(s.p, s.n, pos.p);
        SGPU_LAUNCH(c);
        uint64_t h[8];
        SGPU_TRY(read_u64s(c, pos.p, h, 8));
        uint32_t k;  // index of the first newline that ends a record
        if (spec) {
            uint32_t j = 0;
            while (j < 4 && !(h[j] != ~0ull && h[4 + j] == 1)) j++;
            if (j == 4) return SGPU_OK;  // no "\n+\n" in sight: not canonical here, the exact protocol decides
            k = (2 + j) & 3;             // newline j has role 1 => newline j + 2 (mod 4) has role 3
        } else {
            // the newline that ends the previous shard's last record has global index == 3 (mod 4)
            k = (uint32_t)((3 - (newlines_before & 3)) & 3);
        }
        if (h[k] == ~0ull) return SGPU_OK;  // no record boundary in the buffer: the general path sorts it out
        s0 = h[k] + 1;
        lead_nl = k + 1;
        if (s0 >= s.n || s0 > s.own_len) return SGPU_OK;  // owns nothing (general path: zero records / errors)
    }
    const uint32_t lead = (uint32_t)(s0 & 15);
    const uint64_t skip = s0 - lead;
    const sgpu_status rc = clean_fused_range(c, set, s.p + skip, s.n - skip, lead, s.own_len - skip, s.is_last, reverse,
                                             out, counts, used, ids, want_nl);
    if (ids) ids->base = skip;  // span offsets are relative to the range the kernel saw
    if (want_nl && *used) {
        counts->lead_newlines = lead_nl;
        counts->own_newlines += lead_nl;  // [0, s0) + [s0, own_len)
        counts->speculated = spec ? 1 : 0;
    }
    return rc;
}

}  // namespace sgpu
