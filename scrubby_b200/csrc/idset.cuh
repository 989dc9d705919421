// idset.cuh -- device-side encoding and probe of the exact read-id set.
//
// Replaces std HashSet<String> (SipHash-1-3 + SwissTable) at alignment.rs:62,91,
// classifier.rs:135,274 and utils.rs:251,257, and `read_ids.contains(&id)` at
// cleaner.rs:747,751.
//
// Layout in HBM (round 2): open addressing over 128-byte BUCKETS of eight 16-byte slots -- one L2 line, which is what a
// random DRAM miss costs on B200 whatever is asked for (round 1: 124 B per lookup with 16-, 32- and 64-byte buckets
// alike).  Buckets are grouped into PAGES of 256 (32 KiB): a key's page is the multiply-shift range reduction
// mulhi64(hash, n_pages) -- any number of pages, so the table is sized exactly for its keys -- and its home bucket
// inside the page comes from the hash's low bits.  The probe sequence starts at slot 0 of the home bucket and runs
// linearly, bucket after bucket, WRAPPING INSIDE THE PAGE: a page is a closed little hash table, which is what lets
// the bulk build (idset_build.cu) assemble every page in shared memory and write the table exactly once.  There are
// no deletions, so the occupied slots of a bucket are a prefix of it and a lookup ends at the first empty slot.
// Load factor 0.2 (measured, tools/c4_probe.py on 50 M ids: the fused kernel takes 1.75 / 1.77 / 1.81 / 1.83 / 1.94 ms
// per 3.3 GB at load 0.12 / 0.2 / 0.25 / 0.33 / 0.5 -- lookups that leave the first four slots cost a second round
// trip for the whole warp; the bulk build's page kernel is bound by the keys it places per page, not by the bytes it
// writes: 1.28 ms at load 0.2, 1.59 ms at 0.25).
//   empty  : lo == 0 && hi == 0
//   inline : ids of 1..15 bytes live IN the slot: byte0 = len, bytes 1..15 = id (zero padded).
//            One 16-byte load and a 128-bit compare decide membership exactly.
//   long   : ids of >= 16 bytes: byte0 = 0x80, bytes 1..7 = top 56 bits of a 64-bit hash,
//            hi = (arena offset << 24) | len.  A fingerprint hit is verified against the
//            id bytes in the arena, so there are no false positives.
#pragma once
#include "common.cuh"

namespace sgpu {

constexpr uint32_t IDSET_INLINE_MAX = 15;
#ifndef SGPU_IDSET_LOAD_PCT
#define SGPU_IDSET_LOAD_PCT 20
#endif
constexpr uint64_t IDSET_BUCKET = SGPU_IDSET_BUCKET;      // slots per bucket: 8 x 16 B = one 128-byte line
#ifndef SGPU_IDSET_PAGE_BUCKETS
#define SGPU_IDSET_PAGE_BUCKETS 256
#endif
constexpr uint64_t IDSET_PAGE_BUCKETS = SGPU_IDSET_PAGE_BUCKETS;  // buckets per page (a power of two): 256 = 32 KiB
constexpr uint64_t IDSET_LOAD_PCT = SGPU_IDSET_LOAD_PCT;  // keys <= LOAD_PCT % of the slots
constexpr uint64_t IDSET_MAX_KEY = (1ull << 24) - 1;

struct IdSetView {
    const Slot *table;   // n_pages * 256 buckets * 8 slots, 128-byte aligned (n_pages == 0 -> table == nullptr)
    uint64_t n_pages;
    const uint8_t *arena;
};

// buckets (a whole number of pages) for `keys` ids at the target load
static inline uint64_t idset_buckets_for(uint64_t keys) {
    const uint64_t slots = (keys * 100 + IDSET_LOAD_PCT - 1) / IDSET_LOAD_PCT;
    const uint64_t per_page = IDSET_PAGE_BUCKETS * IDSET_BUCKET;
    const uint64_t pages = (slots + per_page - 1) / per_page;
    return (pages ? pages : 1) * IDSET_PAGE_BUCKETS;
}

#ifdef __CUDACC__

// page / home bucket of a key whose (well mixed) 64-bit hash is h: multiply-shift range reduction over the pages, the
// low bits inside the page; the probe sequence wraps inside the page
__device__ __forceinline__ uint64_t home_page(uint64_t h, uint64_t n_pages) { return __umul64hi(h, n_pages); }
__device__ __forceinline__ uint64_t home_bucket(uint64_t h, uint64_t n_pages) {
    return home_page(h, n_pages) * IDSET_PAGE_BUCKETS + (h & (IDSET_PAGE_BUCKETS - 1));
}
__device__ __forceinline__ uint64_t next_bucket(uint64_t b) {
    return (b & ~(IDSET_PAGE_BUCKETS - 1)) | ((b + 1) & (IDSET_PAGE_BUCKETS - 1));
}
__device__ __forceinline__ uint64_t inline_hash(uint64_t lo, uint64_t hi) {
    return mix64(lo ^ mix64(hi + 0x9E3779B97F4A7C15ULL));
}

__device__ __forceinline__ uint64_t hash_bytes(const uint8_t *p, uint32_t len) {
    uint64_t h = 0x9E3779B97F4A7C15ULL ^ ((uint64_t)len * 0xD6E8FEB86659FD93ULL);
    uint32_t i = 0;
    for (; i + 8 <= len; i += 8) {
        uint64_t w = 0;
#pragma unroll
        for (int b = 0; b < 8; b++) w |= (uint64_t)p[i + b] << (8 * b);
        h = (h ^ w) * 0xFF51AFD7ED558CCDULL;
        h ^= h >> 29;
    }
    uint64_t w = 0;
    for (uint32_t b = 0; i + b < len; b++) w |= (uint64_t)p[i + b] << (8 * b);
    h = (h ^ w) * 0xC4CEB9FE1A85EC53ULL;
    return mix64(h);
}

// hash_bytes() over a key delivered as little-endian 32-bit words: word(k) = bytes 4k .. 4k+3 of the key (bytes past
// the key's end may hold anything).  Same value as hash_bytes(), a fraction of the loads (keys of 16 bytes and more:
// Illumina / ONT read names).
template <typename Words>
__device__ __forceinline__ uint64_t hash_words(Words word, uint32_t len) {
    uint64_t h = 0x9E3779B97F4A7C15ULL ^ ((uint64_t)len * 0xD6E8FEB86659FD93ULL);
    uint32_t i = 0;
    for (; i + 8 <= len; i += 8) {
        const uint64_t w = (uint64_t)word(i >> 2) | ((uint64_t)word((i >> 2) + 1) << 32);
        h = (h ^ w) * 0xFF51AFD7ED558CCDULL;
        h ^= h >> 29;
    }
    const uint32_t rem = len - i;
    uint64_t w = 0;
    if (rem) {
        w = (uint64_t)word(i >> 2);
        if (rem > 4) w |= (uint64_t)word((i >> 2) + 1) << 32;
        w &= (1ull << (8 * rem)) - 1ull;
    }
    h = (h ^ w) * 0xC4CEB9FE1A85EC53ULL;
    return mix64(h);
}
// the words of a key at an arbitrarily aligned GLOBAL address; only words that hold key bytes are read
struct GlobalKeyWords {
    const uint32_t *w;
    uint32_t sh, need;  // misalignment in bits; bytes from the aligned base that belong to the key
    __device__ __forceinline__ GlobalKeyWords(const uint8_t *p, uint32_t len) {
        const uint32_t mis = (uint32_t)((uintptr_t)p & 3u);
        w = reinterpret_cast<const uint32_t *>(p - mis);
        sh = mis * 8u;
        need = mis + len;
    }
    __device__ __forceinline__ uint32_t operator()(uint32_t k) const {
        const uint32_t a = 4u * k < need ? __ldg(w + k) : 0u;
        const uint32_t b = (sh && 4u * (k + 1) < need) ? __ldg(w + k + 1) : 0u;
        return __funnelshift_r(a, b, sh);
    }
};
// key bytes == the arena entry at `e` (16-byte aligned: arena entries are padded to 16)?  word-wise
template <typename Words>
__device__ __forceinline__ bool arena_equal_words(const uint8_t *e, Words word, uint32_t len) {
    const uint32_t *a = reinterpret_cast<const uint32_t *>(e);
    const uint32_t nw = len >> 2, rem = len & 3u;
    for (uint32_t k = 0; k < nw; k++)
        if (__ldg(a + k) != word(k)) return false;
    if (rem) {
        const uint32_t m = (1u << (8 * rem)) - 1u;
        if ((__ldg(a + nw) & m) != (word(nw) & m)) return false;
    }
    return true;
}
constexpr uint32_t IDSET_ARENA_ALIGN = 16;  // arena entries start on 16-byte boundaries (their lengths are padded)
__host__ __device__ __forceinline__ uint32_t arena_padded(uint32_t len) { return (len + IDSET_ARENA_ALIGN - 1) & ~(IDSET_ARENA_ALIGN - 1); }

// builds the slot image of a key and its home hash (home_bucket() turns it into a bucket).  For long keys `hi` is left 0
// (the caller fills offset/len when inserting).
__device__ __forceinline__ void key_image(const uint8_t *p, uint32_t len, uint64_t *lo, uint64_t *hi,
                                          uint64_t *home) {
    if (len <= IDSET_INLINE_MAX) {
        uint64_t a = len, b = 0;
#pragma unroll
        for (uint32_t i = 0; i < 7; i++)
            if (i < len) a |= (uint64_t)p[i] << (8 * (i + 1));
#pragma unroll
        for (uint32_t i = 7; i < 15; i++)
            if (i < len) b |= (uint64_t)p[i] << (8 * (i - 7));
        *lo = a;
        *hi = b;
        *home = inline_hash(a, b);
    } else {
        uint64_t h = hash_bytes(p, len);
        *lo = 0x80ull | (h & ~0xFFull);
        *hi = 0;
        *home = mix64(*lo);
    }
}

// Owner partition of a key among n_parts (1..64) in the hash-partitioned diff: route_owner(home, n_parts) with `home`
// key_image()'s hash.  The set an owner builds from its keys takes the page from home's HIGH bits (home_page) and the
// bucket from its low 8 bits, so the owner is drawn from a fixed bijective remix of home (xor, xorshift-multiply
// rounds): a partition's keys still spread over every page of the owner's set.
__device__ __forceinline__ uint64_t route_remix(uint64_t h) {
    h ^= 0x2545F4914F6CDD1DULL;
    h ^= h >> 30;
    h *= 0xBF58476D1CE4E5B9ULL;
    h ^= h >> 27;
    h *= 0x94D049BB133111EBULL;
    h ^= h >> 31;
    return h;
}
__device__ __forceinline__ uint32_t route_owner(uint64_t home, uint32_t n_parts) {
    return (uint32_t)__umul64hi(route_remix(home), (uint64_t)n_parts);
}

// home hash recomputed from a stored slot (rehash without touching key bytes)
__device__ __forceinline__ uint64_t slot_home(uint64_t lo, uint64_t hi) {
    if ((lo & 0xFF) == 0x80) return mix64(lo);
    return inline_hash(lo, hi);
}

__device__ __forceinline__ bool bytes_equal(const uint8_t *a, const uint8_t *b, uint32_t n) {
    for (uint32_t i = 0; i < n; i++)
        if (a[i] != b[i]) return false;
    return true;
}

__device__ __forceinline__ Slot load_slot(const Slot *p) {
#ifdef SGPU_TBL_NA  // experiment: table lines are used once -- no L1 allocation
    ulonglong2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u64 {%0,%1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(p));
#else
    ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2 *>(p));
#endif
    Slot s;
    s.lo = v.x;
    s.hi = v.y;
    return s;
}

// exact membership of key[0..len), len >= 1
__device__ __forceinline__ bool idset_contains(const IdSetView &v, const uint8_t *key, uint32_t len) {
    if (v.table == nullptr || len > IDSET_MAX_KEY) return false;
    uint64_t lo, hi, home;
    key_image(key, len, &lo, &hi, &home);
    uint64_t b = home_bucket(home, v.n_pages);
    const bool is_inline = len <= IDSET_INLINE_MAX;
    while (true) {
        const Slot *bp = v.table + b * IDSET_BUCKET;
        for (int q = 0; q < (int)IDSET_BUCKET; q++) {
            Slot s = load_slot(bp + q);
            if ((s.lo | s.hi) == 0) return false;
            if (s.lo == lo) {
                if (is_inline) {
                    if (s.hi == hi) return true;
                } else if ((s.hi & 0xFFFFFFull) == len && bytes_equal(v.arena + (s.hi >> 24), key, len)) {
                    return true;
                }
            }
        }
        b = next_bucket(b);
    }
}

#endif  // __CUDACC__

static inline IdSetView view_of(const sgpu_idset *s) {
    IdSetView v;
    v.table = s && s->n_buckets ? s->d_table : nullptr;
    v.n_pages = s ? s->n_buckets / IDSET_PAGE_BUCKETS : 0;
    v.arena = s ? s->d_arena : nullptr;
    return v;
}

}  // namespace sgpu
