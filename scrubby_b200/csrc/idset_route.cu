// idset_route.cu -- the sinks of the ids passes, and the probe of routed id lines.
//
// An ids pass (the single-pass kernel in ids mode, fastq_ids_kernel, fa_record_kernel) ends in (offset, length[, sel])
// spans.  sink_spans() hands them to idset_insert_spans, or ROUTES them for the hash-partitioned diff
// (scrubby_b200/dist.py diff_partitioned): every selected id becomes an "id\n" line in the partition of its owner
// rank, route_owner() in idset.cuh.  One output buffer holds partition 0's lines, then partition 1's, ...; inside a
// partition the lines keep file order, so a partition is a subsequence of the file's ids and routing is reproducible.
//
// Route: one warp per tile of ROUTE_TILE spans.
//   route_count_kernel   : the owner of every selected span, the tile's bytes per partition (a partition-major table
//                          in global memory, the histogram in shared memory) and the partitions' totals
//   exclusive scan of the table (scan.cu)   -> where the tile's lines of each partition start
//   route_scatter_kernel : rounds of 32 spans in order; a span's place is its partition's cursor plus the lengths of the
//                          lower lanes of the same owner (__match_any_sync groups); the group's last lane moves the
//                          cursor; every lane copies its own line
// The single-pass kernel lists its spans in tile completion order: order_spans() puts them in offset order first (a
// bitmap of the span starts, its per-word prefix counts, a scan, then each span's rank).
//
// Probe lines: the '\n' index of a buffer of "id\n" lines (scan.cu), one thread per line probes the set (idset.cuh)
// and selects the absent ids; idset_insert_spans takes them.  Every line counts as one input record.
#include "fastq_records.cuh"

namespace sgpu {

constexpr int ROUTE_WARPS = 4;    // warps (tiles) per block
constexpr int ROUTE_ROUNDS = 16;  // rounds of 32 spans per tile
constexpr uint64_t ROUTE_TILE = 32 * ROUTE_ROUNDS;
constexpr uint32_t ROUTE_MAX_PARTS = 64;
constexpr uint8_t ROUTE_NONE = 0xFF;  // owner of a span that is not selected

__global__ void __launch_bounds__(ROUTE_WARPS * 32)
    route_count_kernel(const uint8_t *src, const uint64_t *off, const uint32_t *len, const uint8_t *sel, uint64_t n,
                       uint32_t n_parts, uint64_t n_tiles, uint8_t *owner, uint64_t *tile_bytes,
                       unsigned long long *totals) {
    __shared__ unsigned long long hb[ROUTE_WARPS][ROUTE_MAX_PARTS];
    __shared__ unsigned int hl[ROUTE_WARPS][ROUTE_MAX_PARTS];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint64_t t = (uint64_t)blockIdx.x * ROUTE_WARPS + w;
    for (uint32_t p = lane; p < ROUTE_MAX_PARTS; p += 32) {
        hb[w][p] = 0;
        hl[w][p] = 0;
    }
    __syncwarp();
    if (t >= n_tiles) return;  // (the whole warp)
    const uint64_t base = t * ROUTE_TILE;
    for (int r = 0; r < ROUTE_ROUNDS; r++) {
        const uint64_t i = base + (uint64_t)r * 32 + lane;
        if (i < n) {
            uint8_t o = ROUTE_NONE;
            if (!sel || sel[i]) {
                const uint32_t l = len[i];
                uint64_t lo, hi, home;
                key_image(src + off[i], l, &lo, &hi, &home);
                o = (uint8_t)route_owner(home, n_parts);
                atomicAdd(&hb[w][o], (unsigned long long)l + 1ull);
                atomicAdd(&hl[w][o], 1u);
            }
            owner[i] = o;
        }
    }
    __syncwarp();
    for (uint32_t p = lane; p < n_parts; p += 32) {
        const unsigned long long b = hb[w][p];
        tile_bytes[(uint64_t)p * n_tiles + t] = b;
        if (b) {
            atomicAdd(&totals[p], b);
            atomicAdd(&totals[ROUTE_MAX_PARTS + p], (unsigned long long)hl[w][p]);
        }
    }
}

__global__ void __launch_bounds__(ROUTE_WARPS * 32)
    route_scatter_kernel(const uint8_t *src, const uint64_t *off, const uint32_t *len, const uint8_t *owner, uint64_t n,
                         uint32_t n_parts, uint64_t n_tiles, const uint64_t *tile_start, uint8_t *lines) {
    __shared__ unsigned long long cur[ROUTE_WARPS][ROUTE_MAX_PARTS];
    __shared__ unsigned int lbytes[ROUTE_WARPS][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint64_t t = (uint64_t)blockIdx.x * ROUTE_WARPS + w;
    if (t >= n_tiles) return;  // (the whole warp)
    for (uint32_t p = lane; p < n_parts; p += 32) cur[w][p] = tile_start[(uint64_t)p * n_tiles + t];
    const uint64_t base = t * ROUTE_TILE;
    for (int r = 0; r < ROUTE_ROUNDS; r++) {
        const uint64_t i = base + (uint64_t)r * 32 + lane;
        uint32_t o = ROUTE_NONE, l = 0;
        if (i < n) {
            o = owner[i];
            if (o != ROUTE_NONE) l = len[i];
        }
        lbytes[w][lane] = o != ROUTE_NONE ? l + 1u : 0u;
        const unsigned peers = __match_any_sync(0xffffffffu, o);
        __syncwarp();  // (also orders the cursor writes of the previous round before the reads below)
        uint64_t pos = 0;
        if (o != ROUTE_NONE) {
            unsigned lower = peers & ((1u << lane) - 1u);
            uint64_t pre = 0;
            while (lower) {
                pre += lbytes[w][__ffs(lower) - 1];
                lower &= lower - 1u;
            }
            pos = cur[w][o] + pre;
        }
        __syncwarp();
        if (o != ROUTE_NONE && (peers >> lane) == 1u) cur[w][o] = pos + l + 1u;  // the group's last lane
        if (o != ROUTE_NONE) {
            const uint8_t *s = src + off[i];
            uint8_t *d = lines + pos;
            for (uint32_t k = 0; k < l; k++) d[k] = s[k];
            d[l] = '\n';
        }
    }
}

// ---------------------------------------------------------------- spans in offset order
constexpr int ORDER_WORDS = 1024;  // bitmap words per block of the rank (32 Kibit: the per-word prefix fits 16 bits)

__global__ void span_mark_kernel(const uint64_t *off, uint64_t n, uint32_t *bits) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) atomicOr(&bits[off[i] >> 5], 1u << (off[i] & 31));
}

__global__ void __launch_bounds__(ORDER_WORDS)
    span_word_prefix_kernel(const uint32_t *bits, uint64_t nw, uint16_t *wpre, uint32_t *block_cnt) {
    __shared__ uint32_t warp_sum[32];
    const uint64_t wi = (uint64_t)blockIdx.x * ORDER_WORDS + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t v = wi < nw ? (uint32_t)__popc(bits[wi]) : 0u;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t x = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += x;
    }
    if (lane == 31) warp_sum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const uint32_t x = warp_sum[lane];
        uint32_t ic = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, ic, d);
            if (lane >= d) ic += y;
        }
        warp_sum[lane] = ic - x;
        if (lane == 31) block_cnt[blockIdx.x] = ic;
    }
    __syncthreads();
    if (wi < nw) wpre[wi] = (uint16_t)(warp_sum[warp] + inc - v);
}

__global__ void span_place_kernel(const uint64_t *off, const uint32_t *len, uint64_t n, const uint32_t *bits,
                                  const uint16_t *wpre, const uint64_t *block_off, uint64_t *off2, uint32_t *len2) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t o = off[i], wi = o >> 5;
    const uint64_t rank = block_off[wi / ORDER_WORDS] + wpre[wi] + __popc(bits[wi] & ((1u << (o & 31)) - 1u));
    off2[rank] = o;
    len2[rank] = len[i];
}

// the n spans (distinct offsets in [0, range)) sorted by offset into off2 / len2
static sgpu_status order_spans(sgpu_ctx *c, uint64_t range, const uint64_t *off, const uint32_t *len, size_t n,
                               DevBuf<uint64_t> &off2, DevBuf<uint32_t> &len2) {
    cudaStream_t st = c->stream;
    const uint64_t nw = range / 32 + 1, nb = ceil_div(nw, (uint64_t)ORDER_WORDS);
    DevBuf<uint32_t> bits, block_cnt;
    DevBuf<uint16_t> wpre;
    DevBuf<uint64_t> block_off;
    SGPU_TRY(bits.alloc(nw, st));
    SGPU_TRY(wpre.alloc(nw, st));
    SGPU_TRY(block_cnt.alloc(nb, st));
    SGPU_TRY(block_off.alloc(nb, st));
    SGPU_TRY(off2.alloc(n, st));
    SGPU_TRY(len2.alloc(n, st));
    SGPU_CUDA(cudaMemsetAsync(bits.p, 0, nw * sizeof(uint32_t), st));
    span_mark_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(off, n, bits.p);
    SGPU_LAUNCH(c);
    span_word_prefix_kernel<<<(unsigned)nb, ORDER_WORDS, 0, st>>>(bits.p, nw, wpre.p, block_cnt.p);
    SGPU_LAUNCH(c);
    SGPU_TRY(exclusive_scan_u32_to_u64(c, block_cnt.p, block_off.p, nb, nullptr));
    span_place_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(off, len, n, bits.p, wpre.p, block_off.p, off2.p, len2.p);
    SGPU_LAUNCH(c);
    SGPU_CUDA(cudaGetLastError());
    return SGPU_OK;
}

// the selected spans as "id\n" lines grouped by owner partition, file order inside a partition (given spans in file
// order); r.n_lines / part_bytes / part_lines are set, SGPU_ERR_CAPACITY when r.cap is too small
static sgpu_status route_spans(sgpu_ctx *c, RouteOut &r, const uint8_t *src, const uint64_t *off, const uint32_t *len,
                               const uint8_t *sel, size_t n) {
    const uint32_t P = r.n_parts;
    memset(r.part_bytes, 0, P * sizeof(uint64_t));
    memset(r.part_lines, 0, P * sizeof(uint64_t));
    r.n_lines = 0;
    if (n == 0) return SGPU_OK;
    cudaStream_t st = c->stream;
    const uint64_t n_tiles = ceil_div(n, ROUTE_TILE);
    DevBuf<uint8_t> owner;
    DevBuf<uint64_t> table, start, totals;
    SGPU_TRY(owner.alloc(n, st));
    SGPU_TRY(table.alloc(P * n_tiles, st));
    SGPU_TRY(start.alloc(P * n_tiles, st));
    SGPU_TRY(totals.alloc(2 * ROUTE_MAX_PARTS, st));
    SGPU_CUDA(cudaMemsetAsync(totals.p, 0, 2 * ROUTE_MAX_PARTS * sizeof(uint64_t), st));
    const unsigned grid = (unsigned)ceil_div(n_tiles, (uint64_t)ROUTE_WARPS);
    route_count_kernel<<<grid, ROUTE_WARPS * 32, 0, st>>>(src, off, len, sel, n, P, n_tiles, owner.p, table.p,
                                                          (unsigned long long *)totals.p);
    SGPU_LAUNCH(c);
    SGPU_TRY(exclusive_scan_u64(c, table.p, start.p, P * n_tiles, nullptr));
    uint64_t h[2 * ROUTE_MAX_PARTS];
    SGPU_TRY(read_u64s(c, totals.p, h, P));
    SGPU_TRY(read_u64s(c, totals.p + ROUTE_MAX_PARTS, h + ROUTE_MAX_PARTS, P));
    uint64_t total = 0;
    for (uint32_t p = 0; p < P; p++) {
        r.part_bytes[p] = h[p];
        r.part_lines[p] = h[ROUTE_MAX_PARTS + p];
        total += h[p];
    }
    r.n_lines = (size_t)total;
    if (total > r.cap) return SGPU_ERR_CAPACITY;
    if (total) {
        route_scatter_kernel<<<grid, ROUTE_WARPS * 32, 0, st>>>(src, off, len, owner.p, n, P, n_tiles, start.p, r.lines);
        SGPU_LAUNCH(c);
    }
    SGPU_CUDA(cudaGetLastError());
    SGPU_CUDA(cudaStreamSynchronize(st));  // scratch buffers are released after this call returns
    return SGPU_OK;
}

sgpu_status sink_spans(sgpu_ctx *c, const SpanSink &k, const uint8_t *d_src, const uint64_t *d_off, const uint32_t *d_len,
                       const uint8_t *d_sel, size_t n, bool in_order, uint64_t range) {
    if (!k.route) return k.into ? idset_insert_spans(c, k.into, d_src, d_off, d_len, d_sel, n) : SGPU_OK;
    if (in_order || n == 0) return route_spans(c, *k.route, d_src, d_off, d_len, d_sel, n);
    DevBuf<uint64_t> off2;
    DevBuf<uint32_t> len2;
    SGPU_TRY(order_spans(c, range, d_off, d_len, n, off2, len2));
    return route_spans(c, *k.route, d_src, off2.p, len2.p, d_sel, n);
}

// ---------------------------------------------------------------- probe lines
// line k of the buffer: [start, end) without its '\n'; absent from the set -> selected.  `set_has_empty`: "" is a
// member of the set (an empty line is then present)
__global__ void __launch_bounds__(128)
    probe_lines_kernel(const uint8_t *buf, uint64_t n, const uint64_t *nlpos, uint64_t n_nl, uint64_t n_lines,
                       IdSetView set, int set_has_empty, uint64_t *key_off, uint32_t *key_len, uint8_t *sel,
                       unsigned long long *n_absent) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool absent = false;
    if (k < n_lines) {
        const uint64_t start = k ? nlpos[k - 1] + 1 : 0, end = k < n_nl ? nlpos[k] : n;
        const uint64_t l = end - start;
        const bool hit = l == 0 ? set_has_empty != 0 : l <= IDSET_MAX_KEY && idset_contains(set, buf + start, (uint32_t)l);
        absent = !hit;
        key_off[k] = start;
        key_len[k] = (uint32_t)(l <= IDSET_MAX_KEY ? l : IDSET_MAX_KEY + 1);
        sel[k] = absent ? 1 : 0;
    }
    const unsigned b = __ballot_sync(0xffffffffu, absent);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(n_absent, (unsigned long long)__popc(b));
}

// "id\n" lines (a last line without '\n' counts too): *n_lines lines, *n_absent of them absent from `probe` (nullptr:
// every line), whose ids go into `into` (nullptr: counted only)
static sgpu_status probe_lines(sgpu_ctx *c, const sgpu_idset *probe, const uint8_t *d_buf, size_t n, sgpu_idset *into,
                               uint64_t *n_lines, uint64_t *n_absent) {
    *n_lines = *n_absent = 0;
    if (n == 0) return SGPU_OK;
    cudaStream_t st = c->stream;
    DevBuf<uint64_t> nlpos, scratch, key_off;
    DevBuf<uint32_t> key_len;
    DevBuf<uint8_t> sel;
    uint64_t n_nl = 0;
    SGPU_TRY(index_newlines(c, d_buf, n, nlpos, &n_nl));
    uint64_t last_nl = 0;
    if (n_nl) SGPU_TRY(read_u64s(c, nlpos.p + n_nl - 1, &last_nl, 1));
    const uint64_t lines = n_nl + ((n_nl == 0 || last_nl + 1 != n) ? 1 : 0);
    SGPU_TRY(scratch.alloc(1, st));
    SGPU_CUDA(cudaMemsetAsync(scratch.p, 0, sizeof(uint64_t), st));
    SGPU_TRY(key_off.alloc(lines, st));
    SGPU_TRY(key_len.alloc(lines, st));
    SGPU_TRY(sel.alloc(lines, st));
    probe_lines_kernel<<<(unsigned)ceil_div(lines, 128), 128, 0, st>>>(
        d_buf, n, nlpos.p, n_nl, lines, view_of(probe), probe && probe->has_empty, key_off.p, key_len.p, sel.p,
        (unsigned long long *)scratch.p);
    SGPU_LAUNCH(c);
    SGPU_TRY(read_u64s(c, scratch.p, n_absent, 1));
    *n_lines = lines;
    if (into && *n_absent) SGPU_TRY(idset_insert_spans(c, into, d_buf, key_off.p, key_len.p, sel.p, lines));
    SGPU_CUDA(cudaStreamSynchronize(st));
    return SGPU_OK;
}

}  // namespace sgpu

using namespace sgpu;

extern "C" {

sgpu_status sgpu_idset_probe_lines_dev(sgpu_ctx *c, const sgpu_idset *probe, const uint8_t *d_lines, size_t n,
                                       sgpu_idset *into, sgpu_counts *counts) {
    if (!c || !counts || (n && !d_lines)) return SGPU_ERR_INVALID_ARG;
    if (n && ((uintptr_t)d_lines & 15)) return SGPU_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(c->mu);
    SGPU_CUDA(cudaSetDevice(c->device));
    uint64_t lines = 0, absent = 0;
    SGPU_TRY(probe_lines(c, probe, d_lines, n, into, &lines, &absent));
    counts->reads_in += lines;
    counts->difference += absent;
    return SGPU_OK;
}

}  // extern "C"
