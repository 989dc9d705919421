// scan.cu -- device-wide exclusive prefix sums (general path bookkeeping) and the '\n' index.
//
// The scans here are the simple reduce / scan-of-sums / downsweep form: they only ever
// touch per-record or per-tile metadata (a few % of the FASTQ bytes).  The fused
// single-pass kernel in fastq_fused.cu carries its own decoupled look-back instead.
#include "common.cuh"

namespace sgpu {

static thread_local char g_cuda_err[512] = "";
void set_cuda_error(cudaError_t e, const char *file, int line) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s (%s) at %s:%d", cudaGetErrorName(e), cudaGetErrorString(e),
             file, line);
}
const char *last_cuda_error_text() { return g_cuda_err; }

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ uint64_t warp_incl_scan(uint64_t v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint64_t t = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += t;
    }
    return v;
}

// block-wide exclusive scan of one value per thread; returns the exclusive prefix, *total = block sum
__device__ __forceinline__ uint64_t block_excl_scan(uint64_t v, uint64_t *total, uint64_t *smem /*>=33*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    uint64_t inc = warp_incl_scan(v, lane);
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint64_t w = lane < nwarps ? smem[lane] : 0;
        uint64_t winc = warp_incl_scan(w, lane);
        smem[lane] = winc - w;
        if (lane == 31) smem[32] = winc;
    }
    __syncthreads();
    uint64_t res = smem[warp] + inc - v;
    *total = smem[32];
    __syncthreads();
    return res;
}

template <typename TIn>
__global__ void __launch_bounds__(SCAN_THREADS) scan_reduce_kernel(const TIn *in, size_t n, uint64_t *block_sums) {
    __shared__ uint64_t sm[40];
    size_t base = (size_t)blockIdx.x * SCAN_TILE;
    uint64_t s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        size_t i = base + (size_t)k * SCAN_THREADS + threadIdx.x;
        if (i < n) s += (uint64_t)in[i];
    }
    uint64_t total;
    block_excl_scan(s, &total, sm);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

template <typename TIn>
__global__ void __launch_bounds__(SCAN_THREADS)
    scan_down_kernel(const TIn *in, uint64_t *out, size_t n, const uint64_t *block_offsets) {
    __shared__ uint64_t sm[40];
    size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
    uint64_t v[SCAN_ITEMS];
    uint64_t s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        size_t i = base + k;
        v[k] = i < n ? (uint64_t)in[i] : 0;
        s += v[k];
    }
    uint64_t total;
    uint64_t pre = block_excl_scan(s, &total, sm) + (block_offsets ? block_offsets[blockIdx.x] : 0);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        size_t i = base + k;
        if (i < n) out[i] = pre;
        pre += v[k];
    }
}

// single block: exclusive scan of up to a few thousand u64 in place, total to *d_total
__global__ void __launch_bounds__(1024) scan_small_kernel(uint64_t *data, size_t n, uint64_t *d_total) {
    __shared__ uint64_t sm[40];
    uint64_t carry = 0;
    for (size_t base = 0; base < n; base += 1024) {
        size_t i = base + threadIdx.x;
        uint64_t v = i < n ? data[i] : 0;
        uint64_t total;
        uint64_t pre = block_excl_scan(v, &total, sm);
        if (i < n) data[i] = carry + pre;
        carry += total;
    }
    if (threadIdx.x == 0 && d_total) *d_total = carry;
}

template <typename TIn>
static sgpu_status scan_impl(sgpu_ctx *c, const TIn *d_in, uint64_t *d_out, size_t n, uint64_t *d_total) {
    cudaStream_t st = c->stream;
    if (n == 0) {
        if (d_total) SGPU_CUDA(cudaMemsetAsync(d_total, 0, 8, st));
        return SGPU_OK;
    }
    size_t nb = ceil_div(n, (size_t)SCAN_TILE);
    DevBuf<uint64_t> sums;
    SGPU_TRY(sums.alloc(nb, st));
    scan_reduce_kernel<TIn><<<(unsigned)nb, SCAN_THREADS, 0, st>>>(d_in, n, sums.p);
    SGPU_LAUNCH(c);
    if (nb <= 16384) {
        scan_small_kernel<<<1, 1024, 0, st>>>(sums.p, nb, d_total);
        SGPU_LAUNCH(c);
    } else {
        SGPU_TRY(scan_impl<uint64_t>(c, sums.p, sums.p, nb, d_total));  // in place is safe: read-before-write per item
    }
    scan_down_kernel<TIn><<<(unsigned)nb, SCAN_THREADS, 0, st>>>(d_in, d_out, n, sums.p);
    SGPU_LAUNCH(c);
    SGPU_CUDA(cudaGetLastError());
    return SGPU_OK;
}

sgpu_status exclusive_scan_u32_to_u64(sgpu_ctx *c, const uint32_t *d_in, uint64_t *d_out, size_t n,
                                      uint64_t *d_total) {
    return scan_impl<uint32_t>(c, d_in, d_out, n, d_total);
}
sgpu_status exclusive_scan_u64(sgpu_ctx *c, const uint64_t *d_in, uint64_t *d_out, size_t n, uint64_t *d_total) {
    return scan_impl<uint64_t>(c, d_in, d_out, n, d_total);
}

sgpu_status read_u64s(sgpu_ctx *c, const void *d_src, uint64_t *h_dst, size_t count) {
    if (count > 64) return SGPU_ERR_INVALID_ARG;
    SGPU_CUDA(cudaMemcpyAsync(c->h_pinned, d_src, count * 8, cudaMemcpyDeviceToHost, c->stream));
    SGPU_CUDA(cudaStreamSynchronize(c->stream));
    memcpy(h_dst, c->h_pinned, count * 8);
    return SGPU_OK;
}

sgpu_status write_u64s(sgpu_ctx *c, void *d_dst, const uint64_t *h_src, size_t count) {
    if (count > 32) return SGPU_ERR_INVALID_ARG;
    memcpy(c->h_pinned + 32, h_src, count * 8);
    SGPU_CUDA(cudaMemcpyAsync(d_dst, c->h_pinned + 32, count * 8, cudaMemcpyHostToDevice, c->stream));
    return SGPU_OK;
}

// ------------------------------------------------------------------------------------
// '\n' index: tile counts -> exclusive scan -> positions
// ------------------------------------------------------------------------------------
constexpr int NL_THREADS = 256;
constexpr int NL_CHUNKS = 4;                          // 16-byte chunks per thread
constexpr int NL_TILE = NL_THREADS * NL_CHUNKS * 16;  // 16 KiB per block iteration

// chunk c of a tile is handled by thread (c % NL_THREADS) in round (c / NL_THREADS): coalesced
__device__ __forceinline__ uint32_t tile_chunk_mask(const uint8_t *buf, size_t n, size_t pos) {
    if (pos >= n) return 0;
    uint4 v = ld_nc_u4(buf + pos);
    uint32_t m = nl_mask16(v);
    size_t rem = n - pos;
    if (rem < 16) m &= (1u << rem) - 1u;
    return m;
}

__global__ void __launch_bounds__(NL_THREADS) nl_count_kernel(const uint8_t *buf, size_t n, uint32_t *tile_counts,
                                                               size_t n_tiles) {
    __shared__ uint64_t sm[40];
    for (size_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        size_t base = t * NL_TILE;
        uint32_t cnt = 0;
#pragma unroll
        for (int k = 0; k < NL_CHUNKS; k++)
            cnt += __popc(tile_chunk_mask(buf, n, base + ((size_t)k * NL_THREADS + threadIdx.x) * 16));
        uint64_t total;
        block_excl_scan(cnt, &total, sm);
        if (threadIdx.x == 0) tile_counts[t] = (uint32_t)total;
    }
}

__global__ void __launch_bounds__(NL_THREADS)
    nl_emit_kernel(const uint8_t *buf, size_t n, const uint64_t *tile_offsets, size_t n_tiles, uint64_t *nlpos) {
    __shared__ uint64_t sm[40];
    for (size_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        size_t base = t * NL_TILE;
        uint32_t m[NL_CHUNKS];
        uint64_t run = tile_offsets[t];
#pragma unroll
        for (int k = 0; k < NL_CHUNKS; k++) {
            size_t pos = base + ((size_t)k * NL_THREADS + threadIdx.x) * 16;
            m[k] = tile_chunk_mask(buf, n, pos);
            uint64_t total;
            uint64_t pre = block_excl_scan(__popc(m[k]), &total, sm);
            uint64_t o = run + pre;
            uint32_t mm = m[k];
            while (mm) {
                int b = __ffs(mm) - 1;
                mm &= mm - 1;
                nlpos[o++] = pos + b;
            }
            run += total;
        }
    }
}

__global__ void nl_sum_kernel(const uint32_t *tile_counts, size_t n_tiles, unsigned long long *total) {
    unsigned long long s = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_tiles; i += (size_t)gridDim.x * blockDim.x)
        s += tile_counts[i];
    for (int d = 16; d; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(total, s);
}

static unsigned nl_grid(sgpu_ctx *c, size_t n_tiles) {
    size_t g = (size_t)c->sm_count * 8;
    return (unsigned)(n_tiles < g ? (n_tiles ? n_tiles : 1) : g);
}

sgpu_status count_newlines(sgpu_ctx *c, const uint8_t *d_buf, size_t n, uint64_t *count) {
    *count = 0;
    if (n == 0) return SGPU_OK;
    if (((uintptr_t)d_buf & 15) != 0) return SGPU_ERR_INVALID_ARG;
    size_t n_tiles = ceil_div(n, (size_t)NL_TILE);
    DevBuf<uint32_t> counts;
    DevBuf<uint64_t> total;
    SGPU_TRY(counts.alloc(n_tiles, c->stream));
    SGPU_TRY(total.alloc(1, c->stream));
    SGPU_CUDA(cudaMemsetAsync(total.p, 0, 8, c->stream));
    nl_count_kernel<<<nl_grid(c, n_tiles), NL_THREADS, 0, c->stream>>>(d_buf, n, counts.p, n_tiles);
    SGPU_LAUNCH(c);
    nl_sum_kernel<<<(unsigned)(ceil_div(n_tiles, 256) < 1024 ? ceil_div(n_tiles, 256) : 1024), 256, 0, c->stream>>>(
        counts.p, n_tiles, (unsigned long long *)total.p);
    SGPU_LAUNCH(c);
    SGPU_CUDA(cudaGetLastError());
    return read_u64s(c, total.p, count, 1);
}

sgpu_status index_newlines(sgpu_ctx *c, const uint8_t *d_buf, size_t n, DevBuf<uint64_t> &nlpos,
                           uint64_t *n_newlines) {
    *n_newlines = 0;
    if (n == 0) return nlpos.alloc(1, c->stream);
    if (((uintptr_t)d_buf & 15) != 0) return SGPU_ERR_INVALID_ARG;
    cudaStream_t st = c->stream;
    size_t n_tiles = ceil_div(n, (size_t)NL_TILE);
    DevBuf<uint32_t> counts;
    DevBuf<uint64_t> offs, total;
    SGPU_TRY(counts.alloc(n_tiles, st));
    SGPU_TRY(offs.alloc(n_tiles, st));
    SGPU_TRY(total.alloc(1, st));
    nl_count_kernel<<<nl_grid(c, n_tiles), NL_THREADS, 0, st>>>(d_buf, n, counts.p, n_tiles);
    SGPU_LAUNCH(c);
    SGPU_TRY(exclusive_scan_u32_to_u64(c, counts.p, offs.p, n_tiles, total.p));
    SGPU_TRY(read_u64s(c, total.p, n_newlines, 1));
    SGPU_TRY(nlpos.alloc((size_t)*n_newlines + 1, st));
    nl_emit_kernel<<<nl_grid(c, n_tiles), NL_THREADS, 0, st>>>(d_buf, n, offs.p, n_tiles, nlpos.p);
    SGPU_LAUNCH(c);
    SGPU_CUDA(cudaGetLastError());
    return SGPU_OK;
}

}  // namespace sgpu
