// Adaptive sampling on the device (spcu_render_adaptive): the per-pixel stopping test at a pass boundary, the neighbourhood
// rule over it (radius > 0), and the stable compaction of the pixels that go on into the next pass's pixel list.  Compiled
// with --fmad=false and without fast-math (Makefile), and every operation of the test is an explicitly rounded intrinsic, so
// that a float32 numpy model (simplepath_b200/adaptive.py) reproduces every decision bit for bit.
#include "ctx.h"
#include "pixel_stats.cuh"

using namespace spcu;

namespace {

constexpr int kBlock = 256; // list entries per CTA of the decide / scatter kernels (8 warps)
constexpr int kScan  = 1024;

// The stopping test of one pixel after n samples: squared standard error of the mean luminance against
// (rel_error * (mean + abs_floor))^2.  Non-finite sums never stop.
__device__ __forceinline__ bool converged(const float* __restrict__ rgb_sum, const float* __restrict__ lum_sumsq, uint32_t pix,
                                          float nf, float rel_error, float abs_floor)
{
    const float R = rgb_sum[3 * pix + 0], G = rgb_sum[3 * pix + 1], B = rgb_sum[3 * pix + 2], Q = lum_sumsq[pix];
    float       m;
    const float se2 = mean_lum_variance(R, G, B, Q, nf, m);
    const float t   = __fmul_rn(rel_error, __fadd_rn(m, abs_floor));
    return isfinite(R) && isfinite(G) && isfinite(B) && isfinite(Q) && se2 <= __fmul_rn(t, t);
}

// block_count[blockIdx.x] = how many of the block's threads have `more` set (every thread of the block calls this).
__device__ __forceinline__ void count_kept(bool more, uint32_t* __restrict__ block_count)
{
    __shared__ uint32_t warp_count[kBlock / 32];
    const unsigned m = __ballot_sync(0xffffffffu, more);
    if ((threadIdx.x & 31) == 0) {
        warp_count[threadIdx.x >> 5] = __popc(m);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t s = 0;
        for (int w = 0; w < kBlock / 32; ++w) s += warp_count[w];
        block_count[blockIdx.x] = s;
    }
}

// Entries [0, n) of `list`, one thread each: a pixel that passes the test gets spp_map[pix] = n_samples; keep[i] = 1 for the
// others.  block_count[b] = how many of block b's entries go on.
__global__ void __launch_bounds__(kBlock) k_adaptive_decide(const uint32_t* __restrict__ list, uint32_t n, const float* __restrict__ rgb_sum,
                                                            const float* __restrict__ lum_sumsq, uint32_t n_samples, float rel_error,
                                                            float abs_floor, uint32_t* __restrict__ spp_map, uint8_t* __restrict__ keep,
                                                            uint32_t* __restrict__ block_count)
{
    const uint32_t i    = blockIdx.x * kBlock + threadIdx.x;
    bool           more = false;
    if (i < n) {
        const uint32_t pix = list[i];
        more               = !converged(rgb_sum, lum_sumsq, pix, static_cast<float>(n_samples), rel_error, abs_floor);
        if (!more) {
            spp_map[pix] = n_samples;
        }
        keep[i] = more ? 1u : 0u;
    }
    count_kept(more, block_count);
}

// ---- the neighbourhood test (radius > 0) -------------------------------------------------------------------------------------
// pass_mask holds one word per 8x8 tile (t = ty * tiles_x + tx); bit (y & 7) * 8 + (x & 7) is the pass flag of pixel (x, y).
// The whole buffer is set to all-ones at the start of a call, so pixels that stopped earlier, pixels of other partitions
// and positions outside the image read as passing.

// Entries [0, n) of `list`: each active pixel's bit = the stopping test of its own sums after n_samples samples.
__global__ void __launch_bounds__(kBlock) k_adaptive_test(const uint32_t* __restrict__ list, uint32_t n, const float* __restrict__ rgb_sum,
                                                          const float* __restrict__ lum_sumsq, uint32_t n_samples, float rel_error,
                                                          float abs_floor, uint32_t width, unsigned long long* __restrict__ pass_mask)
{
    const uint32_t i = blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) {
        return;
    }
    const uint32_t           pix = list[i];
    const uint32_t           x = pix % width, y = pix / width;
    unsigned long long*      word = pass_mask + (y >> 3) * ((width + 7) >> 3) + (x >> 3);
    const unsigned long long bit  = 1ull << ((y & 7u) * 8u + (x & 7u));
    if (converged(rgb_sum, lum_sumsq, pix, static_cast<float>(n_samples), rel_error, abs_floor)) {
        atomicOr(word, bit);
    } else {
        atomicAnd(word, ~bit);
    }
}

// The window of pixel (x, y) as a mask of its tile's word: |dx|, |dy| <= radius, clipped to the tile and to the image.
__device__ __forceinline__ unsigned long long window_mask(uint32_t x, uint32_t y, uint32_t width, uint32_t height, uint32_t radius)
{
    const uint32_t lx = x & 7u, ly = y & 7u;
    const uint32_t x0 = lx > radius ? lx - radius : 0u, x1 = min(min(lx + radius, 7u), lx + (width - 1u - x));
    const uint32_t y0 = ly > radius ? ly - radius : 0u, y1 = min(min(ly + radius, 7u), ly + (height - 1u - y));
    const unsigned long long row  = ((1ull << (x1 - x0 + 1u)) - 1ull) << x0;                                    // bits x0..x1
    const unsigned long long rows = ((~0ull >> (8u * (7u - (y1 - y0)))) << (8u * y0)) & 0x0101010101010101ull; // bit 0 of rows y0..y1
    return rows * row; // row < 256: no carry between bytes
}

// k_adaptive_decide with the neighbourhood rule: the pixel stops iff every pass flag of its window is set.
__global__ void __launch_bounds__(kBlock) k_adaptive_decide_window(const uint32_t* __restrict__ list, uint32_t n, uint32_t width,
                                                                   uint32_t height, uint32_t radius,
                                                                   const unsigned long long* __restrict__ pass_mask, uint32_t n_samples,
                                                                   uint32_t* __restrict__ spp_map, uint8_t* __restrict__ keep,
                                                                   uint32_t* __restrict__ block_count)
{
    const uint32_t i    = blockIdx.x * kBlock + threadIdx.x;
    bool           more = false;
    if (i < n) {
        const uint32_t           pix = list[i];
        const uint32_t           x = pix % width, y = pix / width;
        const unsigned long long win  = window_mask(x, y, width, height, radius);
        const unsigned long long word = pass_mask[(y >> 3) * ((width + 7) >> 3) + (x >> 3)];
        more                          = (word & win) != win;
        if (!more) {
            spp_map[pix] = n_samples;
        }
        keep[i] = more ? 1u : 0u;
    }
    count_kept(more, block_count);
}

// Exclusive scan of the n_blocks block counts, in place, by one CTA: thread t sums a contiguous run of counts, the runs'
// totals are scanned in shared memory, then each run is rewritten as offsets.  *d_total = the number of entries kept.
__global__ void __launch_bounds__(kScan) k_adaptive_scan(uint32_t* __restrict__ block_count, uint32_t n_blocks, uint32_t* __restrict__ d_total)
{
    __shared__ uint32_t run[kScan];
    const uint32_t per = (n_blocks + kScan - 1) / kScan;
    const uint32_t lo = min(threadIdx.x * per, n_blocks), hi = min(lo + per, n_blocks);
    uint32_t       s = 0;
    for (uint32_t b = lo; b < hi; ++b) s += block_count[b];
    run[threadIdx.x] = s;
    __syncthreads();
    for (uint32_t off = 1; off < kScan; off <<= 1) { // Hillis-Steele inclusive scan of the run totals
        const uint32_t add = threadIdx.x >= off ? run[threadIdx.x - off] : 0u;
        __syncthreads();
        run[threadIdx.x] += add;
        __syncthreads();
    }
    uint32_t base = run[threadIdx.x] - s;
    for (uint32_t b = lo; b < hi; ++b) {
        const uint32_t cnt = block_count[b];
        block_count[b]     = base;
        base += cnt;
    }
    if (threadIdx.x == kScan - 1) {
        *d_total = run[kScan - 1];
    }
}

// Kept entries of `list` to out[block offset + rank within the block]: the order of the list (tiles, Morton order inside a
// tile) is preserved.
__global__ void __launch_bounds__(kBlock) k_adaptive_scatter(const uint32_t* __restrict__ list, uint32_t n, const uint8_t* __restrict__ keep,
                                                             const uint32_t* __restrict__ block_offset, uint32_t* __restrict__ out)
{
    __shared__ uint32_t warp_base[kBlock / 32];
    const uint32_t i    = blockIdx.x * kBlock + threadIdx.x;
    const bool     more = i < n && keep[i];
    const unsigned m    = __ballot_sync(0xffffffffu, more);
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        warp_base[warp] = __popc(m);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t s = block_offset[blockIdx.x];
        for (int w = 0; w < kBlock / 32; ++w) {
            const uint32_t c = warp_base[w];
            warp_base[w]     = s;
            s += c;
        }
    }
    __syncthreads();
    if (more) {
        out[warp_base[warp] + __popc(m & ((1u << lane) - 1u))] = list[i];
    }
}

__global__ void __launch_bounds__(kBlock) k_adaptive_fill(const uint32_t* __restrict__ list, uint32_t n, uint32_t value,
                                                          uint32_t* __restrict__ spp_map)
{
    const uint32_t i = blockIdx.x * kBlock + threadIdx.x;
    if (i < n) {
        spp_map[list[i]] = value;
    }
}

} // namespace

size_t spcu::adaptive_scratch_bytes(uint32_t n)
{
    const size_t n_blocks = (static_cast<size_t>(n) + kBlock - 1) / kBlock;
    return (n_blocks + 1) * sizeof(uint32_t) + ((static_cast<size_t>(n) + 3) & ~size_t(3));
}

size_t spcu::adaptive_mask_bytes(uint32_t width, uint32_t height)
{
    return static_cast<size_t>((width + 7) / 8) * ((height + 7) / 8) * sizeof(unsigned long long);
}

cudaError_t spcu::launch_adaptive_compact(const uint32_t* d_list, uint32_t n, const float* d_rgb_sum, const float* d_lum_sumsq,
                                          uint32_t n_samples, float rel_error, float abs_floor, uint32_t width, uint32_t height,
                                          uint32_t radius, unsigned long long* d_pass_mask, uint32_t* d_spp_map,
                                          uint32_t* d_next_list, void* d_scratch, uint32_t* d_n_next, cudaStream_t st)
{
    if (n == 0) {
        return cudaMemsetAsync(d_n_next, 0, sizeof(uint32_t), st);
    }
    const uint32_t n_blocks    = (n + kBlock - 1) / kBlock;
    auto*          block_count = static_cast<uint32_t*>(d_scratch);
    auto*          keep        = reinterpret_cast<uint8_t*>(block_count + n_blocks + 1);
    if (radius == 0) {
        k_adaptive_decide<<<n_blocks, kBlock, 0, st>>>(d_list, n, d_rgb_sum, d_lum_sumsq, n_samples, rel_error, abs_floor, d_spp_map,
                                                       keep, block_count);
    } else { // every pass flag is written before any decision reads one
        k_adaptive_test<<<n_blocks, kBlock, 0, st>>>(d_list, n, d_rgb_sum, d_lum_sumsq, n_samples, rel_error, abs_floor, width,
                                                     d_pass_mask);
        k_adaptive_decide_window<<<n_blocks, kBlock, 0, st>>>(d_list, n, width, height, radius, d_pass_mask, n_samples, d_spp_map,
                                                              keep, block_count);
    }
    k_adaptive_scan<<<1, kScan, 0, st>>>(block_count, n_blocks, d_n_next);
    k_adaptive_scatter<<<n_blocks, kBlock, 0, st>>>(d_list, n, keep, block_count, d_next_list);
    return cudaGetLastError();
}

cudaError_t spcu::launch_adaptive_fill(const uint32_t* d_list, uint32_t n, uint32_t value, uint32_t* d_spp_map, cudaStream_t st)
{
    if (n == 0) {
        return cudaSuccess;
    }
    k_adaptive_fill<<<(n + kBlock - 1) / kBlock, kBlock, 0, st>>>(d_list, n, value, d_spp_map);
    return cudaGetLastError();
}
