// Output side on the device: the per-pixel mean, write_pfm's row order and write_ppm's sRGB quantisation
// (reference main.cpp:100-102, Image/Image.cpp:14-55, Image/Image.h:38-50).  Compiled without fast-math (Makefile): the mean
// is an IEEE division, the sRGB curve uses powf.
#include "ctx.h"

using namespace spcu;

namespace {

// rgb_to_srgb (Image/Image.h:38-45)
__device__ __forceinline__ float to_srgb(float u)
{
    if (u <= 0.0031308f) {
        return __fmul_rn(12.92f, u);
    }
    return __fsub_rn(__fmul_rn(1.055f, powf(u, 1.0f / 2.4f)), 0.055f);
}

__device__ __forceinline__ uint16_t quantise(float c)
{
    const int v = static_cast<int>(__fmul_rn(255.99f, c)); // write_ppm (Image/Image.cpp:22-24)
    return static_cast<uint16_t>(min(max(v, 0), 65535));
}

// One thread per output pixel; output row r holds image row h-1-r (write_ppm / write_pfm iterate j = ny-1 .. 0).
// counts (may be NULL): per-pixel sample counts that replace the uniform `spp` (adaptive sampling); a pixel with 0 samples
// packs as 0.
__global__ void __launch_bounds__(256) k_pack_image(const float* __restrict__ rgb_sum, const uint32_t* __restrict__ counts, uint32_t w,
                                                    uint32_t h, float spp, uint32_t format, float* __restrict__ out_pfm,
                                                    uint16_t* __restrict__ out_ppm)
{
    const size_t n      = static_cast<size_t>(w) * h;
    const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
    for (size_t o = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; o < n; o += stride) {
        const uint32_t r = static_cast<uint32_t>(o / w), x = static_cast<uint32_t>(o - static_cast<size_t>(r) * w);
        const size_t   p = static_cast<size_t>(h - 1 - r) * w + x;
        const size_t   i = p * 3;
        // image(p.x, p.y) /= num_pixel_samples (main.cpp:102; RGB::operator/=(float), math/RGB.h:126-132)
        float m[3] = { 0.0f, 0.0f, 0.0f };
        const float div = counts ? static_cast<float>(counts[p]) : spp;
        if (div != 0.0f) {
            m[0] = __fdiv_rn(rgb_sum[i], div), m[1] = __fdiv_rn(rgb_sum[i + 1], div), m[2] = __fdiv_rn(rgb_sum[i + 2], div);
        }
        if (format == SPCU_IMAGE_PFM) {
            out_pfm[3 * o] = m[0], out_pfm[3 * o + 1] = m[1], out_pfm[3 * o + 2] = m[2];
        } else {
            out_ppm[3 * o] = quantise(to_srgb(m[0])), out_ppm[3 * o + 1] = quantise(to_srgb(m[1])), out_ppm[3 * o + 2] = quantise(to_srgb(m[2]));
        }
    }
}

size_t packed_bytes(size_t n_pixels, uint32_t format)
{
    return n_pixels * 3 * (format == SPCU_IMAGE_PFM ? sizeof(float) : sizeof(uint16_t));
}

} // namespace

// d_rgb_sum: device sums; d_counts (may be NULL): per-pixel divisors in place of spp.  Packs into c->packed and copies the
// result to the host buffer `out`.
int spcu::pack_device_image(spcu_ctx* c, const float* d_rgb_sum, const uint32_t* d_counts, uint32_t w, uint32_t h, uint32_t spp,
                            uint32_t format, void* out)
{
    if (format > SPCU_IMAGE_PPM) {
        return fail(c, SPCU_ERR_INVALID, "unknown image format %u", format);
    }
    if (!out || (spp == 0 && !d_counts) || w == 0 || h == 0) {
        return fail(c, SPCU_ERR_INVALID, "pack image: NULL output, empty image or zero samples");
    }
    const size_t n     = static_cast<size_t>(w) * h;
    const size_t bytes = packed_bytes(n, format);
    CK(c, c->packed.reserve(bytes));
    const unsigned grid = static_cast<unsigned>(std::min<size_t>((n + 255) / 256, static_cast<size_t>(c->sm_count) * 8));
    k_pack_image<<<grid, 256, 0, c->stream>>>(d_rgb_sum, d_counts, w, h, static_cast<float>(spp), format, c->packed.as<float>(),
                                              c->packed.as<uint16_t>());
    CK(c, cudaGetLastError());
    CK(c, cudaMemcpyAsync(out, c->packed.p, bytes, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return SPCU_OK;
}

extern "C" int spcu_pack_image(spcu_ctx* c, const float* rgb_sum, uint32_t width, uint32_t height, uint32_t spp, uint32_t format,
                               void* out)
{
    if (!c) {
        return SPCU_ERR_INVALID;
    }
    if (!rgb_sum) {
        return fail(c, SPCU_ERR_INVALID, "rgb_sum is NULL");
    }
    CK(c, cudaSetDevice(c->device));
    const size_t bytes = static_cast<size_t>(width) * height * 3 * sizeof(float);
    CK(c, c->host_rgb.reserve(std::max<size_t>(bytes, 16)));
    CK(c, cudaMemcpyAsync(c->host_rgb.p, rgb_sum, bytes, cudaMemcpyHostToDevice, c->stream));
    return pack_device_image(c, c->host_rgb.as<float>(), nullptr, width, height, spp, format, out);
}

extern "C" int spcu_pack_image_counts(spcu_ctx* c, const float* rgb_sum, const uint32_t* spp_map, uint32_t width, uint32_t height,
                                      uint32_t format, void* out)
{
    if (!c) {
        return SPCU_ERR_INVALID;
    }
    if (!rgb_sum || !spp_map) {
        return fail(c, SPCU_ERR_INVALID, "rgb_sum or spp_map is NULL");
    }
    CK(c, cudaSetDevice(c->device));
    const size_t n = static_cast<size_t>(width) * height;
    CK(c, c->host_rgb.reserve(std::max<size_t>(n * 3 * sizeof(float), 16)));
    CK(c, c->ad_spp_map.reserve(std::max<size_t>(n * sizeof(uint32_t), 16)));
    CK(c, cudaMemcpyAsync(c->host_rgb.p, rgb_sum, n * 3 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemcpyAsync(c->ad_spp_map.p, spp_map, n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    return pack_device_image(c, c->host_rgb.as<float>(), c->ad_spp_map.as<uint32_t>(), width, height, 0, format, out);
}
