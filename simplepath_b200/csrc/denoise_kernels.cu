// Denoising on the device (spcu_render_guides, spcu_denoise): the first-hit guide buffers of sample 0 and the variance-guided
// edge-avoiding à-trous filter over a frame's sums.  Compiled with --fmad=false and without fast-math (Makefile), and every
// operation of the filter is an explicitly rounded intrinsic with taps summed in a fixed order, so that a float32 numpy model
// (simplepath_b200/denoise.py) reproduces the output bit for bit.  The guide kernel walks the accelerators with the exact
// reference-order walks of trace.cuh, as the extend stage does with SPCU_TRAVERSAL_EXACT.
#include "kernels.h"
#include "pixel_stats.cuh"
#include "shade.cuh"
#include "trace.cuh"

namespace spcu {
namespace {

constexpr int kFilterBlock = 256;

// ---- guides ------------------------------------------------------------------------------------------------------------
// Albedo of a material: a clearcoat's base followed to its one-sample material, then the sum of its BxDFs in table order
// (a Lambert BxDF stores albedo / pi).
__device__ __forceinline__ float3 material_albedo(const DScene& s, uint32_t mat)
{
    for (uint32_t k = 0; k < SPCU_MAX_COAT_DEPTH && s.materials[mat].kind == SPCU_MAT_CLEARCOAT; ++k) {
        mat = s.materials[mat].base;
    }
    const spcu_material& m = s.materials[mat];
    float3               a = make_float3(0.0f, 0.0f, 0.0f);
    for (uint32_t i = 0; i < m.n_bxdfs; ++i) {
        const spcu_bxdf& b = s.bxdfs[m.first_bxdf + i];
        const float      f = b.kind == SPCU_BXDF_LAMBERT ? kPi : 1.0f;
        a.x                = __fadd_rn(a.x, __fmul_rn(b.r[0], f));
        a.y                = __fadd_rn(a.y, __fmul_rn(b.r[1], f));
        a.z                = __fadd_rn(a.z, __fmul_rn(b.r[2], f));
    }
    return a;
}

// One guide record per pixel from the camera ray of sample 0, with the extend stage's rule (Integrator.cpp:558-563):
// intersect_lights with the ray's limits, then intersect with t_max shrunk to the light's distance.
__global__ void __launch_bounds__(kTraceBlock) k_guides(const __grid_constant__ DScene s, spcu_guide* __restrict__ out)
{
    __shared__ int32_t stack[kStackShared * kTraceBlock];
    const uint32_t     n   = s.width * s.height;
    const uint32_t     pix = blockIdx.x * kTraceBlock + threadIdx.x;
    if (pix >= n) {
        return;
    }
    float4 o, d;
    camera_ray(s, pix, 0, o, d);
    const Ray        r{ o.x, o.y, o.z, d.x, d.y, d.z, o.w };
    float            t_max = d.w, beta, gamma;
    const LightPrims lp{ s.lights };
    const int32_t    li = closest_hit<false>(s.lights_accel, lp, r, t_max, beta, gamma, stack + threadIdx.x, nullptr);
    const float      light_t = t_max;
    const GeomPrims  gp{ s.geom_prims, s.geom_meta };
    const int32_t    id = closest_hit<false>(s.geom, gp, r, t_max, beta, gamma, stack + threadIdx.x, nullptr);

    spcu_guide g{};
    if (id >= 0) {
        const HitRec h{ id, t_max, beta, gamma };
        V3           point, nrm;
        uint32_t     mat;
        make_isect<FeatFull>(s, h, v3(o.x, o.y, o.z), v3(d.x, d.y, d.z), point, nrm, mat);
        nrm = normalize(nrm); // (the plane's normal is not normalised by make_isect)
        if (dot(nrm, v3(d.x, d.y, d.z)) > 0.0f) {
            nrm = v3(-nrm.x, -nrm.y, -nrm.z);
        }
        const float3 a = material_albedo(s, mat);
        g              = spcu_guide{ { nrm.x, nrm.y, nrm.z }, t_max, { a.x, a.y, a.z }, id };
    } else if (li >= 0) {
        g.depth = light_t;
        g.id    = -2 - li;
    } else {
        g.depth = light_t; // the ray's t_max
        g.id    = -1;
    }
    out[pix] = g;
}

// ---- filter ------------------------------------------------------------------------------------------------------------
// Per pixel between iterations: col = (mean r, g, b, luminance) and var = the variance of the mean luminance.  A pixel that
// is no tap (empty, or a non-finite sum) has var = -1 and keeps col (0, or sum / n) to the output.

__device__ __forceinline__ float lum(float r, float g, float b)
{
    return __fadd_rn(__fadd_rn(__fmul_rn(0.2126f, r), __fmul_rn(0.7152f, g)), __fmul_rn(0.0722f, b));
}

__global__ void __launch_bounds__(kFilterBlock) k_denoise_init(const float* __restrict__ rgb_sum, const float* __restrict__ lum_sumsq,
                                                               const uint32_t* __restrict__ spp_map, uint32_t spp, uint32_t n_pix,
                                                               float4* __restrict__ col, float* __restrict__ var)
{
    const uint32_t p = blockIdx.x * kFilterBlock + threadIdx.x;
    if (p >= n_pix) {
        return;
    }
    const uint32_t n = spp_map ? spp_map[p] : spp;
    if (n == 0) {
        col[p] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        var[p] = -1.0f;
        return;
    }
    const float nf = static_cast<float>(n);
    const float R = rgb_sum[3 * p + 0], G = rgb_sum[3 * p + 1], B = rgb_sum[3 * p + 2], Q = lum_sumsq[p];
    const float r = __fdiv_rn(R, nf), g = __fdiv_rn(G, nf), b = __fdiv_rn(B, nf);
    if (!(isfinite(R) && isfinite(G) && isfinite(B) && isfinite(Q))) {
        col[p] = make_float4(r, g, b, 0.0f);
        var[p] = -1.0f;
        return;
    }
    float m;
    col[p] = make_float4(r, g, b, lum(r, g, b));
    var[p] = n < 2 ? 0.0f : mean_lum_variance(R, G, B, Q, nf, m);
}

// Class of a guide: 0 geometry, 1 light, 2 miss.
__device__ __forceinline__ int guide_class(int32_t id) { return id >= 0 ? 0 : id == -1 ? 2 : 1; }

__device__ __forceinline__ float bspline(int d) { return d == 0 ? 0.375f : (d == 1 || d == -1) ? 0.25f : 0.0625f; }

// var~ of pixel (x, y): the 3x3 weighted mean of var over the neighbours that are taps, as (sum of w var, sum of w).
__device__ __forceinline__ void prefilter_sums(const float* __restrict__ var, int x, int y, uint32_t width, uint32_t height,
                                               float& pv, float& pw)
{
    pv = 0.0f;
    pw = 0.0f;
    for (int dy = -1; dy <= 1; ++dy) {
        for (int dx = -1; dx <= 1; ++dx) {
            const int qx = x + dx, qy = y + dy;
            if (qx < 0 || qy < 0 || qx >= static_cast<int>(width) || qy >= static_cast<int>(height)) continue;
            const float vq = var[qy * width + qx];
            if (!(vq >= 0.0f)) continue;
            const float w = __fmul_rn(dx == 0 ? 0.5f : 0.25f, dy == 0 ? 0.5f : 0.25f);
            pv            = __fadd_rn(pv, __fmul_rn(w, vq));
            pw            = __fadd_rn(pw, w);
        }
    }
}

// One iteration at step h: col/var in, col_out/var_out (or, for the last iteration, out[p*3+c]) written.
__global__ void __launch_bounds__(kFilterBlock) k_denoise_step(const spcu_guide* __restrict__ guides, const float4* __restrict__ col,
                                                               const float* __restrict__ var, uint32_t width, uint32_t height,
                                                               uint32_t h, float sigma_l, float sigma_z, float sigma_a,
                                                               float4* __restrict__ col_out, float* __restrict__ var_out,
                                                               float* __restrict__ out)
{
    const uint32_t p = blockIdx.x * kFilterBlock + threadIdx.x;
    if (p >= width * height) {
        return;
    }
    const int    x = static_cast<int>(p % width), y = static_cast<int>(p / width);
    const float4 cp = col[p];
    const float  vp = var[p];
    float4       res = cp;
    float        res_var = vp;
    if (vp >= 0.0f) {
        float pv, pw;
        prefilter_sums(var, x, y, width, height, pv, pw);
        const float       l_den = __fadd_rn(__fmul_rn(sigma_l, __fsqrt_rn(__fdiv_rn(pv, pw))), 1e-4f);
        const spcu_guide  gp    = guides[p];
        const int         cls_p = guide_class(gp.id);
        float             sr = 0.0f, sg = 0.0f, sb = 0.0f, sw = 0.0f, sv = 0.0f;
        for (int dy = -2; dy <= 2; ++dy) {
            const int qy = y + dy * static_cast<int>(h);
            if (qy < 0 || qy >= static_cast<int>(height)) continue;
            for (int dx = -2; dx <= 2; ++dx) {
                const int qx = x + dx * static_cast<int>(h);
                if (qx < 0 || qx >= static_cast<int>(width)) continue;
                const uint32_t q  = static_cast<uint32_t>(qy) * width + static_cast<uint32_t>(qx);
                const float    vq = var[q];
                if (!(vq >= 0.0f)) continue;
                const float4 cq = col[q];
                const float  k  = __fmul_rn(bspline(dx), bspline(dy));
                float        w  = k;
                if (dx != 0 || dy != 0) {
                    const spcu_guide gq = guides[q];
                    if (guide_class(gq.id) != cls_p) {
                        w = 0.0f;
                    } else {
                        float wn = 1.0f, az = 0.0f, aa = 0.0f;
                        if (cls_p == 0) {
                            const float dn = __fadd_rn(__fadd_rn(__fmul_rn(gp.normal[0], gq.normal[0]), __fmul_rn(gp.normal[1], gq.normal[1])),
                                                       __fmul_rn(gp.normal[2], gq.normal[2]));
                            wn = fmaxf(0.0f, dn);
#pragma unroll
                            for (int i = 0; i < 7; ++i) wn = __fmul_rn(wn, wn); // ^128
                            const int   m   = max(abs(dx), abs(dy));
                            const float dzn = __fmul_rn(__fmul_rn(sigma_z, gp.depth), static_cast<float>(static_cast<int>(h) * m));
                            az              = __fdiv_rn(fabsf(__fsub_rn(gp.depth, gq.depth)), dzn);
                            const float da  = fmaxf(fmaxf(fabsf(__fsub_rn(gp.albedo[0], gq.albedo[0])), fabsf(__fsub_rn(gp.albedo[1], gq.albedo[1]))),
                                                    fabsf(__fsub_rn(gp.albedo[2], gq.albedo[2])));
                            aa              = __fdiv_rn(da, sigma_a);
                        }
                        const float al  = __fdiv_rn(fabsf(__fsub_rn(cp.w, cq.w)), l_den);
                        const float den = __fadd_rn(__fadd_rn(__fadd_rn(1.0f, __fmul_rn(al, al)), __fmul_rn(az, az)), __fmul_rn(aa, aa));
                        w               = __fdiv_rn(__fmul_rn(k, wn), den);
                    }
                }
                sr = __fadd_rn(sr, __fmul_rn(w, cq.x));
                sg = __fadd_rn(sg, __fmul_rn(w, cq.y));
                sb = __fadd_rn(sb, __fmul_rn(w, cq.z));
                sw = __fadd_rn(sw, w);
                sv = __fadd_rn(sv, __fmul_rn(__fmul_rn(w, w), vq));
            }
        }
        const float r = __fdiv_rn(sr, sw), g = __fdiv_rn(sg, sw), b = __fdiv_rn(sb, sw);
        res     = make_float4(r, g, b, lum(r, g, b));
        res_var = __fdiv_rn(sv, __fmul_rn(sw, sw));
    }
    if (out) {
        out[3 * p + 0] = res.x;
        out[3 * p + 1] = res.y;
        out[3 * p + 2] = res.z;
    } else {
        col_out[p] = res;
        var_out[p] = res_var;
    }
}

// ---- energy-conserving (flux) form: spcu_denoise_conserving ------------------------------------------------------------------
// Three passes per iteration: var~ (k_denoise_prefilter), the weight sums W (k_denoise_wsum) and the exchange of colour
// (k_denoise_flux).  pair_weight is symmetric in its two pixels operand by operand (products, sums, min, max and |a - b|), so
// w_pq from p's pass and w_qp from q's have the same bits, and so do alpha_pq = w_pq / max(W_p, W_q) and alpha_qp.

__global__ void __launch_bounds__(kFilterBlock) k_denoise_prefilter(const float* __restrict__ var, uint32_t width, uint32_t height,
                                                                    float* __restrict__ var_pf)
{
    const uint32_t p = blockIdx.x * kFilterBlock + threadIdx.x;
    if (p >= width * height || !(var[p] >= 0.0f)) {
        return;
    }
    float pv, pw;
    prefilter_sums(var, static_cast<int>(p % width), static_cast<int>(p / width), width, height, pv, pw);
    var_pf[p] = __fdiv_rn(pv, pw);
}

// w_pq of two taps p != q at offset h (dx, dy), k = b[dx] b[dy], hm = h max(|dx|, |dy|); lp, lq luminances, vp, vq their var~.
__device__ __forceinline__ float pair_weight(const spcu_guide& gp, const spcu_guide& gq, float lp, float lq, float vp, float vq, float k,
                                             int hm, float sigma_l, float sigma_z, float sigma_a)
{
    const int cls = guide_class(gp.id);
    if (guide_class(gq.id) != cls) {
        return 0.0f;
    }
    float wn = 1.0f, az = 0.0f, aa = 0.0f;
    if (cls == 0) {
        const float dn = __fadd_rn(__fadd_rn(__fmul_rn(gp.normal[0], gq.normal[0]), __fmul_rn(gp.normal[1], gq.normal[1])),
                                   __fmul_rn(gp.normal[2], gq.normal[2]));
        wn             = fmaxf(0.0f, dn);
#pragma unroll
        for (int i = 0; i < 7; ++i) wn = __fmul_rn(wn, wn); // ^128
        const float dzn = __fmul_rn(__fmul_rn(sigma_z, fminf(gp.depth, gq.depth)), static_cast<float>(hm));
        az              = __fdiv_rn(fabsf(__fsub_rn(gp.depth, gq.depth)), dzn);
        const float da  = fmaxf(fmaxf(fabsf(__fsub_rn(gp.albedo[0], gq.albedo[0])), fabsf(__fsub_rn(gp.albedo[1], gq.albedo[1]))),
                                fabsf(__fsub_rn(gp.albedo[2], gq.albedo[2])));
        aa              = __fdiv_rn(da, sigma_a);
    }
    const float l_den = __fadd_rn(__fmul_rn(sigma_l, __fsqrt_rn(fmaxf(vp, vq))), 1e-4f);
    const float al    = __fdiv_rn(fabsf(__fsub_rn(lp, lq)), l_den);
    const float den   = __fadd_rn(__fadd_rn(__fadd_rn(1.0f, __fmul_rn(al, al)), __fmul_rn(az, az)), __fmul_rn(aa, aa));
    return __fdiv_rn(__fmul_rn(k, wn), den);
}

// W_p: over the taps in row-major order, the centre's k = 9/64 and every other tap's w_pq.  Written for taps only.
__global__ void __launch_bounds__(kFilterBlock) k_denoise_wsum(const spcu_guide* __restrict__ guides, const float4* __restrict__ col,
                                                               const float* __restrict__ var, const float* __restrict__ var_pf,
                                                               uint32_t width, uint32_t height, uint32_t h, float sigma_l,
                                                               float sigma_z, float sigma_a, float* __restrict__ wsum)
{
    const uint32_t p = blockIdx.x * kFilterBlock + threadIdx.x;
    if (p >= width * height || !(var[p] >= 0.0f)) {
        return;
    }
    const int        x = static_cast<int>(p % width), y = static_cast<int>(p / width);
    const float      lp = col[p].w, vp = var_pf[p];
    const spcu_guide gp = guides[p];
    float            sw = 0.0f;
    for (int dy = -2; dy <= 2; ++dy) {
        const int qy = y + dy * static_cast<int>(h);
        if (qy < 0 || qy >= static_cast<int>(height)) continue;
        for (int dx = -2; dx <= 2; ++dx) {
            const int qx = x + dx * static_cast<int>(h);
            if (qx < 0 || qx >= static_cast<int>(width)) continue;
            const uint32_t q = static_cast<uint32_t>(qy) * width + static_cast<uint32_t>(qx);
            if (!(var[q] >= 0.0f)) continue;
            const float k = __fmul_rn(bspline(dx), bspline(dy));
            sw            = __fadd_rn(sw, (dx == 0 && dy == 0) ? k
                                                              : pair_weight(gp, guides[q], lp, col[q].w, vp, var_pf[q], k,
                                                                            static_cast<int>(h) * max(abs(dx), abs(dy)), sigma_l,
                                                                            sigma_z, sigma_a));
        }
    }
    wsum[p] = sw;
}

// One iteration of the flux form at step h: col/var in, col_out/var_out (or, for the last iteration, out[p*3+c]) written.
__global__ void __launch_bounds__(kFilterBlock) k_denoise_flux(const spcu_guide* __restrict__ guides, const float4* __restrict__ col,
                                                               const float* __restrict__ var, const float* __restrict__ var_pf,
                                                               const float* __restrict__ wsum, uint32_t width, uint32_t height,
                                                               uint32_t h, float sigma_l, float sigma_z, float sigma_a,
                                                               float4* __restrict__ col_out, float* __restrict__ var_out,
                                                               float* __restrict__ out)
{
    const uint32_t p = blockIdx.x * kFilterBlock + threadIdx.x;
    if (p >= width * height) {
        return;
    }
    const float4 cp = col[p];
    const float  vp = var[p];
    float4       res = cp;
    float        res_var = vp;
    if (vp >= 0.0f) {
        const int        x = static_cast<int>(p % width), y = static_cast<int>(p / width);
        const float      pf_p = var_pf[p], wp = wsum[p];
        const spcu_guide gp   = guides[p];
        float            sr = 0.0f, sg = 0.0f, sb = 0.0f, sa = 0.0f, sv = 0.0f;
        for (int dy = -2; dy <= 2; ++dy) {
            const int qy = y + dy * static_cast<int>(h);
            if (qy < 0 || qy >= static_cast<int>(height)) continue;
            for (int dx = -2; dx <= 2; ++dx) {
                const int qx = x + dx * static_cast<int>(h);
                if (qx < 0 || qx >= static_cast<int>(width) || (dx == 0 && dy == 0)) continue;
                const uint32_t q  = static_cast<uint32_t>(qy) * width + static_cast<uint32_t>(qx);
                const float    vq = var[q];
                if (!(vq >= 0.0f)) continue;
                const float4 cq = col[q];
                const float  w  = pair_weight(gp, guides[q], cp.w, cq.w, pf_p, var_pf[q], __fmul_rn(bspline(dx), bspline(dy)),
                                              static_cast<int>(h) * max(abs(dx), abs(dy)), sigma_l, sigma_z, sigma_a);
                const float  a  = __fdiv_rn(w, fmaxf(wp, wsum[q]));
                sr              = __fadd_rn(sr, __fmul_rn(a, __fsub_rn(cq.x, cp.x)));
                sg              = __fadd_rn(sg, __fmul_rn(a, __fsub_rn(cq.y, cp.y)));
                sb              = __fadd_rn(sb, __fmul_rn(a, __fsub_rn(cq.z, cp.z)));
                sa              = __fadd_rn(sa, a);
                sv              = __fadd_rn(sv, __fmul_rn(__fmul_rn(a, a), vq));
            }
        }
        const float r = __fadd_rn(cp.x, sr), g = __fadd_rn(cp.y, sg), b = __fadd_rn(cp.z, sb), a0 = __fsub_rn(1.0f, sa);
        res     = make_float4(r, g, b, lum(r, g, b));
        res_var = __fadd_rn(__fmul_rn(__fmul_rn(a0, a0), vp), sv);
    }
    if (out) {
        out[3 * p + 0] = res.x;
        out[3 * p + 1] = res.y;
        out[3 * p + 2] = res.z;
    } else {
        col_out[p] = res;
        var_out[p] = res_var;
    }
}

} // namespace

cudaError_t launch_guides(const DScene& s, spcu_guide* d_out, cudaStream_t st)
{
    const uint32_t n = s.width * s.height;
    if (n == 0) {
        return cudaSuccess;
    }
    k_guides<<<(n + kTraceBlock - 1) / kTraceBlock, kTraceBlock, 0, st>>>(s, d_out);
    return cudaGetLastError();
}

cudaError_t launch_denoise(const spcu_guide* d_guides, const float* d_rgb_sum, const float* d_lum_sumsq, const uint32_t* d_spp_map,
                           uint32_t spp, uint32_t width, uint32_t height, const spcu_denoise_params& p, float4* d_col[2],
                           float* d_var[2], float* d_out, cudaStream_t st)
{
    const uint32_t n = width * height;
    if (n == 0) {
        return cudaSuccess;
    }
    const unsigned grid = (n + kFilterBlock - 1) / kFilterBlock;
    k_denoise_init<<<grid, kFilterBlock, 0, st>>>(d_rgb_sum, d_lum_sumsq, d_spp_map, spp, n, d_col[0], d_var[0]);
    for (uint32_t i = 0; i < p.iterations; ++i) {
        const bool last = i + 1 == p.iterations;
        k_denoise_step<<<grid, kFilterBlock, 0, st>>>(d_guides, d_col[i & 1u], d_var[i & 1u], width, height, 1u << i, p.sigma_l,
                                                      p.sigma_z, p.sigma_a, d_col[(i + 1) & 1u], d_var[(i + 1) & 1u],
                                                      last ? d_out : nullptr);
    }
    return cudaGetLastError();
}

cudaError_t launch_denoise_conserving(const spcu_guide* d_guides, const float* d_rgb_sum, const float* d_lum_sumsq,
                                      const uint32_t* d_spp_map, uint32_t spp, uint32_t width, uint32_t height,
                                      const spcu_denoise_params& p, float4* d_col[2], float* d_var[2], float* d_var_pf, float* d_wsum,
                                      float* d_out, cudaStream_t st)
{
    const uint32_t n = width * height;
    if (n == 0) {
        return cudaSuccess;
    }
    const unsigned grid = (n + kFilterBlock - 1) / kFilterBlock;
    k_denoise_init<<<grid, kFilterBlock, 0, st>>>(d_rgb_sum, d_lum_sumsq, d_spp_map, spp, n, d_col[0], d_var[0]);
    for (uint32_t i = 0; i < p.iterations; ++i) {
        const bool     last = i + 1 == p.iterations;
        const uint32_t in = i & 1u, nx = (i + 1) & 1u, h = 1u << i;
        k_denoise_prefilter<<<grid, kFilterBlock, 0, st>>>(d_var[in], width, height, d_var_pf);
        k_denoise_wsum<<<grid, kFilterBlock, 0, st>>>(d_guides, d_col[in], d_var[in], d_var_pf, width, height, h, p.sigma_l, p.sigma_z,
                                                      p.sigma_a, d_wsum);
        k_denoise_flux<<<grid, kFilterBlock, 0, st>>>(d_guides, d_col[in], d_var[in], d_var_pf, d_wsum, width, height, h, p.sigma_l,
                                                      p.sigma_z, p.sigma_a, d_col[nx], d_var[nx], last ? d_out : nullptr);
    }
    return cudaGetLastError();
}

} // namespace spcu
