/*
 * spcu.h — C-ABI of the B200 path-tracing backend for SimplePath ("CudaIntegrator").
 *
 * This is the drop-in boundary: plain C structs, pointers and sizes; no C++ / torch types.
 * The host side (simplepath_b200/host/, C++ against the reference's own headers) flattens an
 * `sp::Scene` (reference base/Scene.h:47-106) into `spcu_flat_scene` and calls these entry points
 * from `sp::CudaIntegrator`, the new subclass of `sp::Integrator`
 * (reference Integrators/Integrator.h:32-52).  Every entry point cites what it replaces.
 *
 * Conventions
 *  - all functions return SPCU_OK (0) or a negative error code; spcu_last_error() gives text.
 *  - "host" pointers are ordinary CPU memory; "device" pointers live on the context's GPU.
 *  - IDs are *reference order* IDs: geometry prims = the top-level unbounded list of
 *    Scene::m_accelerator_geometry in list order, followed by the BVH leaves' primitives in the
 *    reference's left-to-right depth-first order (shapes/BVHAccelerator.h:62-77,
 *    shapes/ListAccelerator.h:50-62).  Lights likewise over Scene::m_accelerator_lights.
 */
#ifndef SPCU_H
#define SPCU_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPCU_ABI_VERSION 2

/* ---- error codes ------------------------------------------------------------------------- */
#define SPCU_OK 0
#define SPCU_ERR_INVALID (-1)   /* bad argument / malformed scene                              */
#define SPCU_ERR_CUDA (-2)      /* CUDA runtime error (no CPU fallback exists)                 */
#define SPCU_ERR_NO_SCENE (-3)  /* call needs spcu_upload_scene first                          */
#define SPCU_ERR_LIMIT (-4)     /* scene exceeds a compiled-in limit (stack depth, bxdfs, ...) */
#define SPCU_ERR_INTERNAL (-5)  /* a kernel's bounded wait / iteration cap ran out (protocol fault); the result is void */

/* ---- primitive / light / material kinds -------------------------------------------------- */
#define SPCU_PRIM_TRIANGLE 0u /* shapes/Triangle.h:69-246 (vertices pre-transformed to world) */
#define SPCU_PRIM_SPHERE 1u   /* shapes/Sphere.h:13-150   (unit sphere in object space)       */
#define SPCU_PRIM_PLANE 2u    /* shapes/Plane.h:12-100    (y = 0 in object space, unbounded)  */

#define SPCU_LIGHT_SPHERE 0u    /* Lights/Light.h:336-388 SphereLight                */
#define SPCU_LIGHT_ENV_CONST 1u /* Lights/Light.h:120-177 EnvironmentLight           */
#define SPCU_LIGHT_ENV_IBL 2u   /* Lights/Light.h:179-334 ImageBasedEnvironmentLight */

#define SPCU_BXDF_LAMBERT 0u    /* materials/Material.h:313-350 */
#define SPCU_BXDF_MICROFACET 1u /* materials/Material.h:386-454 + BeckmannDistribution :213-267 */
#define SPCU_BXDF_SPECULAR 2u   /* materials/Material.h:352-383 */

#define SPCU_MAT_ONE_SAMPLE 0u /* materials/Material.h:533-718 OneSampleMaterial */
#define SPCU_MAT_CLEARCOAT 1u  /* materials/Material.h:723-806 ClearcoatMaterial */

#define SPCU_MAX_BXDFS 4u      /* per OneSampleMaterial (the .sp parser creates at most 2) */
#define SPCU_MAX_COAT_DEPTH 4u /* nesting of clearcoat-over-clearcoat                      */
#define SPCU_MAX_BVH_DEPTH 96u /* traversal stack capacity                                 */

/* ---- integrators (reference Integrators/Integrator.h:18-28) ------------------------------- */
#define SPCU_INTEGRATOR_ITERATIVE_RRNEE 0u   /* Integrator.cpp:550-635 (north star)  */
#define SPCU_INTEGRATOR_BRUTE_FORCE_RR 1u    /* Integrator.cpp:211-266               */
#define SPCU_INTEGRATOR_DIRECT_LIGHTING 2u   /* Integrator.cpp:277-312               */
#define SPCU_INTEGRATOR_WHITTED 3u           /* Integrator.cpp:314-368 (tail recursion over specular bounces, unrolled) */

/* ---- rays and hits ------------------------------------------------------------------------ */
/* One query: sp::Ray (math/Ray.h:21-49) + sp::RayLimits (math/Ray.h:13-19). 32 bytes. */
typedef struct spcu_ray {
    float ox, oy, oz, t_min;
    float dx, dy, dz, t_max;
} spcu_ray;

/* Result of a closest-hit query. id = -1 and t = the query's t_max when nothing was hit. */
typedef struct spcu_hit {
    int32_t id;
    float   t;
} spcu_hit;

/* ---- flattened acceleration structure ------------------------------------------------------ */
/*
 * One internal node of shapes/BVHAccelerator.h (NodeInternal :36-93): the bounds of BOTH children
 * (the reference tests a child's own bounds before descending, :67 / :84) and their links.
 *   box = { lo0.x lo0.y lo0.z hi0.x | hi0.y hi0.z lo1.x lo1.y | lo1.z hi1.x hi1.y hi1.z }
 *   child[k] >= 0 : index of an internal node
 *   child[k] <  0 : leaf; first primitive = ~child[k], number of primitives = count[k] & 0x7fffffff,
 *                   bit 31 of count[k] set when the leaf holds a non-triangle primitive
 * 64 bytes = four 16-byte vector loads, one cache-line half.
 */
typedef struct spcu_bvh_node {
    float    box[12];
    int32_t  child[2];
    uint32_t count[2];
} spcu_bvh_node;

#define SPCU_LEAF_COUNT_MASK 0x7fffffffu
#define SPCU_LEAF_MIXED_FLAG 0x80000000u

/*
 * Intersection data of one primitive, 48 bytes (three 16-byte loads).
 *   triangle     : p0.xyz _ | p1.xyz _ | p2.xyz _           (world space, Triangle.h:99-101)
 *   sphere/plane : world_to_object, column major + affine:
 *                  c0.x c0.y c0.z c1.x | c1.y c1.z c2.x c2.y | c2.z a.x a.y a.z
 */
typedef struct spcu_prim_geom {
    float v[12];
} spcu_prim_geom;

/*
 * Shading data of one primitive, 48 bytes, read once per accepted closest hit.
 *   triangle     : n0.xyz _ | n1.xyz _ | n2.xyz _           (Triangle.h:148-155)
 *   sphere/plane : normal matrix inverse(object_to_world.linear).transposed(), column major:
 *                  c0.xyz _ | c1.xyz _ | c2.xyz _            (math/LinearSpace3x3.h:163-167)
 */
typedef struct spcu_prim_shade {
    float v[12];
} spcu_prim_shade;

/* meta word of a primitive: bits 0-1 kind (SPCU_PRIM_*), bits 2-31 material index */
#define SPCU_META_KIND(m) ((m) & 3u)
#define SPCU_META_MATERIAL(m) ((m) >> 2)
#define SPCU_MAKE_META(kind, material) (((uint32_t)(material) << 2) | ((uint32_t)(kind) & 3u))

/* One accelerator = reference ListAccelerator [unbounded..., BVHAccelerator(bounded)]
 * built by internal::create_acceleration_structure (base/Scene.h:27-45). */
typedef struct spcu_accel {
    uint32_t n_prims;     /* unbounded + bounded                                            */
    uint32_t n_unbounded; /* prims [0, n_unbounded) are scanned linearly first              */
    uint32_t n_nodes;     /* internal nodes                                                 */
    int32_t  root;        /* >= 0 internal node; < 0 leaf with first prim ~root             */
    uint32_t root_count;  /* leaf root: count (+ mixed flag); the root's own bounds are never
                             tested (BVHAccelerator.h:132-148)                              */
    uint32_t max_depth;   /* deepest internal-node nesting, for the traversal stack         */
    const spcu_bvh_node* nodes; /* [n_nodes]                                                */
} spcu_accel;

/* ---- materials ----------------------------------------------------------------------------- */
typedef struct spcu_bxdf {
    uint32_t kind;           /* SPCU_BXDF_*                                                     */
    float    r[3];           /* Lambert: albedo/pi (m_albedo, Material.h:317); microfacet/specular: m_r */
    float    alpha_x;        /* BeckmannDistribution::m_alpha_x (after roughness_to_alpha)      */
    float    alpha_y;
    float    ior;            /* MicrofacetReflection::m_ior                                     */
    uint32_t sample_visible; /* MicrofacetDistribution::m_sample_visible_area                   */
} spcu_bxdf;

typedef struct spcu_material {
    uint32_t kind;        /* SPCU_MAT_*                                     */
    uint32_t n_bxdfs;     /* one-sample: number of BxDFs                    */
    uint32_t first_bxdf;  /* one-sample: index into bxdfs[]                 */
    uint32_t base;        /* clearcoat: index of the base material          */
    float    ior;         /* clearcoat: m_ior                               */
    float    specular[3]; /* clearcoat: m_specular_color                    */
} spcu_material;

/* ---- lights -------------------------------------------------------------------------------- */
typedef struct spcu_light {
    uint32_t kind; /* SPCU_LIGHT_* */
    float    radiance[3];
    /* sphere light: Sphere::m_object_to_world and inverse (12 floats each, layout of spcu_prim_geom)
     * and the normal matrix (9 floats, column major) */
    float world_to_object[12];
    float object_to_world[12];
    float normal_xf[9];
    /* image based light: m_light_to_world linear and inverse (column major 3x3) */
    float    light_to_world[9];
    float    world_to_light[9];
    uint32_t img_w, img_h; /* radiance image (after modify_image), row major RGB in float_pool */
    uint32_t nu, nv;       /* Distribution2D resolution (= 2*img_w, 2*img_h)                   */
    float    marg_integral;
    uint32_t _pad;
    uint64_t img_off;       /* [img_h][img_w][3]                                                */
    uint64_t cond_func_off; /* [nv][nu]      Distribution1D::m_function of each conditional     */
    uint64_t cond_cdf_off;  /* [nv][nu+1]    Distribution1D::m_cdf (reference-built, incl. its
                               shifted normalisation, math/Distribution1D.h:42-43)              */
    uint64_t cond_int_off;  /* [nv]          m_function_integral of each conditional            */
    uint64_t marg_func_off; /* [nv]                                                             */
    uint64_t marg_cdf_off;  /* [nv+1]                                                           */
} spcu_light;

/* ---- whole scene --------------------------------------------------------------------------- */
typedef struct spcu_flat_scene {
    uint32_t abi_version; /* SPCU_ABI_VERSION */
    /* render parameters: Scene::{image_width,image_height,russian_roulette_depth,max_depth} */
    uint32_t width, height;
    uint32_t rr_depth, max_depth;
    /* PerspectiveCamera m_transform (Cameras/Camera.h:99-129): col0 col1 col2 affine, xyz each */
    float camera[12];

    /* geometry (Scene::m_accelerator_geometry) */
    spcu_accel             geom;
    const spcu_prim_geom*  geom_prims; /* [geom.n_prims] */
    const spcu_prim_shade* geom_shade; /* [geom.n_prims] */
    const uint32_t*        geom_meta;  /* [geom.n_prims] */

    /* lights (Scene::m_accelerator_lights); "prims" of this accelerator are lights[] entries */
    spcu_accel        lights_accel;
    uint32_t          n_lights;
    uint32_t          _pad0;
    const spcu_light* lights;      /* [n_lights] in accelerator (ID) order                     */
    const uint32_t*   light_order; /* [n_lights] Scene::m_lights (for_each_light) order → ID   */

    uint32_t             n_materials;
    uint32_t             n_bxdfs;
    const spcu_material* materials;
    const spcu_bxdf*     bxdfs;

    uint64_t     n_pool; /* floats */
    const float* float_pool;
} spcu_flat_scene;

/* ---- work partition and render outputs ------------------------------------------------------ */
/*
 * What one GPU renders.  The unit is the reference's 8x8 tile (base/Tile.h:12, TileScheduler.h:66-82,
 * row major over tiles).  This rank renders tiles t with  t % tile_stride == tile_offset  and, for
 * each of their pixels, samples [sample_begin, sample_end) of spp_total.
 */
typedef struct spcu_partition {
    uint32_t tile_offset;
    uint32_t tile_stride;
    uint32_t sample_begin;
    uint32_t sample_end;
    uint32_t spp_total; /* jitter table length; samples are indexed globally */
    uint32_t integrator; /* SPCU_INTEGRATOR_* */
    uint64_t seed;
} spcu_partition;

/* Per-stage device counters of one render call. */
typedef struct spcu_stats {
    uint64_t paths;               /* camera samples started                                       */
    uint64_t rays_closest;        /* Scene::intersect queries (geometry accelerator)              */
    uint64_t rays_any;            /* Scene::intersect_p queries (geometry half)                   */
    uint64_t rays_lights;         /* Scene::intersect_lights queries (lights accelerator)         */
    uint64_t nodes_visited;       /* internal nodes fetched by geometry queries                   */
    uint64_t prims_tested;        /* triangle tests by geometry queries                           */
    uint64_t xf_prims_tested;     /* sphere / plane tests by geometry queries                     */
    uint64_t shade_calls;         /* Material::sample/eval/pdf evaluations                        */
    uint64_t kernel_launches;     /* kernels launched by this call                                */
    float    device_ms;           /* CUDA-event time of the wavefront loop                        */
    float    trace_ms;            /* ... of which extend/any-hit traversal kernels                */
    float    shade_ms;            /* ... of which shading / NEE kernels                           */
    float    _pad;
} spcu_stats;

typedef struct spcu_ctx spcu_ctx;

/* ---- entry points ---------------------------------------------------------------------------- */

/* Create / destroy a context bound to one CUDA device.  Replaces nothing in the reference (it has no
 * device); owned by CudaIntegrator's constructor / destructor. */
int  spcu_create(int device, spcu_ctx** out);
void spcu_destroy(spcu_ctx* ctx);
const char* spcu_last_error(const spcu_ctx* ctx); /* ctx may be NULL: last creation error */
int  spcu_abi_version(void);

/* Copy a flattened scene (host pointers) to the device.  Replaces the in-memory object graph handed to
 * Integrator::integrate (Scene&, base/Scene.h:47-106).  jitter = spp x 2 floats from
 * RSequenceSampler::get_next_2D (math/Sampler.h:158-162, main.cpp:67-71,96). */
int spcu_upload_scene(spcu_ctx* ctx, const spcu_flat_scene* scene, const float* jitter, uint32_t spp);

/* Scene::intersect (base/Scene.h:74-77) over a batch: closest geometry hit, reference order, exact
 * arithmetic.  rays/hits are host pointers. */
int spcu_trace_closest(spcu_ctx* ctx, const spcu_ray* rays, uint64_t n, spcu_hit* hits);
/* Scene::intersect_p (base/Scene.h:79-82): geometry OR lights accelerator any-hit. out[i] = 0/1. */
int spcu_trace_any(spcu_ctx* ctx, const spcu_ray* rays, uint64_t n, uint8_t* out);
/* Scene::intersect_lights (base/Scene.h:69-72): closest light (ID order of lights[]) and distance. */
int spcu_trace_lights(spcu_ctx* ctx, const spcu_ray* rays, uint64_t n, spcu_hit* hits);
/* Scene::intersect through the ORDERED walk (nearer child first; the renderer's extend stage uses it when
 * SPCU_OPT_TRAVERSAL = SPCU_TRAVERSAL_ORDERED).  Same boxes, primitive tests and arithmetic as spcu_trace_closest; the
 * answers differ only on epsilon ties (counted by tests/test_gpu_trace.py and stated in DESIGN.md).  counters (may be
 * NULL) = { internal nodes visited, triangle tests, sphere/plane tests }. */
int spcu_trace_closest_fast(spcu_ctx* ctx, const spcu_ray* rays, uint64_t n, spcu_hit* hits, uint64_t counters[3]);

/* The same queries through the RENDERER's traversal stages — the kernels a frame actually runs (the two-kernel extend / shadow
 * stages: set-up + root for all rays, then the persistent walk with lane refill and warp-wide leaf steps) — so that the parity
 * tests can hold them to the oracle on arbitrary ray batches.
 *   spcu_extend_batch: Integrator.cpp:558-563 — Scene::intersect_lights with the ray's limits, then Scene::intersect with t_max
 *     shrunk to the light's distance.  hits[i] = closest geometry primitive under that limit (id -1, t = the shrunk limit on a
 *     miss); light_hits[i] (may be NULL) = the light (id -1, t = the ray's t_max when none).  traversal = SPCU_TRAVERSAL_EXACT
 *     (reference order: bit-exact IDs and distances) or SPCU_TRAVERSAL_ORDERED (the render default: epsilon ties may differ).
 *   spcu_shadow_batch: Integrator.cpp:503 — Scene::intersect_p of a light sample's visibility ray. out[i] = 0/1. */
int spcu_extend_batch(spcu_ctx* ctx, const spcu_ray* rays, uint64_t n, uint32_t traversal, spcu_hit* hits, spcu_hit* light_hits);
int spcu_shadow_batch(spcu_ctx* ctx, const spcu_ray* rays, uint64_t n, uint8_t* occluded);

/* Camera::generate_ray for (pixel, sample) pairs (Cameras/Camera.h:119-129 + main.cpp:96-98):
 * rays[i] for pixel index pix[i] (= y*width+x) and sample index smp[i]. host pointers. */
int spcu_generate_rays(spcu_ctx* ctx, const uint32_t* pix, const uint32_t* smp, uint64_t n, spcu_ray* rays);

/* render_thread + Integrator::integrate over a partition (main.cpp:77-107, Integrator.cpp:550-635):
 * rgb_sum[(y*w+x)*3+c] += sum over this partition's samples of L; lum_sumsq[y*w+x] += sum of
 * luminance(L)^2 (may be NULL).  Host buffers, full image size, accumulated into (caller zeroes). */
int spcu_render(spcu_ctx* ctx, const spcu_partition* part, float* rgb_sum, float* lum_sumsq,
                spcu_stats* stats);
/* Same work, but the outputs are OVERWRITTEN with this partition's sums (pixels outside the partition become 0): nothing
 * is uploaded, the caller need not zero anything.  What CudaIntegrator::render_frame calls for a whole frame; with
 * page-locked output buffers the device→host copy runs at PCIe speed. */
int spcu_render_frame(spcu_ctx* ctx, const spcu_partition* part, float* rgb_sum, float* lum_sumsq,
                      spcu_stats* stats);
/* Same, accumulating into DEVICE buffers (so the caller can reduce them across GPUs with NCCL before
 * the single device→host copy).  stream = cudaStream_t as void*, NULL for the default stream. */
int spcu_render_device(spcu_ctx* ctx, const spcu_partition* part, float* d_rgb_sum, float* d_lum_sumsq,
                       spcu_stats* stats, void* stream);

/* ---- adaptive sampling --------------------------------------------------------------------------------------------------
 * Renders each pixel until the standard error of its mean luminance meets a target, instead of the same sample count
 * everywhere.  Replaces nothing in the reference (it renders num_pixel_samples for every pixel, main.cpp:90-102).
 * The partition's sample_end is the budget (the most samples any pixel gets); sample_begin must be 0.  Passes end at fixed
 * sample counts that depend only on these parameters, never on the image:
 *   s_0 = min(min_spp, sample_end),  s_{k+1} = min(s_k + pass_spp, sample_end).
 * Pass 0 renders samples [0, s_0) of every pixel of the partition; at each boundary s_k < sample_end every pixel still active
 * is tested with n = s_k, and the pass after it renders [s_k, s_{k+1}) of the pixels that failed the test only.  The test,
 * float32 with one rounding per operation (R, G, B = the pixel's rgb_sum, Q = its lum_sumsq):
 *   L = (0.2126 R + 0.7152 G) + 0.0722 B;  m = L / n;  d = Q / n - m m;  v = d > 0 ? d (n / (n - 1)) : 0;
 *   pass  <=>  R, G, B, Q finite  and  v / n <= (rel_error (m + abs_floor))^2
 * With radius 0 an active pixel stops at s_k iff it passes.  With radius r > 0 it stops iff every pixel q of its window
 *   W(p) = { q : |x_q - x_p| <= r, |y_q - y_p| <= r, q in the same 8x8 tile as p, q inside the image }
 * passes, where a pixel that stopped at an earlier boundary counts as passing and every other one is tested with n = s_k.
 * All of a boundary's tests are made before any of its decisions, so the decisions do not depend on thread order.  r >= 7
 * makes the window the whole tile: a tile then stops at one boundary.  n_p cannot decrease as r grows.
 * So pixel p gets samples [0, n_p) with min(min_spp, sample_end) <= n_p <= sample_end, and its sums equal bit for bit those
 * of a fixed render of [0, n_p): the result does not depend on the tile partition, the batch shape or the kernel
 * organisation (a window never leaves its tile, and a tile belongs to one partition).  What stopping on an estimated
 * variance does to the mean, and what the window does about it, is measured in DESIGN.md §11. */
typedef struct spcu_adaptive {
    uint32_t min_spp;   /* samples before the first test, >= 2                                              */
    uint32_t pass_spp;  /* samples added per pass, >= 1                                                     */
    float    rel_error; /* target standard error relative to the mean luminance, finite, >= 0             */
    float    abs_floor; /* added to the mean in the target, so that near-black pixels can stop; finite, >= 0 */
    uint32_t radius;    /* half-width of the window of the stopping rule, 0..7 (0: each pixel on its own)         */
} spcu_adaptive;

/* Adaptive render of a tile partition into host buffers, OVERWRITTEN like spcu_render_frame's: rgb_sum / lum_sumsq (may be
 * NULL) as there, spp_map[y*w+x] = n_p (0 outside the partition).  n_passes (may be NULL) = passes rendered.  stats are
 * summed over the passes, device_ms covers the whole call.  SPCU_ERR_INVALID for parameters outside the rules above or
 * sample_begin != 0; the context stays usable. */
int spcu_render_adaptive(spcu_ctx* ctx, const spcu_partition* part, const spcu_adaptive* ad, float* rgb_sum, float* lum_sumsq,
                         uint32_t* spp_map, uint32_t* n_passes, spcu_stats* stats);
/* Same into DEVICE buffers of the image's size on `stream` (cudaStream_t as void*, NULL = default stream), also
 * overwritten; d_lum_sumsq may be NULL.  With tile partitions the ranks' sums can then be added by spcu_reduce_to_root (and
 * their spp maps, which are 0 outside each rank's tiles, likewise by the caller).  The call synchronises once per pass: the
 * host needs the number of active pixels to shape the next pass. */
int spcu_render_adaptive_device(spcu_ctx* ctx, const spcu_partition* part, const spcu_adaptive* ad, float* d_rgb_sum,
                                float* d_lum_sumsq, uint32_t* d_spp_map, uint32_t* n_passes, spcu_stats* stats, void* stream);

/* ---- denoising -----------------------------------------------------------------------------------------------------------
 * Turns a low-sample frame into a smoother image: the spatial filter of SVGF (an edge-avoiding à-trous wavelet filter whose
 * luminance term is scaled by each pixel's standard deviation), guided by the first hit of each pixel's camera ray.  Replaces
 * nothing in the reference (it divides the sums by the sample count, main.cpp:100-102).  DESIGN.md §12 has the measurements.
 *
 * Guide buffers: one record per pixel of the uploaded scene's image, from the camera ray of sample 0 (the ray a render traces
 * first), with the extend stage's rule and the exact walk: intersect_lights with the ray's limits, then intersect with t_max
 * shrunk to the light's distance; a geometry hit under that limit wins, else a light hit, else the ray missed.  id and depth
 * equal what spcu_extend_batch(camera ray of (pix, 0), SPCU_TRAVERSAL_EXACT) returns. */
typedef struct spcu_guide {
    float   normal[3]; /* unit shading normal of the first geometry hit, facing the camera; 0 otherwise             */
    float   depth;     /* distance of the accepted hit (geometry or light); the ray's t_max (FLT_MAX) on a miss     */
    float   albedo[3]; /* one-sample material (a clearcoat's base, followed): sum over its BxDFs in table order of
                          r * pi (Lambert) or r (microfacet, specular), float32; 0 for light hits and misses         */
    int32_t id;        /* >= 0 geometry primitive (reference-order ID); -2 - k light k (ID order); -1 miss          */
} spcu_guide;          /* 32 bytes */
/* Host out[h*w] / device d_out[h*w] (on `stream`, cudaStream_t as void*, NULL = default stream), overwritten. */
int spcu_render_guides(spcu_ctx* ctx, spcu_guide* out);
int spcu_render_guides_device(spcu_ctx* ctx, spcu_guide* d_out, void* stream);

/* The filter, float32 with one rounding per operation and taps summed in a fixed order (a numpy model reproduces it bit for
 * bit).  Per pixel p with n = n_p samples (spp_map[p], or spp):
 *   n = 0: empty — outputs 0 and is never a tap.  R, G, B or Q (lum_sumsq) not finite: outputs sum / n and is never a tap.
 *   otherwise c = sum / n per channel, l = (0.2126 c_R + 0.7152 c_G) + 0.0722 c_B, var = the variance of the mean luminance
 *   of the adaptive test (spcu_adaptive above: v / n), 0 when n < 2.
 * Iteration i = 0 .. iterations-1, step h = 2^i:
 *   var~_p = 3x3 weighted mean of var over the neighbours that are taps (centre 1/4, edges 1/8, corners 1/16, row-major sums);
 *   taps q = p + h (dx, dy), dx, dy in -2..2, row-major, skipped outside the image or when not a tap;
 *   k = b[dx] b[dy], b = (1/16, 1/4, 3/8, 1/4, 1/16); the centre's w = k; for another tap:
 *     classes of p and q differ (geometry hit, light hit, miss): w = 0; else
 *     both geometry: w_n = max(0, (n_x n'_x + n_y n'_y) + n_z n'_z)^128 (seven squarings),
 *                    a_z = |z_p - z_q| / ((sigma_z z_p) (h max(|dx|, |dy|))),  a_a = max_c |alb_p,c - alb_q,c| / sigma_a;
 *     otherwise w_n = 1, a_z = a_a = 0;
 *     a_l = |l_p - l_q| / (sigma_l sqrt(var~_p) + 1e-4);   w = (k w_n) / (((1 + a_l a_l) + a_z a_z) + a_a a_a);
 *   S_c += w c_q, S_w += w, S_v += (w w) var_q;  c' = S_c / S_w, var' = S_v / (S_w S_w), l' from c'.
 * The output is c' after the last iteration: the denoised MEAN colour out[(y*w+x)*3+c]. */
typedef struct spcu_denoise_params {
    uint32_t iterations; /* 1..8; iteration i uses step 2^i                        */
    float    sigma_l;    /* luminance, in standard deviations; finite, > 0        */
    float    sigma_z;    /* relative depth change per pixel of offset; finite, > 0 */
    float    sigma_a;    /* albedo difference; finite, > 0                         */
} spcu_denoise_params;
/* From a frame's sums (host buffers of the image's size; spp_map NULL = every pixel has `spp` samples).  The guides are
 * computed inside from the uploaded scene.  Outputs overwritten.  SPCU_ERR_INVALID for parameters outside the ranges above,
 * lum_sumsq NULL, or spp 0 without a map; the context stays usable. */
int spcu_denoise(spcu_ctx* ctx, const float* rgb_sum, const float* lum_sumsq, const uint32_t* spp_map, uint32_t spp,
                 const spcu_denoise_params* p, float* out);
/* Same on DEVICE buffers, enqueued on `stream` (cudaStream_t as void*, NULL = default stream); d_out may be d_rgb_sum. */
int spcu_denoise_device(spcu_ctx* ctx, const float* d_rgb_sum, const float* d_lum_sumsq, const uint32_t* d_spp_map,
                        uint32_t spp, const spcu_denoise_params* p, float* d_out, void* stream);

/* ---- multi-GPU: accumulators summed into rank 0 with NCCL over NVLink (SURVEY.md §8e) ------------------------------------
 * The scene is replicated (every rank uploads it), the work is partitioned by spcu_partition (tiles or sample ranges), there
 * is no exchange during tracing; ONE ncclReduce(sum, root 0) per accumulator ends a frame.  Replaces nothing in the reference
 * (its image is one process's Array2D, main.cpp:100-102).
 *   one process per GPU : rank 0 calls spcu_comm_unique_id, the launcher hands the bytes to every rank (MPI / torchrun /
 *                         a file), every rank calls spcu_comm_init_rank(ctx, nranks, rank, id) — a collective.
 *   one process, n GPUs : spcu_comm_init_all over n contexts (rank i = ctxs[i]); afterwards every context is driven from its
 *                         own host thread (what sp::CudaIntegrator does with SPCU_DEVICES=n).
 * spcu_reduce_to_root: in place on DEVICE buffers of the image's size, on `stream`; every rank calls it, rank 0's buffers hold
 * the sums afterwards.  A context without a communicator is a world of one rank (no-op).
 * spcu_render_frame_reduced = spcu_render_frame of this rank's partition + the reduction + the single device->host copy on
 * rank 0 (the other ranks may pass NULL host pointers); with_sumsq must agree on all ranks. */
#define SPCU_NCCL_ID_BYTES 128
int  spcu_comm_unique_id(uint8_t id[SPCU_NCCL_ID_BYTES]);
int  spcu_comm_init_rank(spcu_ctx* ctx, int nranks, int rank, const uint8_t id[SPCU_NCCL_ID_BYTES]);
int  spcu_comm_init_all(spcu_ctx** ctxs, int n);
void spcu_comm_destroy(spcu_ctx* ctx);
int  spcu_comm_rank(const spcu_ctx* ctx);
int  spcu_comm_size(const spcu_ctx* ctx);
int  spcu_reduce_to_root(spcu_ctx* ctx, float* d_rgb_sum, float* d_lum_sumsq, void* stream);
int  spcu_render_frame_reduced(spcu_ctx* ctx, const spcu_partition* part, int with_sumsq, float* rgb_sum, float* lum_sumsq,
                               spcu_stats* stats);

/* Upper bound of paths kept in flight per wavefront batch (0 = default). */
int spcu_set_wavefront_size(spcu_ctx* ctx, uint64_t n_paths);

/* Instrumentation switches (all default 0 = off; they never change results).
 *   SPCU_OPT_COUNT_NODES : spcu_stats.{nodes_visited,prims_tested,xf_prims_tested} are counted (per-thread
 *                          counters in the traversal loops; off in timed runs).
 *   SPCU_OPT_STAGE_TIMING: spcu_stats.{trace_ms,shade_ms} are measured with one CUDA-event pair per launch. */
#define SPCU_OPT_COUNT_NODES 0u
#define SPCU_OPT_STAGE_TIMING 1u
/*   SPCU_OPT_PIPELINE    : which kernel organisation renders (same stages, same random numbers, same estimator):
 *                          SPCU_PIPELINE_WAVEFRONT = one kernel per stage with compacted queues in HBM between them;
 *                          SPCU_PIPELINE_PATHS = one persistent kernel per batch, a thread carries a path in registers
 *                          and regenerates it in place; SPCU_PIPELINE_SMWAVE = the SM-local wavefront: one persistent
 *                          CTA per SM keeps path state and per-stage work queues in shared memory, warps run one stage
 *                          for up to 32 queued paths at a time; SPCU_PIPELINE_AUTO (default) = whichever measures
 *                          faster for the uploaded scene's feature set (DESIGN.md, profiles/): SMWAVE for analytic
 *                          scenes, WAVEFRONT for scenes with a BVH. */
#define SPCU_OPT_PIPELINE 2u
/*   SPCU_OPT_TRAVERSAL   : closest-hit walk of the RENDERER's extend stage: SPCU_TRAVERSAL_ORDERED (default) = nearer child
 *                          first (see spcu_trace_closest_fast): about half the node visits, answers differ from the
 *                          reference-order walk on epsilon ties only (counted by tests/test_gpu_trace.py and by bench.py's
 *                          `ordered_walk` object, stated in DESIGN.md); SPCU_TRAVERSAL_EXACT = the reference's own order,
 *                          bit-exact IDs.  spcu_trace_closest is always the exact walk; with SPCU_OPT_COUNT_NODES the
 *                          renderer also walks in reference order (the counters are defined on that walk). */
#define SPCU_OPT_TRAVERSAL 3u
/*   SPCU_OPT_GENERIC_KERNELS : 1 = always run the kernels compiled for every scene feature (default 0: spcu_upload_scene picks
 *                          the smallest compiled feature set that covers the scene).  Takes effect at the next upload. */
#define SPCU_OPT_GENERIC_KERNELS 4u
/*   SPCU_OPT_BATCH_LANES : how many wavefront batches of one render call are in flight at the same time, each with its own
 *                          wavefront state on its own CUDA stream (0 = default: 4; 1 = one batch after the other).  The
 *                          kernels of a batch leave issue slots idle — the walks wait on dependent fetches, every launch
 *                          has a tail — and the kernels of another batch fill them (DESIGN.md).  Batches still add their
 *                          samples to the accumulators in batch order (event-ordered resolve kernels): images are
 *                          bit-identical for every value.  Only the queue wavefront uses it; per-launch timing and node
 *                          counting render with one lane. */
#define SPCU_OPT_BATCH_LANES 5u
#define SPCU_OPT_COUNT_ 6u
#define SPCU_TRAVERSAL_EXACT 0u
#define SPCU_TRAVERSAL_ORDERED 1u
#define SPCU_PIPELINE_WAVEFRONT 0u
#define SPCU_PIPELINE_PATHS 1u
#define SPCU_PIPELINE_SMWAVE 2u
#define SPCU_PIPELINE_AUTO 3u
int spcu_set_option(spcu_ctx* ctx, uint32_t option, uint32_t value);
/* The kernel organisation (SPCU_PIPELINE_*) the next render of the uploaded scene will run: SPCU_OPT_PIPELINE with
 * SPCU_PIPELINE_AUTO resolved.  -1 without a scene. */
int spcu_resolved_pipeline(const spcu_ctx* ctx);

/* Per-kernel breakdown of the LAST render call (needs SPCU_OPT_STAGE_TIMING = 1 for `ms`): one entry per wavefront
 * stage, in pipeline order.  items = queue entries the stage processed (paths, rays or vertices), counted on the device. */
typedef struct spcu_stage_time {
    char     name[24];
    uint64_t launches;
    uint64_t items;
    float    ms;
    uint32_t traverses; /* 1 for extend / shadow / mis_trace */
} spcu_stage_time;
#define SPCU_MAX_STAGES 16u
int spcu_stage_times(spcu_ctx* ctx, spcu_stage_time* out, uint32_t capacity, uint32_t* n_out);

/* Bytes of scene data resident on the device after spcu_upload_scene (what one upload copies host->device). */
uint64_t spcu_scene_bytes(const spcu_ctx* ctx);

/* spcu_trace_closest plus the traversal work it did, summed over the batch: counters = { internal nodes visited,
 * triangle tests, sphere/plane tests } — the N_node / N_tri / N_xf of the byte model in DESIGN.md. */
int spcu_trace_closest_counted(spcu_ctx* ctx, const spcu_ray* rays, uint64_t n, spcu_hit* hits, uint64_t counters[3]);

/* ---- acceleration-structure construction on the device (SURVEY.md §8(f) rank 1) ------------------------------------- */
/* World bounds of one bounded primitive, Hitable::get_world_bounds (shapes/Hitable.h:32-35): lower xyz, upper xyz. */
typedef struct spcu_bounds {
    float lo[3];
    float hi[3];
} spcu_bounds;

/* BVHAccelerator(first, last) (shapes/BVHAccelerator.h:123-129) = construct (:175-209): a node over [first, last) holds
 * the merged bounds of its primitives (math/BBox.h:60-64, folded in range order); <= k_max_leaf_elements (4, :211)
 * primitives make a leaf; otherwise the range is std::partition'ed (libstdc++'s bidirectional Hoare scheme, whose
 * resulting ORDER is part of the contract because primitive IDs are positions) by
 * center(prim bounds)[d] < center(node bounds)[d] with d = max_dim(size(node bounds)) (math/Vector3.h:653-670), and a
 * partition with an empty side makes a leaf of any size.
 *   bounds[n]        primitive bounds in the order the reference holds them BEFORE construction (host)
 *   non_triangle[n]  may be NULL; 1 marks a sphere (sets SPCU_LEAF_MIXED_FLAG on its leaf)
 *   first_id         ID of leaf position 0 (= spcu_accel.n_unbounded of the accelerator being built)
 *   order[n]         out: order[k] = index into bounds[] of the primitive at leaf position k (ID first_id + k)
 *   nodes[capacity]  out: internal nodes in the flattener's numbering (depth-first pre-order, left subtree first);
 *                    at most max(n, 1) - 1 are produced
 *   accel            out: n_prims, n_unbounded, n_nodes, root, root_count, max_depth (nodes = the caller's pointer)
 *   device_ms        out, may be NULL: CUDA-event time of the construction kernels (copies excluded)
 * Produces, bit for bit, the arrays the flattener emits for the tree the reference builds from the same sequence
 * (oracle/ref_harness.cpp spref_build_bvh; tests/test_gpu_build.py).  Finite, non-NaN bounds with lo <= hi are required;
 * SPCU_ERR_LIMIT when the tree is deeper than SPCU_MAX_BVH_DEPTH or needs more than `capacity` nodes. */
int spcu_build_bvh(spcu_ctx* ctx, const spcu_bounds* bounds, uint32_t n, const uint8_t* non_triangle, uint32_t first_id,
                   uint32_t* order, spcu_bvh_node* nodes, uint32_t capacity, spcu_accel* accel, float* device_ms);

/* spcu_upload_scene for a scene whose geometry accelerator has NOT been built: create_acceleration_structure + the
 * flattener's walk (base/Scene.h:27-45; shapes/BVHAccelerator.h:123-209) happen on the device.  scene->geom_prims / geom_shade /
 * geom_meta hold the primitives in PRE-construction order: [0, geom.n_unbounded) the top-level list (planes), then the bounded
 * primitives as the reference holds them before BVHAccelerator(first, last); scene->geom.{n_prims, n_unbounded} are read, the
 * other fields of scene->geom are ignored.  Triangle bounds are computed on the device; `bounds` ([n_prims - n_unbounded], may
 * be NULL when every bounded primitive is a triangle) supplies the world bounds of the others (spheres:
 * TransformableShape::get_world_bounds_impl, shapes/Shape.h:61-64).  order ([n_prims - n_unbounded], may be NULL): order[k] =
 * pre-construction index (within the bounded range) of the primitive that received ID n_unbounded + k.  built (may be NULL):
 * header of the accelerator now resident (nodes = NULL).  The resident scene is bit-identical to what spcu_upload_scene gets
 * from the flattener for the tree the reference builds from the same sequence. */
int spcu_upload_scene_build(spcu_ctx* ctx, const spcu_flat_scene* scene, const float* jitter, uint32_t spp,
                            const spcu_bounds* bounds, uint32_t* order, spcu_accel* built);

/* Triangle::get_world_bounds_impl (shapes/Triangle.h:228-237): BBox::extend over the three world-space vertices of
 * tris[i] (layout of spcu_prim_geom), in vertex order.  Host pointers. */
int spcu_triangle_bounds(spcu_ctx* ctx, const spcu_prim_geom* tris, uint32_t n, spcu_bounds* out);

/* ---- output side on the device (SURVEY.md §8(f) rank 4) ------------------------------------------------------------- */
/* What the reference writes after render(): image(x, y) /= num_pixel_samples (main.cpp:100-102), then sp::write
 * (Image/Image.cpp:14-55).  Both formats store rows bottom-up (j = ny-1 .. 0).
 *   SPCU_IMAGE_PFM : out = float[h][w][3], the payload of write_pfm (:40-55) on a little-endian host: sum / spp
 *   SPCU_IMAGE_PPM : out = uint16_t[h][w][3], the numbers write_ppm prints (:14-29): int(255.99f * rgb_to_srgb(sum / spp))
 *                    (Image/Image.h:38-50), clamped to [0, 65535]; half the device->host bytes of the float sums */
#define SPCU_IMAGE_PFM 0u
#define SPCU_IMAGE_PPM 1u
/* Packs host-resident per-pixel sums (rgb_sum[(y*w+x)*3+c], as spcu_render returns them). */
int spcu_pack_image(spcu_ctx* ctx, const float* rgb_sum, uint32_t width, uint32_t height, uint32_t spp, uint32_t format, void* out);
/* spcu_pack_image with a per-pixel divisor: spp_map[y*w+x] (host, as spcu_render_adaptive returns it) in place of spp.  A
 * pixel with 0 samples packs as 0. */
int spcu_pack_image_counts(spcu_ctx* ctx, const float* rgb_sum, const uint32_t* spp_map, uint32_t width, uint32_t height,
                           uint32_t format, void* out);
/* spcu_render_frame + packing of the device-resident sums: only the packed image crosses to the host.  The divisor is the
 * partition's sample count (sample_end - sample_begin). */
int spcu_render_image(spcu_ctx* ctx, const spcu_partition* part, uint32_t format, void* out, spcu_stats* stats);

/* ---- mesh ingest on the device (SURVEY.md §8(f) rank 3) ------------------------------------------------------------- */
/* What read_ply does once the vertex and face lists are read (base/PlyReader.cpp:487-531) followed by Mesh's constructor
 * (shapes/Triangle.h:25-51): face normals by compensated cross product, zero-area faces dropped, vertex normals = normalised
 * sum of the kept faces' normals in face order ((0,1,0) for an empty sum), vertices and normals to world space, and the
 * pre-gathered triangle records of this header in face order — the pre-construction order spcu_upload_scene_build takes.
 *   vertices[nv*3], faces[nf*3]   object-space positions and the indices of the triangular faces, as the parser read them
 *   object_to_world[12]           AffineSpace, layout c0.xyz c1.xyz c2.xyz affine.xyz (as spcu_prim_geom's transform)
 *   normal_xf[9]                  inverse(linear).transposed(), column major: what LinearSpace3x3::operator()(Normal3)
 *                                 (math/LinearSpace3x3.h:163-167) builds on every call — computed once by the host
 *   prims / shade / meta [nf]     out; the first *n_kept entries are valid (meta = triangle | material)
 *   world_vertices / world_normals [nv*3]  out, may be NULL: Mesh::m_vertices / m_normals
 * Positions, the set of kept faces and their order are bit-exact; normals agree with the reference to a few ulp because
 * normalize() multiplies by an SSE rsqrtss estimate there (math/Math.h:205-227). */
int spcu_ingest_mesh(spcu_ctx* ctx, const float* vertices, uint32_t nv, const uint32_t* faces, uint32_t nf,
                     const float object_to_world[12], const float normal_xf[9], uint32_t material, spcu_prim_geom* prims,
                     spcu_prim_shade* shade, uint32_t* meta, uint32_t* n_kept, float* world_vertices, float* world_normals,
                     float* device_ms);

/* The STL flavour (base/STLReader.cpp:60-137): vertices[] is the parser's de-duplicated vertex list (VertexIndexer, :18-36, host
 * side), faces[] its index triples, face_normals[nf*3] the normals stored in the file.  A stored normal is used unless it
 * is_zero (every component within 1e-5 of 0: math/Vector3.h:644-647), then the cross product; a face whose normal still is_zero
 * adds nothing to the vertex normals but — its indices were pushed before the test (:95-96) — STAYS in the mesh: *n_kept = nf. */
int spcu_ingest_mesh_stl(spcu_ctx* ctx, const float* vertices, uint32_t nv, const uint32_t* faces, uint32_t nf,
                         const float* face_normals, const float object_to_world[12], const float normal_xf[9], uint32_t material,
                         spcu_prim_geom* prims, spcu_prim_shade* shade, uint32_t* meta, uint32_t* n_kept, float* world_vertices,
                         float* world_normals, float* device_ms);

#ifdef __cplusplus
}
#endif
#endif /* SPCU_H */
