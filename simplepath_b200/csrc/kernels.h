// Host-callable launchers of the backend's kernels.  Each .cu translation unit defines its own kernels (no
// relocatable device code); the C-ABI layer (spcu_api.cu) only sees these functions.
#pragma once

#include "device_scene.h"
#include "features.h"

namespace spcu {

// ---- trace_kernels.cu (compiled with --fmad=false; exact, reference-order traversal) ---------------------------
void launch_trace_closest(const DScene& s, const spcu_ray* d_rays, uint64_t n, spcu_hit* d_hits, TraceCounters* d_cnt,
                          cudaStream_t st);
// the ordered ("fast") walk: nearer child first, ties towards the higher reference-order ID (trace.cuh)
void launch_trace_closest_ordered(const DScene& s, const spcu_ray* d_rays, uint64_t n, spcu_hit* d_hits, TraceCounters* d_cnt,
                                  cudaStream_t st);
void launch_trace_any(const DScene& s, const spcu_ray* d_rays, uint64_t n, uint8_t* d_out, cudaStream_t st);
void launch_trace_lights(const DScene& s, const spcu_ray* d_rays, uint64_t n, spcu_hit* d_hits, cudaStream_t st);

// Ray batches through the wavefront's own traversal stages (spcu_extend_batch / spcu_shadow_batch): slot i <- ray i.
void launch_batch_fill(const DWave& w, const spcu_ray* d_rays, uint32_t n, uint32_t* queue, uint32_t* d_n_queue, bool shadow,
                       cudaStream_t st);
void launch_batch_gather_extend(const DWave& w, uint32_t n, spcu_hit* d_hits, spcu_hit* d_light_hits, cudaStream_t st);

// Wavefront stages that traverse.  `queue` holds path slots; n_queue is read on the device (no host sync).
// d_cursor (extend, shadow): a zeroed uint32 in device memory, the stage's global work cursor.
// extend: Scene::intersect_lights then Scene::intersect for every queued path (Integrator.cpp:558-563).
// q_walk / d_n_walk: a queue (and its zeroed length) for the two-kernel form — `begin` finishes the rays that end at the root
// of the BVH and parks the others there for the persistent `walk` kernel; NULL: one kernel.  Returns the kernels launched.
// adv (only where extend_fuses_advance() says so): `queue` is the previous depth's queue of LIVE vertices and `begin` runs
// their `advance` stage first (throughput, Russian roulette, next ray) — launch_advance is then not called for that depth.
struct AdvanceArgs
{
    uint64_t seed;
    uint32_t depth; // of the vertex the path leaves
};
bool extend_fuses_advance(const struct Launch& l, const uint32_t* q_walk, const TraceCounters* d_cnt);
int launch_extend(const struct Launch& l, const DScene& s, const DWave& w, const uint32_t* queue, const uint32_t* d_n_queue,
                  uint32_t max_n, uint32_t* d_cursor, const SortedQueue& sorted, bool ordered, uint32_t* q_walk,
                  uint32_t* d_n_walk, unsigned long long* d_counters, TraceCounters* d_cnt, const AdvanceArgs* adv = nullptr);
// shadow: Scene::intersect_p of the light-sample visibility ray (Integrator.cpp:503).
// Unoccluded entries are compacted into q_lit (may be NULL: then only the per-slot flag is written).
int launch_shadow(const struct Launch& l, const DScene& s, const DWave& w, const uint32_t* queue, const uint32_t* d_n_queue,
                  uint32_t max_n, uint32_t light_index, uint32_t* d_cursor, uint32_t* q_lit, uint32_t* d_n_lit, uint32_t* q_walk,
                  uint32_t* d_n_walk, unsigned long long* d_counters, TraceCounters* d_cnt);
// mis: Scene::intersect_lights then, on a light hit, Scene::intersect_p of the BSDF-sampled ray (Integrator.cpp:531-532).
// d_cursor / q_walk / d_n_walk as for launch_shadow (begin + persistent walk); returns the kernels launched.
int launch_mis_trace(const struct Launch& l, const DScene& s, const DWave& w, const uint32_t* queue,
                     const uint32_t* d_n_queue, uint32_t max_n, uint32_t* d_cursor, uint32_t* q_walk, uint32_t* d_n_walk,
                     unsigned long long* d_counters, TraceCounters* d_cnt);

// ---- build_kernels.cu: the 4-wide copy of the resident binary nodes (8 x float4 per node, trace.cuh) ------------------------
// d_big: room for n_prims / (kWideSmallLeafMax + 1) + 1 entries; d_n_big: one counter (zeroed here)
void launch_build_wide(const float4* d_nodes, uint32_t n, float4* d_wide, int2* d_big, uint32_t* d_n_big, int sm_count, cudaStream_t st);

// ---- shade_kernels.cu ------------------------------------------------------------------------------------------
struct RenderParams
{
    uint64_t seed;
    uint32_t integrator;
    uint32_t depth;       // current path depth
    uint32_t light_index; // index into light_order of the light handled by the NEE stages
};

// Grid of a persistent-style wavefront kernel: enough CTAs to fill every SM at the kernel's occupancy, never more than
// the queue can feed.  (The queue length itself lives on the device; max_n is its upper bound.)
unsigned wavefront_grid(uint32_t max_n, int block, int ctas_per_sm, int sm_count);

void launch_generate_rays(const DScene& s, const uint32_t* d_pix, const uint32_t* d_smp, uint64_t n, spcu_ray* d_rays,
                          cudaStream_t st);

struct Launch
{
    int          sm_count;
    cudaStream_t stream;
    int          features; // FeatFull::id / FeatAnalytic::id (features.h): which instantiation of the kernels the scene needs
};

// raygen: fills slots [0, n_pix*n_samples) from the pixel list and the sample range, and the initial queue (main.cpp:90-98).
void launch_raygen(const Launch& l, const DScene& s, const DWave& w, const uint32_t* d_pix_list, uint32_t n_pix,
                   uint32_t sample_begin, uint32_t n_samples, uint32_t* queue, uint32_t* d_n_queue,
                   unsigned long long* d_counters);
// shade: hit/miss handling + primary BSDF sample S0 (Integrator.cpp:558-572,627-632); surviving paths go to q_live.  Then
// Light::sample for every light (Integrator.cpp:497-501): usable samples of light l go to q_shadow[l * capacity ...] /
// d_n_shadow[l], their LightRec to w.light[l * capacity + slot].  q_shadow == NULL: no light sampling (brute force).
void launch_shade(const Launch& l, const DScene& s, const DWave& w, const RenderParams& p, const SortedQueue& sorted,
                  uint32_t max_n, uint32_t* q_live, uint32_t* d_n_live, uint32_t* q_shadow, uint32_t* d_n_shadow,
                  unsigned long long* d_counters);
// nee_bsdf: light-strategy term, second BSDF sample, Light::pdf; paths needing the BSDF-strategy ray go to q_mis
// (Integrator.cpp:503-530).
void launch_nee_bsdf(const Launch& l, const DScene& s, const DWave& w, const RenderParams& p, const uint32_t* q_shadow,
                     const uint32_t* d_n_shadow, uint32_t max_n, uint32_t* q_mis, uint32_t* d_n_mis,
                     unsigned long long* d_counters);
// nee_mis_accumulate: adds the vertex's direct-light estimate for this light after the mis trace (Integrator.cpp:531-538).
void launch_nee_mis_accumulate(const Launch& l, const DScene& s, const DWave& w, const uint32_t* q_mis,
                               const uint32_t* d_n_mis, uint32_t max_n, unsigned long long* d_counters);
// direct: DirectLightingIntegrator's per-light term after the shadow trace (Integrator.cpp:296-306).
void launch_direct_accumulate(const Launch& l, const DScene& s, const DWave& w, const RenderParams& p,
                              const uint32_t* q_shadow, const uint32_t* d_n_shadow, uint32_t max_n,
                              unsigned long long* d_counters);
// advance: throughput update, Russian roulette, next segment (Integrator.cpp:601-626); survivors go to q_next.
void launch_advance(const Launch& l, const DScene& s, const DWave& w, const RenderParams& p, const uint32_t* q_live,
                    const uint32_t* d_n_live, uint32_t max_n, uint32_t* q_next, uint32_t* d_n_next,
                    unsigned long long* d_counters);
// whitted_advance: the Whitted integrator's BSDF sample; specular samples continue as the next segment (Integrator.cpp:357-363).
void launch_whitted_advance(const Launch& l, const DScene& s, const DWave& w, const RenderParams& p, const uint32_t* q_live,
                            const uint32_t* d_n_live, uint32_t max_n, uint32_t* q_next, uint32_t* d_n_next,
                            unsigned long long* d_counters);
// resolve: per pixel, add this batch's samples in sample order to the accumulators (main.cpp:100).
// d_radiance[(k * n_pix + i) * stride] = radiance sample k of pixel-list entry i (float4 units).
void launch_resolve(const Launch& l, const float4* d_radiance, uint32_t stride, const uint32_t* d_pix_list, uint32_t n_pix,
                    uint32_t n_samples, float* d_rgb_sum, float* d_lum_sumsq, unsigned long long* d_counters);
// ---- path_kernels.cu ------------------------------------------------------------------------------------------------
// The persistent path kernel: every slot of the batch from camera to termination in one launch; d_radiance[slot] = L.
void launch_paths(const Launch& l, const DScene& s, const uint32_t* d_pix_list, uint32_t n_pix, uint32_t sample_begin,
                  uint32_t n_samples, uint64_t seed, uint32_t integrator, float4* d_radiance, unsigned long long* d_counters,
                  TraceCounters* d_cnt);

// ---- smwave_kernels.cu -----------------------------------------------------------------------------------------------
// The SM-local wavefront: one persistent CTA per SM keeps its paths' state and the per-stage work queues in shared
// memory; same contract as launch_paths.  smwave_supports: path depth and light count fit the packed per-path flags.
bool        smwave_supports(const DScene& s);
cudaError_t launch_smwave(const Launch& l, const DScene& s, const uint32_t* d_pix_list, uint32_t n_pix, uint32_t sample_begin,
                          uint32_t n_samples, uint64_t seed, uint32_t integrator, float4* d_radiance,
                          unsigned long long* d_counters, TraceCounters* d_cnt);

// ---- adaptive_kernels.cu (exact float32 arithmetic: --fmad=false, no fast-math) ----------------------------------------------
// The stopping test of spcu_render_adaptive at a pass boundary, for list entries [0, n) after n_samples samples: pixels that
// pass get d_spp_map[pix] = n_samples, the others are copied, in list order, to d_next_list; *d_n_next = how many.
// radius > 0: a pixel stops only if every pixel of its window (|dx|, |dy| <= radius, clipped to its 8x8 tile and the image)
// passes; d_pass_mask (adaptive_mask_bytes, one word per tile, set to all-ones at the start of the call) holds the pass
// flags between boundaries.  radius == 0 launches the per-pixel test only and does not touch d_pass_mask.
// d_scratch: adaptive_scratch_bytes(n) bytes.  Enqueue only.
size_t      adaptive_scratch_bytes(uint32_t n);
size_t      adaptive_mask_bytes(uint32_t width, uint32_t height);
cudaError_t launch_adaptive_compact(const uint32_t* d_list, uint32_t n, const float* d_rgb_sum, const float* d_lum_sumsq,
                                    uint32_t n_samples, float rel_error, float abs_floor, uint32_t width, uint32_t height,
                                    uint32_t radius, unsigned long long* d_pass_mask, uint32_t* d_spp_map, uint32_t* d_next_list,
                                    void* d_scratch, uint32_t* d_n_next, cudaStream_t st);
// d_spp_map[d_list[i]] = value for i < n
cudaError_t launch_adaptive_fill(const uint32_t* d_list, uint32_t n, uint32_t value, uint32_t* d_spp_map, cudaStream_t st);

// ---- denoise_kernels.cu (exact float32 arithmetic: --fmad=false, no fast-math) -------------------------------------------------
// spcu_render_guides: d_out[pix] for every pixel of the image (spcu_guide, include/spcu.h).  Enqueue only.
cudaError_t launch_guides(const DScene& s, spcu_guide* d_out, cudaStream_t st);
// spcu_denoise's filter (include/spcu.h) over width x height pixels: d_col / d_var are the two ping-pong buffers of the
// iterations (n float4 / n float each), d_out[pix*3+c] the result (may alias d_rgb_sum).  Parameters already checked.  Enqueue only.
cudaError_t launch_denoise(const spcu_guide* d_guides, const float* d_rgb_sum, const float* d_lum_sumsq, const uint32_t* d_spp_map,
                           uint32_t spp, uint32_t width, uint32_t height, const spcu_denoise_params& p, float4* d_col[2],
                           float* d_var[2], float* d_out, cudaStream_t st);

// pixel list of one rank: tiles t with t % stride == offset, 8x8 tiles row major (TileScheduler.h:66-82)
uint32_t    count_partition_pixels(uint32_t width, uint32_t height, uint32_t tile_offset, uint32_t tile_stride);
// d_tile_prefix_scratch: one uint32 per owned tile.  Synchronises the stream.
cudaError_t build_pixel_list(uint32_t width, uint32_t height, uint32_t tile_offset, uint32_t tile_stride,
                             uint32_t* d_pix_list, uint32_t* d_tile_prefix_scratch, cudaStream_t st);

} // namespace spcu
