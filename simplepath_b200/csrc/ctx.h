// Private to the backend's host code: the context behind the opaque spcu_ctx handle and error plumbing.
#pragma once

#include "kernels.h"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

namespace spcu {

// Grow-only device allocation that frees itself.
struct DevBuf
{
    void*  p     = nullptr;
    size_t bytes = 0;

    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes)
    {
        o.p     = nullptr;
        o.bytes = 0;
    }
    ~DevBuf() { release(); }

    cudaError_t reserve(size_t n)
    {
        if (n <= bytes) {
            return cudaSuccess;
        }
        if (p) {
            cudaFree(p);
            p     = nullptr;
            bytes = 0;
        }
        const cudaError_t e = cudaMalloc(&p, n);
        if (e == cudaSuccess) {
            bytes = n;
        }
        return e;
    }

    void release()
    {
        if (p) {
            cudaFree(p);
        }
        p     = nullptr;
        bytes = 0;
    }

    template <typename T>
    T* as() const
    {
        return static_cast<T*>(p);
    }
};

constexpr int      kNumQueues      = 7;        // cur, next, live, shadow, lit, mis, walk
constexpr int      kMaxQueueCounts = 4096;     // device queue-length words zeroed once per batch
constexpr uint64_t kBatchRays      = 1u << 22; // rays per chunk of the batch query entry points
constexpr uint32_t kMaxMaterialSegments = 15;  // materials beyond share the last segment

constexpr int      kMaxBatchLanes  = 8;        // SPCU_OPT_BATCH_LANES
constexpr int      kDefaultBatchLanes = 4;

// Wavefront state of one batch in flight (SPCU_OPT_BATCH_LANES): records, queues, queue counts and the material-sorted queue,
// carved from one allocation and laid out again for every call's batch capacity (spcu_render.cu lay_out_lane).
// Lane 0 runs on the call's stream (`stream` stays NULL); lanes 1..k on their own.
struct WaveLane
{
    DevBuf       mem;
    DWave        wave{};
    uint32_t*    queues[kNumQueues] = {};
    uint32_t*    queue_counts       = nullptr; // uint32[kMaxQueueCounts]
    uint32_t*    sorted             = nullptr; // [n_segments][wave.capacity]: the hand-over between extend and shade
    cudaStream_t stream   = nullptr;
    cudaEvent_t  resolved = nullptr; // recorded after each of the lane's resolve kernels

    void release() { mem.release(); }
};

} // namespace spcu

struct spcu_ctx
{
    int          device = 0;
    std::string  err;
    cudaStream_t stream = nullptr;
    cudaEvent_t  ev0 = nullptr, ev1 = nullptr;
    int          sm_count = 148;
    void*        nccl_comm   = nullptr; // ncclComm_t of this context's rank (comm.cu); NULL: single GPU
    int          comm_rank   = 0;
    int          comm_nranks = 1;
    bool         scratch_in_use = false;   // a render has been enqueued: its last event is ev1 on scratch_stream
    cudaStream_t scratch_stream = nullptr;

    // scene
    bool         have_scene = false;
    spcu::DScene ds{};
    spcu::DevBuf geom_wide; // 4-wide copy of geom_nodes (built at upload)
    spcu::DevBuf geom_big;  // its side table of oversized leaves + the slot counter (device_scene.h)
    spcu::DevBuf geom_nodes, geom_prims, geom_shade, geom_meta, light_nodes, lights, light_order, materials, bxdfs, pool,
        jitter;
    uint64_t scene_bytes = 0;
    spcu_accel built_geom{}; // geometry accelerator header of the resident scene (nodes = NULL: they live on the device)

    // batch-query scratch
    spcu::DevBuf q_rays, q_out, q_aux, q_cnt;

    // wavefront
    uint64_t                  wavefront_size = 0; // 0 = default
    std::vector<spcu::WaveLane> lanes = std::vector<spcu::WaveLane>(1); // lanes[0]: the context's own
    spcu::DevBuf              counters;     // unsigned long long[kNumCounters] followed by TraceCounters
    spcu::DevBuf              pix_list;
    uint32_t                  pix_list_offset = ~0u, pix_list_stride = 0, pix_list_n = 0;
    spcu::DevBuf              host_rgb, host_sq; // device accumulators of the host-buffer entry point
    spcu::DevBuf              packed;            // packed output image (spcu_render_image / spcu_pack_image)
    // adaptive sampling (spcu_render_adaptive): ping-pong active pixel lists, the per-pixel sample counts, a lum_sumsq
    // accumulator for callers that pass none, the compaction's scratch + active count, the per-tile pass flags of the
    // neighbourhood test (radius > 0), and the call's event pair
    spcu::DevBuf              ad_list[2], ad_spp_map, ad_sq, ad_scratch, ad_mask;
    cudaEvent_t               ad_ev[2] = { nullptr, nullptr };
    // denoising (spcu_denoise): the guide buffers and the ping-pong colour / variance buffers of the filter's iterations
    spcu::DevBuf              dn_guides, dn_col[2], dn_var[2];
    void*                     stage[2]    = { nullptr, nullptr }; // page-locked staging of large host->device copies
    cudaEvent_t               stage_ev[2] = { nullptr, nullptr };
    bool                      stage_busy[2] = { false, false };
    spcu::DevBuf              path_radiance;     // float4 per slot of a batch (SPCU_PIPELINE_PATHS)
    uint32_t                  n_materials = 0;
    int                       features    = 0; // feature set of the uploaded scene (features.h)

    uint32_t                 options[SPCU_OPT_COUNT_] = {};
    std::vector<cudaEvent_t> stage_events; // pairs, when SPCU_OPT_STAGE_TIMING is on
    std::vector<int>         stage_kinds;  // spcu::Stage of each pair
    spcu_stage_time          stage_report[spcu::kNumStages] = {};
};

namespace spcu {

int fail(spcu_ctx* c, int code, const char* fmt, ...);
int need_scene(spcu_ctx* c);
// spcu_api.cu: host->device copy on the context's stream.  Large copies from pageable memory go through two page-locked
// staging buffers (CPU memcpy of chunk k+1 overlaps the DMA of chunk k); the source is fully consumed when the call returns.
int copy_to_device(spcu_ctx* c, void* dst, const void* src, size_t bytes);
// image_kernels.cu: mean, row order and sRGB quantisation of device-resident sums, result copied to the host buffer `out`
// d_counts (may be NULL): per-pixel sample counts dividing the sums in place of spp
int pack_device_image(spcu_ctx* c, const float* d_rgb_sum, const uint32_t* d_counts, uint32_t w, uint32_t h, uint32_t spp,
                      uint32_t format, void* out);
// build_kernels.cu: geometry of an UNBUILT scene -> bounds, BVH and leaf-order gather on the device (spcu_upload_scene_build)
int build_scene_geometry(spcu_ctx* c, const spcu_flat_scene* s, const spcu_bounds* extra_bounds, uint32_t* order_out,
                         spcu_accel* built, bool* proper_boxes);

#define CK(ctx, call)                                                                                                     \
    do {                                                                                                                  \
        const cudaError_t e_ = (call);                                                                                    \
        if (e_ != cudaSuccess) {                                                                                          \
            return spcu::fail((ctx), SPCU_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
        }                                                                                                                 \
    } while (0)

} // namespace spcu
