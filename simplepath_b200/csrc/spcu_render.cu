// spcu_render / spcu_render_device: host orchestration of the wavefront loop.
//
// One call renders a partition (a set of 8x8 tiles x a sample range) in batches of at most `wavefront_size` paths:
//
//   raygen -> for depth in [0, max_depth):  extend -> shade (+ all light samples) -> { per light: shadow -> nee_bsdf -> mis ->
//             nee_mis_accumulate } -> advance        -> resolve (per-pixel sums, in sample order)
//
// Every stage is a persistent-style kernel reading its queue length from device memory, so a batch is enqueued without
// any host synchronisation; queues are compacted on the device (warp ballot + one atomic per warp).
#include "ctx.h"

#include <chrono>
#include <cmath>

using namespace spcu;

namespace {

enum Queue { kQCur = 0, kQNext, kQLive, kQShadow, kQLit, kQMis, kQWalk };
constexpr int    kCounterBlock = kNumCounters + kNumStages; // + per-stage item counters
constexpr size_t kCounterBytes = kCounterBlock * sizeof(unsigned long long) + sizeof(TraceCounters);

const char* const kStageNames[kNumStages] = { "raygen",   "extend",    "shade",     "nee_light",         "shadow",           "nee_bsdf",
                                              "mis_trace", "nee_mis_accumulate", "direct_accumulate", "advance", "resolve", "paths" };
inline bool stage_traverses(int st) { return st == kStExtend || st == kStShadow || st == kStMisTrace; }

int queue_fault(spcu_ctx* c, unsigned long long n_faults)
{
    return fail(c, SPCU_ERR_INTERNAL, "%llu kernel(s) gave up on a bounded wait (queue protocol fault); the image is void", n_faults);
}

// segments of the material-sorted queue: one per material (materials beyond the last share it) + the miss segment
uint32_t material_segments(const spcu_ctx* c) { return std::min<uint32_t>(c->n_materials, kMaxMaterialSegments) + 1u; }

// The lane's wavefront state for batches of `capacity` slots (also the stride of the per-light planes and material segments),
// every array at a 256-byte-aligned offset of the lane's one allocation, as cudaMalloc would place it.  The allocation only
// grows: a smaller batch reuses it with its own stride.
int lay_out_lane(spcu_ctx* c, WaveLane& lane, uint32_t capacity, uint32_t n_segments)
{
    const size_t planes = std::max(1u, c->ds.n_lights); // light records and the shadow queue: one plane per light
    auto         carve  = [&](uintptr_t base) {
        size_t off  = 0;
        auto   take = [&](auto*& ptr, size_t n) {
            ptr = reinterpret_cast<std::remove_reference_t<decltype(ptr)>>(base + off);
            off += (n * sizeof *ptr + 255) & ~size_t(255);
        };
        DWave& w = lane.wave;
        take(w.path, capacity);
        take(w.ray, capacity);
        take(w.vertex, capacity);
        take(w.extend, capacity);
        take(w.s0, capacity);
        take(w.light, capacity * planes);
        take(w.mis, capacity);
        take(w.occluded, capacity);
        for (int i = 0; i < kNumQueues; ++i) {
            take(lane.queues[i], capacity * (i == kQShadow ? planes : 1u));
        }
        take(lane.queue_counts, kMaxQueueCounts);
        take(lane.sorted, static_cast<size_t>(n_segments) * capacity);
        return off;
    };
    CK(c, lane.mem.reserve(carve(0)));
    carve(reinterpret_cast<uintptr_t>(lane.mem.p));
    lane.wave.capacity = capacity;
    return SPCU_OK;
}

// Lane k of SPCU_OPT_BATCH_LANES laid out for this call's batches.  Lane 0 must get its memory.  A lane k >= 1 that cannot
// is not an error: it is released and the render goes on with the lanes before it.
int ensure_lane(spcu_ctx* c, size_t k, uint32_t capacity, uint32_t n_segments)
{
    WaveLane& lane = c->lanes[k];
    if (k > 0 && !lane.stream) {
        CK(c, cudaStreamCreateWithFlags(&lane.stream, cudaStreamNonBlocking));
    }
    if (!lane.resolved) {
        CK(c, cudaEventCreateWithFlags(&lane.resolved, cudaEventDisableTiming));
    }
    const int rc = lay_out_lane(c, lane, capacity, n_segments);
    if (rc != SPCU_OK && k > 0) {
        cudaGetLastError(); // (out of memory is sticky-free; clear it)
        lane.release();
    }
    return rc;
}

// Batch shape for `target` slots: the whole pixel list x as many samples as fit, or a slice of the pixel list x one sample.
struct BatchShape
{
    uint32_t pix, smp;
};

BatchShape batch_shape(uint32_t n_pix, uint32_t n_samples, uint64_t target)
{
    if (n_pix > target) {
        return { static_cast<uint32_t>(target), 1 };
    }
    return { n_pix, static_cast<uint32_t>(std::min<uint64_t>(n_samples, std::max<uint64_t>(1, target / n_pix))) };
}

// The wavefront state, queues and counters are context-owned scratch: work on ANOTHER stream than the previous render's must
// not start before that render has finished with them (ev1 is recorded at the end of every render).
int wait_for_scratch(spcu_ctx* c, cudaStream_t st)
{
    if (c->scratch_in_use && c->scratch_stream != st) {
        CK(c, cudaStreamWaitEvent(st, c->ev1, 0));
    }
    return SPCU_OK;
}

int ensure_pixel_list(spcu_ctx* c, const spcu_partition& part)
{
    if (c->pix_list_stride == part.tile_stride && c->pix_list_offset == part.tile_offset) {
        return SPCU_OK;
    }
    const uint32_t w = c->ds.width, h = c->ds.height;
    const uint32_t n_pix   = count_partition_pixels(w, h, part.tile_offset, part.tile_stride);
    const uint32_t n_tiles = ((w + 7) / 8) * ((h + 7) / 8);
    const uint32_t owned   = part.tile_offset < n_tiles ? (n_tiles - part.tile_offset + part.tile_stride - 1) / part.tile_stride : 0;
    // pixel list followed by the per-tile prefix scratch
    CK(c, c->pix_list.reserve((static_cast<size_t>(n_pix) + owned + 1) * sizeof(uint32_t)));
    CK(c, build_pixel_list(w, h, part.tile_offset, part.tile_stride, c->pix_list.as<uint32_t>(),
                           c->pix_list.as<uint32_t>() + n_pix, c->stream));
    c->pix_list_offset = part.tile_offset;
    c->pix_list_stride = part.tile_stride;
    c->pix_list_n      = n_pix;
    return SPCU_OK;
}

// Optional per-launch timing: an event pair around every kernel launch, summed per stage kind afterwards.
struct StageTimer
{
    spcu_ctx*    c;
    bool         on;
    cudaStream_t st;
    size_t       used = 0;

    void begin(int kind)
    {
        ++launches[kind];
        if (!on) return;
        if (used + 2 > c->stage_events.size()) {
            cudaEvent_t a, b;
            cudaEventCreate(&a);
            cudaEventCreate(&b);
            c->stage_events.push_back(a);
            c->stage_events.push_back(b);
        }
        c->stage_kinds.resize(c->stage_events.size() / 2);
        c->stage_kinds[used / 2] = kind;
        cudaEventRecord(c->stage_events[used], st);
    }
    void end()
    {
        if (!on) return;
        cudaEventRecord(c->stage_events[used + 1], st);
        used += 2;
    }
    uint64_t launches[kNumStages] = {};

    void collect(float& trace_ms, float& shade_ms)
    {
        trace_ms = shade_ms = 0.0f;
        for (size_t i = 0; i < used; i += 2) {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, c->stage_events[i], c->stage_events[i + 1]);
            const int st = c->stage_kinds[i / 2];
            c->stage_report[st].ms += ms;
            (stage_traverses(st) ? trace_ms : shade_ms) += ms;
        }
    }
};

// Device counters -> spcu_stats (+ the per-stage report).  Synchronises `st`.
int read_back_stats(spcu_ctx* c, cudaStream_t st, spcu_stats* stats, uint64_t launches, StageTimer& timer)
{
    auto* d_counters = c->counters.as<unsigned long long>();
    CK(c, cudaEventSynchronize(c->ev1));
    unsigned long long h[kCounterBlock];
    TraceCounters      tc{};
    CK(c, cudaMemcpyAsync(h, d_counters, sizeof h, cudaMemcpyDeviceToHost, st));
    CK(c, cudaMemcpyAsync(&tc, d_counters + kCounterBlock, sizeof tc, cudaMemcpyDeviceToHost, st));
    CK(c, cudaStreamSynchronize(st));
    stats->paths           = h[kCntPaths];
    stats->rays_closest    = h[kCntRaysClosest];
    stats->rays_any        = h[kCntRaysAny];
    stats->rays_lights     = h[kCntRaysLights];
    stats->shade_calls     = h[kCntShadeCalls];
    stats->nodes_visited   = tc.nodes;
    stats->prims_tested    = tc.tris;
    stats->xf_prims_tested = tc.xf;
    stats->kernel_launches = launches;
    if (h[kCntErrors]) {
        return queue_fault(c, h[kCntErrors]);
    }
    CK(c, cudaEventElapsedTime(&stats->device_ms, c->ev0, c->ev1));
    for (int i = 0; i < kNumStages; ++i) {
        spcu_stage_time& r = c->stage_report[i];
        std::memset(&r, 0, sizeof r);
        std::snprintf(r.name, sizeof r.name, "%s", kStageNames[i]);
        r.launches  = timer.launches[i];
        r.items     = h[kNumCounters + i];
        r.traverses = stage_traverses(i) ? 1u : 0u;
    }
    timer.collect(stats->trace_ms, stats->shade_ms);
    return SPCU_OK;
}

// SPCU_PIPELINE_AUTO: the organisation that measures faster for the scene's feature set (DESIGN.md §4)
uint32_t resolve_pipeline(const spcu_ctx* c)
{
    const uint32_t pipeline = c->options[SPCU_OPT_PIPELINE];
    if (pipeline != SPCU_PIPELINE_AUTO) {
        return pipeline;
    }
    return (c->features == FeatAnalytic::id && smwave_supports(c->ds)) ? SPCU_PIPELINE_SMWAVE : SPCU_PIPELINE_WAVEFRONT;
}

// Argument checks of a render call, ordering of the context's scratch after earlier renders on other streams, and the
// partition's pixel list (c->pix_list, c->pix_list_n).  st = the stream the call runs on.
int prepare_render(spcu_ctx* c, const spcu_partition* part, const float* d_rgb_sum, cudaStream_t caller_stream, bool have_caller_stream,
                   cudaStream_t& st)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!part || !d_rgb_sum) {
        return fail(c, SPCU_ERR_INVALID, "partition or accumulator is NULL");
    }
    const DScene& s = c->ds;
    if (part->tile_stride == 0 || part->tile_offset >= part->tile_stride) {
        return fail(c, SPCU_ERR_INVALID, "bad tile partition %u/%u", part->tile_offset, part->tile_stride);
    }
    if (part->sample_begin > part->sample_end || part->sample_end > part->spp_total || part->spp_total > s.spp) {
        return fail(c, SPCU_ERR_INVALID, "bad sample range [%u,%u) of %u (jitter table holds %u)", part->sample_begin,
                    part->sample_end, part->spp_total, s.spp);
    }
    if (part->integrator > SPCU_INTEGRATOR_WHITTED) {
        return fail(c, SPCU_ERR_INVALID, "unknown integrator %u", part->integrator);
    }
    // The caller's stream (spcu_render_device) orders this call after the caller's earlier work on that stream.
    st = have_caller_stream ? caller_stream : c->stream;
    if (int rc = wait_for_scratch(c, st); rc != SPCU_OK) return rc;
    c->scratch_in_use = true;
    c->scratch_stream = st;
    return ensure_pixel_list(c, *part);
}

// The batch loop of every pipeline: samples [sample_begin, sample_begin + n_samples) of the n_pix pixels of d_pix_list (n_pix,
// n_samples > 0), added to the accumulators in sample order.  One batch is the persistent path / SM-local kernel on the call's
// stream, or the queue wavefront's stage chain on lane `batch % n_lanes`; then its resolve.
int render_batches(spcu_ctx* c, const spcu_partition* part, const uint32_t* d_pix_list, uint32_t n_pix, uint32_t sample_begin,
                   uint32_t n_samples, float* d_rgb_sum, float* d_lum_sumsq, spcu_stats* stats, cudaStream_t st)
{
    const DScene&  s        = c->ds;
    const uint32_t pipeline = resolve_pipeline(c);
    if (pipeline == SPCU_PIPELINE_SMWAVE && !smwave_supports(s)) {
        return fail(c, SPCU_ERR_INVALID, "SPCU_PIPELINE_SMWAVE: max_depth %u / %u lights exceed its packed path flags",
                    s.max_depth, s.n_lights);
    }
    const bool wavefront = pipeline == SPCU_PIPELINE_WAVEFRONT;
    // the persistent kernels keep 16 B of radiance per slot, the queue wavefront its whole state
    const BatchShape shape    = batch_shape(n_pix, n_samples, c->wavefront_size ? c->wavefront_size : wavefront ? 1ull << 24 : 1ull << 27);
    const uint32_t   capacity = shape.pix * shape.smp;
    CK(c, c->counters.reserve(kCounterBytes));
    auto*          d_counters = c->counters.as<unsigned long long>();
    TraceCounters* d_cnt      = c->options[SPCU_OPT_COUNT_NODES] ? reinterpret_cast<TraceCounters*>(d_counters + kCounterBlock) : nullptr;
    StageTimer     timer{ c, c->options[SPCU_OPT_STAGE_TIMING] != 0, st };
    uint64_t       launches = 0;

    const uint32_t n_lights    = s.n_lights;
    const uint32_t max_depth   = part->integrator == SPCU_INTEGRATOR_DIRECT_LIGHTING ? std::min(1u, s.max_depth) : s.max_depth;
    const bool     nee         = part->integrator == SPCU_INTEGRATOR_ITERATIVE_RRNEE;
    const bool     whitted     = part->integrator == SPCU_INTEGRATOR_WHITTED;
    const bool     direct      = part->integrator == SPCU_INTEGRATOR_DIRECT_LIGHTING || whitted; // per-light direct term
    const uint32_t n_segments  = material_segments(c);
    const uint32_t counts_need = 1 + max_depth * (4 + 7 * n_lights + n_segments);
    // ---- batches in flight (SPCU_OPT_BATCH_LANES) of the queue wavefront: lane 0 on the call's stream -----------------------
    uint32_t n_lanes = 1;
    if (wavefront) {
        if (counts_need > static_cast<uint32_t>(kMaxQueueCounts)) {
            return fail(c, SPCU_ERR_LIMIT, "max_depth x lights needs %u queue counters (limit %d)", counts_need, kMaxQueueCounts);
        }
        const uint64_t n_batches  = static_cast<uint64_t>((n_pix + shape.pix - 1) / shape.pix) * ((n_samples + shape.smp - 1) / shape.smp);
        uint32_t       want_lanes = c->options[SPCU_OPT_BATCH_LANES] ? c->options[SPCU_OPT_BATCH_LANES] : kDefaultBatchLanes;
        if (timer.on || d_cnt) {
            want_lanes = 1; // per-launch events and the node counters describe one batch at a time
        }
        want_lanes = static_cast<uint32_t>(std::min<uint64_t>({ want_lanes, kMaxBatchLanes, n_batches }));
        if (c->lanes.size() < want_lanes) {
            c->lanes.resize(want_lanes);
        }
        if (int rc = ensure_lane(c, 0, capacity, n_segments); rc != SPCU_OK) return rc;
        while (n_lanes < want_lanes && ensure_lane(c, n_lanes, capacity, n_segments) == SPCU_OK) {
            ++n_lanes; // (not enough memory for another lane: render with the ones we have)
        }
    } else {
        CK(c, c->path_radiance.reserve(static_cast<size_t>(capacity) * sizeof(float4)));
    }

    // raygen and the stage chain of one batch of the queue wavefront: slots [0, np x ns) on `lane`
    auto stage_chain = [&](WaveLane& lane, const Launch& L, const uint32_t* d_pix, uint32_t np, uint32_t sample0, uint32_t ns) {
        const uint32_t max_n    = np * ns;
        uint32_t**     q        = lane.queues;
        uint32_t*      d_counts = lane.queue_counts;
        CK(c, cudaMemsetAsync(d_counts, 0, counts_need * sizeof(uint32_t), L.stream));
        uint32_t next_count = 0;
        auto     new_count  = [&]() { return d_counts + next_count++; };

        uint32_t* n_cur = new_count();
        timer.begin(kStRaygen);
        launch_raygen(L, s, lane.wave, d_pix, np, sample0, ns, q[kQCur], n_cur, d_counters);
        timer.end();
        ++launches;

        uint32_t* q_cur  = q[kQCur];
        uint32_t* q_next = q[kQNext];
        // advance (of depth d) + the set-up of extend (of depth d + 1) as ONE kernel where the extend stage has a `begin`
        // kernel to put it in; the live queue of depth d then goes to extend directly
        const bool fuse_advance    = !whitted && extend_fuses_advance(L, q[kQWalk], d_cnt);
        bool       pending_advance = false;
        for (uint32_t depth = 0; depth < max_depth; ++depth) {
            RenderParams p{ part->seed, part->integrator, depth, 0 };
            SortedQueue  sorted{ lane.sorted, d_counts + next_count, n_segments, capacity };
            next_count += n_segments;
            timer.begin(kStExtend);
            uint32_t*         cursor = new_count();
            const AdvanceArgs adv{ part->seed, depth - 1u };
            launches += launch_extend(L, s, lane.wave, q_cur, n_cur, max_n, cursor, sorted,
                                      // (node counting is DEFINED on the reference-order walk: DESIGN.md byte model)
                                      c->options[SPCU_OPT_TRAVERSAL] == SPCU_TRAVERSAL_ORDERED && !d_cnt, q[kQWalk], new_count(),
                                      d_counters, d_cnt, pending_advance ? &adv : nullptr);
            pending_advance = false;
            timer.end();
            uint32_t* n_live   = new_count();
            uint32_t* n_shadow = d_counts + next_count; // one shadow queue (and counter) per light
            next_count += n_lights;
            uint32_t* q_shadow = (nee || direct) ? q[kQShadow] : nullptr;
            timer.begin(kStShade);
            launch_shade(L, s, lane.wave, p, sorted, max_n, q[kQLive], n_live, q_shadow, n_shadow, d_counters);
            timer.end();
            launches += 1;
            if (nee || direct) {
                for (uint32_t li = 0; li < n_lights; ++li) {
                    p.light_index        = li;
                    uint32_t* q_shadow_l = q_shadow + static_cast<size_t>(li) * capacity;
                    uint32_t* n_lit      = direct ? nullptr : new_count();
                    timer.begin(kStShadow);
                    uint32_t* cursor_l = new_count();
                    launches += launch_shadow(L, s, lane.wave, q_shadow_l, n_shadow + li, max_n, li, cursor_l,
                                              direct ? nullptr : q[kQLit], n_lit, q[kQWalk], new_count(), d_counters, d_cnt);
                    timer.end();
                    if (direct) {
                        timer.begin(kStDirectAccumulate);
                        launch_direct_accumulate(L, s, lane.wave, p, q_shadow_l, n_shadow + li, max_n, d_counters);
                        timer.end();
                        ++launches;
                        continue;
                    }
                    uint32_t* n_mis = new_count();
                    timer.begin(kStNeeBsdf);
                    launch_nee_bsdf(L, s, lane.wave, p, q[kQLit], n_lit, max_n, q[kQMis], n_mis, d_counters);
                    timer.end();
                    timer.begin(kStMisTrace);
                    uint32_t* cursor_m = new_count();
                    launches += launch_mis_trace(L, s, lane.wave, q[kQMis], n_mis, max_n, cursor_m, q[kQWalk], new_count(), d_counters, d_cnt);
                    timer.end();
                    timer.begin(kStNeeMisAccumulate);
                    launch_nee_mis_accumulate(L, s, lane.wave, q[kQMis], n_mis, max_n, d_counters);
                    timer.end();
                    launches += 2;
                }
            }
            if (direct && !whitted) {
                break;
            }
            if (fuse_advance) {
                // the live queue is read by the next depth's extend (and rewritten only by the shade stage after it):
                // two buffers in turn, so that this depth's q_live is intact while the next one's is being filled
                q_cur           = q[kQLive];
                n_cur           = n_live;
                pending_advance = true;
                std::swap(q[kQLive], q[kQNext]);
                continue;
            }
            uint32_t* n_next = new_count();
            timer.begin(kStAdvance);
            if (whitted) {
                launch_whitted_advance(L, s, lane.wave, p, q[kQLive], n_live, max_n, q_next, n_next, d_counters);
            } else {
                launch_advance(L, s, lane.wave, p, q[kQLive], n_live, max_n, q_next, n_next, d_counters);
            }
            timer.end();
            ++launches;
            std::swap(q_cur, q_next);
            n_cur = n_next;
        }
        return SPCU_OK;
    };

    CK(c, cudaMemsetAsync(d_counters, 0, kCounterBytes, st));
    CK(c, cudaEventRecord(c->ev0, st));
    for (uint32_t k = 1; k < n_lanes; ++k) { // the other lanes start after whatever the call's stream held before
        CK(c, cudaStreamWaitEvent(c->lanes[k].stream, c->ev0, 0));
    }
    uint64_t batch = 0;
    for (uint32_t pb = 0; pb < n_pix; pb += shape.pix) {
        const uint32_t np = std::min(shape.pix, n_pix - pb);
        for (uint32_t sb = 0; sb < n_samples; sb += shape.smp, ++batch) {
            const uint32_t ns   = std::min(shape.smp, n_samples - sb);
            const uint64_t k    = batch % n_lanes;
            WaveLane&      lane = c->lanes[k];
            const Launch   L{ c->sm_count, k ? lane.stream : st, c->features };
            if (wavefront) {
                if (int rc = stage_chain(lane, L, d_pix_list + pb, np, sample_begin + sb, ns); rc != SPCU_OK) return rc;
            } else {
                timer.begin(kStPaths);
                if (pipeline == SPCU_PIPELINE_SMWAVE) {
                    CK(c, launch_smwave(L, s, d_pix_list + pb, np, sample_begin + sb, ns, part->seed, part->integrator,
                                        c->path_radiance.as<float4>(), d_counters, d_cnt));
                } else {
                    launch_paths(L, s, d_pix_list + pb, np, sample_begin + sb, ns, part->seed, part->integrator,
                                 c->path_radiance.as<float4>(), d_counters, d_cnt);
                }
                timer.end();
                ++launches;
            }
            // batches add their samples to the accumulators in batch order, whichever lane ran them: this resolve waits for the
            // previous batch's (the float sums, and so the image, do not depend on the number of lanes)
            if (n_lanes > 1 && batch > 0) {
                CK(c, cudaStreamWaitEvent(L.stream, c->lanes[(batch - 1) % n_lanes].resolved, 0));
            }
            timer.begin(kStResolve);
            launch_resolve(L, wavefront ? &lane.wave.path->L : c->path_radiance.as<float4>(), wavefront ? 2 : 1, d_pix_list + pb, np,
                           ns, d_rgb_sum, d_lum_sumsq, d_counters);
            timer.end();
            ++launches;
            if (n_lanes > 1) {
                CK(c, cudaEventRecord(lane.resolved, L.stream));
            }
            CK(c, cudaGetLastError());
        }
    }
    for (uint32_t k = 1; k < n_lanes; ++k) { // join: the call's stream ends after every lane's last resolve
        CK(c, cudaStreamWaitEvent(st, c->lanes[k].resolved, 0));
    }
    CK(c, cudaEventRecord(c->ev1, st));

    if (stats) {
        if (int rc = read_back_stats(c, st, stats, launches, timer); rc != SPCU_OK) return rc;
        if (!wavefront) {
            c->stage_report[kStPaths].items = stats->paths;
        }
    }
    return SPCU_OK;
}

int render_impl(spcu_ctx* c, const spcu_partition* part, float* d_rgb_sum, float* d_lum_sumsq, spcu_stats* stats,
                cudaStream_t caller_stream, bool have_caller_stream)
{
    cudaStream_t st = nullptr;
    if (int rc = prepare_render(c, part, d_rgb_sum, caller_stream, have_caller_stream, st); rc != SPCU_OK) return rc;
    const uint32_t n_pix     = c->pix_list_n;
    const uint32_t n_samples = part->sample_end - part->sample_begin;
    if (stats) {
        std::memset(stats, 0, sizeof *stats);
    }
    if (n_pix == 0 || n_samples == 0) {
        return SPCU_OK;
    }
    return render_batches(c, part, c->pix_list.as<uint32_t>(), n_pix, part->sample_begin, n_samples, d_rgb_sum, d_lum_sumsq, stats,
                          st);
}

// the counters and kernel times of one adaptive pass, added to the call's (its device_ms is timed over the whole call)
void add_stats(spcu_stats& total, const spcu_stats& pass)
{
    total.paths += pass.paths;
    total.rays_closest += pass.rays_closest;
    total.rays_any += pass.rays_any;
    total.rays_lights += pass.rays_lights;
    total.nodes_visited += pass.nodes_visited;
    total.prims_tested += pass.prims_tested;
    total.xf_prims_tested += pass.xf_prims_tested;
    total.shade_calls += pass.shade_calls;
    total.kernel_launches += pass.kernel_launches;
    total.trace_ms += pass.trace_ms;
    total.shade_ms += pass.shade_ms;
}

// spcu_render_adaptive(_device): the pass loop over shrinking pixel lists (schedule and stopping test: include/spcu.h).  Pass 0
// renders the partition's own list (c->pix_list, read only); after it the active pixels ping-pong between c->ad_list[0/1].
int adaptive_impl(spcu_ctx* c, const spcu_partition* part, const spcu_adaptive* ad, float* d_rgb_sum, float* d_lum_sumsq,
                  uint32_t* d_spp_map, uint32_t* n_passes, spcu_stats* stats, cudaStream_t caller_stream, bool have_caller_stream)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!ad || !d_spp_map) {
        return fail(c, SPCU_ERR_INVALID, "adaptive parameters or spp map is NULL");
    }
    if (ad->min_spp < 2 || ad->pass_spp < 1 || !std::isfinite(ad->rel_error) || !(ad->rel_error >= 0.0f) ||
        !std::isfinite(ad->abs_floor) || !(ad->abs_floor >= 0.0f)) {
        return fail(c, SPCU_ERR_INVALID, "bad adaptive parameters: min_spp %u (>= 2), pass_spp %u (>= 1), rel_error %g, abs_floor %g "
                    "(finite, >= 0)", ad->min_spp, ad->pass_spp, ad->rel_error, ad->abs_floor);
    }
    if (ad->radius > 7) {
        return fail(c, SPCU_ERR_INVALID, "bad adaptive window radius %u (0..7: the window is clipped to the pixel's 8x8 tile)",
                    ad->radius);
    }
    if (part && part->sample_begin != 0) {
        return fail(c, SPCU_ERR_INVALID, "adaptive rendering starts at sample 0 (sample_begin %u)", part->sample_begin);
    }
    cudaStream_t st = nullptr;
    if (int rc = prepare_render(c, part, d_rgb_sum, caller_stream, have_caller_stream, st); rc != SPCU_OK) return rc;

    const size_t n_pixels = static_cast<size_t>(c->ds.width) * c->ds.height;
    float*       d_sq     = d_lum_sumsq;
    if (!d_sq) { // the stopping test needs the sums of squares
        CK(c, c->ad_sq.reserve(n_pixels * sizeof(float)));
        d_sq = c->ad_sq.as<float>();
    }
    for (auto& e : c->ad_ev) {
        if (!e) CK(c, cudaEventCreate(&e));
    }
    CK(c, cudaEventRecord(c->ad_ev[0], st));
    CK(c, cudaMemsetAsync(d_rgb_sum, 0, n_pixels * 3 * sizeof(float), st));
    CK(c, cudaMemsetAsync(d_sq, 0, n_pixels * sizeof(float), st));
    CK(c, cudaMemsetAsync(d_spp_map, 0, n_pixels * sizeof(uint32_t), st));
    spcu_stats total{};
    uint32_t   passes = 0;
    const uint32_t  budget = part->sample_end;
    const uint32_t* list   = c->pix_list.as<uint32_t>();
    uint32_t        n      = c->pix_list_n;
    if (n > 0 && budget > 0) {
        for (auto& l : c->ad_list) {
            CK(c, l.reserve(static_cast<size_t>(n) * sizeof(uint32_t)));
        }
        CK(c, c->ad_scratch.reserve(sizeof(uint32_t) + adaptive_scratch_bytes(n))); // active count, then the compaction's scratch
        uint32_t* d_n_next = c->ad_scratch.as<uint32_t>();
        if (ad->radius > 0) { // all pass: pixels that stop keep their set bit, those never tested are outside every window
            const size_t mask_bytes = adaptive_mask_bytes(c->ds.width, c->ds.height);
            CK(c, c->ad_mask.reserve(mask_bytes));
            CK(c, cudaMemsetAsync(c->ad_mask.p, 0xff, mask_bytes, st));
        }
        uint32_t  begin = 0, end = std::min(ad->min_spp, budget);
        for (;;) {
            spcu_stats ps{}; // (read back after every pass: the fault counter is checked there)
            if (int rc = render_batches(c, part, list, n, begin, end - begin, d_rgb_sum, d_sq, &ps, st); rc != SPCU_OK) return rc;
            ++passes;
            add_stats(total, ps);
            if (end >= budget) {
                break;
            }
            uint32_t* next = c->ad_list[passes & 1u].as<uint32_t>(); // never the list being read (pass 0 reads c->pix_list)
            CK(c, launch_adaptive_compact(list, n, d_rgb_sum, d_sq, end, ad->rel_error, ad->abs_floor, c->ds.width, c->ds.height,
                                          ad->radius, c->ad_mask.as<unsigned long long>(), d_spp_map, next, d_n_next + 1, d_n_next, st));
            total.kernel_launches += ad->radius > 0 ? 4 : 3;
            CK(c, cudaMemcpyAsync(&n, d_n_next, sizeof n, cudaMemcpyDeviceToHost, st));
            CK(c, cudaStreamSynchronize(st)); // the next pass's batches are shaped by the number of active pixels
            list = next;
            if (n == 0) {
                break;
            }
            begin = end;
            end   = std::min(end + ad->pass_spp, budget);
        }
        CK(c, launch_adaptive_fill(list, n, budget, d_spp_map, st)); // still active when the budget ran out
    }
    CK(c, cudaEventRecord(c->ad_ev[1], st));
    if (stats) {
        CK(c, cudaEventSynchronize(c->ad_ev[1]));
        CK(c, cudaEventElapsedTime(&total.device_ms, c->ad_ev[0], c->ad_ev[1]));
        *stats = total;
    }
    if (n_passes) {
        *n_passes = passes;
    }
    return SPCU_OK;
}

// spcu_render_adaptive_predicted(_device): rounds over bucketed pixel lists (grid, prediction and stopping rule:
// include/spcu.h).  Round 0 renders the partition's own list; after it the pixels still going ping-pong between
// c->ad_list[0/1], bucket-contiguous, each pixel's grid index in c->ad_level.  One render call per non-empty bucket.
int adaptive_predicted_impl(spcu_ctx* c, const spcu_partition* part, const spcu_adaptive_predicted* ap, float* d_rgb_sum,
                            float* d_lum_sumsq, uint32_t* d_spp_map, uint32_t* n_rounds, uint32_t* n_calls, spcu_stats* stats,
                            cudaStream_t caller_stream, bool have_caller_stream)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!ap || !d_spp_map) {
        return fail(c, SPCU_ERR_INVALID, "adaptive parameters or spp map is NULL");
    }
    if (ap->min_spp < 2 || ap->max_step < 1 || ap->max_step > 8 || !std::isfinite(ap->rel_error) || !(ap->rel_error >= 0.0f) ||
        !std::isfinite(ap->abs_floor) || !(ap->abs_floor >= 0.0f)) {
        return fail(c, SPCU_ERR_INVALID, "bad adaptive parameters: min_spp %u (>= 2), max_step %u (1..8), rel_error %g, abs_floor %g "
                    "(finite, >= 0)", ap->min_spp, ap->max_step, ap->rel_error, ap->abs_floor);
    }
    if (ap->radius > 7) {
        return fail(c, SPCU_ERR_INVALID, "bad adaptive window radius %u (0..7: the window is clipped to the pixel's 8x8 tile)",
                    ap->radius);
    }
    if (part && part->sample_begin != 0) {
        return fail(c, SPCU_ERR_INVALID, "adaptive rendering starts at sample 0 (sample_begin %u)", part->sample_begin);
    }
    cudaStream_t st = nullptr;
    if (int rc = prepare_render(c, part, d_rgb_sum, caller_stream, have_caller_stream, st); rc != SPCU_OK) return rc;

    const size_t n_pixels = static_cast<size_t>(c->ds.width) * c->ds.height;
    float*       d_sq     = d_lum_sumsq;
    if (!d_sq) { // the stopping test needs the sums of squares
        CK(c, c->ad_sq.reserve(n_pixels * sizeof(float)));
        d_sq = c->ad_sq.as<float>();
    }
    for (auto& e : c->ad_ev) {
        if (!e) CK(c, cudaEventCreate(&e));
    }
    CK(c, cudaEventRecord(c->ad_ev[0], st));
    CK(c, cudaMemsetAsync(d_rgb_sum, 0, n_pixels * 3 * sizeof(float), st));
    CK(c, cudaMemsetAsync(d_sq, 0, n_pixels * sizeof(float), st));
    CK(c, cudaMemsetAsync(d_spp_map, 0, n_pixels * sizeof(uint32_t), st));
    spcu_stats     total{};
    uint32_t       rounds = 0, calls = 0;
    const uint32_t budget = part->sample_end;
    // the grid g_0 = min(min_spp, budget), g_{i+1} = min(2 g_i, budget): at most 32 counts below 2^32
    std::vector<uint32_t> g{ std::min(ap->min_spp, budget) };
    while (g.back() < budget) {
        g.push_back(static_cast<uint32_t>(std::min<uint64_t>(2ull * g.back(), budget)));
    }
    const uint32_t  last = static_cast<uint32_t>(g.size() - 1);
    const uint32_t* list = c->pix_list.as<uint32_t>();
    const uint32_t  n    = c->pix_list_n;
    auto            render = [&](const uint32_t* l, uint32_t np, uint32_t begin, uint32_t end) {
        spcu_stats ps{}; // (read back after every call: the fault counter is checked there)
        if (int rc = render_batches(c, part, l, np, begin, end - begin, d_rgb_sum, d_sq, &ps, st); rc != SPCU_OK) return rc;
        ++calls;
        add_stats(total, ps);
        return SPCU_OK;
    };
    if (n > 0 && budget > 0) {
        if (int rc = render(list, n, 0, g[0]); rc != SPCU_OK) return rc;
        rounds = 1;
        if (last == 0) {
            CK(c, launch_adaptive_fill(list, n, budget, d_spp_map, st));
        } else {
            const uint32_t n_buckets = adaptive_predict_buckets(last, ap->max_step);
            for (auto& l : c->ad_list) {
                CK(c, l.reserve(static_cast<size_t>(n) * sizeof(uint32_t)));
            }
            // bucket offsets + total, then the rounds' scratch
            const size_t offsets_bytes = (static_cast<size_t>(n_buckets) + 1) * sizeof(uint32_t);
            CK(c, c->ad_scratch.reserve(offsets_bytes + adaptive_predict_scratch_bytes(n, n_buckets)));
            CK(c, c->ad_level.reserve(n_pixels));
            CK(c, cudaMemsetAsync(c->ad_level.p, 0, n_pixels, st));
            auto* d_offsets = c->ad_scratch.as<uint32_t>();
            void* d_scratch = static_cast<char*>(c->ad_scratch.p) + offsets_bytes;
            if (ap->radius > 0) { // all pass: pixels that stop set their bit, those never tested are outside every window
                const size_t mask_bytes = adaptive_mask_bytes(c->ds.width, c->ds.height);
                CK(c, c->ad_mask.reserve(mask_bytes));
                CK(c, cudaMemsetAsync(c->ad_mask.p, 0xff, mask_bytes, st));
            }
            struct Range
            {
                uint32_t offset, count, n_samples;
            };
            std::vector<Range>    tested{ { 0, n, g[0] } }; // the entries of `list` to test, by their count
            std::vector<uint32_t> h_offsets(n_buckets + 1);
            uint32_t              n_test = n, next_k = 1;
            while (n_test > 0) {
                uint32_t* next = c->ad_list[next_k].as<uint32_t>(); // never the list being read (round 0 reads c->pix_list)
                next_k ^= 1u;
                if (ap->radius > 0) { // every pass flag is written before any decision reads one
                    for (const Range& r : tested) {
                        CK(c, launch_adaptive_test(list + r.offset, r.count, d_rgb_sum, d_sq, r.n_samples, ap->rel_error, ap->abs_floor,
                                                   c->ds.width, c->ad_mask.as<unsigned long long>(), st));
                    }
                    total.kernel_launches += tested.size();
                }
                CK(c, launch_adaptive_predict(list, n_test, d_rgb_sum, d_sq, g[0], budget, last, ap->max_step, ap->rel_error, ap->abs_floor,
                                              c->ds.width, c->ds.height, ap->radius, c->ad_mask.as<unsigned long long>(),
                                              c->ad_level.as<uint8_t>(), d_spp_map, next, d_scratch, d_offsets, st));
                total.kernel_launches += 3;
                CK(c, cudaMemcpyAsync(h_offsets.data(), d_offsets, h_offsets.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
                CK(c, cudaStreamSynchronize(st)); // the round's calls are shaped by its buckets
                list = next;
                tested.clear();
                bool rendered = false;
                for (uint32_t j = 0; j < last; ++j) { // calls in a fixed order: j ascending, then t
                    for (uint32_t t = j + 1; t <= std::min(j + ap->max_step, last); ++t) {
                        const uint32_t b    = adaptive_predict_bucket(j, t, last, ap->max_step);
                        const uint32_t size = h_offsets[b + 1] - h_offsets[b];
                        if (size == 0) {
                            continue;
                        }
                        if (int rc = render(list + h_offsets[b], size, g[j], g[t]); rc != SPCU_OK) return rc;
                        rendered = true;
                        if (t < last) {
                            tested.push_back({ h_offsets[b], size, g[t] });
                        }
                    }
                }
                rounds += rendered ? 1u : 0u;
                n_test = h_offsets[adaptive_predict_bucket(0, last, last, ap->max_step)]; // the buckets of t < last come first
            }
        }
    }
    CK(c, cudaEventRecord(c->ad_ev[1], st));
    if (stats) {
        CK(c, cudaEventSynchronize(c->ad_ev[1]));
        CK(c, cudaEventElapsedTime(&total.device_ms, c->ad_ev[0], c->ad_ev[1]));
        *stats = total;
    }
    if (n_rounds) {
        *n_rounds = rounds;
    }
    if (n_calls) {
        *n_calls = calls;
    }
    return SPCU_OK;
}

// The host-buffer entry points synchronise anyway: they also read the fault counter (kCntErrors) when no stats were asked
// for, so a kernel that gave up on a bounded wait fails the call instead of returning a void image.
int sync_and_check_faults(spcu_ctx* c, bool already_checked)
{
    unsigned long long faults = 0;
    if (!already_checked && c->counters.p) {
        CK(c, cudaMemcpyAsync(&faults, c->counters.as<unsigned long long>() + kCntErrors, sizeof faults, cudaMemcpyDeviceToHost,
                              c->stream));
    }
    CK(c, cudaStreamSynchronize(c->stream));
    return faults ? queue_fault(c, faults) : SPCU_OK;
}

// The host-buffer entry points: device accumulators for the image (c->host_rgb, and c->host_sq `with_sumsq`), zeroed or, where
// rgb_in (and sq_in) are given, holding those host arrays; `render(d_rgb_sum, d_lum_sumsq)` enqueues the call's work on the
// context's stream; the accumulators go back to rgb_sum / lum_sumsq where those are not NULL, and the call ends in the fault check.
template <typename Render>
int host_buffer_render(spcu_ctx* c, bool with_sumsq, const float* rgb_in, const float* sq_in, float* rgb_sum, float* lum_sumsq,
                       bool already_checked, Render&& render)
{
    const size_t sq_bytes = static_cast<size_t>(c->ds.width) * c->ds.height * sizeof(float), rgb_bytes = 3 * sq_bytes;
    CK(c, c->host_rgb.reserve(rgb_bytes));
    float* d_sq = nullptr;
    if (with_sumsq) {
        CK(c, c->host_sq.reserve(sq_bytes));
        d_sq = c->host_sq.as<float>();
    }
    if (rgb_in) {
        CK(c, cudaMemcpyAsync(c->host_rgb.p, rgb_in, rgb_bytes, cudaMemcpyHostToDevice, c->stream));
        if (d_sq) CK(c, cudaMemcpyAsync(d_sq, sq_in, sq_bytes, cudaMemcpyHostToDevice, c->stream));
    } else {
        CK(c, cudaMemsetAsync(c->host_rgb.p, 0, rgb_bytes, c->stream));
        if (d_sq) CK(c, cudaMemsetAsync(d_sq, 0, sq_bytes, c->stream));
    }
    if (int rc = render(c->host_rgb.as<float>(), d_sq); rc != SPCU_OK) return rc;
    if (rgb_sum) CK(c, cudaMemcpyAsync(rgb_sum, c->host_rgb.p, rgb_bytes, cudaMemcpyDeviceToHost, c->stream));
    if (lum_sumsq && d_sq) CK(c, cudaMemcpyAsync(lum_sumsq, d_sq, sq_bytes, cudaMemcpyDeviceToHost, c->stream));
    return sync_and_check_faults(c, already_checked);
}

// spcu_denoise(_device) and, `conserve`, spcu_denoise_conserving(_device): guides into c->dn_guides, then the filter through
// the ping-pong buffers c->dn_col / c->dn_var (and, for the flux form, c->dn_var_pf / c->dn_wsum).  Those are context scratch
// like the renders' (wait_for_scratch): a call on another stream starts after the previous user is done.
int denoise_impl(spcu_ctx* c, const float* d_rgb_sum, const float* d_lum_sumsq, const uint32_t* d_spp_map, uint32_t spp,
                 const spcu_denoise_params* p, float* d_out, cudaStream_t st, bool conserve)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!p || !d_rgb_sum || !d_lum_sumsq || !d_out) {
        return fail(c, SPCU_ERR_INVALID, "parameters, rgb_sum, lum_sumsq or out is NULL");
    }
    if (p->iterations < 1 || p->iterations > 8 || !std::isfinite(p->sigma_l) || !(p->sigma_l > 0.0f) || !std::isfinite(p->sigma_z) ||
        !(p->sigma_z > 0.0f) || !std::isfinite(p->sigma_a) || !(p->sigma_a > 0.0f)) {
        return fail(c, SPCU_ERR_INVALID, "bad denoise parameters: iterations %u (1..8), sigma_l %g, sigma_z %g, sigma_a %g (finite, > 0)",
                    p->iterations, p->sigma_l, p->sigma_z, p->sigma_a);
    }
    if (!d_spp_map && spp == 0) {
        return fail(c, SPCU_ERR_INVALID, "spp is 0 and there is no spp map");
    }
    const size_t n = static_cast<size_t>(c->ds.width) * c->ds.height;
    CK(c, c->dn_guides.reserve(n * sizeof(spcu_guide)));
    float4* col[2];
    float*  var[2];
    for (int k = 0; k < 2; ++k) {
        CK(c, c->dn_col[k].reserve(n * sizeof(float4)));
        CK(c, c->dn_var[k].reserve(n * sizeof(float)));
        col[k] = c->dn_col[k].as<float4>();
        var[k] = c->dn_var[k].as<float>();
    }
    if (conserve) {
        CK(c, c->dn_var_pf.reserve(n * sizeof(float)));
        CK(c, c->dn_wsum.reserve(n * sizeof(float)));
    }
    if (int rc = wait_for_scratch(c, st); rc != SPCU_OK) return rc;
    CK(c, launch_guides(c->ds, c->dn_guides.as<spcu_guide>(), st));
    if (conserve) {
        CK(c, launch_denoise_conserving(c->dn_guides.as<spcu_guide>(), d_rgb_sum, d_lum_sumsq, d_spp_map, spp, c->ds.width, c->ds.height,
                                        *p, col, var, c->dn_var_pf.as<float>(), c->dn_wsum.as<float>(), d_out, st));
    } else {
        CK(c, launch_denoise(c->dn_guides.as<spcu_guide>(), d_rgb_sum, d_lum_sumsq, d_spp_map, spp, c->ds.width, c->ds.height, *p, col,
                             var, d_out, st));
    }
    CK(c, cudaEventRecord(c->ev1, st));
    c->scratch_in_use = true;
    c->scratch_stream = st;
    return SPCU_OK;
}

// spcu_denoise / spcu_denoise_conserving: the sums go up into the host-buffer accumulators, the filter writes the mean colour
// over the colour sums there, and that buffer comes back to `out`.
int denoise_host(spcu_ctx* c, const float* rgb_sum, const float* lum_sumsq, const uint32_t* spp_map, uint32_t spp,
                 const spcu_denoise_params* p, float* out, bool conserve)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!rgb_sum || !lum_sumsq || !out) {
        return fail(c, SPCU_ERR_INVALID, "rgb_sum, lum_sumsq or out is NULL");
    }
    const size_t n = static_cast<size_t>(c->ds.width) * c->ds.height;
    return host_buffer_render(c, true, rgb_sum, lum_sumsq, out, nullptr, true, [&](float* d_rgb_sum, float* d_sq) {
        uint32_t* d_map = nullptr;
        if (spp_map) {
            CK(c, c->ad_spp_map.reserve(n * sizeof(uint32_t)));
            d_map = c->ad_spp_map.as<uint32_t>();
            CK(c, cudaMemcpyAsync(d_map, spp_map, n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
        }
        return denoise_impl(c, d_rgb_sum, d_sq, d_map, spp, p, d_rgb_sum, c->stream, conserve);
    });
}

} // namespace

extern "C" {

int spcu_render_device(spcu_ctx* c, const spcu_partition* part, float* d_rgb_sum, float* d_lum_sumsq, spcu_stats* stats,
                       void* stream)
{
    // stream == NULL means the legacy default stream, as in the CUDA runtime
    return render_impl(c, part, d_rgb_sum, d_lum_sumsq, stats, static_cast<cudaStream_t>(stream), true);
}

int spcu_render_adaptive_device(spcu_ctx* c, const spcu_partition* part, const spcu_adaptive* ad, float* d_rgb_sum, float* d_lum_sumsq,
                                uint32_t* d_spp_map, uint32_t* n_passes, spcu_stats* stats, void* stream)
{
    return adaptive_impl(c, part, ad, d_rgb_sum, d_lum_sumsq, d_spp_map, n_passes, stats, static_cast<cudaStream_t>(stream), true);
}

int spcu_render_adaptive(spcu_ctx* c, const spcu_partition* part, const spcu_adaptive* ad, float* rgb_sum, float* lum_sumsq,
                         uint32_t* spp_map, uint32_t* n_passes, spcu_stats* stats)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!rgb_sum || !spp_map) {
        return fail(c, SPCU_ERR_INVALID, "rgb_sum or spp_map is NULL");
    }
    const size_t map_bytes = static_cast<size_t>(c->ds.width) * c->ds.height * sizeof(uint32_t);
    CK(c, c->ad_spp_map.reserve(map_bytes));
    // (every pass's fault counter has been read)
    return host_buffer_render(c, true, nullptr, nullptr, rgb_sum, lum_sumsq, true, [&](float* d_rgb_sum, float* d_sq) {
        if (int rc = adaptive_impl(c, part, ad, d_rgb_sum, d_sq, c->ad_spp_map.as<uint32_t>(), n_passes, stats, nullptr, false);
            rc != SPCU_OK) {
            return rc;
        }
        CK(c, cudaMemcpyAsync(spp_map, c->ad_spp_map.p, map_bytes, cudaMemcpyDeviceToHost, c->stream));
        return SPCU_OK;
    });
}

int spcu_render_adaptive_predicted_device(spcu_ctx* c, const spcu_partition* part, const spcu_adaptive_predicted* ap, float* d_rgb_sum,
                                          float* d_lum_sumsq, uint32_t* d_spp_map, uint32_t* n_rounds, uint32_t* n_calls,
                                          spcu_stats* stats, void* stream)
{
    return adaptive_predicted_impl(c, part, ap, d_rgb_sum, d_lum_sumsq, d_spp_map, n_rounds, n_calls, stats,
                                   static_cast<cudaStream_t>(stream), true);
}

int spcu_render_adaptive_predicted(spcu_ctx* c, const spcu_partition* part, const spcu_adaptive_predicted* ap, float* rgb_sum,
                                   float* lum_sumsq, uint32_t* spp_map, uint32_t* n_rounds, uint32_t* n_calls, spcu_stats* stats)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!rgb_sum || !spp_map) {
        return fail(c, SPCU_ERR_INVALID, "rgb_sum or spp_map is NULL");
    }
    const size_t map_bytes = static_cast<size_t>(c->ds.width) * c->ds.height * sizeof(uint32_t);
    CK(c, c->ad_spp_map.reserve(map_bytes));
    // (every call's fault counter has been read)
    return host_buffer_render(c, true, nullptr, nullptr, rgb_sum, lum_sumsq, true, [&](float* d_rgb_sum, float* d_sq) {
        if (int rc = adaptive_predicted_impl(c, part, ap, d_rgb_sum, d_sq, c->ad_spp_map.as<uint32_t>(), n_rounds, n_calls, stats,
                                             nullptr, false);
            rc != SPCU_OK) {
            return rc;
        }
        CK(c, cudaMemcpyAsync(spp_map, c->ad_spp_map.p, map_bytes, cudaMemcpyDeviceToHost, c->stream));
        return SPCU_OK;
    });
}

int spcu_render(spcu_ctx* c, const spcu_partition* part, float* rgb_sum, float* lum_sumsq, spcu_stats* stats)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!rgb_sum) {
        return fail(c, SPCU_ERR_INVALID, "rgb_sum is NULL");
    }
    return host_buffer_render(c, lum_sumsq != nullptr, rgb_sum, lum_sumsq, rgb_sum, lum_sumsq, stats != nullptr, [&](float* d_rgb_sum, float* d_sq) {
        return render_impl(c, part, d_rgb_sum, d_sq, stats, nullptr, false);
    });
}

int spcu_render_guides_device(spcu_ctx* c, spcu_guide* d_out, void* stream)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!d_out) {
        return fail(c, SPCU_ERR_INVALID, "out is NULL");
    }
    CK(c, launch_guides(c->ds, d_out, static_cast<cudaStream_t>(stream)));
    return SPCU_OK;
}

int spcu_render_guides(spcu_ctx* c, spcu_guide* out)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!out) {
        return fail(c, SPCU_ERR_INVALID, "out is NULL");
    }
    const size_t bytes = static_cast<size_t>(c->ds.width) * c->ds.height * sizeof(spcu_guide);
    CK(c, c->dn_guides.reserve(bytes));
    if (int rc = wait_for_scratch(c, c->stream); rc != SPCU_OK) return rc;
    CK(c, launch_guides(c->ds, c->dn_guides.as<spcu_guide>(), c->stream));
    CK(c, cudaMemcpyAsync(out, c->dn_guides.p, bytes, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return SPCU_OK;
}

int spcu_denoise_device(spcu_ctx* c, const float* d_rgb_sum, const float* d_lum_sumsq, const uint32_t* d_spp_map, uint32_t spp,
                        const spcu_denoise_params* p, float* d_out, void* stream)
{
    return denoise_impl(c, d_rgb_sum, d_lum_sumsq, d_spp_map, spp, p, d_out, static_cast<cudaStream_t>(stream), false);
}

int spcu_denoise(spcu_ctx* c, const float* rgb_sum, const float* lum_sumsq, const uint32_t* spp_map, uint32_t spp,
                 const spcu_denoise_params* p, float* out)
{
    return denoise_host(c, rgb_sum, lum_sumsq, spp_map, spp, p, out, false);
}

int spcu_denoise_conserving_device(spcu_ctx* c, const float* d_rgb_sum, const float* d_lum_sumsq, const uint32_t* d_spp_map,
                                   uint32_t spp, const spcu_denoise_params* p, float* d_out, void* stream)
{
    return denoise_impl(c, d_rgb_sum, d_lum_sumsq, d_spp_map, spp, p, d_out, static_cast<cudaStream_t>(stream), true);
}

int spcu_denoise_conserving(spcu_ctx* c, const float* rgb_sum, const float* lum_sumsq, const uint32_t* spp_map, uint32_t spp,
                            const spcu_denoise_params* p, float* out)
{
    return denoise_host(c, rgb_sum, lum_sumsq, spp_map, spp, p, out, true);
}

int spcu_resolved_pipeline(const spcu_ctx* c)
{
    return (c && c->have_scene) ? static_cast<int>(resolve_pipeline(c)) : -1;
}

int spcu_render_frame(spcu_ctx* c, const spcu_partition* part, float* rgb_sum, float* lum_sumsq, spcu_stats* stats)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!rgb_sum) {
        return fail(c, SPCU_ERR_INVALID, "rgb_sum is NULL");
    }
    return host_buffer_render(c, lum_sumsq != nullptr, nullptr, nullptr, rgb_sum, lum_sumsq, stats != nullptr, [&](float* d_rgb_sum, float* d_sq) {
        return render_impl(c, part, d_rgb_sum, d_sq, stats, nullptr, false);
    });
}

int spcu_render_frame_reduced(spcu_ctx* c, const spcu_partition* part, int with_sumsq, float* rgb_sum, float* lum_sumsq,
                              spcu_stats* stats)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    const bool root = c->comm_rank == 0;
    if (root && (!rgb_sum || (with_sumsq && !lum_sumsq))) {
        return fail(c, SPCU_ERR_INVALID, "rank 0 needs the host buffers");
    }
    return host_buffer_render(c, with_sumsq != 0, nullptr, nullptr, root ? rgb_sum : nullptr, root ? lum_sumsq : nullptr, stats != nullptr,
                              [&](float* d_rgb_sum, float* d_sq) {
                                  if (int rc = render_impl(c, part, d_rgb_sum, d_sq, stats, nullptr, false); rc != SPCU_OK) return rc;
                                  return spcu_reduce_to_root(c, d_rgb_sum, d_sq, c->stream);
                              });
}

int spcu_render_image(spcu_ctx* c, const spcu_partition* part, uint32_t format, void* out, spcu_stats* stats)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (!part || part->sample_end <= part->sample_begin) {
        return fail(c, SPCU_ERR_INVALID, "empty sample range");
    }
    if (int rc = host_buffer_render(c, false, nullptr, nullptr, nullptr, nullptr, stats != nullptr,
                                    [&](float* d_rgb_sum, float*) { return render_impl(c, part, d_rgb_sum, nullptr, stats, nullptr, false); });
        rc != SPCU_OK) {
        return rc;
    }
    return pack_device_image(c, c->host_rgb.as<float>(), nullptr, c->ds.width, c->ds.height, part->sample_end - part->sample_begin, format,
                             out);
}

// Ray batches through the renderer's own traversal stages: the kernels a frame runs (begin + persistent walk, lane refill,
// pair leaf steps), not the one-thread-per-ray kernels behind spcu_trace_*.  They borrow lane 0 of the render's wavefront
// state (shadow rays use light plane 0).
static int stage_batch(spcu_ctx* c, const spcu_ray* rays, uint64_t n, uint32_t traversal, spcu_hit* hits, spcu_hit* light_hits,
                       uint8_t* occluded)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    const bool shadow = occluded != nullptr;
    if (n && (!rays || (!shadow && !hits))) {
        return fail(c, SPCU_ERR_INVALID, "NULL ray or result buffer");
    }
    if (traversal > SPCU_TRAVERSAL_ORDERED) {
        return fail(c, SPCU_ERR_INVALID, "unknown traversal %u", traversal);
    }
    const cudaStream_t st = c->stream;
    if (int rc = wait_for_scratch(c, st); rc != SPCU_OK) return rc;
    const uint32_t chunk      = static_cast<uint32_t>(std::min<uint64_t>(std::max<uint64_t>(n, 1), kBatchRays));
    const uint32_t n_segments = material_segments(c);
    WaveLane&      lane       = c->lanes[0];
    if (int rc = lay_out_lane(c, lane, chunk, n_segments); rc != SPCU_OK) return rc;
    CK(c, c->counters.reserve(kCounterBytes));
    CK(c, c->q_rays.reserve(static_cast<size_t>(chunk) * sizeof(spcu_ray)));
    CK(c, c->q_out.reserve(static_cast<size_t>(chunk) * sizeof(spcu_hit)));
    CK(c, c->q_aux.reserve(static_cast<size_t>(chunk) * sizeof(spcu_hit)));
    auto*        d_counters = c->counters.as<unsigned long long>();
    uint32_t*    d_counts   = lane.queue_counts;
    const Launch L{ c->sm_count, st, c->features };
    for (uint64_t done = 0; done < n; done += chunk) {
        const uint32_t m = static_cast<uint32_t>(std::min<uint64_t>(chunk, n - done));
        CK(c, cudaMemcpyAsync(c->q_rays.p, rays + done, static_cast<size_t>(m) * sizeof(spcu_ray), cudaMemcpyHostToDevice, st));
        CK(c, cudaMemsetAsync(d_counts, 0, (8 + n_segments) * sizeof(uint32_t), st));
        CK(c, cudaMemsetAsync(d_counters, 0, kCounterBytes, st));
        uint32_t* n_cur = d_counts + 0;
        launch_batch_fill(lane.wave, c->q_rays.as<spcu_ray>(), m, lane.queues[kQCur], n_cur, shadow, st);
        if (shadow) {
            launch_shadow(L, c->ds, lane.wave, lane.queues[kQCur], n_cur, m, 0, d_counts + 1, nullptr, nullptr, lane.queues[kQWalk],
                          d_counts + 2, d_counters, nullptr);
            CK(c, cudaGetLastError());
            CK(c, cudaMemcpyAsync(occluded + done, lane.wave.occluded, m, cudaMemcpyDeviceToHost, st));
        } else {
            SortedQueue sorted{ lane.sorted, d_counts + 8, n_segments, chunk };
            launch_extend(L, c->ds, lane.wave, lane.queues[kQCur], n_cur, m, d_counts + 1, sorted, traversal == SPCU_TRAVERSAL_ORDERED,
                          lane.queues[kQWalk], d_counts + 2, d_counters, nullptr);
            launch_batch_gather_extend(lane.wave, m, c->q_out.as<spcu_hit>(), light_hits ? c->q_aux.as<spcu_hit>() : nullptr, st);
            CK(c, cudaGetLastError());
            CK(c, cudaMemcpyAsync(hits + done, c->q_out.p, static_cast<size_t>(m) * sizeof(spcu_hit), cudaMemcpyDeviceToHost, st));
            if (light_hits) {
                CK(c, cudaMemcpyAsync(light_hits + done, c->q_aux.p, static_cast<size_t>(m) * sizeof(spcu_hit), cudaMemcpyDeviceToHost, st));
            }
        }
        if (int rc = sync_and_check_faults(c, false); rc != SPCU_OK) return rc;
    }
    return SPCU_OK;
}

int spcu_extend_batch(spcu_ctx* c, const spcu_ray* rays, uint64_t n, uint32_t traversal, spcu_hit* hits, spcu_hit* light_hits)
{
    return stage_batch(c, rays, n, traversal, hits, light_hits, nullptr);
}

int spcu_shadow_batch(spcu_ctx* c, const spcu_ray* rays, uint64_t n, uint8_t* occluded)
{
    if (n && !occluded) {
        return fail(c, SPCU_ERR_INVALID, "NULL result buffer");
    }
    uint8_t dummy = 0;
    return stage_batch(c, rays, n, SPCU_TRAVERSAL_EXACT, nullptr, nullptr, occluded ? occluded : &dummy);
}

int spcu_stage_times(spcu_ctx* c, spcu_stage_time* out, uint32_t capacity, uint32_t* n_out)
{
    if (!c || !out || !n_out) {
        return fail(c, SPCU_ERR_INVALID, "NULL argument");
    }
    const uint32_t n = std::min<uint32_t>(capacity, kNumStages);
    std::memcpy(out, c->stage_report, n * sizeof(spcu_stage_time));
    *n_out = n;
    return SPCU_OK;
}

} // extern "C"
