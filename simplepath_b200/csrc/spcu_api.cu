// The C-ABI of include/spcu.h: context, scene upload, batch queries and the wavefront render loop.
// Host code only; kernels live in trace_kernels.cu (exact arithmetic) and shade_kernels.cu.
// There is no CPU fallback anywhere in this file: every entry point either runs CUDA kernels or returns an error.
#include "ctx.h"

#include <cmath>

using namespace spcu;

namespace spcu {

static thread_local std::string g_create_error;

int fail(spcu_ctx* c, int code, const char* fmt, ...)
{
    char    buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) {
        c->err = buf;
    } else {
        g_create_error = buf;
    }
    return code;
}

int copy_to_device(spcu_ctx* c, void* dst, const void* src, size_t bytes)
{
    constexpr size_t kChunk = 32u << 20, kThreshold = 64u << 20;
    if (bytes < kThreshold) {
        CK(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
        return SPCU_OK;
    }
    // A pageable cudaMemcpy of gigabytes (the 28 M-triangle scene is 2.8 GB) runs at ~4 GB/s; staged by hand it is bound by
    // the CPU's memcpy instead.
    for (int i = 0; i < 2; ++i) {
        if (!c->stage[i]) {
            CK(c, cudaMallocHost(&c->stage[i], kChunk));
            CK(c, cudaEventCreateWithFlags(&c->stage_ev[i], cudaEventDisableTiming));
        }
    }
    const char* from = static_cast<const char*>(src);
    char*       to   = static_cast<char*>(dst);
    int         i    = 0;
    for (size_t off = 0; off < bytes; off += kChunk, i ^= 1) {
        const size_t n = std::min(kChunk, bytes - off);
        if (c->stage_busy[i]) {
            CK(c, cudaEventSynchronize(c->stage_ev[i])); // the DMA out of this buffer has finished
        }
        std::memcpy(c->stage[i], from + off, n);
        CK(c, cudaMemcpyAsync(to + off, c->stage[i], n, cudaMemcpyHostToDevice, c->stream));
        CK(c, cudaEventRecord(c->stage_ev[i], c->stream));
        c->stage_busy[i] = true;
    }
    return SPCU_OK;
}

int need_scene(spcu_ctx* c)
{
    if (!c) {
        return SPCU_ERR_INVALID;
    }
    if (!c->have_scene) {
        return fail(c, SPCU_ERR_NO_SCENE, "no scene uploaded");
    }
    CK(c, cudaSetDevice(c->device));
    return SPCU_OK;
}

} // namespace spcu

namespace {

template <typename T>
int upload(spcu_ctx* c, DevBuf& buf, const T* src, size_t n)
{
    const size_t bytes = std::max<size_t>(n * sizeof(T), 16); // never a null device pointer
    CK(c, buf.reserve(bytes));
    if (n) {
        if (!src) {
            return fail(c, SPCU_ERR_INVALID, "scene array is NULL but its count is %zu", n);
        }
        if (const int rc = copy_to_device(c, buf.p, src, n * sizeof(T)); rc != SPCU_OK) {
            return rc;
        }
        c->scene_bytes += n * sizeof(T);
    }
    return SPCU_OK;
}

// every child box finite with lo <= hi (what the reference's construction always produces: bounds are folded min / max)
bool boxes_are_proper(const spcu_accel& a)
{
    for (uint32_t i = 0; i < a.n_nodes; ++i) {
        const float* b = a.nodes[i].box;
        for (int k = 0; k < 2; ++k) {
            for (int d = 0; d < 3; ++d) {
                const float lo = b[6 * k + d], hi = b[6 * k + 3 + d];
                if (!(std::isfinite(lo) && std::isfinite(hi) && lo <= hi)) {
                    return false;
                }
            }
        }
    }
    return true;
}

int validate_accel(spcu_ctx* c, const spcu_accel& a, const char* what)
{
    if (a.n_unbounded > a.n_prims) {
        return fail(c, SPCU_ERR_INVALID, "%s: n_unbounded > n_prims", what);
    }
    if (a.n_nodes >= (1u << 30) || a.n_prims >= (1u << 30)) { // traversal cursors keep a flag in bit 30 (trace_kernels.cu)
        return fail(c, SPCU_ERR_LIMIT, "%s: more than 2^30 nodes or primitives", what);
    }
    if (a.max_depth > SPCU_MAX_BVH_DEPTH) {
        return fail(c, SPCU_ERR_LIMIT, "%s: BVH depth %u exceeds SPCU_MAX_BVH_DEPTH", what, a.max_depth);
    }
    if (a.root >= 0 && static_cast<uint32_t>(a.root) >= a.n_nodes) {
        return fail(c, SPCU_ERR_INVALID, "%s: root out of range", what);
    }
    if (a.n_nodes > 0 && !a.nodes) {
        return fail(c, SPCU_ERR_INVALID, "%s: nodes is NULL but n_nodes is %u", what, a.n_nodes);
    }
    auto leaf_ok = [&](int32_t link, uint32_t count) {
        const uint64_t first = static_cast<uint32_t>(~link);
        return first + (count & SPCU_LEAF_COUNT_MASK) <= a.n_prims;
    };
    if (a.root < 0 && !leaf_ok(a.root, a.root_count)) {
        return fail(c, SPCU_ERR_INVALID, "%s: root leaf out of range", what);
    }
    // The traversal stacks (trace.cuh) push without a bound check, so the depth they are sized for is DERIVED here, not
    // taken from the header: children always follow their parent, one forward pass gives every node its nesting level.
    std::vector<uint8_t> level(a.n_nodes, 0);
    uint32_t             depth = 0;
    if (a.root >= 0) {
        level[a.root] = 1;
    }
    for (uint32_t i = 0; i < a.n_nodes; ++i) {
        for (int k = 0; k < 2; ++k) {
            const int32_t link = a.nodes[i].child[k];
            if (link >= 0 ? (static_cast<uint32_t>(link) >= a.n_nodes || static_cast<uint32_t>(link) <= i)
                          : !leaf_ok(link, a.nodes[i].count[k])) {
                return fail(c, SPCU_ERR_INVALID, "%s: node %u child %d out of range", what, i, k);
            }
            if (link >= 0 && level[i]) {
                if (level[i] >= SPCU_MAX_BVH_DEPTH) {
                    return fail(c, SPCU_ERR_LIMIT, "%s: BVH deeper than SPCU_MAX_BVH_DEPTH (%u) at node %d", what,
                                SPCU_MAX_BVH_DEPTH, link);
                }
                level[link] = std::max<uint8_t>(level[link], static_cast<uint8_t>(level[i] + 1));
            }
        }
        depth = std::max<uint32_t>(depth, level[i]);
    }
    if (depth != a.max_depth) {
        return fail(c, SPCU_ERR_INVALID, "%s: header says max_depth %u but the nodes nest %u deep", what, a.max_depth, depth);
    }
    return SPCU_OK;
}

// Smallest compiled feature set (features.h) that covers the scene.
int scene_features(const spcu_flat_scene& s)
{
    bool analytic = s.geom.n_nodes == 0 && s.lights_accel.n_nodes == 0;
    for (uint32_t i = 0; analytic && i < s.geom.n_prims; ++i) {
        analytic = SPCU_META_KIND(s.geom_meta[i]) != SPCU_PRIM_TRIANGLE;
    }
    for (uint32_t i = 0; analytic && i < s.n_bxdfs; ++i) {
        // the selection weight of a lone Lambert BxDF is lum(rho) / lum(rho), rho = r * pi: exactly 1 iff that is normal
        const float* r   = s.bxdfs[i].r;
        const float  pi  = 3.14159265358979323846f;
        const float  lum = 0.2126f * (r[0] * pi) + 0.7152f * (r[1] * pi) + 0.0722f * (r[2] * pi);
        analytic = s.bxdfs[i].kind == SPCU_BXDF_LAMBERT && std::isnormal(lum) && std::isnormal(lum / 16.0f);
    }
    for (uint32_t i = 0; analytic && i < s.n_materials; ++i) {
        const spcu_material& m = s.materials[i];
        analytic = m.kind == SPCU_MAT_ONE_SAMPLE ? m.n_bxdfs == 1
                                                 : (m.base < s.n_materials && s.materials[m.base].kind == SPCU_MAT_ONE_SAMPLE);
    }
    for (uint32_t i = 0; analytic && i < s.n_lights; ++i) {
        analytic = s.lights[i].kind != SPCU_LIGHT_ENV_IBL;
    }
    return analytic ? FeatAnalytic::id : FeatFull::id;
}

DAccel device_accel(const spcu_accel& a, const DevBuf& nodes, bool proper_boxes)
{
    DAccel d;
    d.wide         = nullptr;
    d.big          = nullptr;
    d.proper_boxes = proper_boxes ? 1u : 0u;
    d.nodes       = nodes.as<const float4>();
    d.root        = a.root;
    d.root_count  = a.root_count;
    d.n_unbounded = a.n_unbounded;
    d.n_prims     = a.n_prims;
    return d;
}

} // namespace

// =====================================================================================================================
extern "C" {

int spcu_abi_version(void)
{
    return SPCU_ABI_VERSION;
}

const char* spcu_last_error(const spcu_ctx* ctx)
{
    return ctx ? ctx->err.c_str() : spcu::g_create_error.c_str();
}

int spcu_create(int device, spcu_ctx** out)
{
    if (!out) {
        return fail(nullptr, SPCU_ERR_INVALID, "out is NULL");
    }
    *out      = nullptr;
    int count = 0;
    if (const cudaError_t e = cudaGetDeviceCount(&count); e != cudaSuccess || count == 0) {
        return fail(nullptr, SPCU_ERR_CUDA, "no CUDA device: %s (this backend has no CPU fallback)",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (device < 0 || device >= count) {
        return fail(nullptr, SPCU_ERR_INVALID, "device %d out of range [0,%d)", device, count);
    }
    CK(nullptr, cudaSetDevice(device));
    cudaDeviceProp prop{};
    CK(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        return fail(nullptr, SPCU_ERR_CUDA, "device %d is sm_%d%d; this library holds sm_100a code only", device, prop.major,
                    prop.minor);
    }
    auto* c     = new spcu_ctx;
    c->options[SPCU_OPT_PIPELINE]  = SPCU_PIPELINE_AUTO;
    c->options[SPCU_OPT_TRAVERSAL] = SPCU_TRAVERSAL_ORDERED;
    c->device   = device;
    c->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess) {
        const int rc = fail(nullptr, SPCU_ERR_CUDA, "stream/event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
        if (c->ev1) cudaEventDestroy(c->ev1);
        if (c->ev0) cudaEventDestroy(c->ev0);
        if (c->stream) cudaStreamDestroy(c->stream);
        delete c;
        return rc;
    }
    *out = c;
    return SPCU_OK;
}

void spcu_destroy(spcu_ctx* c)
{
    if (!c) {
        return;
    }
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    spcu_comm_destroy(c);
    for (auto& lane : c->lanes) {
        if (lane.stream) cudaStreamSynchronize(lane.stream);
        if (lane.resolved) cudaEventDestroy(lane.resolved);
        if (lane.stream) cudaStreamDestroy(lane.stream);
    }
    for (auto e : c->ad_ev) {
        if (e) cudaEventDestroy(e);
    }
    for (auto e : c->stage_events) {
        cudaEventDestroy(e);
    }
    for (int i = 0; i < 2; ++i) {
        if (c->stage[i]) {
            cudaFreeHost(c->stage[i]);
            cudaEventDestroy(c->stage_ev[i]);
        }
    }
    cudaEventDestroy(c->ev0);
    cudaEventDestroy(c->ev1);
    cudaStreamDestroy(c->stream);
    delete c; // (its device buffers free themselves)
}

int spcu_set_option(spcu_ctx* c, uint32_t option, uint32_t value)
{
    if (!c || option >= SPCU_OPT_COUNT_) {
        return fail(c, SPCU_ERR_INVALID, "unknown option %u", option);
    }
    c->options[option] = value;
    return SPCU_OK;
}

int spcu_set_wavefront_size(spcu_ctx* c, uint64_t n_paths)
{
    if (!c) {
        return SPCU_ERR_INVALID;
    }
    if (n_paths > (1ull << 28)) {
        return fail(c, SPCU_ERR_LIMIT, "wavefront of %llu paths exceeds 2^28", static_cast<unsigned long long>(n_paths));
    }
    c->wavefront_size = n_paths;
    return SPCU_OK;
}

// spcu_upload_scene (build = false) and spcu_upload_scene_build (build = true: the geometry arrives unbuilt).
static int upload_impl(spcu_ctx* c, const spcu_flat_scene* s, const float* jitter, uint32_t spp, bool build,
                       const spcu_bounds* bounds, uint32_t* order)
{
    if (!c) {
        return SPCU_ERR_INVALID;
    }
    if (!s || s->abi_version != SPCU_ABI_VERSION) {
        return fail(c, SPCU_ERR_INVALID, "scene is NULL or has a different ABI version");
    }
    if (s->width == 0 || s->height == 0 || static_cast<uint64_t>(s->width) * s->height > (1ull << 31)) {
        return fail(c, SPCU_ERR_INVALID, "bad image size %ux%u", s->width, s->height);
    }
    if (spp > 0 && !jitter) {
        return fail(c, SPCU_ERR_INVALID, "jitter table is NULL");
    }
    if (!build) {
        if (int rc = validate_accel(c, s->geom, "geometry accelerator"); rc != SPCU_OK) return rc;
    } else if (s->geom.n_unbounded > s->geom.n_prims || s->geom.n_prims >= (1u << 30)) {
        return fail(c, SPCU_ERR_INVALID, "geometry: n_unbounded > n_prims, or more than 2^30 primitives");
    }
    // every array with a non-zero count must be there BEFORE the loops below read it
    if ((s->geom.n_prims && (!s->geom_meta || !s->geom_prims || !s->geom_shade)) || (s->n_materials && !s->materials) ||
        (s->n_bxdfs && !s->bxdfs) || (s->n_lights && (!s->lights || !s->light_order)) || (s->n_pool && !s->float_pool)) {
        return fail(c, SPCU_ERR_INVALID, "a scene array is NULL but its count is not 0");
    }
    if (int rc = validate_accel(c, s->lights_accel, "lights accelerator"); rc != SPCU_OK) return rc;
    if (s->lights_accel.n_prims != s->n_lights) {
        return fail(c, SPCU_ERR_INVALID, "lights accelerator holds %u prims but n_lights is %u", s->lights_accel.n_prims,
                    s->n_lights);
    }
    for (uint32_t i = 0; i < s->geom.n_prims; ++i) {
        if (SPCU_META_MATERIAL(s->geom_meta[i]) >= s->n_materials || SPCU_META_KIND(s->geom_meta[i]) > SPCU_PRIM_PLANE) {
            return fail(c, SPCU_ERR_INVALID, "primitive %u: bad kind or material index", i);
        }
        if (build && !bounds && i >= s->geom.n_unbounded && SPCU_META_KIND(s->geom_meta[i]) != SPCU_PRIM_TRIANGLE) {
            return fail(c, SPCU_ERR_INVALID, "primitive %u is bounded and not a triangle: its world bounds must be supplied", i);
        }
    }
    for (uint32_t i = 0; i < s->n_materials; ++i) {
        const spcu_material& m = s->materials[i];
        if (m.kind == SPCU_MAT_ONE_SAMPLE) {
            if (m.n_bxdfs == 0 || m.n_bxdfs > SPCU_MAX_BXDFS || static_cast<uint64_t>(m.first_bxdf) + m.n_bxdfs > s->n_bxdfs) {
                return fail(c, SPCU_ERR_LIMIT, "material %u: bad BxDF range", i);
            }
        } else if (m.kind == SPCU_MAT_CLEARCOAT) {
            // the flattener emits bases before the materials that coat them: chains are finite
            if (m.base >= i) {
                return fail(c, SPCU_ERR_INVALID, "material %u: clearcoat base must precede it", i);
            }
            uint32_t depth = 1, b = m.base;
            while (s->materials[b].kind == SPCU_MAT_CLEARCOAT) {
                b = s->materials[b].base;
                if (++depth >= SPCU_MAX_COAT_DEPTH) {
                    return fail(c, SPCU_ERR_LIMIT, "material %u: clearcoat nesting too deep", i);
                }
            }
        } else {
            return fail(c, SPCU_ERR_INVALID, "material %u: unknown kind", i);
        }
    }
    std::vector<bool> light_seen(s->n_lights, false); // light_order is a permutation: every light sampled exactly once
    for (uint32_t i = 0; i < s->n_lights; ++i) {
        if (s->lights[i].kind > SPCU_LIGHT_ENV_IBL || s->light_order[i] >= s->n_lights || light_seen[s->light_order[i]]) {
            return fail(c, SPCU_ERR_INVALID, "light %u: bad kind, or light_order is not a permutation", i);
        }
        light_seen[s->light_order[i]] = true;
    }
    CK(c, cudaSetDevice(c->device));
    c->have_scene  = false;
    c->scene_bytes = 0;
    int        rc;
    spcu_accel geom        = s->geom;
    bool       geom_proper = true;
    if (build) {
        if ((rc = build_scene_geometry(c, s, bounds, order, &geom, &geom_proper)) != SPCU_OK) return rc;
    } else {
        geom_proper = boxes_are_proper(s->geom);
        if ((rc = upload(c, c->geom_nodes, s->geom.nodes, s->geom.n_nodes)) != SPCU_OK) return rc;
        if ((rc = upload(c, c->geom_prims, s->geom_prims, s->geom.n_prims)) != SPCU_OK) return rc;
        if ((rc = upload(c, c->geom_shade, s->geom_shade, s->geom.n_prims)) != SPCU_OK) return rc;
        if ((rc = upload(c, c->geom_meta, s->geom_meta, s->geom.n_prims)) != SPCU_OK) return rc;
    }
    if ((rc = upload(c, c->light_nodes, s->lights_accel.nodes, s->lights_accel.n_nodes)) != SPCU_OK) return rc;
    if ((rc = upload(c, c->lights, s->lights, s->n_lights)) != SPCU_OK) return rc;
    if ((rc = upload(c, c->light_order, s->light_order, s->n_lights)) != SPCU_OK) return rc;
    if ((rc = upload(c, c->materials, s->materials, s->n_materials)) != SPCU_OK) return rc;
    if ((rc = upload(c, c->bxdfs, s->bxdfs, s->n_bxdfs)) != SPCU_OK) return rc;
    if ((rc = upload(c, c->pool, s->float_pool, s->n_pool)) != SPCU_OK) return rc;
    if ((rc = upload(c, c->jitter, jitter, static_cast<size_t>(spp) * 2)) != SPCU_OK) return rc;
    // the 4-wide copy of the geometry tree for the ordered / any-hit walks (a packed child holds a node index, or a first
    // primitive / side-table slot in 27 bits: device_scene.h)
    const bool wide = geom.n_nodes > 0 && geom.n_nodes < (1u << 31) && geom.n_prims <= kWidePayloadMask && geom_proper;
    if (wide) {
        const size_t big_entries = geom.n_prims / (kWideSmallLeafMax + 1u) + 1u;
        CK(c, c->geom_wide.reserve(static_cast<size_t>(geom.n_nodes) * 128));
        CK(c, c->geom_big.reserve(big_entries * sizeof(int2) + sizeof(uint32_t)));
        launch_build_wide(c->geom_nodes.as<const float4>(), geom.n_nodes, c->geom_wide.as<float4>(), c->geom_big.as<int2>(),
                          reinterpret_cast<uint32_t*>(c->geom_big.as<int2>() + big_entries), c->sm_count, c->stream);
        CK(c, cudaGetLastError());
    }
    CK(c, cudaStreamSynchronize(c->stream));

    DScene& d = c->ds;
    d.width     = s->width;
    d.height    = s->height;
    d.rr_depth  = s->rr_depth;
    d.max_depth = s->max_depth;
    std::memcpy(d.camera, s->camera, sizeof d.camera);
    d.geom         = device_accel(geom, c->geom_nodes, geom_proper);
    d.geom.wide    = wide ? c->geom_wide.as<const float4>() : nullptr;
    d.geom.big     = wide ? c->geom_big.as<const int2>() : nullptr;
    d.geom_prims   = c->geom_prims.as<const float4>();
    d.geom_shade   = c->geom_shade.as<const float4>();
    d.geom_meta    = c->geom_meta.as<const uint32_t>();
    d.lights_accel = device_accel(s->lights_accel, c->light_nodes, boxes_are_proper(s->lights_accel));
    d.n_lights     = s->n_lights;
    d.lights       = c->lights.as<const spcu_light>();
    d.light_order  = c->light_order.as<const uint32_t>();
    d.materials    = c->materials.as<const spcu_material>();
    d.bxdfs        = c->bxdfs.as<const spcu_bxdf>();
    d.pool         = c->pool.as<const float>();
    d.jitter       = c->jitter.as<const float>();
    d.spp          = spp;
    c->n_materials = s->n_materials;
    spcu_flat_scene as_built = *s;
    as_built.geom            = geom;
    c->features    = c->options[SPCU_OPT_GENERIC_KERNELS] ? FeatFull::id : scene_features(as_built);
    c->built_geom  = geom;
    c->built_geom.nodes = nullptr;
    c->have_scene      = true;
    c->pix_list_stride = 0; // invalidate the cached pixel list
    return SPCU_OK;
}

int spcu_upload_scene(spcu_ctx* c, const spcu_flat_scene* s, const float* jitter, uint32_t spp)
{
    return upload_impl(c, s, jitter, spp, false, nullptr, nullptr);
}

int spcu_upload_scene_build(spcu_ctx* c, const spcu_flat_scene* s, const float* jitter, uint32_t spp, const spcu_bounds* bounds,
                            uint32_t* order, spcu_accel* built)
{
    const int rc = upload_impl(c, s, jitter, spp, true, bounds, order);
    if (rc == SPCU_OK && built) {
        *built = c->built_geom;
    }
    return rc;
}

uint64_t spcu_scene_bytes(const spcu_ctx* c)
{
    return c ? c->scene_bytes : 0;
}

// ---- batch queries -----------------------------------------------------------------------------------------------------
enum class Query { closest, closest_ordered, lights, any };

static int run_query(spcu_ctx* c, Query q, const spcu_ray* rays, uint64_t n, void* out, uint64_t* counters3)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (n && (!rays || !out)) {
        return fail(c, SPCU_ERR_INVALID, "NULL ray or result buffer");
    }
    const size_t out_elem = (q == Query::any) ? sizeof(uint8_t) : sizeof(spcu_hit);
    const uint64_t chunk  = std::min<uint64_t>(n, kBatchRays);
    CK(c, c->q_rays.reserve(std::max<size_t>(chunk, 1) * sizeof(spcu_ray)));
    CK(c, c->q_out.reserve(std::max<size_t>(chunk, 1) * out_elem));
    TraceCounters* d_cnt = nullptr;
    if (counters3) {
        CK(c, c->q_cnt.reserve(sizeof(TraceCounters)));
        d_cnt = c->q_cnt.as<TraceCounters>();
        CK(c, cudaMemsetAsync(d_cnt, 0, sizeof(TraceCounters), c->stream));
    }
    for (uint64_t done = 0; done < n; done += chunk) {
        const uint64_t m = std::min(chunk, n - done);
        CK(c, cudaMemcpyAsync(c->q_rays.p, rays + done, m * sizeof(spcu_ray), cudaMemcpyHostToDevice, c->stream));
        switch (q) {
        case Query::closest:
            launch_trace_closest(c->ds, c->q_rays.as<spcu_ray>(), m, c->q_out.as<spcu_hit>(), d_cnt, c->stream);
            break;
        case Query::closest_ordered:
            launch_trace_closest_ordered(c->ds, c->q_rays.as<spcu_ray>(), m, c->q_out.as<spcu_hit>(), d_cnt, c->stream);
            break;
        case Query::lights:
            launch_trace_lights(c->ds, c->q_rays.as<spcu_ray>(), m, c->q_out.as<spcu_hit>(), c->stream);
            break;
        case Query::any:
            launch_trace_any(c->ds, c->q_rays.as<spcu_ray>(), m, c->q_out.as<uint8_t>(), c->stream);
            break;
        }
        CK(c, cudaGetLastError());
        CK(c, cudaMemcpyAsync(static_cast<char*>(out) + done * out_elem, c->q_out.p, m * out_elem, cudaMemcpyDeviceToHost,
                              c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
    }
    if (counters3) {
        TraceCounters h{};
        CK(c, cudaMemcpy(&h, d_cnt, sizeof h, cudaMemcpyDeviceToHost));
        counters3[0] = h.nodes;
        counters3[1] = h.tris;
        counters3[2] = h.xf;
    }
    return SPCU_OK;
}

int spcu_trace_closest(spcu_ctx* c, const spcu_ray* rays, uint64_t n, spcu_hit* hits)
{
    return run_query(c, Query::closest, rays, n, hits, nullptr);
}

int spcu_trace_closest_counted(spcu_ctx* c, const spcu_ray* rays, uint64_t n, spcu_hit* hits, uint64_t counters[3])
{
    return run_query(c, Query::closest, rays, n, hits, counters);
}

int spcu_trace_closest_fast(spcu_ctx* c, const spcu_ray* rays, uint64_t n, spcu_hit* hits, uint64_t counters[3])
{
    return run_query(c, Query::closest_ordered, rays, n, hits, counters);
}

int spcu_trace_lights(spcu_ctx* c, const spcu_ray* rays, uint64_t n, spcu_hit* hits)
{
    return run_query(c, Query::lights, rays, n, hits, nullptr);
}

int spcu_trace_any(spcu_ctx* c, const spcu_ray* rays, uint64_t n, uint8_t* out)
{
    return run_query(c, Query::any, rays, n, out, nullptr);
}

int spcu_generate_rays(spcu_ctx* c, const uint32_t* pix, const uint32_t* smp, uint64_t n, spcu_ray* rays)
{
    if (int rc = need_scene(c); rc != SPCU_OK) return rc;
    if (n && (!pix || !smp || !rays)) {
        return fail(c, SPCU_ERR_INVALID, "NULL buffer");
    }
    const uint64_t n_pixels = static_cast<uint64_t>(c->ds.width) * c->ds.height;
    for (uint64_t i = 0; i < n; ++i) {
        if (pix[i] >= n_pixels || smp[i] >= c->ds.spp) {
            return fail(c, SPCU_ERR_INVALID, "entry %llu: pixel or sample index out of range", static_cast<unsigned long long>(i));
        }
    }
    const uint64_t chunk = std::min<uint64_t>(n, kBatchRays);
    CK(c, c->q_rays.reserve(std::max<size_t>(chunk, 1) * sizeof(spcu_ray)));
    CK(c, c->q_aux.reserve(std::max<size_t>(chunk, 1) * 2 * sizeof(uint32_t)));
    uint32_t* d_pix = c->q_aux.as<uint32_t>();
    uint32_t* d_smp = d_pix + chunk;
    for (uint64_t done = 0; done < n; done += chunk) {
        const uint64_t m = std::min(chunk, n - done);
        CK(c, cudaMemcpyAsync(d_pix, pix + done, m * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
        CK(c, cudaMemcpyAsync(d_smp, smp + done, m * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
        launch_generate_rays(c->ds, d_pix, d_smp, m, c->q_rays.as<spcu_ray>(), c->stream);
        CK(c, cudaGetLastError());
        CK(c, cudaMemcpyAsync(rays + done, c->q_rays.p, m * sizeof(spcu_ray), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
    }
    return SPCU_OK;
}

} // extern "C"
