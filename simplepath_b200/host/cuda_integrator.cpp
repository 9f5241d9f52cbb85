#include "cuda_integrator.h"

#include "flat_scene.h"

#include "base/Scene.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <stdexcept>
#include <thread>
#include <unistd.h>
#include <cstdio>

namespace sp {
namespace {

std::string g_selected_inner = "iterative_rrnee";

std::uint32_t integrator_code(const std::string& name)
{
    if (name == "iterative_rrnee") return SPCU_INTEGRATOR_ITERATIVE_RRNEE;
    if (name == "brute_force_iterative_rr") return SPCU_INTEGRATOR_BRUTE_FORCE_RR;
    if (name == "direct_lighting") return SPCU_INTEGRATOR_DIRECT_LIGHTING;
    if (name == "whitted") return SPCU_INTEGRATOR_WHITTED;
    throw std::runtime_error("CudaIntegrator: no device path for integrator '" + name + "'");
}

unsigned env_unsigned(const char* name, unsigned fallback)
{
    const char* v = std::getenv(name);
    return (v && *v) ? static_cast<unsigned>(std::strtoul(v, nullptr, 10)) : fallback;
}

// Called from string_to_integrator_type while main() reads its arguments, i.e. BEFORE the scene file is parsed: from here on
// Scene's constructor leaves the geometry accelerator unbuilt (the hunk in base/Scene.h) and render_sum builds it on the device.
// SPCU_BUILD_ON_DEVICE=0 keeps the reference's own construction; =verify keeps it AND rebuilds on the device to compare.
void arm_deferred_construction()
{
    const char* v = std::getenv("SPCU_BUILD_ON_DEVICE");
    internal::g_defer_geometry_accelerator = !(v && (*v == '0' || std::string(v) == "verify"));
}

void leave_now(int status, void*)
{
    std::fflush(nullptr);
    _exit(status);
}

} // namespace
} // namespace sp

void spb200::arm_exit_guard()
{
    static std::once_flag once;
    std::call_once(once, [] { on_exit(&sp::leave_now, nullptr); });
}

namespace sp {

struct CudaIntegrator::Device
{
    spcu_ctx* ctx = nullptr;
    int       index;

    explicit Device(int index_)
    : index(index_)
    {
        if (spcu_create(index, &ctx) != SPCU_OK) {
            throw std::runtime_error(std::string("CudaIntegrator: ") + spcu_last_error(nullptr));
        }
    }
    ~Device() { spcu_destroy(ctx); }
    Device(const Device&)            = delete;
    Device& operator=(const Device&) = delete;

    void check(int rc, const char* what) const
    {
        if (rc != SPCU_OK) {
            throw std::runtime_error(std::string("CudaIntegrator: ") + what + ": " + spcu_last_error(ctx));
        }
    }
};

bool CudaIntegrator::select(std::string_view name)
{
    constexpr std::string_view prefix = "cuda";
    if (!name.starts_with(prefix)) {
        return false;
    }
    name.remove_prefix(prefix.size());
    if (name.empty()) {
        g_selected_inner = "iterative_rrnee";
        arm_deferred_construction();
        return true;
    }
    if (name.front() != '_') {
        return false;
    }
    name.remove_prefix(1);
    integrator_code(std::string(name)); // throws for names without a device path
    g_selected_inner = std::string(name);
    arm_deferred_construction();
    return true;
}

CudaIntegrator::CudaIntegrator()
: CudaIntegrator(Options{ .device    = static_cast<int>(env_unsigned("SPCU_DEVICE", 0)),
                          .n_devices = static_cast<int>(env_unsigned("SPCU_DEVICES", 1)),
                          .spp       = env_unsigned("SPCU_SPP", 16),
                          .inner     = g_selected_inner,
                          .seed      = env_unsigned("SPCU_SEED", 0) })
{
}

CudaIntegrator::CudaIntegrator(Options options)
: m_options(std::move(options))
{
    integrator_code(m_options.inner);
    spb200::arm_exit_guard(); // the scene has been parsed by now: see flat_scene.h
    if (m_options.n_devices < 1) {
        throw std::runtime_error("CudaIntegrator: n_devices must be >= 1");
    }
}

CudaIntegrator::~CudaIntegrator() = default;

// Sum of radiance samples per pixel, row major W*H*3.
void CudaIntegrator::render_sum(const Scene& scene, unsigned spp, std::vector<float>& rgb_sum, std::vector<std::uint32_t>* spp_map,
                                float rel_error, std::uint32_t radius, std::vector<float>* lum_sumsq) const
{
    if (m_devices.empty()) {
        for (int i = 0; i < m_options.n_devices; ++i) {
            m_devices.push_back(std::make_unique<Device>(m_options.device + i));
        }
        if (m_devices.size() > 1) { // one NCCL communicator over the devices: the frame is summed on device 0 (SURVEY §8e)
            std::vector<spcu_ctx*> ctxs;
            for (const auto& d : m_devices) {
                ctxs.push_back(d->ctx);
            }
            if (spcu_comm_init_all(ctxs.data(), static_cast<int>(ctxs.size())) != SPCU_OK) {
                throw std::runtime_error(std::string("CudaIntegrator: spcu_comm_init_all: ") + spcu_last_error(m_devices[0]->ctx));
            }
        }
    }
    // one host thread per device, for the upload as for the render
    auto on_every_device = [this](auto&& work) {
        const auto               n = m_devices.size();
        std::vector<std::string> errors(n);
        auto                     guarded = [&](std::size_t k) {
            try {
                work(k);
            } catch (const std::exception& e) {
                errors[k] = e.what();
            }
        };
        if (n == 1) {
            guarded(0);
        } else {
            std::vector<std::thread> threads;
            for (std::size_t k = 0; k < n; ++k) {
                threads.emplace_back(guarded, k);
            }
            for (auto& t : threads) {
                t.join();
            }
        }
        for (const auto& e : errors) {
            if (!e.empty()) {
                throw std::runtime_error(e);
            }
        }
    };
    if (m_uploaded_scene != &scene || m_uploaded_spp != spp) {
        const auto t0 = std::chrono::steady_clock::now();
        // The flattened copy only lives for the duration of the upload: nothing of `scene` is retained.
        const spb200::FlatScene  flat   = spb200::flatten_scene(scene);
        const std::vector<float> jitter = spb200::jitter_table(spp);
        // SPCU_BUILD_ON_DEVICE=1: hand the geometry over UNBUILT and let the device construct the acceleration structure
        // (spcu_upload_scene_build).  The flattener lists the bounded primitives in leaf order, and construction from the
        // leaf order is a fixed point of BVHAccelerator::construct (Hoare's partition does not move a partitioned range),
        // so the device must arrive at exactly the tree the reference built: checked, header and primitive order.
        const char* bod             = std::getenv("SPCU_BUILD_ON_DEVICE");
        const bool  build_on_device = bod && std::string(bod) == "verify";
        on_every_device([&](std::size_t k) { // the replicas are uploaded concurrently (lucy: 3.4 GB per device)
            const auto& d = m_devices[k];
            if (flat.geom_unbuilt) { // the reference never built this tree: BVHAccelerator::construct runs on the device
                spcu_accel built{};
                d->check(spcu_upload_scene_build(d->ctx, &flat.view, jitter.data(), spp, flat.geom_bounds.data(), nullptr, &built),
                         "spcu_upload_scene_build");
                std::fprintf(stderr, "CudaIntegrator: acceleration structure built on device %d (never on the host): %u primitives, "
                                     "%u nodes, depth %u\n", d->index, built.n_prims, built.n_nodes, built.max_depth);
                return;
            }
            if (!build_on_device) {
                d->check(spcu_upload_scene(d->ctx, &flat.view, jitter.data(), spp), "spcu_upload_scene");
                return;
            }
            const spcu_accel&     want = flat.view.geom;
            std::vector<uint32_t> order(want.n_prims - want.n_unbounded);
            spcu_accel            built{};
            d->check(spcu_upload_scene_build(d->ctx, &flat.view, jitter.data(), spp, nullptr, order.data(), &built),
                     "spcu_upload_scene_build");
            bool same = built.n_prims == want.n_prims && built.n_unbounded == want.n_unbounded && built.n_nodes == want.n_nodes &&
                        built.root == want.root && built.root_count == want.root_count && built.max_depth == want.max_depth;
            for (uint32_t k = 0; same && k < order.size(); ++k) {
                same = order[k] == k;
            }
            if (!same) {
                throw std::runtime_error("CudaIntegrator: the device-built acceleration structure differs from the reference's");
            }
            std::fprintf(stderr, "CudaIntegrator: acceleration structure built on device %d: %u primitives, %u nodes, depth %u\n",
                         d->index, built.n_prims, built.n_nodes, built.max_depth);
        });
        m_uploaded_scene = &scene;
        m_uploaded_spp   = spp;
        m_upload_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    }
    const std::size_t n = static_cast<std::size_t>(scene.image_width) * scene.image_height * 3u;
    rgb_sum.resize(n); // spcu_render_frame overwrites: nothing to zero, nothing to upload
    float* sq = nullptr;
    if (lum_sumsq) {
        lum_sumsq->resize(n / 3u);
        sq = lum_sumsq->data();
    }

    const auto           n_dev = static_cast<std::uint32_t>(m_devices.size());
    const std::uint32_t  code  = integrator_code(m_options.inner);
    if (spp_map) { // (one device: render_frame checks)
        // passes of 16 samples (fewer when the budget is smaller); the first test needs at least 2 samples
        const std::uint32_t  k = std::min(16u, spp);
        const spcu_adaptive  ad{ std::max(2u, k), k, rel_error, 0.0f, radius };
        const spcu_partition part{ 0u, 1u, 0u, spp, spp, code, m_options.seed };
        spp_map->resize(n / 3u);
        std::uint32_t passes = 0;
        m_devices[0]->check(spcu_render_adaptive(m_devices[0]->ctx, &part, &ad, rgb_sum.data(), sq, spp_map->data(), &passes, &m_stats),
                            "spcu_render_adaptive");
        std::uint64_t early = 0;
        for (const std::uint32_t c : *spp_map) {
            early += c < spp ? 1u : 0u;
        }
        const double pixels = static_cast<double>(spp_map->size());
        std::fprintf(stderr, "CudaIntegrator: adaptive sampling to %g, window radius %u: %u passes, mean %.2f spp of %u, %.1f %% of pixels "
                     "stopped early\n", rel_error, radius, passes, static_cast<double>(m_stats.paths) / pixels, spp,
                     100.0 * static_cast<double>(early) / pixels);
        return;
    }
    std::vector<spcu_stats> stats(n_dev);
    // Tile-interleaved partition (base/TileScheduler.h:66-82 order): device k renders tiles t with t % n == k.  Disjoint
    // pixels, so the sum over devices is exact (every other device contributes +0): the per-device accumulators are summed on
    // device 0 by ncclReduce over NVLink (spcu_render_frame_reduced) and ONE frame crosses to the host.
    on_every_device([&](std::size_t k) {
        const spcu_partition part{ static_cast<std::uint32_t>(k), n_dev, 0u, spp, spp, code, m_options.seed };
        m_devices[k]->check(spcu_render_frame_reduced(m_devices[k]->ctx, &part, sq ? 1 : 0, k == 0 ? rgb_sum.data() : nullptr,
                                                      k == 0 ? sq : nullptr, &stats[k]),
                            "spcu_render_frame_reduced");
    });
    m_stats = stats[0];
    for (std::uint32_t k = 1; k < n_dev; ++k) {
        m_stats.paths += stats[k].paths;
        m_stats.rays_closest += stats[k].rays_closest;
        m_stats.rays_any += stats[k].rays_any;
        m_stats.rays_lights += stats[k].rays_lights;
        m_stats.shade_calls += stats[k].shade_calls;
        m_stats.kernel_launches += stats[k].kernel_launches;
        m_stats.device_ms = std::max(m_stats.device_ms, stats[k].device_ms);
    }
}

bool CudaIntegrator::render_frame(const Scene& scene, unsigned spp, Image& image) const
{
    if (spp == 0) {
        throw std::runtime_error("CudaIntegrator: samples per pixel must be >= 1");
    }
    // SPCU_DENOISE=1: the image is the denoised mean (spcu_denoise on device 0, with Context.denoise's defaults)
    bool denoise = false;
    if (const char* d = std::getenv("SPCU_DENOISE"); d && *d) {
        if (std::string(d) != "1") {
            throw std::runtime_error(std::string("CudaIntegrator: SPCU_DENOISE must be 1 (or unset), not '") + d + "'");
        }
        denoise = true;
    }
    std::vector<float>         sum;
    std::vector<float>         sumsq; // SPCU_DENOISE: the filter's variance estimate needs the sums of squared luminance
    std::vector<std::uint32_t> counts; // SPCU_ADAPTIVE=<rel_error>: --samples is the budget, each pixel has its own count
    if (const char* adaptive = std::getenv("SPCU_ADAPTIVE"); adaptive && *adaptive) {
        char*       end = nullptr;
        const float rel = std::strtof(adaptive, &end);
        if (end == adaptive || *end != '\0') {
            throw std::runtime_error(std::string("CudaIntegrator: SPCU_ADAPTIVE must be a relative standard error, not '") + adaptive + "'");
        }
        std::uint32_t radius = 0; // SPCU_ADAPTIVE_RADIUS=<0..7>: a pixel stops only when its window in its tile has converged
        if (const char* r = std::getenv("SPCU_ADAPTIVE_RADIUS"); r && *r) {
            char*               r_end = nullptr;
            const unsigned long v     = std::strtoul(r, &r_end, 10);
            if (r_end == r || *r_end != '\0' || *r < '0' || *r > '9' || v > 7) {
                throw std::runtime_error(std::string("CudaIntegrator: SPCU_ADAPTIVE_RADIUS must be a window radius from 0 to 7, not '") + r +
                                         "'");
            }
            radius = static_cast<std::uint32_t>(v);
        }
        if (m_options.n_devices > 1) {
            throw std::runtime_error("CudaIntegrator: SPCU_ADAPTIVE renders on one device; unset SPCU_DEVICES or set it to 1");
        }
        render_sum(scene, spp, sum, &counts, rel, radius, denoise ? &sumsq : nullptr);
    } else {
        render_sum(scene, spp, sum, nullptr, 0.0f, 0, denoise ? &sumsq : nullptr);
    }
    const auto  w   = static_cast<std::size_t>(scene.image_width);
    const auto  h   = static_cast<std::size_t>(scene.image_height);
    if (denoise) { // after the reduction: device 0 holds the scene, the frame's sums go back to it once more
        const spcu_denoise_params p{ 5u, 8.0f, 0.1f, 0.1f }; // Context.denoise's defaults (DESIGN.md §12)
        std::vector<float>        mean(sum.size());
        const auto                t0 = std::chrono::steady_clock::now();
        m_devices[0]->check(spcu_denoise(m_devices[0]->ctx, sum.data(), sumsq.data(), counts.empty() ? nullptr : counts.data(), spp, &p,
                                         mean.data()),
                            "spcu_denoise");
        const double ms = 1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        std::fprintf(stderr, "CudaIntegrator: denoised (%u iterations, sigma_l %g, sigma_z %g, sigma_a %g) in %.2f ms\n", p.iterations,
                     static_cast<double>(p.sigma_l), static_cast<double>(p.sigma_z), static_cast<double>(p.sigma_a), ms);
        sum.swap(mean);
        counts.assign(w * h, 1u); // the means, divided by 1 below (exact)
    }
    for (std::size_t y = 0; y < h; ++y) {
        for (std::size_t x = 0; x < w; ++x) {
            const float* p = &sum[(y * w + x) * 3u];
            // image(p) += L ... ; image(p) /= num_pixel_samples (main.cpp:100-102)
            RGB         c{ p[0], p[1], p[2] };
            const float div = counts.empty() ? static_cast<float>(spp) : static_cast<float>(counts[y * w + x]);
            c /= div;
            image(x, y) = c;
        }
    }
    return true;
}

RGB CudaIntegrator::integrate_impl(const Ray&, const Scene& scene, MemoryArena&, Sampler&, const Point2& pixel_coords) const
{
    std::call_once(m_lazy_once, [&] {
        render_sum(scene, m_options.spp, m_lazy_mean);
        const float div = static_cast<float>(m_options.spp);
        for (float& v : m_lazy_mean) {
            v /= div;
        }
    });
    const int x = std::clamp(static_cast<int>(std::floor(pixel_coords.x)), 0, scene.image_width - 1);
    const int y = std::clamp(static_cast<int>(std::floor(pixel_coords.y)), 0, scene.image_height - 1);
    const float* p = &m_lazy_mean[(static_cast<std::size_t>(y) * scene.image_width + x) * 3u];
    return RGB{ p[0], p[1], p[2] };
}

} // namespace sp
