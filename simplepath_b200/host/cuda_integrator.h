// sp::CudaIntegrator — the B200 wavefront path tracer behind the reference's Integrator interface
// (Integrators/Integrator.h:32-52).  It owns an opaque device context (include/spcu.h) and nothing of the Scene.
//
// The reference's interface is per ray (`integrate(ray, scene, arena, sampler, pixel)` called spp times per pixel from
// N threads, main.cpp:77-107); a GPU renders whole frames.  Two entry points bridge that (SURVEY.md §8b):
//   * render_frame(scene, spp, image)  — what the driver's render() calls when it sees a CudaIntegrator
//     (the one-line dispatch of INTEGRATION.md); fills `image` with the per-pixel means, like render_thread does.
//   * integrate_impl(...)              — for an UNMODIFIED render loop: the first call renders the whole frame on the
//     GPU (std::call_once), every call returns the converged mean of the pixel `pixel_coords` falls in, so the stock
//     loop's `sum of spp calls / spp` reproduces it.
// Errors of the C layer surface as std::runtime_error, which main()'s catch blocks already print (main.cpp:398-404).
#pragma once

#include "spcu.h"

#include "Integrators/Integrator.h"
#include "Image/Image.h"

#include <memory>
#include <mutex>
#include <string>
#include <string_view>
#include <vector>

namespace sp {

class CudaIntegrator final : public Integrator
{
public:
    struct Options
    {
        int         device     = 0;                 // first CUDA device
        int         n_devices  = 1;                 // tile-interleaved across devices [device, device + n_devices)
        unsigned    spp        = 16;                // samples per pixel of the lazy whole-frame render (integrate_impl)
        std::string inner      = "iterative_rrnee"; // iterative_rrnee | brute_force_iterative_rr | direct_lighting | whitted
        std::uint64_t seed     = 0;
    };

    CudaIntegrator();                    // options from the name given to select() and the SPCU_* environment
    explicit CudaIntegrator(Options options);
    ~CudaIntegrator() override;

    // "cuda", "cuda_direct_lighting", "cuda_brute_force_iterative_rr", "cuda_whitted": remembers which reference integrator the next
    // default-constructed CudaIntegrator reproduces.  Returns false for names that are not ours.
    static bool select(std::string_view name);

    // Renders `scene` at `spp` samples per pixel into `image` (per-pixel means).  Always returns true; throws on error.
    bool render_frame(const Scene& scene, unsigned spp, Image& image) const;

    [[nodiscard]] const spcu_stats& last_stats() const noexcept { return m_stats; }
    [[nodiscard]] double last_upload_seconds() const noexcept { return m_upload_seconds; }

private:
    RGB integrate_impl(const Ray&, const Scene& scene, MemoryArena&, Sampler&, const Point2& pixel_coords) const override;

    // spp_map != NULL: adaptive sampling (spcu_render_adaptive, one device) to the standard error `rel_error` with the window
    // radius `radius` of the stopping rule, spp the budget; *spp_map = the samples each pixel received.  max_step > 0: with
    // predicted counts instead (spcu_render_adaptive_predicted), at most max_step doublings per round.
    // lum_sumsq != NULL: also the per-pixel sums of squared luminance (W*H), which the denoiser needs
    void render_sum(const Scene& scene, unsigned spp, std::vector<float>& rgb_sum, std::vector<std::uint32_t>* spp_map = nullptr,
                    float rel_error = 0.0f, std::uint32_t radius = 0, std::vector<float>* lum_sumsq = nullptr,
                    std::uint32_t max_step = 0) const;

    struct Device;
    Options                              m_options;
    mutable std::vector<std::unique_ptr<Device>> m_devices;
    mutable const Scene*                 m_uploaded_scene = nullptr;
    mutable unsigned                     m_uploaded_spp   = 0;
    mutable spcu_stats                   m_stats{};
    mutable double                       m_upload_seconds = 0.0;
    mutable std::once_flag               m_lazy_once;
    mutable std::vector<float>           m_lazy_mean; // W*H*3, per-pixel means of the lazy render
};

} // namespace sp
