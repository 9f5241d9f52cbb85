"""The render kernels in steady state: every lane draws many paths one after another, as in the benchmark frame.

The golden scenes of test_gpu_render.py hold at most a few thousand paths, which the persistent kernels take in one
fill: no lane of k_paths ever draws a second path, no slot of k_smwave ever regenerates, and the queue wavefront's
grid-stride loops run once.  Here every render is sized from the device's SM count so that each lane draws several
paths, and is checked three ways:
 * per pixel against the oracle at 1920x1080 (the benchmark frame's first and last sample);
 * bit for bit against the same render cut into batches small enough that every lane draws one path (a pixel's sums
   do not depend on batch shape, DESIGN.md §11), on every golden scene, pipeline and integrator, and at 1080p;
 * adaptive sampling at 1080p, where the compaction scan sums runs of several block counts, against the numpy model
   and fixed renders.
"""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from simplepath_b200 import adaptive, capi, host, rsequence
from simplepath_b200.flat import FlatSceneData

pytestmark = pytest.mark.gpu
SCENES = ["g_spheres", "g_spheres_ibl", "g_example", "g_bunny", "g_elf", "g_chain", "g_lights"]
INTEGRATORS = ["iterative_rrnee", "brute_force_iterative_rr", "direct_lighting", "whitted"]
PIPELINES = {"wavefront": capi.PIPELINE_WAVEFRONT, "paths": capi.PIPELINE_PATHS, "smwave": capi.PIPELINE_SMWAVE}
WITH_AUTO = dict(PIPELINES, auto=capi.PIPELINE_AUTO)
SEED = 0  # bench.py's default

# ---- how many paths the persistent kernels hold at once -----------------------------------------------------------------
# k_paths (csrc/path_kernels.cu) runs one path per thread in CTAs of kPathBlock = 128 threads, at most occupancy x SMs CTAs
# (wavefront_grid), and an SM holds at most 2048 threads.
PATH_BLOCK = 128
THREADS_PER_SM = 2048
# k_smwave (csrc/smwave_kernels.cu) runs one CTA per SM holding P paths; resident_paths caps P at 32 * (kRing - 8), kRing = 64.
SMWAVE_RING = 64
SMWAVE_MAX_PATHS = 32 * (SMWAVE_RING - 8)


def sm_count() -> int:
    return torch.cuda.get_device_properties(0).multi_processor_count


def resident_bound(sms: int) -> int:
    """An upper bound on the paths either persistent kernel holds at once on `sms` SMs."""
    return sms * max(THREADS_PER_SM, SMWAVE_MAX_PATHS)


def assert_steady_state(n_paths: int, sms: int) -> None:
    """Enough paths that every lane of either persistent kernel draws several of them."""
    need = 4 * resident_bound(sms)
    assert n_paths >= need, f"{n_paths} paths do not reach steady state on {sms} SMs (need {need})"


def assert_one_path_per_lane(batch_paths: int, sms: int) -> None:
    """Few enough paths per batch that k_paths gives every lane at most one (ceil(n / grid) <= 128 slots per CTA), k_smwave
    takes them all in its first fill and the queue wavefront's stage kernels run one grid-stride iteration."""
    assert batch_paths <= PATH_BLOCK * sms, f"a batch of {batch_paths} paths gives some lane a second path on {sms} SMs"


def lum(c):
    return 0.2126 * c[..., 0] + 0.7152 * c[..., 1] + 0.0722 * c[..., 2]


@pytest.fixture(scope="module")
def sms(built):
    return sm_count()


@pytest.fixture(scope="module")
def workloads():
    """Full-resolution workload scenes, loaded once."""
    cache = {}

    def get(name):
        if name not in cache:
            if not host.loadable(name):
                pytest.skip(f"{name} cannot be loaded here")
            cache[name] = host.workload(name)
        return cache[name]
    return get


def upload(ctx, flat, jitter, pipeline):
    ctx.set_option(capi.OPT_PIPELINE, pipeline)
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), jitter, keepalive=flat)


@pytest.fixture
def restore(ctx):
    """Whatever a test sets, the next one starts from the natural batch shape and the queue wavefront."""
    yield
    ctx.set_wavefront_size(0)
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_WAVEFRONT)


def render_or_skip(ctx, part, pipeline):
    """ctx.render(part); SMWAVE packs depth and light cursor into one word and rejects scenes that overflow it."""
    try:
        return ctx.render(part)
    except capi.SpcuError as e:
        if pipeline == capi.PIPELINE_SMWAVE and "SPCU_PIPELINE_SMWAVE" in str(e):
            pytest.skip(str(e))
        raise


# ---- 1. per pixel against the oracle at 1920x1080 ------------------------------------------------------------------------
FULL_SCENES = ["c2_example_scene", "c3_bunny", "c4_elf"]
FULL_SPP = 256  # the benchmark frame's sample count: its jitter table
WINDOWS = [(0, 1), (255, 256)]


@pytest.fixture(scope="module")
def oracle_frames(oracle_port, workloads):
    """The oracle's render of (scene, sample window) with iterative_rrnee, once each."""
    cache = {}

    def get(name, window):
        if (name, window) not in cache:
            flat = workloads(name)
            part = capi.Partition(0, 1, window[0], window[1], FULL_SPP, capi.INTEGRATORS["iterative_rrnee"], SEED)
            cache[name, window] = oracle_port.render(flat.pointer(), rsequence.jitter_table(FULL_SPP), part,
                                                     threads=os.cpu_count())
        return cache[name, window]
    return get


@pytest.mark.parametrize("pipeline", list(WITH_AUTO))
@pytest.mark.parametrize("window", WINDOWS, ids=lambda w: f"s{w[0]}")
@pytest.mark.parametrize("name", FULL_SCENES)
def test_full_resolution_per_pixel_vs_oracle(ctx, sms, workloads, oracle_frames, restore, name, window, pipeline):
    """The bars of test_gpu_render.py::test_per_pixel_vs_oracle, on the benchmark's frame size."""
    flat = workloads(name)
    code = WITH_AUTO[pipeline]
    upload(ctx, flat, rsequence.jitter_table(FULL_SPP), code)
    part = ctx.partition(spp=FULL_SPP, sample_begin=window[0], sample_end=window[1], seed=SEED)
    n_paths = flat.width * flat.height * (window[1] - window[0])
    assert_steady_state(n_paths, sms)
    rgb, sq, st = render_or_skip(ctx, part, code)
    want, want_sq, want_st = oracle_frames(name, window)
    assert st["paths"] == want_st["paths"] == n_paths
    bad_rgb = (np.abs(rgb - want) > 2e-3 * (1.0 + np.abs(want))).any(axis=-1)
    bad_sq = np.abs(sq - want_sq) > 2e-3 * (1.0 + np.abs(want_sq))
    bad = bad_rgb | bad_sq
    mean_err = abs(lum(rgb).mean() - lum(want).mean()) / lum(want).mean()
    # A scale error of the sums smaller than the per-pixel band (say 1e-3) passes the bars above; the median relative
    # difference over the pixels that agree sees it.  Measured on a B200 on all 24 cases: exactly 0 for both.
    lit = ~bad & (want_sq > 0)
    bias_lum = float(np.median(lum(rgb)[lit] / lum(want)[lit] - 1.0))
    bias_sq = float(np.median(sq[lit] / want_sq[lit] - 1.0))
    print(f"\n{name} samples [{window[0]},{window[1]}) {pipeline} ({ctx.resolved_pipeline()}): {bad.mean():.4%} of pixels "
          f"differ (rgb {bad_rgb.mean():.4%}, lum_sumsq {bad_sq.mean():.4%}); mean luminance {mean_err:.4%} off; median "
          f"relative difference of the agreeing pixels: luminance {bias_lum:+.2e}, lum_sumsq {bias_sq:+.2e}; "
          + "; ".join(f"{k} {st[k]} vs {want_st[k]}" for k in ("rays_closest", "rays_lights", "shade_calls")))
    assert bad.mean() < 0.005, f"{name}: {bad.mean():.3%} of pixels differ from the oracle"
    assert abs(lum(rgb).mean() - lum(want).mean()) <= 0.002 * lum(want).mean() + 1e-6
    assert abs(bias_lum) < 1e-4 and abs(bias_sq) < 1e-4, (bias_lum, bias_sq)
    for key in ("rays_closest", "rays_lights"):
        assert abs(st[key] - want_st[key]) <= 0.005 * want_st[key] + 8, (key, st[key], want_st[key])
    assert abs(st["shade_calls"] - want_st["shade_calls"]) <= 0.008 * want_st["shade_calls"] + 8


# ---- 2. steady state equals one path per lane, bit for bit ---------------------------------------------------------------
COUNTERS = ("paths", "rays_closest", "rays_any", "rays_lights", "shade_calls")


def assert_same_render(ctx, part, code, small, label):
    """The natural batch shape against batches of `small` paths: the same sums to the bit, the same work counted."""
    natural = render_or_skip(ctx, part, code)
    ctx.set_wavefront_size(small)
    one = ctx.render(part)
    ctx.set_wavefront_size(0)
    assert natural[0].tobytes() == one[0].tobytes(), f"{label}: rgb sums depend on the batch shape"
    assert natural[1].tobytes() == one[1].tobytes(), f"{label}: lum_sumsq depends on the batch shape"
    for key in COUNTERS:
        assert natural[2][key] == one[2][key], (label, key, natural[2][key], one[2][key])
    print(f"\n{label}: {natural[1].size * 4} sums and {len(COUNTERS)} counters equal; "
          f"{natural[2]['kernel_launches']} against {one[2]['kernel_launches']} launches")


@pytest.mark.parametrize("integrator", INTEGRATORS)
@pytest.mark.parametrize("pipeline", list(PIPELINES))
@pytest.mark.parametrize("name", SCENES)
def test_golden_steady_state_equals_one_path_per_lane(ctx, sms, restore, name, pipeline, integrator):
    """A golden scene rendered to ~1000 spp: one sample of every pixel per batch against the natural shape."""
    flat = FlatSceneData.load(GOLDEN / f"{name}.flat.npz")
    n_pix = flat.width * flat.height
    spp = -(-4 * resident_bound(sms) // n_pix)
    assert_steady_state(n_pix * spp, sms)
    assert_one_path_per_lane(n_pix, sms)
    code = PIPELINES[pipeline]
    upload(ctx, flat, rsequence.jitter_table(spp), code)
    assert_same_render(ctx, ctx.partition(spp=spp, integrator=integrator, seed=SEED), code, n_pix,
                       f"{name}/{pipeline}/{integrator} at {spp} spp")


STEADY_1080P_SPP = 72  # 64 + 8 samples in the persistent kernels' 2^27-path batches; nine 8-sample batches of the queue wavefront
SMALL_1080P = 1 << 14  # pixels of one sample per batch


@pytest.mark.parametrize("pipeline", list(WITH_AUTO))
@pytest.mark.parametrize("name", ["c2_example_scene", "c3_bunny"])
def test_1080p_steady_state_equals_one_path_per_lane(ctx, sms, workloads, restore, name, pipeline):
    flat = workloads(name)
    assert_steady_state(flat.width * flat.height * STEADY_1080P_SPP, sms)
    assert_one_path_per_lane(SMALL_1080P, sms)
    code = WITH_AUTO[pipeline]
    upload(ctx, flat, rsequence.jitter_table(STEADY_1080P_SPP), code)
    assert_same_render(ctx, ctx.partition(spp=STEADY_1080P_SPP, seed=SEED), code, SMALL_1080P,
                       f"{name}/{pipeline} at {STEADY_1080P_SPP} spp")


# ---- 3. adaptive sampling, exact, at 1080p -------------------------------------------------------------------------------
BUDGET, MIN_SPP, PASS_SPP, FLOOR = 64, 16, 16, 1e-3
CANDIDATE_ERRORS = (1.0, 0.5, 0.3, 0.2, 0.1, 0.05, 0.02, 0.01)
SCAN_THREADS, SCAN_BLOCK = 1024, 256  # kScan, kBlock of csrc/adaptive_kernels.cu


@pytest.fixture(scope="module")
def bunny_fixed(ctx, sms, workloads):
    """c3_bunny at 1080p on AUTO with fixed renders of [0, b) at every pass boundary b."""
    flat = workloads("c3_bunny")
    assert_steady_state(flat.width * flat.height * MIN_SPP, sms)
    upload(ctx, flat, rsequence.jitter_table(BUDGET), capi.PIPELINE_AUTO)
    fixed = {}
    for b in adaptive.boundaries(BUDGET, MIN_SPP, PASS_SPP):
        rgb, sq, _ = ctx.render_frame(ctx.partition(spp=BUDGET, sample_end=b, seed=SEED))
        fixed[b] = (rgb, sq)
    return flat, fixed


@pytest.mark.parametrize("radius", [0, 2])
def test_1080p_adaptive_is_exact(ctx, bunny_fixed, restore, radius):
    flat, fixed = bunny_fixed
    shape = (flat.height, flat.width)
    # the first pass's list holds every pixel: more block counts than scan threads, so a thread sums a run of several
    assert -(-shape[0] * shape[1] // SCAN_BLOCK) > SCAN_THREADS
    whole = np.ones(shape, dtype=bool)

    def model(e):
        return adaptive.spp_map(lambda n: fixed[n], whole, BUDGET, MIN_SPP, PASS_SPP, e, FLOOR, radius=radius)

    best, best_n = None, 0  # as test_gpu_adaptive.py's exercising_error
    for e in CANDIDATE_ERRORS:
        u = np.unique(model(e))
        if MIN_SPP in u and BUDGET in u and len(u) > best_n:
            best, best_n = e, len(u)
    assert best is not None and best_n >= 3, "no candidate error exercises the schedule"
    want = model(best)
    upload(ctx, flat, rsequence.jitter_table(BUDGET), capi.PIPELINE_AUTO)
    rgb, sq, spp_map, st = ctx.render_adaptive(ctx.partition(spp=BUDGET, seed=SEED), best, min_spp=MIN_SPP,
                                               pass_spp=PASS_SPP, abs_floor=FLOOR, radius=radius)
    counts = {int(n): int((want == n).sum()) for n in np.unique(want)}
    print(f"\nc3_bunny adaptive radius {radius}, rel_error {best}: pixels per count {counts}, {st['passes']} passes")
    assert np.array_equal(spp_map, want), f"{(spp_map != want).sum()} pixels decided otherwise than the model"
    for n in np.unique(spp_map):
        sel = spp_map == n
        want_rgb, want_sq = fixed[int(n)]
        assert rgb[sel].tobytes() == want_rgb[sel].tobytes(), f"sums of the pixels with {n} samples"
        assert sq[sel].tobytes() == want_sq[sel].tobytes(), f"sums of squares of the pixels with {n} samples"
    assert st["paths"] == int(spp_map.sum(dtype=np.uint64))
