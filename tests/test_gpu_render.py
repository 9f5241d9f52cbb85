"""Parity of the CUDA wavefront renderer (through spcu_render) with the oracle and with the reference's golden renders.

Two bars:
 * per pixel against the oracle's restatement, which draws the SAME counter-based random numbers: images must agree
   up to rounding (different libm / rsqrt / FMA contraction), except for the few paths that a rounding difference
   sends down another branch (a Russian-roulette or BxDF-selection comparison landing on the other side);
 * statistically against the REAL reference (tests/golden/*.render.npz, its own mt19937_64 streams): per-pixel
   z-scores of the luminance means from RunningStats-style variances.
"""
import numpy as np
import pytest

from conftest import GOLDEN
from simplepath_b200 import capi
from simplepath_b200.flat import FlatSceneData

pytestmark = pytest.mark.gpu
SCENES = ["g_spheres", "g_spheres_ibl", "g_example", "g_bunny", "g_elf", "g_chain", "g_lights"]
INTEGRATORS = ["iterative_rrnee", "brute_force_iterative_rr", "direct_lighting", "whitted"]


def lum(c):
    return 0.2126 * c[..., 0] + 0.7152 * c[..., 1] + 0.0722 * c[..., 2]


PIPELINES = {"smwave": capi.PIPELINE_SMWAVE, "paths": capi.PIPELINE_PATHS, "wavefront": capi.PIPELINE_WAVEFRONT}
CURRENT = {"pipeline": capi.PIPELINE_WAVEFRONT}


@pytest.fixture(scope="module", params=[(s, p) for p in PIPELINES for s in SCENES], ids=lambda sp: f"{sp[0]}-{sp[1]}")
def scene(request, ctx):
    """(scene, kernel organisation): every test below runs against both the persistent path kernel and the
    queue-based wavefront pipeline."""
    name, pipeline = request.param
    flat = FlatSceneData.load(GOLDEN / f"{name}.flat.npz")
    vec = np.load(GOLDEN / f"{name}.vectors.npz")
    CURRENT["pipeline"] = PIPELINES[pipeline]
    yield name, flat, vec
    CURRENT["pipeline"] = capi.PIPELINE_WAVEFRONT
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_WAVEFRONT)


def upload(ctx, flat, jitter):
    ctx.set_option(capi.OPT_PIPELINE, CURRENT["pipeline"])
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), jitter, keepalive=flat)


@pytest.mark.parametrize("integrator", INTEGRATORS)
def test_per_pixel_vs_oracle(ctx, oracle_port, scene, integrator):
    name, flat, vec = scene
    jitter = vec["jitter"]
    spp = jitter.shape[0]
    upload(ctx, flat, jitter)
    part = ctx.partition(spp=spp, integrator=integrator, seed=20261018)
    rgb, sq, st = ctx.render(part)
    want, want_sq, want_st = oracle_port.render(flat.pointer(), jitter, part)
    assert st["paths"] == want_st["paths"] == flat.width * flat.height * spp
    # stated tolerance: a pixel "agrees" when every channel, and its sum of squared luminance, is within 2e-3 * (1 + |oracle|)
    # of the oracle's sum.
    # The bounds below are 3-4x the worst case measured over all 84 (scene, pipeline, integrator) combinations
    # (profiles/scripts/parity_margins.py -> profiles/r03t_parity_margins.jsonl: 0.13 % of pixels, 0.035 % of the mean
    # luminance, 0.24 % of the shade calls, 0.09 % / 0.04 % of the light / any-hit queries, closest-hit counts equal).
    tol = 2e-3 * (1.0 + np.abs(want))
    bad = (np.abs(rgb - want) > tol).any(axis=-1) | (np.abs(sq - want_sq) > 2e-3 * (1.0 + np.abs(want_sq)))
    assert bad.mean() < 0.005, f"{name}/{integrator}: {bad.mean():.2%} of pixels differ from the oracle"
    assert abs(lum(rgb).mean() - lum(want).mean()) <= 0.002 * lum(want).mean() + 1e-6
    # a scale error below the per-pixel band (a 1e-3 one passes it) moves the median relative difference of the pixels that
    # agree, which rounding alone leaves at 0 (measured at 1080p: tests/test_gpu_render_steady_state.py)
    lit = ~bad & (want_sq > 0)
    assert abs(np.median(sq[lit] / want_sq[lit] - 1.0)) < 1e-4 and abs(np.median(lum(rgb)[lit] / lum(want)[lit] - 1.0)) < 1e-4
    # identical random numbers => identical path structure except for those few paths
    for key in ("rays_closest", "rays_lights"):
        assert abs(st[key] - want_st[key]) <= 0.005 * want_st[key] + 8, (key, st[key], want_st[key])
    assert abs(st["shade_calls"] - want_st["shade_calls"]) <= 0.008 * want_st["shade_calls"] + 8
    # (direct lighting / whitted: the reference skips the shadow query when f == 0; the wavefront pipeline traces it anyway
    # — measured: at most 3.7 % more any-hit queries)
    assert abs(st["rays_any"] - want_st["rays_any"]) <= (0.10 if integrator in ("direct_lighting", "whitted") else 0.005) * want_st["rays_any"] + 8


@pytest.mark.parametrize("integrator", INTEGRATORS)
def test_statistical_vs_reference_render(ctx, scene, integrator):
    """|z| of per-pixel luminance means, reference (N_ref samples, RunningStats variance) vs CUDA (N samples,
    sum / sum-of-squares).  Stated bar: mean z within +-0.1, fewer than 0.5 % of pixels beyond 4 sigma, image mean within
    5 standard errors."""
    name, flat, vec = scene
    path = GOLDEN / f"{name}.render.npz"
    if not path.exists():
        pytest.skip("no golden render for this scene")
    gold = np.load(path)
    n_ref = int(gold[f"{integrator}.spp"])
    spp = n_ref  # equal sample counts: with skewed (firefly) pixel distributions unequal counts bias z itself
    from simplepath_b200 import rsequence
    jitter = rsequence.jitter_table(spp)
    upload(ctx, flat, jitter)
    rgb, sq, st = ctx.render(ctx.partition(spp=spp, integrator=integrator, seed=99))
    mean = lum(rgb / spp)
    var = np.maximum(sq / spp - mean ** 2, 0.0) * spp / (spp - 1)
    ref_mean, ref_var = gold[f"{integrator}.lum_mean"], gold[f"{integrator}.lum_var"]
    se = np.sqrt(var / spp + ref_var / n_ref) + 1e-4
    z = (mean - ref_mean) / se
    assert abs(z.mean()) < 0.1, f"{name}/{integrator}: mean z {z.mean():+.3f}"
    assert (np.abs(z) > 4).mean() < 0.005, f"{name}/{integrator}: {(np.abs(z) > 4).mean():.3%} beyond 4 sigma"
    # whole-image mean: difference within 5 standard errors of the image mean (pixels are independent)
    se_img = np.sqrt((se ** 2).sum()) / se.size
    assert abs(mean.mean() - ref_mean.mean()) < 5.0 * se_img, f"{name}/{integrator}: image mean off"


def test_pipelines_agree(ctx, scene):
    """The two kernel organisations run the same estimator on the same random numbers: images agree per pixel up to
    rounding (they are different instruction schedules of the same arithmetic)."""
    name, flat, vec = scene
    jitter = vec["jitter"]
    upload(ctx, flat, jitter)
    imgs = {}
    for pname, code in PIPELINES.items():
        ctx.set_option(capi.OPT_PIPELINE, code)
        imgs[pname], _, _ = ctx.render(ctx.partition(seed=77))
    ctx.set_option(capi.OPT_PIPELINE, CURRENT["pipeline"])
    b = imgs["wavefront"]
    for other in ("paths", "smwave"):
        a   = imgs[other]
        bad = (np.abs(a - b) > 2e-3 * (1.0 + np.abs(b))).any(axis=-1)
        assert bad.mean() < 0.02, f"{name}: {other} differs from the queue wavefront on {bad.mean():.2%} of the pixels"


def test_ordered_traversal_renders_the_same_image(ctx, scene):
    """SPCU_TRAVERSAL_ORDERED changes which boxes are visited, not what is hit (up to epsilon ties)."""
    name, flat, vec = scene
    if CURRENT["pipeline"] != capi.PIPELINE_WAVEFRONT:
        pytest.skip("the ordered walk is an option of the wavefront's extend stage")
    jitter = vec["jitter"]
    upload(ctx, flat, jitter)
    ctx.set_option(capi.OPT_TRAVERSAL, capi.TRAVERSAL_EXACT)
    try:
        exact, _, st_e = ctx.render(ctx.partition(seed=123))
    finally:
        ctx.set_option(capi.OPT_TRAVERSAL, capi.TRAVERSAL_ORDERED)  # the render default
    fast, _, st_f = ctx.render(ctx.partition(seed=123))
    differing = (exact != fast).any(axis=-1).mean()
    assert differing < 0.002, f"{name}: {differing:.3%} of pixels differ between the exact and the ordered walk"
    assert abs(st_e["rays_closest"] - st_f["rays_closest"]) <= 0.001 * st_e["rays_closest"] + 4


def test_partitions_are_exact(ctx, scene):
    """Tile partitions touch disjoint pixels and sample ranges accumulate in sample order, so any split of the work
    — by tiles, by samples, or into small wavefronts — gives the bit-identical image (SURVEY.md §8e)."""
    name, flat, vec = scene
    jitter = vec["jitter"]
    spp = jitter.shape[0]
    upload(ctx, flat, jitter)
    whole, whole_sq, _ = ctx.render(ctx.partition(spp=spp, seed=5))

    tiles = np.zeros_like(whole)
    tiles_sq = np.zeros_like(whole_sq)
    for rank in range(3):
        r, s, _ = ctx.render(ctx.partition(spp=spp, seed=5, rank=rank, world=3))
        tiles += r
        tiles_sq += s
    assert tiles.tobytes() == whole.tobytes() and tiles_sq.tobytes() == whole_sq.tobytes()

    part_a = ctx.partition(spp=spp, seed=5, sample_begin=0, sample_end=1)
    part_b = ctx.partition(spp=spp, seed=5, sample_begin=1, sample_end=spp)
    acc, acc_sq, _ = ctx.render(part_a)
    acc, acc_sq, _ = ctx.render(part_b, into=(acc, acc_sq))
    assert acc.tobytes() == whole.tobytes() and acc_sq.tobytes() == whole_sq.tobytes()

    ctx.set_wavefront_size(777)
    small, small_sq, st = ctx.render(ctx.partition(spp=spp, seed=5))
    assert small.tobytes() == whole.tobytes() and small_sq.tobytes() == whole_sq.tobytes()
    # ... and however many of those batches are in flight at once (SPCU_OPT_BATCH_LANES: the default is 4): the resolve
    # kernels are event-ordered, so the per-pixel sums add up in batch order on every lane count
    for lanes in (1, 2, 3, 8):
        ctx.set_option(capi.OPT_BATCH_LANES, lanes)
        laned, laned_sq, st_l = ctx.render(ctx.partition(spp=spp, seed=5))
        assert laned.tobytes() == whole.tobytes() and laned_sq.tobytes() == whole_sq.tobytes(), f"{lanes} lanes"
        assert st_l["paths"] == st["paths"] and st_l["rays_closest"] == st["rays_closest"] and st_l["rays_any"] == st["rays_any"]
    ctx.set_option(capi.OPT_BATCH_LANES, 0)
    ctx.set_wavefront_size(0)


def test_progressive_passes(ctx, scene):
    """Multi-pass rendering (the reference's TileScheduler hands out (tile, pass); base/TileScheduler.h:58-86): every pass adds
    its sample range to the same accumulators, each preview is exactly the frame rendered up to that sample, and the last
    one is the one-call frame bit for bit."""
    name, flat, vec = scene
    jitter = vec["jitter"]
    spp = jitter.shape[0]
    upload(ctx, flat, jitter)
    whole, whole_sq, st = ctx.render(ctx.partition(spp=spp, seed=11))
    seen, paths = [], 0
    for done, rgb, sq, st_p in ctx.render_passes(3, spp=spp, seed=11):
        seen.append(done)
        paths += st_p["paths"]
        upto, upto_sq, _ = ctx.render(ctx.partition(spp=spp, seed=11, sample_begin=0, sample_end=done))
        assert rgb.tobytes() == upto.tobytes() and sq.tobytes() == upto_sq.tobytes(), f"{name}: preview after {done} samples"
    assert seen[-1] == spp and seen == sorted(set(seen)) and paths == st["paths"]
    assert rgb.tobytes() == whole.tobytes() and sq.tobytes() == whole_sq.tobytes()


@pytest.mark.parametrize("integrator", INTEGRATORS)
def test_feature_specialised_kernels_render_the_same_image(ctx, scene, integrator):
    """spcu_upload_scene picks kernels compiled for the scene's feature set (csrc/features.h: no BVH / triangles /
    microfacet / image-based light code for analytic scenes).  A feature that is absent only removes never-taken branches,
    so the image must agree with the kernels compiled for everything; compilers may schedule the surviving arithmetic
    differently (FMA contraction in the shading TUs), hence rounding-level tolerance and equal ray counts within 0.1 %."""
    name, flat, vec = scene
    jitter = vec["jitter"]
    upload(ctx, flat, jitter)
    part = ctx.partition(integrator=integrator, seed=4242)
    special, _, st_s = ctx.render(part)
    ctx.set_option(capi.OPT_GENERIC_KERNELS, 1)
    try:
        upload(ctx, flat, jitter)  # the feature set is chosen at upload
        generic, _, st_g = ctx.render(part)
    finally:
        ctx.set_option(capi.OPT_GENERIC_KERNELS, 0)
        upload(ctx, flat, jitter)
    bad = (np.abs(special - generic) > 2e-3 * (1.0 + np.abs(generic))).any(axis=-1)
    assert bad.mean() < 0.01, f"{name}/{integrator}: {bad.mean():.2%} of pixels differ between feature sets"
    for key in ("rays_closest", "rays_any", "rays_lights", "shade_calls"):
        assert abs(st_s[key] - st_g[key]) <= 0.001 * st_g[key] + 4, (key, st_s[key], st_g[key])


def test_render_frame_overwrites_and_equals_render(ctx, scene):
    """spcu_render_frame = spcu_render into zeroed buffers, without the upload: bitwise the same sums, whatever the
    output buffers held before; pixels outside a tile partition come back as 0."""
    name, flat, vec = scene
    upload(ctx, flat, vec["jitter"])
    part = ctx.partition(seed=31, rank=1, world=2)
    want, want_sq, st_w = ctx.render(part)
    junk = (np.full_like(want, np.nan), np.full_like(want_sq, 7.0))
    got, got_sq, st_g = ctx.render_frame(part, out=junk)
    assert got.tobytes() == want.tobytes() and got_sq.tobytes() == want_sq.tobytes()
    assert st_g["paths"] == st_w["paths"]


def test_seed_changes_the_image_and_repeats_exactly(ctx, scene):
    name, flat, vec = scene
    jitter = vec["jitter"]
    upload(ctx, flat, jitter)
    a, _, _ = ctx.render(ctx.partition(seed=1))
    b, _, _ = ctx.render(ctx.partition(seed=1))
    c, _, _ = ctx.render(ctx.partition(seed=2))
    assert a.tobytes() == b.tobytes()
    assert a.tobytes() != c.tobytes()


def test_counters_with_node_counting(ctx, oracle_port, scene):
    """Traversal work counted on the device equals the oracle's count on the reference topology, for the primary rays
    (depth 0 is identical on both sides: same camera rays up to normalize())."""
    name, flat, vec = scene
    jitter = vec["jitter"]
    upload(ctx, flat, jitter)
    ctx.set_option(capi.OPT_COUNT_NODES, 1)
    try:
        part = ctx.partition(integrator="iterative_rrnee", seed=3)
        _, _, st = ctx.render(part)
        _, _, want = oracle_port.render(flat.pointer(), jitter, part)
    finally:
        ctx.set_option(capi.OPT_COUNT_NODES, 0)
    for key in ("nodes_visited", "prims_tested", "xf_prims_tested"):
        assert abs(st[key] - want[key]) <= 0.02 * want[key] + 16, (key, st[key], want[key])


def test_bad_partitions_are_rejected(ctx, scene):
    name, flat, vec = scene
    upload(ctx, flat, vec["jitter"])
    spp = vec["jitter"].shape[0]
    with pytest.raises(capi.SpcuError):
        ctx.render(ctx.partition(spp=spp, rank=2, world=2))
    with pytest.raises(capi.SpcuError):
        ctx.render(ctx.partition(spp=spp + 1))  # longer than the jitter table
    with pytest.raises(capi.SpcuError):
        ctx.render(capi.Partition(0, 1, 0, spp, spp, 9, 0))  # unknown integrator
