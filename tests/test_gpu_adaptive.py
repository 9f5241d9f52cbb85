"""Adaptive sampling (spcu_render_adaptive) on the device.

Random numbers are keyed by (pixel, global sample index) and the resolve kernel adds a pixel's samples in sample order,
so the sums of a pixel that received samples [0, n) equal, bit for bit, those of a fixed render of [0, n).  The stopping
test is float32 with one rounding per operation, so the numpy model (simplepath_b200/adaptive.py) run on those fixed
renders' sums reproduces every decision.  Both are checked exactly here, on every golden scene and kernel organisation,
and the images are held statistically against the reference's converged renders.
"""
import numpy as np
import pytest

from conftest import GOLDEN
from simplepath_b200 import adaptive, capi, host, rsequence
from simplepath_b200.flat import FlatSceneData

pytestmark = pytest.mark.gpu
SCENES = ["g_spheres", "g_spheres_ibl", "g_example", "g_bunny", "g_elf", "g_chain", "g_lights"]
PIPELINES = {"smwave": capi.PIPELINE_SMWAVE, "paths": capi.PIPELINE_PATHS, "wavefront": capi.PIPELINE_WAVEFRONT}
BUDGET, MIN_SPP, PASS_SPP, FLOOR, SEED = 64, 4, 4, 1e-3, 20261020
CANDIDATE_ERRORS = (1.0, 0.5, 0.3, 0.2, 0.1, 0.05, 0.02, 0.01)


@pytest.fixture(scope="module", params=[(s, p) for p in PIPELINES for s in SCENES], ids=lambda sp: f"{sp[0]}-{sp[1]}")
def scene(request, ctx):
    """(scene, kernel organisation, fixed renders of samples [0, b) at every pass boundary b of the schedule)."""
    name, pipeline = request.param
    flat = FlatSceneData.load(GOLDEN / f"{name}.flat.npz")
    ctx.set_option(capi.OPT_PIPELINE, PIPELINES[pipeline])
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), rsequence.jitter_table(BUDGET), keepalive=flat)
    fixed = {}
    for b in adaptive.boundaries(BUDGET, MIN_SPP, PASS_SPP):
        rgb, sq, _ = ctx.render_frame(ctx.partition(spp=BUDGET, sample_end=b, seed=SEED))
        fixed[b] = (rgb, sq)
    yield name, flat, fixed
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_WAVEFRONT)


def model_map(fixed, partition, rel_error, abs_floor=FLOOR):
    return adaptive.spp_map(lambda n: fixed[n], partition, BUDGET, MIN_SPP, PASS_SPP, rel_error, abs_floor)


def exercising_error(fixed, shape):
    """The target error whose map (by the model) holds the most distinct counts, min_spp and the budget among them: the
    test must see pixels stop at the first test, in between, and run to the budget."""
    best, best_n = None, 0
    whole = np.ones(shape, dtype=bool)
    for e in CANDIDATE_ERRORS:
        u = np.unique(model_map(fixed, whole, e))
        if MIN_SPP in u and BUDGET in u and len(u) > best_n:
            best, best_n = e, len(u)
    assert best is not None and best_n >= 3, "no candidate error exercises the schedule on this scene"
    return best


def assert_sums_are_fixed_renders(fixed, rgb, sq, spp_map):
    for n in np.unique(spp_map):
        sel = spp_map == n
        want_rgb, want_sq = fixed[int(n)]
        assert rgb[sel].tobytes() == want_rgb[sel].tobytes(), f"sums of the pixels with {n} samples"
        assert sq[sel].tobytes() == want_sq[sel].tobytes(), f"sums of squares of the pixels with {n} samples"


def passes_of(spp_map):
    """Passes the schedule runs for a whole-frame map: up to the boundary of the last pixel to stop."""
    b = adaptive.boundaries(BUDGET, MIN_SPP, PASS_SPP)
    return b.index(int(spp_map.max())) + 1


def test_sums_and_decisions_are_exact(ctx, scene):
    name, flat, fixed = scene
    shape = (flat.height, flat.width)
    rel = exercising_error(fixed, shape)
    part = ctx.partition(spp=BUDGET, seed=SEED)
    rgb, sq, spp_map, st = ctx.render_adaptive(part, rel, min_spp=MIN_SPP, pass_spp=PASS_SPP, abs_floor=FLOOR)
    want = model_map(fixed, np.ones(shape, dtype=bool), rel)
    assert np.array_equal(spp_map, want), f"{name}: {(spp_map != want).sum()} pixels decided otherwise than the model"
    u = np.unique(spp_map)
    assert len(u) >= 3 and MIN_SPP in u and BUDGET in u, u
    assert_sums_are_fixed_renders(fixed, rgb, sq, spp_map)
    assert st["paths"] == int(spp_map.sum(dtype=np.uint64))
    assert st["passes"] == passes_of(spp_map)


def test_zero_error_stops_only_zero_variance_pixels(ctx, scene):
    name, flat, fixed = scene
    part = ctx.partition(spp=BUDGET, seed=SEED)
    rgb, sq, spp_map, st = ctx.render_adaptive(part, 0.0, min_spp=MIN_SPP, pass_spp=PASS_SPP, abs_floor=0.0)
    want = model_map(fixed, np.ones(spp_map.shape, dtype=bool), 0.0, 0.0)
    assert np.array_equal(spp_map, want)
    assert_sums_are_fixed_renders(fixed, rgb, sq, spp_map)
    assert st["paths"] == int(spp_map.sum(dtype=np.uint64))


def test_invariant_to_batches_lanes_and_tiles(ctx, scene):
    name, flat, fixed = scene
    rel = exercising_error(fixed, (flat.height, flat.width))
    kw = dict(min_spp=MIN_SPP, pass_spp=PASS_SPP, abs_floor=FLOOR)
    part = ctx.partition(spp=BUDGET, seed=SEED)
    rgb, sq, spp_map, st = ctx.render_adaptive(part, rel, **kw)
    try:
        for lanes in (1, 2, 4):
            ctx.set_option(capi.OPT_BATCH_LANES, lanes)
            r, s, m, _ = ctx.render_adaptive(part, rel, **kw)
            assert r.tobytes() == rgb.tobytes() and s.tobytes() == sq.tobytes() and np.array_equal(m, spp_map), f"{lanes} lanes"
        ctx.set_option(capi.OPT_BATCH_LANES, 0)
        ctx.set_wavefront_size(777)
        r, s, m, st_small = ctx.render_adaptive(part, rel, **kw)
        assert r.tobytes() == rgb.tobytes() and s.tobytes() == sq.tobytes() and np.array_equal(m, spp_map), "wavefront 777"
        assert st_small["paths"] == st["paths"]
    finally:
        ctx.set_option(capi.OPT_BATCH_LANES, 0)
        ctx.set_wavefront_size(0)
    tiles, tiles_sq, tiles_map, paths = np.zeros_like(rgb), np.zeros_like(sq), np.zeros_like(spp_map), 0
    for rank in range(3):
        r, s, m, st_t = ctx.render_adaptive(ctx.partition(spp=BUDGET, seed=SEED, rank=rank, world=3), rel, **kw)
        assert not (m.astype(bool) & tiles_map.astype(bool)).any(), "tile partitions overlap"
        tiles += r
        tiles_sq += s
        tiles_map += m
        paths += st_t["paths"]
    assert tiles.tobytes() == rgb.tobytes() and tiles_sq.tobytes() == sq.tobytes() and np.array_equal(tiles_map, spp_map)
    assert paths == st["paths"]


def test_budget_equal_to_min_spp_is_a_fixed_render(ctx, scene):
    name, flat, fixed = scene
    part = ctx.partition(spp=BUDGET, sample_end=MIN_SPP, seed=SEED)
    rgb, sq, spp_map, st = ctx.render_adaptive(part, 0.5, min_spp=MIN_SPP, pass_spp=PASS_SPP)
    want_rgb, want_sq = fixed[MIN_SPP]
    assert rgb.tobytes() == want_rgb.tobytes() and sq.tobytes() == want_sq.tobytes()
    assert (spp_map == MIN_SPP).all() and st["passes"] == 1
    assert st["paths"] == flat.width * flat.height * MIN_SPP


def _bunny(ctx):
    flat = FlatSceneData.load(GOLDEN / "g_bunny.flat.npz")
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_AUTO)
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), rsequence.jitter_table(BUDGET), keepalive=flat)
    return flat


def test_pack_image_with_counts(ctx):
    _bunny(ctx)
    rgb, _, spp_map, _ = ctx.render_adaptive(ctx.partition(spp=BUDGET, seed=3, rank=1, world=2), 0.1, min_spp=4, pass_spp=4)
    assert (spp_map == 0).any() and len(np.unique(spp_map)) >= 3  # pixels of the other rank's tiles, and several counts
    for fmt in (capi.IMAGE_PFM, capi.IMAGE_PPM):
        uniform = np.full(spp_map.shape, 7, dtype=np.uint32)
        assert ctx.pack_image(rgb, uniform, fmt).tobytes() == ctx.pack_image(rgb, 7, fmt).tobytes()
    pfm = ctx.pack_image(rgb, spp_map, capi.IMAGE_PFM)
    with np.errstate(invalid="ignore", divide="ignore"):
        want = np.where(spp_map[..., None] > 0, rgb / spp_map[..., None].astype(np.float32), np.float32(0)).astype(np.float32)
    assert pfm.tobytes() == want[::-1].tobytes()  # rows bottom-up
    ppm = ctx.pack_image(rgb, spp_map, capi.IMAGE_PPM)
    for k in np.unique(spp_map):
        sel = (spp_map == k)[::-1]
        if k == 0:
            assert (ppm[sel] == 0).all()
        else:
            assert ppm[sel].tobytes() == ctx.pack_image(rgb, int(k), capi.IMAGE_PPM)[sel].tobytes()


BAD = [dict(min_spp=1), dict(min_spp=0), dict(pass_spp=0), dict(rel_error=-0.1), dict(rel_error=float("nan")),
       dict(rel_error=float("inf")), dict(abs_floor=-1e-3), dict(abs_floor=float("nan")), dict(abs_floor=float("inf"))]


@pytest.mark.parametrize("bad", BAD + [dict(sample_begin=1)], ids=lambda d: ",".join(f"{k}={v}" for k, v in d.items()))
def test_bad_parameters_are_rejected_and_leave_the_context_usable(ctx, bad):
    _bunny(ctx)
    part = ctx.partition(spp=BUDGET, seed=9, sample_end=16)
    before = ctx.render_frame(part)[:2]
    kw = dict(rel_error=0.1, min_spp=4, pass_spp=4, abs_floor=0.0)
    kw.update({k: v for k, v in bad.items() if k != "sample_begin"})
    bad_part = ctx.partition(spp=BUDGET, seed=9, sample_begin=bad.get("sample_begin", 0), sample_end=16)
    with pytest.raises(capi.SpcuError):
        ctx.render_adaptive(bad_part, kw.pop("rel_error"), **kw)
    after = ctx.render_frame(part)[:2]
    assert before[0].tobytes() == after[0].tobytes() and before[1].tobytes() == after[1].tobytes()
    rgb, sq, m, _ = ctx.render_adaptive(part, 0.1, min_spp=4, pass_spp=4)
    assert m.max() <= 16 and m.min() >= 4


# ---- statistics against the reference's converged renders (as tests/test_gpu_converged.py) ------------------------------------
EPS = 1e-3
# config -> (scene, budget, target error).  Bunny at 0.01: at looser targets its pixels stop before they have drawn one of the
# rare bright paths, and the bound does not hold (measured at 0.05: relMSE 1.69x the expected, mean luminance -7.8 %;
# profiles/r05b_adaptive_bias.jsonl, DESIGN.md §11).
CONVERGED = {"c2": ("c2_example_scene", 64, 0.05), "c3": ("c3_bunny", 256, 0.01), "c4": ("c4_elf", 64, 0.05)}


def lum(c):
    return 0.2126 * c[..., 0] + 0.7152 * c[..., 1] + 0.0722 * c[..., 2]


def block_mean(a, b):
    h, w = a.shape[:2]
    return a.reshape(h // b, b, w // b, b, *a.shape[2:]).mean(axis=(1, 3))


@pytest.mark.parametrize("cfg", list(CONVERGED))
def test_relmse_against_the_reference_render(ctx, cfg):
    """Expected relMSE as in test_gpu_converged.py with each block's mean of 1 / n_p in place of 1 / spp.  Stopping on an
    estimated variance can bias a pixel's mean in principle; this bound is where that would show (DESIGN.md)."""
    scene, budget, rel = CONVERGED[cfg]
    path = GOLDEN / f"converged_{cfg}.npz"
    if not path.exists():
        pytest.skip(f"{path.name} not generated")
    if not host.loadable(scene):
        pytest.skip(f"{scene} cannot be loaded here")
    gold = np.load(path)
    b, n_ref = int(gold["block"]), int(gold["spp"])
    flat = host.workload(scene)
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_AUTO)
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), rsequence.jitter_table(budget), keepalive=flat)
    rgb, _, spp_map, st = ctx.render_adaptive(ctx.partition(spp=budget, seed=20261018), rel, min_spp=16, pass_spp=16,
                                              want_sumsq=False)
    n = spp_map.astype(np.float64)
    assert st["paths"] == int(spp_map.sum(dtype=np.uint64)) and (n >= 16).all()
    mine = block_mean(lum(rgb.astype(np.float64) / n[..., None]), b)
    ref, var = gold["lum"].astype(np.float64), gold["lum_var"].astype(np.float64)
    denom = ref ** 2 + EPS
    relmse = float(((mine - ref) ** 2 / denom).mean())
    expected = float((var / (b * b) * (block_mean(1.0 / n, b) + 1.0 / n_ref) / denom).mean())
    print(f"\n{cfg}: adaptive rel_error {rel}, budget {budget}: mean spp {n.mean():.1f}, {st['passes']} passes; relMSE "
          f"{relmse:.3e}, expected {expected:.3e} (ratio {relmse / expected:.2f}); mean luminance {mine.mean():.5f} vs "
          f"{ref.mean():.5f}")
    assert relmse <= 1.5 * expected + 1e-5, f"{cfg}: relMSE {relmse:.3e} vs expected {expected:.3e}"
    assert abs(mine.mean() - ref.mean()) <= 0.01 * ref.mean()
