"""Adaptive sampling with the neighbourhood rule (spcu_adaptive.radius > 0) on the device.

A pixel stops only when every pixel of its window, clipped to its 8x8 tile and the image, passes the per-pixel test.  The
tests are all made before the decisions of a boundary, so the numpy model (simplepath_b200/adaptive.py) run on fixed renders'
sums reproduces every decision, and since a window never leaves its tile the sums still equal a fixed render of [0, n_p)
whatever the partition, lanes or wavefront size.  Both are checked exactly on every golden scene and kernel organisation,
and the images are held statistically against the reference's converged renders.
"""
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN
from simplepath_b200 import adaptive, capi, host, rsequence, scenes
from simplepath_b200.flat import FlatSceneData

pytestmark = pytest.mark.gpu
SCENES = ["g_spheres", "g_spheres_ibl", "g_example", "g_bunny", "g_elf", "g_chain", "g_lights"]
PIPELINES = {"smwave": capi.PIPELINE_SMWAVE, "paths": capi.PIPELINE_PATHS, "wavefront": capi.PIPELINE_WAVEFRONT}
BUDGET, MIN_SPP, PASS_SPP, FLOOR, SEED = 64, 4, 4, 1e-3, 20261021
CANDIDATE_ERRORS = (2.0, 1.0, 0.5, 0.3, 0.2, 0.1, 0.05, 0.02, 0.01)
RADII = (1, 2, 7)


@pytest.fixture(scope="module", params=[(s, p) for p in PIPELINES for s in SCENES], ids=lambda sp: f"{sp[0]}-{sp[1]}")
def window_scene(request, ctx):
    """(scene, fixed renders of samples [0, b) at every pass boundary b, target errors that exercise the r = 1 schedule)."""
    name, pipeline = request.param
    flat = FlatSceneData.load(GOLDEN / f"{name}.flat.npz")
    ctx.set_option(capi.OPT_PIPELINE, PIPELINES[pipeline])
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), rsequence.jitter_table(BUDGET), keepalive=flat)
    fixed = {}
    for b in adaptive.boundaries(BUDGET, MIN_SPP, PASS_SPP):
        rgb, sq, _ = ctx.render_frame(ctx.partition(spp=BUDGET, sample_end=b, seed=SEED))
        fixed[b] = (rgb, sq)
    yield name, flat, fixed, window_errors(fixed, (flat.height, flat.width))
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_WAVEFRONT)


def model_map(fixed, partition, rel_error, radius):
    return adaptive.spp_map(lambda n: fixed[n], partition, BUDGET, MIN_SPP, PASS_SPP, rel_error, FLOOR, radius=radius)


def relative_error(fixed, n):
    """Per pixel, the smallest target error at which its sums after n samples would pass (float64, approximate): the
    standard error of the mean luminance over (mean + abs_floor); inf where a sum is not finite."""
    rgb, sq = (a.astype(np.float64) for a in fixed[n])
    with np.errstate(all="ignore"):
        m = (0.2126 * rgb[..., 0] + 0.7152 * rgb[..., 1] + 0.0722 * rgb[..., 2]) / n
        v = np.maximum(sq / n - m * m, 0.0) * n / (n - 1)
        e = np.sqrt(v / n) / (m + FLOOR)
    return np.where(np.isfinite(rgb).all(axis=-1) & np.isfinite(sq) & np.isfinite(e), e, np.inf)


def window_errors(fixed, shape):
    """Target errors at which the r = 1 maps (by the model) hold min_spp, the budget and counts in between.  One error where
    one can (the map with the most distinct counts); otherwise two, one map holding min_spp and one the budget.  On a scene
    whose noise is much the same everywhere a single error cannot: a whole window passes at min_spp only above `lo`, while
    some pixel fails at every boundary only below `hi` < `lo`.  Besides fixed candidates, errors around both bounds are tried."""
    first = relative_error(fixed, MIN_SPP)
    levels = np.unique(first[np.isfinite(first)])
    lo_i, hi_i = 0, len(levels) - 1  # smallest level at which some r = 1 window passes entirely
    while lo_i < hi_i:
        mid = (lo_i + hi_i) // 2
        if adaptive.window_all(first <= levels[mid], 1).any():
            hi_i = mid
        else:
            lo_i = mid + 1
    lo = float(levels[lo_i]) if len(levels) else np.inf
    tests = [b for b in adaptive.boundaries(BUDGET, MIN_SPP, PASS_SPP) if b < BUDGET]
    hi = float(np.min([relative_error(fixed, b) for b in tests], axis=0).max())
    bounds = [x for x in (lo, hi) if 0 < x < np.inf]
    grid = np.geomspace(min(bounds) / 2, max(bounds) * 2, 24).tolist() if bounds else []
    whole = np.ones(shape, dtype=bool)
    counts = {e: set(np.unique(model_map(fixed, whole, e, 1)).tolist()) for e in list(CANDIDATE_ERRORS) + grid}

    def most(keep):
        ok = [e for e, u in counts.items() if keep(u)]
        return max(ok, key=lambda e: len(counts[e])) if ok else None

    both = most(lambda u: MIN_SPP in u and BUDGET in u and len(u) >= 3)
    if both is not None:
        return [both]
    errors = [e for e in (most(lambda u: MIN_SPP in u and len(u) >= 2), most(lambda u: BUDGET in u and len(u) >= 2)) if e is not None]
    seen = set().union(*(counts[e] for e in errors))
    assert MIN_SPP in seen and BUDGET in seen and len(seen) >= 3, \
        f"no candidate errors exercise the r = 1 schedule on this scene (lo {lo}, hi {hi})"
    return errors


def assert_sums_are_fixed_renders(fixed, rgb, sq, spp_map):
    for n in np.unique(spp_map):
        sel = spp_map == n
        want_rgb, want_sq = fixed[int(n)]
        assert rgb[sel].tobytes() == want_rgb[sel].tobytes(), f"sums of the pixels with {n} samples"
        assert sq[sel].tobytes() == want_sq[sel].tobytes(), f"sums of squares of the pixels with {n} samples"


def tile_constant(m):
    h, w = m.shape
    return all(len(np.unique(m[y:y + 8, x:x + 8])) == 1 for y in range(0, h, 8) for x in range(0, w, 8))


def test_decisions_and_sums_are_exact_for_every_radius(ctx, window_scene):
    name, flat, fixed, errors = window_scene
    whole = np.ones((flat.height, flat.width), dtype=bool)
    part = ctx.partition(spp=BUDGET, seed=SEED)
    kw = dict(min_spp=MIN_SPP, pass_spp=PASS_SPP, abs_floor=FLOOR)
    seen = set()
    for rel in errors:
        maps = {0: ctx.render_adaptive(part, rel, **kw)[2]}
        assert np.array_equal(maps[0], model_map(fixed, whole, rel, 0))
        for r in RADII:
            rgb, sq, spp_map, st = ctx.render_adaptive(part, rel, radius=r, **kw)
            want = model_map(fixed, whole, rel, r)
            assert np.array_equal(spp_map, want), \
                f"{name}, rel_error {rel}, radius {r}: {(spp_map != want).sum()} pixels decided otherwise than the model"
            assert_sums_are_fixed_renders(fixed, rgb, sq, spp_map)
            assert st["paths"] == int(spp_map.sum(dtype=np.uint64))
            maps[r] = spp_map
        seen |= set(np.unique(maps[1]).tolist())
        for lo, hi in zip((0,) + RADII, RADII):
            assert (maps[lo] <= maps[hi]).all(), f"{name}: radius {hi} stops a pixel earlier than radius {lo}"
        assert tile_constant(maps[7])
    assert len(seen) >= 3 and MIN_SPP in seen and BUDGET in seen, seen


def test_invariant_to_batches_lanes_and_tiles(ctx, window_scene):
    name, flat, fixed, errors = window_scene
    rel = errors[0]
    kw = dict(min_spp=MIN_SPP, pass_spp=PASS_SPP, abs_floor=FLOOR, radius=2)
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


def _bunny(ctx):
    flat = FlatSceneData.load(GOLDEN / "g_bunny.flat.npz")
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_AUTO)
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), rsequence.jitter_table(BUDGET), keepalive=flat)
    return flat


@pytest.mark.parametrize("radius", [8, 2 ** 32 - 1])
def test_radius_beyond_the_tile_is_rejected_and_leaves_the_context_usable(ctx, radius):
    _bunny(ctx)
    part = ctx.partition(spp=BUDGET, seed=9, sample_end=16)
    kw = dict(min_spp=4, pass_spp=4, abs_floor=0.0)
    before = ctx.render_adaptive(part, 0.1, radius=2, **kw)
    with pytest.raises(capi.SpcuError, match="radius"):
        ctx.render_adaptive(part, 0.1, radius=radius, **kw)
    after = ctx.render_adaptive(part, 0.1, radius=2, **kw)
    for a, b in zip(before[:3], after[:3]):
        assert a.tobytes() == b.tobytes()


# ---- statistics against the reference's converged renders (the metric and bound of test_gpu_adaptive.py) ---------------------
EPS = 1e-3
RADIUS = 2  # the radius DESIGN.md §11 recommends
# config -> (scene, budget, target error).  Bunny at 0.1, the loosest target measured: with radius 2 its relMSE is 1.15x the
# expected and its mean luminance -0.69 %, against 1.88x and -10.1 % per pixel (profiles/r06a_adaptive_window_bias.jsonl).
CONVERGED = {"c2": ("c2_example_scene", 64, 0.05), "c3": ("c3_bunny", 256, 0.1), "c4": ("c4_elf", 64, 0.05)}


def lum(c):
    return 0.2126 * c[..., 0] + 0.7152 * c[..., 1] + 0.0722 * c[..., 2]


def block_mean(a, b):
    h, w = a.shape[:2]
    return a.reshape(h // b, b, w // b, b, *a.shape[2:]).mean(axis=(1, 3))


@pytest.mark.parametrize("cfg", list(CONVERGED))
def test_relmse_with_the_window_against_the_reference_render(ctx, cfg):
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
                                              want_sumsq=False, radius=RADIUS)
    n = spp_map.astype(np.float64)
    assert st["paths"] == int(spp_map.sum(dtype=np.uint64)) and (n >= 16).all()
    mine = block_mean(lum(rgb.astype(np.float64) / n[..., None]), b)
    ref, var = gold["lum"].astype(np.float64), gold["lum_var"].astype(np.float64)
    denom = ref ** 2 + EPS
    relmse = float(((mine - ref) ** 2 / denom).mean())
    expected = float((var / (b * b) * (block_mean(1.0 / n, b) + 1.0 / n_ref) / denom).mean())
    print(f"\n{cfg}: adaptive rel_error {rel}, radius {RADIUS}, budget {budget}: mean spp {n.mean():.1f}, {st['passes']} passes; "
          f"relMSE {relmse:.3e}, expected {expected:.3e} (ratio {relmse / expected:.2f}); mean luminance {mine.mean():.5f} vs "
          f"{ref.mean():.5f}")
    assert relmse <= 1.5 * expected + 1e-5, f"{cfg}: relMSE {relmse:.3e} vs expected {expected:.3e}"
    assert abs(mine.mean() - ref.mean()) <= 0.01 * ref.mean()


# ---- the drop-in with SPCU_ADAPTIVE_RADIUS ------------------------------------------------------------------------------------
needs_plugin = pytest.mark.skipif(not host.DRIVER.exists() or not host.available(),
                                  reason="host plugin not built (needs the reference sources)")


@needs_plugin
def test_driver_with_a_window_writes_the_same_image(ctx, tmp_path):
    sp = scenes.ensure("g_bunny", tmp_path)
    spp, rel = 64, 0.1
    env = dict(os.environ, SPCU_SEED="11", SPCU_ADAPTIVE=str(rel), SPCU_ADAPTIVE_RADIUS="2")
    proc = subprocess.run([str(host.DRIVER), "--samples", str(spp), "--integrator", "cuda", sp.name], cwd=tmp_path, env=env,
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert proc.returncode == 0, proc.stdout[-2000:]
    assert "radius 2" in proc.stdout
    img = scenes.read_pfm(tmp_path / "image.pfm")

    flat = host.parse(sp)
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_AUTO)
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), host.jitter(spp), keepalive=flat)
    rgb, _, spp_map, _ = ctx.render_adaptive(ctx.partition(spp=spp, integrator="iterative_rrnee", seed=11), rel, min_spp=16,
                                             pass_spp=16, want_sumsq=False, radius=2)
    want = ctx.pack_image(rgb, spp_map, capi.IMAGE_PFM)[::-1]  # packed rows are bottom-up, read_pfm's top-down
    assert img.tobytes() == np.ascontiguousarray(want).tobytes()


@needs_plugin
@pytest.mark.parametrize("value", ["9", "two", "-1"])
def test_driver_rejects_a_bad_radius(tmp_path, value):
    sp = scenes.ensure("g_bunny", tmp_path)
    env = dict(os.environ, SPCU_ADAPTIVE="0.1", SPCU_ADAPTIVE_RADIUS=value)
    proc = subprocess.run([str(host.DRIVER), "--samples", "16", "--integrator", "cuda", sp.name], cwd=tmp_path, env=env,
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert proc.returncode != 0 and "SPCU_ADAPTIVE_RADIUS" in proc.stdout
