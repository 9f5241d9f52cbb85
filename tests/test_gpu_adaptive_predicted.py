"""Adaptive sampling with predicted sample counts (spcu_render_adaptive_predicted) on the device.

A pixel's count is on the doubling grid min_spp, 2 min_spp, ... up to the budget, and every round's tests are made before its
decisions, so the numpy model (simplepath_b200/adaptive.py) run on fixed renders' sums at the grid counts reproduces every
decision and every move; the ranges a pixel renders are contiguous, so its sums equal a fixed render of [0, n_p) whatever the
partition, lanes, wavefront size or kernel organisation.  Both are checked exactly on every golden scene and kernel
organisation, and the images are held statistically against the reference's converged renders.
"""
import ctypes as C
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
BUDGET, MIN_SPP, FLOOR, SEED = 64, 4, 1e-3, 20261022
GRID = adaptive.grid(BUDGET, MIN_SPP)  # 4, 8, 16, 32, 64
CANDIDATE_ERRORS = (2.0, 1.0, 0.5, 0.3, 0.2, 0.1, 0.05, 0.02, 0.01, 0.005)
CASES = [(r, m) for r in (0, 2) for m in (1, 4)]  # (radius, max_step)


@pytest.fixture(scope="module", params=[(s, p) for p in PIPELINES for s in SCENES], ids=lambda sp: f"{sp[0]}-{sp[1]}")
def grid_scene(request, ctx):
    """(scene, fixed renders of samples [0, g) at every grid count g, target errors whose maps hold g_0, the budget and
    counts in between)."""
    name, pipeline = request.param
    flat = FlatSceneData.load(GOLDEN / f"{name}.flat.npz")
    ctx.set_option(capi.OPT_PIPELINE, PIPELINES[pipeline])
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), rsequence.jitter_table(BUDGET), keepalive=flat)
    fixed = {}
    for g in GRID:
        rgb, sq, _ = ctx.render_frame(ctx.partition(spp=BUDGET, sample_end=g, seed=SEED))
        fixed[g] = (rgb, sq)
    yield name, flat, fixed, pick_errors(fixed, (flat.height, flat.width))
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_WAVEFRONT)


def model_map(fixed, partition, rel_error, radius, max_step, budget=BUDGET, min_spp=MIN_SPP):
    return adaptive.predicted_spp_map(lambda n: fixed[n], partition, budget, min_spp, max_step, rel_error, FLOOR, radius=radius)


def pick_errors(fixed, shape):
    """One target error whose radius-0, max_step-4 map holds g_0, the budget and a count in between, where one exists (the
    one with the most distinct counts); otherwise one that holds g_0 and one that holds the budget."""
    whole = np.ones(shape, dtype=bool)
    counts = {e: set(np.unique(model_map(fixed, whole, e, 0, 4)).tolist()) for e in CANDIDATE_ERRORS}

    def most(keep):
        ok = [e for e, u in counts.items() if keep(u)]
        return max(ok, key=lambda e: len(counts[e])) if ok else None

    both = most(lambda u: GRID[0] in u and BUDGET in u and len(u) >= 3)
    if both is not None:
        return [both]
    errors = [e for e in (most(lambda u: GRID[0] in u and len(u) >= 2), most(lambda u: BUDGET in u and len(u) >= 2)) if e is not None]
    seen = set().union(*(counts[e] for e in errors))
    assert GRID[0] in seen and BUDGET in seen and len(seen) >= 3, f"no candidate error exercises the grid: {counts}"
    return errors


def assert_sums_are_fixed_renders(fixed, rgb, sq, spp_map):
    for n in np.unique(spp_map):
        sel = spp_map == n
        want_rgb, want_sq = fixed[int(n)]
        assert rgb[sel].tobytes() == want_rgb[sel].tobytes(), f"sums of the pixels with {n} samples"
        assert sq[sel].tobytes() == want_sq[sel].tobytes(), f"sums of squares of the pixels with {n} samples"


def test_decisions_and_sums_are_exact(ctx, grid_scene):
    name, flat, fixed, errors = grid_scene
    whole = np.ones((flat.height, flat.width), dtype=bool)
    part = ctx.partition(spp=BUDGET, seed=SEED)
    seen = set()
    for rel in errors:
        for radius, max_step in CASES:
            rgb, sq, spp_map, st = ctx.render_adaptive_predicted(part, rel, min_spp=MIN_SPP, max_step=max_step, abs_floor=FLOOR,
                                                                 radius=radius)
            want = model_map(fixed, whole, rel, radius, max_step)
            assert np.array_equal(spp_map, want), \
                f"{name}, rel_error {rel}, radius {radius}, max_step {max_step}: {(spp_map != want).sum()} pixels differ from the model"
            assert_sums_are_fixed_renders(fixed, rgb, sq, spp_map)
            assert st["paths"] == int(spp_map.sum(dtype=np.uint64))
            assert 1 <= st["rounds"] <= len(GRID) and st["calls"] >= st["rounds"]
            if radius == 0 and max_step == 4:
                seen |= set(np.unique(spp_map).tolist())
    assert GRID[0] in seen and BUDGET in seen and len(seen) >= 3, seen


def test_invariant_to_batches_lanes_and_tiles(ctx, grid_scene):
    name, flat, fixed, errors = grid_scene
    rel = errors[0]
    kw = dict(min_spp=MIN_SPP, max_step=4, abs_floor=FLOOR, radius=2)
    part = ctx.partition(spp=BUDGET, seed=SEED)
    rgb, sq, spp_map, st = ctx.render_adaptive_predicted(part, rel, **kw)
    try:
        for lanes in (1, 2, 4):
            ctx.set_option(capi.OPT_BATCH_LANES, lanes)
            r, s, m, _ = ctx.render_adaptive_predicted(part, rel, **kw)
            assert r.tobytes() == rgb.tobytes() and s.tobytes() == sq.tobytes() and np.array_equal(m, spp_map), f"{lanes} lanes"
        ctx.set_option(capi.OPT_BATCH_LANES, 0)
        ctx.set_wavefront_size(777)
        r, s, m, st_small = ctx.render_adaptive_predicted(part, rel, **kw)
        assert r.tobytes() == rgb.tobytes() and s.tobytes() == sq.tobytes() and np.array_equal(m, spp_map), "wavefront 777"
        assert st_small["paths"] == st["paths"]
    finally:
        ctx.set_option(capi.OPT_BATCH_LANES, 0)
        ctx.set_wavefront_size(0)
    tiles, tiles_sq, tiles_map, paths = np.zeros_like(rgb), np.zeros_like(sq), np.zeros_like(spp_map), 0
    for rank in range(3):
        r, s, m, st_t = ctx.render_adaptive_predicted(ctx.partition(spp=BUDGET, seed=SEED, rank=rank, world=3), rel, **kw)
        assert not (m.astype(bool) & tiles_map.astype(bool)).any(), "tile partitions overlap"
        tiles += r
        tiles_sq += s
        tiles_map += m
        paths += st_t["paths"]
    assert tiles.tobytes() == rgb.tobytes() and tiles_sq.tobytes() == sq.tobytes() and np.array_equal(tiles_map, spp_map)
    assert paths == st["paths"]


def test_two_point_grid_is_the_pass_schedule(ctx, grid_scene):
    """budget = 2 min_spp: the grid is {min_spp, 2 min_spp}, and every max_step gives what spcu_render_adaptive gives with
    pass_spp = min_spp, byte for byte."""
    name, flat, fixed, errors = grid_scene
    part = ctx.partition(spp=BUDGET, sample_end=2 * MIN_SPP, seed=SEED)
    for rel in errors + [0.2]:
        for radius in (0, 2):
            want = ctx.render_adaptive(part, rel, min_spp=MIN_SPP, pass_spp=MIN_SPP, abs_floor=FLOOR, radius=radius)
            for max_step in (1, 4, 8):
                got = ctx.render_adaptive_predicted(part, rel, min_spp=MIN_SPP, max_step=max_step, abs_floor=FLOOR, radius=radius)
                for a, b in zip(got[:3], want[:3]):
                    assert a.tobytes() == b.tobytes(), f"{name}, rel_error {rel}, radius {radius}, max_step {max_step}"


def test_budget_of_min_spp_is_a_fixed_render(ctx, grid_scene):
    name, flat, fixed, errors = grid_scene
    part = ctx.partition(spp=BUDGET, sample_end=MIN_SPP, seed=SEED)
    rgb, sq, spp_map, st = ctx.render_adaptive_predicted(part, errors[0], min_spp=MIN_SPP, radius=2)
    assert rgb.tobytes() == fixed[MIN_SPP][0].tobytes() and sq.tobytes() == fixed[MIN_SPP][1].tobytes()
    assert (spp_map == MIN_SPP).all() and st["rounds"] == 1 and st["calls"] == 1


def _bunny(ctx):
    flat = FlatSceneData.load(GOLDEN / "g_bunny.flat.npz")
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_AUTO)
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), rsequence.jitter_table(BUDGET), keepalive=flat)
    return flat


@pytest.mark.parametrize("bad", [dict(min_spp=1), dict(min_spp=0), dict(max_step=0), dict(max_step=9), dict(radius=8),
                                 dict(radius=2 ** 32 - 1), dict(rel_error=-0.1), dict(rel_error=float("nan")),
                                 dict(abs_floor=float("inf")), dict(abs_floor=-1.0), dict(sample_begin=4)],
                         ids=lambda d: "-".join(f"{k}={v}" for k, v in d.items()))
def test_rejections_leave_the_context_usable(ctx, bad):
    _bunny(ctx)
    good = dict(min_spp=4, max_step=4, abs_floor=0.0, radius=2, rel_error=0.1)
    part = ctx.partition(spp=BUDGET, seed=9, sample_end=32)
    before = ctx.render_adaptive_predicted(part, **good)
    args = {**good, **bad}
    if "sample_begin" in args:
        bad_part = ctx.partition(spp=BUDGET, seed=9, sample_end=32)
        bad_part.sample_begin = args.pop("sample_begin")
    else:
        bad_part = part
    with pytest.raises(capi.SpcuError):
        ctx.render_adaptive_predicted(bad_part, **args)
    after = ctx.render_adaptive_predicted(part, **good)
    for a, b in zip(before[:3], after[:3]):
        assert a.tobytes() == b.tobytes()


@pytest.mark.parametrize("radius", [0, 2])
def test_device_entry_point_equals_the_host_one(ctx, radius):
    import torch
    _bunny(ctx)
    part = ctx.partition(spp=BUDGET, seed=17)
    kw = dict(min_spp=4, max_step=4, abs_floor=1e-3, radius=radius)
    runs = [(e, ctx.render_adaptive_predicted(part, e, **kw)) for e in (1.0, 0.5, 0.3, 0.2, 0.1, 0.05, 0.02)]
    rel, (want, want_sq, want_map, st_w) = max(runs, key=lambda r: len(np.unique(r[1][2])))
    assert len(np.unique(want_map)) >= 3, np.unique(want_map)

    rgb = torch.zeros((ctx.height, ctx.width, 3), dtype=torch.float32, device="cuda")
    sq = torch.zeros((ctx.height, ctx.width), dtype=torch.float32, device="cuda")
    spp_map = torch.zeros((ctx.height, ctx.width), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ap = capi.AdaptivePredicted(kw["min_spp"], rel, kw["abs_floor"], radius, kw["max_step"])
    rounds, calls, st = C.c_uint32(), C.c_uint32(), capi.Stats()
    ctx._check(ctx.lib.spcu_render_adaptive_predicted_device(ctx.h, C.byref(part), C.byref(ap), C.c_void_p(rgb.data_ptr()),
                                                             C.c_void_p(sq.data_ptr()), C.c_void_p(spp_map.data_ptr()),
                                                             C.byref(rounds), C.byref(calls), C.byref(st), None),
               "spcu_render_adaptive_predicted_device")
    torch.cuda.synchronize()
    assert rgb.cpu().numpy().tobytes() == want.tobytes() and sq.cpu().numpy().tobytes() == want_sq.tobytes()
    assert np.array_equal(spp_map.cpu().numpy().view(np.uint32), want_map)
    assert rounds.value == st_w["rounds"] and calls.value == st_w["calls"] and st.paths == st_w["paths"]


# ---- statistics against the reference's converged renders (the metric and bounds of test_gpu_adaptive_window.py) ------------
EPS = 1e-3
CONVERGED = {"c2": ("c2_example_scene", 64, 0.05), "c3": ("c3_bunny", 256, 0.1), "c4": ("c4_elf", 64, 0.05)}
# Radius 2, as the pass schedule's test.  Larger steps stop more of bunny's pixels before a rare bright path shows up in their
# window: at 0.1 its mean luminance is -0.69 % with max_step 1, -0.84 % with 2 and -1.79 % with 4 or 8, outside the bound
# (profiles/r09a_adaptive_predicted_probe.jsonl, DESIGN.md §11.1).  The bound is held for the steps that keep it.
STEPS_WITHIN_BOUND = (1, 2)


def lum(c):
    return 0.2126 * c[..., 0] + 0.7152 * c[..., 1] + 0.0722 * c[..., 2]


def block_mean(a, b):
    h, w = a.shape[:2]
    return a.reshape(h // b, b, w // b, b, *a.shape[2:]).mean(axis=(1, 3))


@pytest.mark.parametrize("max_step", STEPS_WITHIN_BOUND)
@pytest.mark.parametrize("cfg", list(CONVERGED))
def test_relmse_against_the_reference_render(ctx, cfg, max_step):
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
    rgb, _, spp_map, st = ctx.render_adaptive_predicted(ctx.partition(spp=budget, seed=20261018), rel, min_spp=16,
                                                        max_step=max_step, want_sumsq=False, radius=2)
    n = spp_map.astype(np.float64)
    assert st["paths"] == int(spp_map.sum(dtype=np.uint64)) and (n >= 16).all()
    mine = block_mean(lum(rgb.astype(np.float64) / n[..., None]), b)
    ref, var = gold["lum"].astype(np.float64), gold["lum_var"].astype(np.float64)
    denom = ref ** 2 + EPS
    relmse = float(((mine - ref) ** 2 / denom).mean())
    expected = float((var / (b * b) * (block_mean(1.0 / n, b) + 1.0 / n_ref) / denom).mean())
    print(f"\n{cfg}: predicted counts, rel_error {rel}, radius 2, max_step {max_step}, budget {budget}: mean spp {n.mean():.1f}, "
          f"{st['rounds']} rounds, {st['calls']} calls; relMSE {relmse:.3e}, expected {expected:.3e} (ratio {relmse / expected:.2f}); "
          f"mean luminance {mine.mean():.5f} vs {ref.mean():.5f}")
    assert relmse <= 1.5 * expected + 1e-5, f"{cfg}: relMSE {relmse:.3e} vs expected {expected:.3e}"
    assert abs(mine.mean() - ref.mean()) <= 0.01 * ref.mean()


# ---- the drop-in with SPCU_ADAPTIVE_STEP --------------------------------------------------------------------------------------
needs_plugin = pytest.mark.skipif(not host.DRIVER.exists() or not host.available(),
                                  reason="host plugin not built (needs the reference sources)")


def _driver(tmp_path, spp, **env):
    sp = scenes.ensure("g_bunny", tmp_path)
    proc = subprocess.run([str(host.DRIVER), "--samples", str(spp), "--integrator", "cuda", sp.name], cwd=tmp_path,
                          env=dict(os.environ, **env), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    return sp, proc


@needs_plugin
def test_driver_with_predicted_counts_writes_the_same_image(ctx, tmp_path):
    spp, rel = 64, 0.1
    sp, proc = _driver(tmp_path, spp, SPCU_SEED="11", SPCU_ADAPTIVE=str(rel), SPCU_ADAPTIVE_RADIUS="2", SPCU_ADAPTIVE_STEP="3")
    assert proc.returncode == 0, proc.stdout[-2000:]
    assert "max step 3" in proc.stdout and "rounds" in proc.stdout and "render calls" in proc.stdout
    img = scenes.read_pfm(tmp_path / "image.pfm")

    flat = host.parse(sp)
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_AUTO)
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), host.jitter(spp), keepalive=flat)
    rgb, _, spp_map, _ = ctx.render_adaptive_predicted(ctx.partition(spp=spp, integrator="iterative_rrnee", seed=11), rel, min_spp=16,
                                                       max_step=3, want_sumsq=False, radius=2)
    want = ctx.pack_image(rgb, spp_map, capi.IMAGE_PFM)[::-1]  # packed rows are bottom-up, read_pfm's top-down
    assert img.tobytes() == np.ascontiguousarray(want).tobytes()


@needs_plugin
def test_driver_without_a_step_keeps_the_pass_schedule(tmp_path):
    _, with_unset = _driver(tmp_path, 32, SPCU_SEED="5", SPCU_ADAPTIVE="0.1")
    assert with_unset.returncode == 0, with_unset.stdout[-2000:]
    assert "passes" in with_unset.stdout and "max step" not in with_unset.stdout
    img = scenes.read_pfm(tmp_path / "image.pfm")
    _, with_empty = _driver(tmp_path, 32, SPCU_SEED="5", SPCU_ADAPTIVE="0.1", SPCU_ADAPTIVE_STEP="")
    assert with_empty.returncode == 0 and "max step" not in with_empty.stdout
    assert scenes.read_pfm(tmp_path / "image.pfm").tobytes() == img.tobytes()


@needs_plugin
@pytest.mark.parametrize("value", ["0", "9", "two", "-1", "4x"])
def test_driver_rejects_a_bad_step(tmp_path, value):
    _, proc = _driver(tmp_path, 16, SPCU_ADAPTIVE="0.1", SPCU_ADAPTIVE_STEP=value)
    assert proc.returncode != 0 and "SPCU_ADAPTIVE_STEP" in proc.stdout
