"""Adaptive sampling with predicted sample counts without a GPU: the numpy model (simplepath_b200/adaptive.py) against a
per-pixel restatement of the contract in include/spcu.h, the properties the contract states, and the ctypes mirror of
spcu_adaptive_predicted."""
import ctypes
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT
from simplepath_b200 import adaptive

F = np.float32
H, W = 19, 21  # partial tiles on the right and at the bottom


@pytest.mark.parametrize("budget,min_spp,want", [
    (256, 16, [16, 32, 64, 128, 256]),
    (100, 16, [16, 32, 64, 100]),
    (16, 16, [16]),
    (10, 16, [10]),
    (32, 16, [16, 32]),
    (2 ** 32 - 1, 2, [2 ** k for k in range(1, 32)] + [2 ** 32 - 1]),
])
def test_grid(budget, min_spp, want):
    assert adaptive.grid(budget, min_spp) == want
    assert len(want) <= 32  # min_spp >= 2: the device keeps a grid index in one byte and bounds its buckets by this


def _random_sums(seed, budget, shape=(H, W), special=True):
    """Per-pixel samples with a spread of noise levels (grey radiance, so luminance = value), some zero-variance, empty and
    non-finite pixels, and their sums at any n."""
    rng = np.random.default_rng(seed)
    scale = rng.choice([0.0, 0.02, 0.1, 0.3, 1.0, 3.0], size=shape)
    samples = (0.5 + scale[..., None] * rng.standard_normal((*shape, budget))).astype(F)
    if special:
        samples[rng.random(shape) < 0.05, :] = 0.5  # zero variance
        samples[rng.random(shape) < 0.03, :] = 0.0  # empty: mean and variance 0
        nan = rng.random(shape) < 0.02
        samples[nan, rng.integers(0, budget)] = np.inf  # a non-finite sample from then on
    cum = np.cumsum(samples, axis=-1, dtype=F)
    cum2 = np.cumsum(samples * samples, axis=-1, dtype=F)

    def sums_at(n):
        return np.repeat(cum[..., n - 1][..., None], 3, axis=-1), cum2[..., n - 1]

    return sums_at


def _scalar_need(rgb, q, n, rel, floor):
    """need for one pixel, straight from the contract (float32, one rounding per operation)."""
    R, G, B = (F(x) for x in rgb)
    q, nf = F(q), F(n)
    with np.errstate(all="ignore"):
        L = F(F(F(0.2126) * R) + F(F(0.7152) * G)) + F(F(0.0722) * B)
        m = F(L / nf)
        d = F(F(q / nf) - F(m * m))
        v = F(d * F(nf / F(nf - F(1)))) if d > 0 else F(0)
        T = F(F(rel) * F(m + F(floor)))
        TT = F(T * T)
        need = F(v / TT)
    if not all(np.isfinite([R, G, B, q])) or not (TT > 0) or not np.isfinite(TT) or not np.isfinite(need):
        return F(np.inf)
    return need


def _scalar_target(need, j, g, max_step):
    upper = min(j + max_step, len(g) - 1)
    for i in range(j + 1, upper + 1):
        if F(g[i]) >= need:
            return i
    return upper


@pytest.mark.parametrize("seed", range(3))
def test_need_and_target_match_the_contract_pixel_by_pixel(seed):
    budget, min_spp = 256, 4
    g = adaptive.grid(budget, min_spp)
    sums_at = _random_sums(seed, budget)
    rng = np.random.default_rng(100 + seed)
    for n in g[:-1]:
        rgb, sq = sums_at(n)
        for rel, floor in ((0.1, 0.0), (0.05, 0.03), (0.0, 0.0), (0.3, 1e-3)):
            need = adaptive.need(rgb, sq, n, rel, floor)
            assert need.dtype == F
            for y in range(H):
                for x in range(W):
                    want = _scalar_need(rgb[y, x], sq[y, x], n, rel, floor)
                    assert need[y, x].tobytes() == want.tobytes(), (n, rel, y, x)
            j = rng.integers(0, len(g) - 1, size=(H, W))
            for max_step in (1, 2, 4, 8):
                t = adaptive.target_level(need, j, g, max_step)
                want = np.array([[_scalar_target(need[y, x], j[y, x], g, max_step) for x in range(W)] for y in range(H)])
                assert np.array_equal(t, want)
                assert ((t > j) & (t - j <= max_step) & (t <= len(g) - 1)).all()
    assert np.isinf(adaptive.need(*sums_at(g[0]), g[0], 0.0, 0.0)).all(), "T = 0: need is +inf"


def _scalar_map(sums_at, partition, budget, min_spp, max_step, rel, floor, radius):
    """The rounds of the contract, one pixel at a time: test every active pixel below the budget at its own count, then decide
    each one from the window's flags, then move the ones that go on."""
    g = adaptive.grid(budget, min_spp)
    last = len(g) - 1
    h, w = partition.shape
    level = {p: 0 for p in zip(*np.nonzero(partition))}
    passed = np.ones((h, w), dtype=bool)
    out = np.zeros((h, w), dtype=np.uint32)
    while level:
        for p in [p for p, j in level.items() if j == last]:
            out[p], passed[p] = budget, True
            del level[p]
        need = {}
        for p, j in level.items():
            rgb, sq = sums_at(g[j])
            passed[p] = bool(adaptive.converged(rgb[p], sq[p], g[j], rel, floor))
            need[p] = _scalar_need(rgb[p], sq[p], g[j], rel, floor)
        moves = {}
        for (y, x), j in level.items():
            win = [(qy, qx) for qy in range(max(0, y - radius), min(h, y + radius + 1))
                   for qx in range(max(0, x - radius), min(w, x + radius + 1)) if (qy >> 3, qx >> 3) == (y >> 3, x >> 3)]
            if all(passed[q] for q in win):
                out[y, x] = g[j]
                moves[(y, x)] = None
            else:
                moves[(y, x)] = j + 1 if passed[y, x] else _scalar_target(need[(y, x)], j, g, max_step)
        for p, t in moves.items():
            if t is None:
                del level[p]
            else:
                level[p] = t
    return out


@pytest.mark.parametrize("radius", [0, 1, 2])
@pytest.mark.parametrize("max_step", [1, 3, 8])
def test_model_matches_the_rounds_pixel_by_pixel(radius, max_step):
    budget, min_spp = 128, 4
    sums_at = _random_sums(7 + radius, budget)
    part = np.ones((H, W), dtype=bool)
    part[8:16, 0:8] = False  # one tile outside the partition
    for rel in (0.05, 0.2):
        want = _scalar_map(sums_at, part, budget, min_spp, max_step, rel, 1e-3, radius)
        got = adaptive.predicted_spp_map(sums_at, part, budget, min_spp, max_step, rel, 1e-3, radius=radius)
        assert np.array_equal(got, want)


@pytest.mark.parametrize("seed", range(4))
def test_counts_are_on_the_grid_and_never_fall_as_the_radius_grows(seed):
    budget, min_spp = 256, 4
    g = adaptive.grid(budget, min_spp)
    sums_at = _random_sums(seed, budget)
    part = np.ones((H, W), dtype=bool)
    for max_step in (1, 2, 4, 8):
        for rel in (0.02, 0.1, 0.4):
            maps = [adaptive.predicted_spp_map(sums_at, part, budget, min_spp, max_step, rel, 1e-3, radius=r) for r in range(8)]
            assert set(np.unique(maps[0]).tolist()) <= set(g)
            for r in range(7):
                assert set(np.unique(maps[r + 1]).tolist()) <= set(g)
                assert (maps[r] <= maps[r + 1]).all(), f"max_step {max_step}, rel {rel}: radius {r + 1} stops a pixel earlier"
            assert (maps[0] >= min(min_spp, budget)).all() and (maps[0] <= budget).all()
    spread = adaptive.predicted_spp_map(sums_at, part, budget, min_spp, 4, 0.1, 1e-3)
    assert len(np.unique(spread)) >= 4, "the sums must exercise the grid"


@pytest.mark.parametrize("max_step", range(1, 9))
def test_two_point_grid_is_the_pass_schedule(max_step):
    min_spp = 8
    budget = 2 * min_spp
    assert adaptive.grid(budget, min_spp) == [min_spp, budget]
    part = np.ones((H, W), dtype=bool)
    part[:8, 8:16] = False
    for seed in range(3):
        sums_at = _random_sums(seed, budget)
        for radius in (0, 2):
            for rel in (0.05, 0.2, 0.5):
                want = adaptive.spp_map(sums_at, part, budget, min_spp, min_spp, rel, 1e-3, radius=radius)
                got = adaptive.predicted_spp_map(sums_at, part, budget, min_spp, max_step, rel, 1e-3, radius=radius)
                assert np.array_equal(got, want)


def test_budget_of_min_spp_renders_every_pixel_once():
    sums_at = _random_sums(0, 16)
    part = np.ones((H, W), dtype=bool)
    part[8:, 8:16] = False
    got = adaptive.predicted_spp_map(sums_at, part, 16, 16, 4, 0.1, 0.0)
    assert np.array_equal(got, np.where(part, 16, 0).astype(np.uint32))


def test_ctypes_mirror_matches_the_header(built):
    from simplepath_b200 import capi
    probe = r'''
    #include "spcu.h"
    #include <stddef.h>
    #include <stdio.h>
    int main(void){ printf("%zu %zu %zu %zu %zu %zu %d\n", sizeof(spcu_adaptive_predicted),
        offsetof(spcu_adaptive_predicted, min_spp), offsetof(spcu_adaptive_predicted, rel_error),
        offsetof(spcu_adaptive_predicted, abs_floor), offsetof(spcu_adaptive_predicted, radius),
        offsetof(spcu_adaptive_predicted, max_step), SPCU_ABI_VERSION); return 0; }
    '''
    with tempfile.TemporaryDirectory() as d:
        src = f"{d}/p.c"
        open(src, "w").write(probe)
        subprocess.check_call(["gcc", "-I", str(ROOT / "include"), src, "-o", f"{d}/p"])
        got = [int(x) for x in subprocess.check_output([f"{d}/p"]).split()]
    A = capi.AdaptivePredicted
    assert got == [ctypes.sizeof(A), A.min_spp.offset, A.rel_error.offset, A.abs_floor.offset, A.radius.offset,
                   A.max_step.offset, 2]
    assert capi.ABI_VERSION == 2
