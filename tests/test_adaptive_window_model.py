"""The neighbourhood rule of adaptive sampling without a GPU: the numpy model's clipped windows (simplepath_b200/adaptive.py)
against the definition in include/spcu.h, the properties that follow from it, and the ctypes mirror of the `radius` field."""
import ctypes
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT
from simplepath_b200 import adaptive

H, W = 19, 21  # neither a multiple of 8: partial tiles on the right and at the bottom


def window(y, x, h, w, r):
    """W(p) straight from the definition: the pixels q with |x_q - x_p| <= r, |y_q - y_p| <= r, in p's 8x8 tile, in the image."""
    return [(qy, qx) for qy in range(h) for qx in range(w)
            if abs(qx - x) <= r and abs(qy - y) <= r and (qx >> 3, qy >> 3) == (x >> 3, y >> 3)]


@pytest.mark.parametrize("r", range(9))
def test_window_all_matches_the_definition(r):
    rng = np.random.default_rng(r)
    passed = rng.random((H, W)) < 0.93
    got = adaptive.window_all(passed, r)
    want = np.array([[all(passed[q] for q in window(y, x, H, W, r)) for x in range(W)] for y in range(H)])
    assert np.array_equal(got, want)


def _single_failure(y, x, r):
    passed = np.ones((H, W), dtype=bool)
    passed[y, x] = False
    return ~adaptive.window_all(passed, r)  # the pixels whose window holds (y, x)


def test_windows_are_clipped_at_tile_edges():
    blocked = _single_failure(7, 7, 2)  # last pixel of tile (0, 0)
    want = np.zeros((H, W), dtype=bool)
    want[5:8, 5:8] = True  # nothing of tiles (1, 0), (0, 1) or (1, 1), although they are within 2
    assert np.array_equal(blocked, want)
    blocked = _single_failure(8, 8, 1)  # first pixel of tile (1, 1)
    want = np.zeros((H, W), dtype=bool)
    want[8:10, 8:10] = True
    assert np.array_equal(blocked, want)


def test_windows_are_clipped_at_image_edges_and_on_partial_tiles():
    blocked = _single_failure(0, 0, 3)  # image corner
    want = np.zeros((H, W), dtype=bool)
    want[0:4, 0:4] = True
    assert np.array_equal(blocked, want)
    blocked = _single_failure(H - 1, W - 1, 7)  # partial corner tile: columns 16..20, rows 16..18
    want = np.zeros((H, W), dtype=bool)
    want[16:H, 16:W] = True
    assert np.array_equal(blocked, want)
    # a partial tile's window at r = 7 is the part of the tile inside the image: all of it passing lets every pixel stop
    passed = np.zeros((H, W), dtype=bool)
    passed[16:, 16:] = True
    stops = adaptive.window_all(passed, 7)
    assert stops[16:, 16:].all() and not stops[:16].any() and not stops[:, :16].any()


def _random_sums(seed, budget=32, shape=(H, W)):
    """Per-pixel samples with a spread of noise levels (grey radiance, so luminance = value) and their sums at any n."""
    rng = np.random.default_rng(seed)
    scale = rng.choice([0.0, 0.05, 0.3, 1.0, 3.0], size=shape)
    samples = (0.5 + scale[..., None] * rng.standard_normal((*shape, budget))).astype(np.float32)
    samples[rng.random(shape) < 0.05, :] = 0.5  # some zero-variance pixels

    def sums_at(n):
        v = samples[..., :n]
        return np.repeat(v.sum(axis=-1, dtype=np.float32)[..., None], 3, axis=-1), (v * v).sum(axis=-1, dtype=np.float32)

    return sums_at


def _reference_map(sums_at, partition, budget, min_spp, pass_spp, rel_error, abs_floor):
    """The per-pixel schedule as it stood before the window was added (radius 0)."""
    out = np.zeros(partition.shape, dtype=np.uint32)
    active = partition.copy()
    for s in adaptive.boundaries(budget, min_spp, pass_spp):
        if s >= budget or not active.any():
            break
        rgb, sq = sums_at(s)
        done = active & adaptive.converged(rgb, sq, s, rel_error, abs_floor)
        out[done] = s
        active &= ~done
    out[active] = budget
    return out


@pytest.mark.parametrize("seed", range(4))
def test_radius_zero_is_the_per_pixel_rule(seed):
    sums_at = _random_sums(seed)
    part = np.ones((H, W), dtype=bool)
    part[:8, 8:16] = False  # one tile outside the partition
    for rel in (0.02, 0.1, 0.5):
        want = _reference_map(sums_at, part, 32, 4, 4, rel, 1e-3)
        assert np.array_equal(adaptive.spp_map(sums_at, part, 32, 4, 4, rel, 1e-3), want)
        assert np.array_equal(adaptive.spp_map(sums_at, part, 32, 4, 4, rel, 1e-3, radius=0), want)


def _tile_constant(m):
    h, w = m.shape
    for ty in range(0, h, 8):
        for tx in range(0, w, 8):
            if len(np.unique(m[ty:ty + 8, tx:tx + 8])) != 1:
                return False
    return True


@pytest.mark.parametrize("seed", range(4))
def test_maps_are_monotone_in_the_radius_and_tile_constant_at_seven(seed):
    sums_at = _random_sums(seed)
    part = np.ones((H, W), dtype=bool)
    for rel in (0.05, 0.2, 0.5):
        maps = [adaptive.spp_map(sums_at, part, 32, 4, 4, rel, 1e-3, radius=r) for r in range(8)]
        assert len(np.unique(maps[0])) >= 3, "the sums must exercise the schedule"
        for r in range(7):
            assert (maps[r] <= maps[r + 1]).all(), f"rel_error {rel}: radius {r + 1} stops a pixel earlier than radius {r}"
        assert _tile_constant(maps[7])
        assert np.array_equal(maps[7], adaptive.spp_map(sums_at, part, 32, 4, 4, rel, 1e-3, radius=100))


def test_a_stopped_pixel_counts_as_passing_for_its_neighbours():
    """Pixel a passes at every boundary; b, its neighbour, fails at the first and passes from the second on.  With r = 1 a
    waits for b, and once b has stopped neither blocks the other."""
    shape = (1, 2)
    noisy_then_flat = [1.0, 0.0, 1.0, 0.0] + [0.5] * 60

    def sums_at(n):
        v = np.array([[[0.5] * n, noisy_then_flat[:n]]], dtype=np.float32)
        return np.repeat(v.sum(axis=-1, dtype=np.float32)[..., None], 3, axis=-1), (v * v).sum(axis=-1, dtype=np.float32)

    part = np.ones(shape, dtype=bool)
    m0 = adaptive.spp_map(sums_at, part, 64, 4, 4, 0.2, 0.0)
    m1 = adaptive.spp_map(sums_at, part, 64, 4, 4, 0.2, 0.0, radius=1)
    assert m0[0, 0] == 4 and m0[0, 1] > 4
    assert m1[0, 0] == m1[0, 1] == m0[0, 1]


def test_ctypes_mirror_of_the_radius_matches_the_header(built):
    from simplepath_b200 import capi
    probe = r'''
    #include "spcu.h"
    #include <stddef.h>
    #include <stdio.h>
    int main(void){ printf("%zu %zu %zu %d\n", sizeof(spcu_adaptive), offsetof(spcu_adaptive, radius), sizeof(((spcu_adaptive*)0)->radius),
        SPCU_ABI_VERSION); return 0; }
    '''
    with tempfile.TemporaryDirectory() as d:
        src = f"{d}/p.c"
        open(src, "w").write(probe)
        subprocess.check_call(["gcc", "-I", str(ROOT / "include"), src, "-o", f"{d}/p"])
        got = [int(x) for x in subprocess.check_output([f"{d}/p"]).split()]
    A = capi.Adaptive
    assert got == [ctypes.sizeof(A), A.radius.offset, A.radius.size, capi.ABI_VERSION]
