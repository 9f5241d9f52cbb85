"""Adaptive sampling without a GPU: the numpy model's schedule and stopping test (simplepath_b200/adaptive.py), and the
ctypes mirror of spcu_adaptive against the C header."""
import ctypes
import subprocess
import tempfile

import numpy as np

from conftest import ROOT
from simplepath_b200 import adaptive


def test_schedule_boundaries():
    assert adaptive.boundaries(64, 4, 4) == list(range(4, 65, 4))
    assert adaptive.boundaries(64, 16, 20) == [16, 36, 56, 64]  # the last pass is cut at the budget
    assert adaptive.boundaries(8, 16, 4) == [8]                 # min_spp >= budget: one pass of the whole budget
    assert adaptive.boundaries(16, 16, 4) == [16]
    assert adaptive.boundaries(5, 2, 1) == [2, 3, 4, 5]


def _sums(values):
    """rgb_sum / lum_sumsq of per-pixel samples (grey radiance, so luminance = value)."""
    v = np.asarray(values, dtype=np.float32)
    rgb = np.repeat(v.sum(axis=-1, dtype=np.float32)[..., None], 3, axis=-1)
    return rgb, (v * v).sum(axis=-1, dtype=np.float32)


def test_zero_variance_stops_even_at_zero_error():
    rgb, sq = _sums([[1.0, 1.0, 1.0, 1.0], [0.0, 0.0, 0.0, 0.0], [1.0, 0.0, 1.0, 0.0]])
    assert adaptive.converged(rgb, sq, 4, 0.0, 0.0).tolist() == [True, True, False]
    assert adaptive.converged(rgb, sq, 4, 10.0, 0.0).tolist() == [True, True, True]


def test_abs_floor_lets_dark_pixels_stop():
    rgb, sq = _sums([[0.0, 0.0, 0.0, 1e-3]])
    assert not adaptive.converged(rgb, sq, 4, 0.1, 0.0)[0]
    assert adaptive.converged(rgb, sq, 4, 0.1, 0.1)[0]


def test_non_finite_sums_never_stop():
    rgb = np.ones((5, 3), dtype=np.float32)
    sq = np.ones(5, dtype=np.float32)
    rgb[0, 0], rgb[1, 1], rgb[2, 2], sq[3] = np.inf, np.nan, -np.inf, np.nan
    got = adaptive.converged(rgb, sq, 4, 1e30, 1e30)
    assert got.tolist() == [False, False, False, False, True]


def test_model_map_follows_the_schedule():
    """A pixel stops at the first boundary where its sums pass; pixels outside the partition get 0, the rest the budget."""
    rng = np.random.default_rng(0)
    samples = rng.random((4, 6, 32), dtype=np.float32)
    samples[0, :] = 0.5          # row 0: zero variance, stops at min_spp
    samples[1, :] *= 1e3         # row 1: noisy, runs to the budget
    part = np.ones((4, 6), dtype=bool)
    part[3] = False

    def sums_at(n):
        return _sums(samples[..., :n])

    m = adaptive.spp_map(sums_at, part, 32, 4, 8, 0.05, 0.0)
    assert (m[0] == 4).all() and (m[3] == 0).all()
    assert set(np.unique(m[:3])) <= {4, 12, 20, 28, 32}
    for y, x in zip(*np.nonzero(part)):
        n = int(m[y, x])
        for b in adaptive.boundaries(32, 4, 8):
            if b >= n:
                break
            rgb, sq = sums_at(b)
            assert not adaptive.converged(rgb[y, x], sq[y, x], b, 0.05, 0.0)  # did not stop earlier
        if n < 32:
            rgb, sq = sums_at(n)
            assert adaptive.converged(rgb[y, x], sq[y, x], n, 0.05, 0.0)


def test_ctypes_mirror_of_spcu_adaptive_matches_the_header(built):
    from simplepath_b200 import capi
    probe = r'''
    #include "spcu.h"
    #include <stddef.h>
    #include <stdio.h>
    int main(void){ printf("%zu %zu %zu %zu %zu\n", sizeof(spcu_adaptive), offsetof(spcu_adaptive, min_spp),
        offsetof(spcu_adaptive, pass_spp), offsetof(spcu_adaptive, rel_error), offsetof(spcu_adaptive, abs_floor)); return 0; }
    '''
    with tempfile.TemporaryDirectory() as d:
        src = f"{d}/p.c"
        open(src, "w").write(probe)
        subprocess.check_call(["gcc", "-I", str(ROOT / "include"), src, "-o", f"{d}/p"])
        got = [int(x) for x in subprocess.check_output([f"{d}/p"]).split()]
    A = capi.Adaptive
    assert got == [ctypes.sizeof(A), A.min_spp.offset, A.pass_spp.offset, A.rel_error.offset, A.abs_floor.offset]
