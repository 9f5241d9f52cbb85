"""Numpy model of adaptive sampling (spcu_render_adaptive, include/spcu.h): the pass schedule, the per-pixel stopping test and
the neighbourhood rule over it.

The test is float32 with one rounding per operation, as the device computes it (csrc/adaptive_kernels.cu), so the model
reproduces every decision bit for bit from the same sums.
"""
from __future__ import annotations

import numpy as np

F = np.float32


def boundaries(budget: int, min_spp: int, pass_spp: int) -> list[int]:
    """Sample counts at which the passes end: s_0 = min(min_spp, budget), s_{k+1} = min(s_k + pass_spp, budget)."""
    s = [min(min_spp, budget)]
    while s[-1] < budget:
        s.append(min(s[-1] + pass_spp, budget))
    return s


def converged(rgb_sum: np.ndarray, lum_sumsq: np.ndarray, n: int, rel_error: float, abs_floor: float) -> np.ndarray:
    """Pixels whose sums after n samples pass the stopping test: squared standard error of the mean luminance <=
    (rel_error * (mean + abs_floor))^2, and all four sums finite."""
    rgb_sum = np.asarray(rgb_sum, dtype=F)
    Q = np.asarray(lum_sumsq, dtype=F)
    R, G, B = rgb_sum[..., 0], rgb_sum[..., 1], rgb_sum[..., 2]
    nf = F(n)
    with np.errstate(all="ignore"):
        L = (F(0.2126) * R + F(0.7152) * G) + F(0.0722) * B
        m = L / nf
        d = Q / nf - m * m
        v = np.where(d > F(0), d * (nf / (nf - F(1))), F(0)).astype(F)
        se2 = v / nf
        t = F(rel_error) * (m + F(abs_floor))
        ok = se2 <= t * t
    return ok & np.isfinite(R) & np.isfinite(G) & np.isfinite(B) & np.isfinite(Q)


def window_all(passed: np.ndarray, radius: int) -> np.ndarray:
    """For every pixel p of a bool [H, W] map: whether `passed` holds on all of its window W(p) = {q : |x_q - x_p| <= radius,
    |y_q - y_p| <= radius, q in the same 8x8 tile as p (tiles_x = ceil(W / 8), tile of (x, y) = (x >> 3, y >> 3)), q inside
    the image}.  A rectangle's AND is taken along x, then along y; positions outside the image count as passing."""
    h, w = passed.shape
    th, tw = -(-h // 8), -(-w // 8)
    a = np.ones((th * 8, tw * 8), dtype=bool)
    a[:h, :w] = passed
    a = a.reshape(th, 8, tw, 8)  # [tile y, y & 7, tile x, x & 7]
    for axis in (3, 1):
        out = a.copy()
        for d in range(1, min(radius, 7) + 1):
            lo = [slice(None)] * 4
            hi = [slice(None)] * 4
            lo[axis], hi[axis] = slice(0, 8 - d), slice(d, 8)
            out[tuple(lo)] &= a[tuple(hi)]  # neighbour at +d inside the tile
            out[tuple(hi)] &= a[tuple(lo)]  # neighbour at -d
        a = out
    return a.reshape(th * 8, tw * 8)[:h, :w]


def spp_map(sums_at, partition: np.ndarray, budget: int, min_spp: int, pass_spp: int, rel_error: float,
            abs_floor: float, radius: int = 0) -> np.ndarray:
    """The per-pixel sample counts n_p the schedule gives.  sums_at(n) -> (rgb_sum [H,W,3], lum_sumsq [H,W]) of a fixed render
    of samples [0, n); partition: bool [H,W], the pixels the call renders (the others get 0).  At each boundary every active
    pixel is tested first; then an active pixel stops iff every pixel of its window (window_all) passes, a pixel that
    stopped earlier or lies outside the partition counting as passing."""
    out = np.zeros(partition.shape, dtype=np.uint32)
    active = partition.copy()
    passed = np.ones(partition.shape, dtype=bool)
    for s in boundaries(budget, min_spp, pass_spp):
        if s >= budget or not active.any():
            break
        rgb, sq = sums_at(s)
        passed = np.where(active, converged(rgb, sq, s, rel_error, abs_floor), passed)
        done = active & window_all(passed, radius)
        out[done] = s
        active &= ~done
    out[active] = budget
    return out
