"""Numpy model of adaptive sampling (spcu_render_adaptive, include/spcu.h): the pass schedule and the per-pixel stopping test.

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


def spp_map(sums_at, partition: np.ndarray, budget: int, min_spp: int, pass_spp: int, rel_error: float,
            abs_floor: float) -> np.ndarray:
    """The per-pixel sample counts n_p the schedule gives.  sums_at(n) -> (rgb_sum [H,W,3], lum_sumsq [H,W]) of a fixed render
    of samples [0, n); partition: bool [H,W], the pixels the call renders (the others get 0)."""
    out = np.zeros(partition.shape, dtype=np.uint32)
    active = partition.copy()
    for s in boundaries(budget, min_spp, pass_spp):
        if s >= budget or not active.any():
            break
        rgb, sq = sums_at(s)
        done = active & converged(rgb, sq, s, rel_error, abs_floor)
        out[done] = s
        active &= ~done
    out[active] = budget
    return out
