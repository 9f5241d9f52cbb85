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


def _test_terms(rgb_sum, lum_sumsq, n: int, rel_error: float, abs_floor: float):
    """The stopping test's terms after n samples: (v, T^2, all four sums finite), v the unbiased luminance variance and
    T = rel_error * (mean + abs_floor)."""
    rgb_sum = np.asarray(rgb_sum, dtype=F)
    Q = np.asarray(lum_sumsq, dtype=F)
    R, G, B = rgb_sum[..., 0], rgb_sum[..., 1], rgb_sum[..., 2]
    nf = F(n)
    with np.errstate(all="ignore"):
        L = (F(0.2126) * R + F(0.7152) * G) + F(0.0722) * B
        m = L / nf
        d = Q / nf - m * m
        v = np.where(d > F(0), d * (nf / (nf - F(1))), F(0)).astype(F)
        t = F(rel_error) * (m + F(abs_floor))
        tt = t * t
    return v, tt, np.isfinite(R) & np.isfinite(G) & np.isfinite(B) & np.isfinite(Q)


def converged(rgb_sum: np.ndarray, lum_sumsq: np.ndarray, n: int, rel_error: float, abs_floor: float) -> np.ndarray:
    """Pixels whose sums after n samples pass the stopping test: squared standard error of the mean luminance <=
    (rel_error * (mean + abs_floor))^2, and all four sums finite."""
    v, tt, finite = _test_terms(rgb_sum, lum_sumsq, n, rel_error, abs_floor)
    with np.errstate(all="ignore"):
        ok = v / F(n) <= tt
    return ok & finite


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


# ---- predicted sample counts (spcu_render_adaptive_predicted) ----------------------------------------------------------------
def grid(budget: int, min_spp: int) -> list[int]:
    """The counts a pixel can hold: g_0 = min(min_spp, budget), g_{i+1} = min(2 g_i, budget), up to the budget."""
    g = [min(min_spp, budget)]
    while g[-1] < budget:
        g.append(min(2 * g[-1], budget))
    return g


def need(rgb_sum, lum_sumsq, n: int, rel_error: float, abs_floor: float) -> np.ndarray:
    """The sample count at which the stopping test would pass, predicted from the sums after n samples: v / T^2 with the
    test's own v and T (float32, one rounding per operation); +inf where T^2 is 0 or not finite, the quotient is not finite
    or a sum is not finite."""
    v, tt, finite = _test_terms(rgb_sum, lum_sumsq, n, rel_error, abs_floor)
    with np.errstate(all="ignore"):
        q = (v / tt).astype(F)
    ok = finite & (tt > F(0)) & np.isfinite(tt) & np.isfinite(q)
    return np.where(ok, q, F(np.inf)).astype(F)


def target_level(need_: np.ndarray, j: np.ndarray, g: list[int], max_step: int) -> np.ndarray:
    """t = the smallest grid index i in (j, min(j + max_step, last)] with float32(g_i) >= need, else that upper end."""
    last = len(g) - 1
    gf = np.array(g, dtype=F)
    upper = np.minimum(j + max_step, last)
    t = upper.copy()
    for s in range(max_step, 0, -1):  # the smallest index that qualifies is written last
        i = j + s
        ok = (i <= upper) & (gf[np.minimum(i, last)] >= need_)
        t = np.where(ok, i, t)
    return t


def predicted_spp_map(sums_at, partition: np.ndarray, budget: int, min_spp: int, max_step: int, rel_error: float,
                      abs_floor: float, radius: int = 0) -> np.ndarray:
    """The per-pixel sample counts n_p of the predicted schedule.  sums_at(n) -> (rgb_sum [H,W,3], lum_sumsq [H,W]) of a fixed
    render of samples [0, n) for any n of grid(budget, min_spp); partition: bool [H,W] (the other pixels get 0).  Every round
    tests each active pixel below the budget with n = its count g_j, then decides as spp_map does (a stopped pixel, one at the
    budget or one outside the partition counts as passing).  A pixel that does not stop moves to grid index j + 1 when it
    passed its own test, else to target_level(need); one that reaches the budget stops there."""
    g = grid(budget, min_spp)
    last = len(g) - 1
    out = np.zeros(partition.shape, dtype=np.uint32)
    level = np.zeros(partition.shape, dtype=np.int64)
    active = partition.copy()
    passed = np.ones(partition.shape, dtype=bool)
    need_ = np.full(partition.shape, np.inf, dtype=F)
    while active.any():
        end = active & (level == last)
        out[end] = budget
        passed[end] = True
        active &= ~end
        if not active.any():
            break
        for j in np.unique(level[active]):
            sel = active & (level == j)
            rgb, sq = sums_at(g[j])
            passed = np.where(sel, converged(rgb, sq, g[j], rel_error, abs_floor), passed)
            need_ = np.where(sel, need(rgb, sq, g[j], rel_error, abs_floor), need_)
        done = active & window_all(passed, radius)
        out[done] = np.array(g, dtype=np.uint32)[level[done]]
        active &= ~done
        t = np.where(passed, level + 1, target_level(need_, level, g, max_step))
        level = np.where(active, t, level)
    return out
