"""Numpy model of the denoiser (spcu_render_guides / spcu_denoise / spcu_denoise_conserving, include/spcu.h): the guides'
albedo rule and the variance-guided à-trous filter, in its gather form and its energy-conserving flux form.

Everything is float32 with one rounding per operation, as the device computes it (csrc/denoise_kernels.cu), and taps are
added one after the other in the filter's order, so the model reproduces the device's output bit for bit from the same sums
and guides.
"""
from __future__ import annotations

import numpy as np

from .capi import DENOISE_DEFAULTS

F = np.float32
MATERIAL_DTYPE = np.dtype([("kind", "<u4"), ("n_bxdfs", "<u4"), ("first_bxdf", "<u4"), ("base", "<u4"), ("ior", "<f4"),
                           ("specular", "<f4", 3)])
BXDF_DTYPE = np.dtype([("kind", "<u4"), ("r", "<f4", 3), ("alpha_x", "<f4"), ("alpha_y", "<f4"), ("ior", "<f4"),
                       ("sample_visible", "<u4")])
MAT_CLEARCOAT, BXDF_LAMBERT, MAX_COAT_DEPTH = 1, 0, 4
PI = F(3.14159265358979323846)
B3 = (F(1 / 16), F(1 / 4), F(3 / 8), F(1 / 4), F(1 / 16))  # à-trous B-spline weights of offsets -2..2


def material_albedos(flat) -> np.ndarray:
    """Albedo [n_materials, 3] of every material of a FlatSceneData: a clearcoat's base followed to its one-sample material,
    then the sum over its BxDFs in table order of r * pi (Lambert, stored as albedo / pi) or r (microfacet, specular)."""
    mats = flat.arrays["materials"].view(MATERIAL_DTYPE).reshape(-1)
    bxdfs = flat.arrays["bxdfs"].view(BXDF_DTYPE).reshape(-1)
    out = np.zeros((mats.shape[0], 3), dtype=F)
    for i in range(mats.shape[0]):
        m = i
        for _ in range(MAX_COAT_DEPTH):
            if mats[m]["kind"] != MAT_CLEARCOAT:
                break
            m = int(mats[m]["base"])
        a = np.zeros(3, dtype=F)
        for k in range(int(mats[m]["n_bxdfs"])):
            b = bxdfs[int(mats[m]["first_bxdf"]) + k]
            a = a + b["r"].astype(F) * (PI if b["kind"] == BXDF_LAMBERT else F(1))
        out[i] = a
    return out


def _lum(r, g, b):
    return (F(0.2126) * r + F(0.7152) * g) + F(0.0722) * b


def _shift(a: np.ndarray, dx: int, dy: int, fill):
    """out[y, x] = a[y + dy, x + dx], `fill` outside the image."""
    h, w = a.shape[:2]
    out = np.full_like(a, fill)
    if abs(dx) >= w or abs(dy) >= h:
        return out
    ys, yd = slice(max(dy, 0), h + min(dy, 0)), slice(max(-dy, 0), h + min(-dy, 0))
    xs, xd = slice(max(dx, 0), w + min(dx, 0)), slice(max(-dx, 0), w + min(-dx, 0))
    out[yd, xd] = a[ys, xs]
    return out


def prepare(rgb_sum: np.ndarray, lum_sumsq: np.ndarray, spp) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(colour [H, W, 3] = sum / n, variance [H, W] of the mean luminance, tap [H, W] bool) before the first iteration.
    Empty pixels have colour 0, pixels with a non-finite sum colour sum / n; neither is a tap."""
    rgb_sum = np.asarray(rgb_sum, dtype=F)
    Q = np.asarray(lum_sumsq, dtype=F)
    n = np.broadcast_to(np.asarray(spp, dtype=np.uint32), Q.shape)
    nf = n.astype(F)
    R, G, B = rgb_sum[..., 0], rgb_sum[..., 1], rgb_sum[..., 2]
    with np.errstate(all="ignore"):
        col = rgb_sum / nf[..., None]
        L = _lum(R, G, B)
        m = L / nf
        d = Q / nf - m * m
        v = np.where(d > F(0), d * (nf / (nf - F(1))), F(0)).astype(F)
        var = np.where(n < 2, F(0), v / nf).astype(F)
    empty = n == 0
    col[empty] = F(0)
    tap = ~empty & np.isfinite(R) & np.isfinite(G) & np.isfinite(B) & np.isfinite(Q)
    return col.astype(F), var, tap


def prefilter(var: np.ndarray, tap: np.ndarray) -> np.ndarray:
    """var~ [H, W]: the 3x3 weighted mean (1/4, 1/8, 1/16) of var over the neighbours that are taps, summed row-major."""
    pv = np.zeros_like(var)
    pw = np.zeros_like(var)
    with np.errstate(all="ignore"):
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                ok = _shift(tap, dx, dy, False)
                w = F(0.5 if dx == 0 else 0.25) * F(0.5 if dy == 0 else 0.25)
                pv = np.where(ok, pv + w * _shift(var, dx, dy, F(0)), pv)
                pw = np.where(ok, pw + w, pw)
        return pv / pw


def _guide_fields(guides):
    """(normal, depth, albedo, class) of the guides; class 0 geometry hit, 1 light hit, 2 miss."""
    gid = np.asarray(guides["id"])
    return (np.asarray(guides["normal"], dtype=F), np.asarray(guides["depth"], dtype=F), np.asarray(guides["albedo"], dtype=F),
            np.where(gid >= 0, 0, np.where(gid == -1, 2, 1)))


def denoise(guides: np.ndarray, rgb_sum: np.ndarray, lum_sumsq: np.ndarray, spp, iterations: int = DENOISE_DEFAULTS["iterations"],
            sigma_l: float = DENOISE_DEFAULTS["sigma_l"], sigma_z: float = DENOISE_DEFAULTS["sigma_z"],
            sigma_a: float = DENOISE_DEFAULTS["sigma_a"], conserve_energy: bool = False) -> np.ndarray:
    """The filter of spcu_denoise: denoised mean colour [H, W, 3] from the guides [H, W] (capi.GUIDE_DTYPE) and a frame's sums;
    spp = the samples of every pixel (int) or the per-pixel counts [H, W].  conserve_energy: the flux form of
    spcu_denoise_conserving (conserving_iteration)."""
    if conserve_energy:
        col, var, tap = prepare(rgb_sum, lum_sumsq, spp)
        for it in range(iterations):
            col, var = conserving_iteration(guides, col, var, tap, 1 << it, sigma_l, sigma_z, sigma_a)
        return col
    sigma_l, sigma_z, sigma_a = F(sigma_l), F(sigma_z), F(sigma_a)
    col, var, tap = prepare(rgb_sum, lum_sumsq, spp)
    lum = _lum(col[..., 0], col[..., 1], col[..., 2])
    nrm, depth, alb, cls = _guide_fields(guides)
    geo = cls == 0
    with np.errstate(all="ignore"):
        for it in range(iterations):
            h = 1 << it
            l_den = sigma_l * np.sqrt(prefilter(var, tap)) + F(1e-4)
            S = np.zeros_like(col)
            Sw = np.zeros_like(var)
            Sv = np.zeros_like(var)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    ok = _shift(tap, dx * h, dy * h, False)
                    cq = _shift(col, dx * h, dy * h, F(0))
                    vq = _shift(var, dx * h, dy * h, F(0))
                    k = B3[dx + 2] * B3[dy + 2]
                    if dx == 0 and dy == 0:
                        w = np.full_like(var, k)
                    else:
                        lq = _shift(lum, dx * h, dy * h, F(0))
                        same = _shift(cls, dx * h, dy * h, -1) == cls
                        nq = _shift(nrm, dx * h, dy * h, F(0))
                        dn = (nrm[..., 0] * nq[..., 0] + nrm[..., 1] * nq[..., 1]) + nrm[..., 2] * nq[..., 2]
                        wn = np.maximum(F(0), dn)
                        for _ in range(7):
                            wn = wn * wn
                        zq = _shift(depth, dx * h, dy * h, F(0))
                        az = np.abs(depth - zq) / ((sigma_z * depth) * F(h * max(abs(dx), abs(dy))))
                        aq = _shift(alb, dx * h, dy * h, F(0))
                        da = np.maximum(np.maximum(np.abs(alb[..., 0] - aq[..., 0]), np.abs(alb[..., 1] - aq[..., 1])),
                                        np.abs(alb[..., 2] - aq[..., 2]))
                        aa = da / sigma_a
                        wn, az, aa = (np.where(geo, x, d).astype(F) for x, d in ((wn, F(1)), (az, F(0)), (aa, F(0))))
                        al = np.abs(lum - lq) / l_den
                        w = np.where(same, (k * wn) / (((F(1) + al * al) + az * az) + aa * aa), F(0)).astype(F)
                    S = np.where(ok[..., None], S + w[..., None] * cq, S)
                    Sw = np.where(ok, Sw + w, Sw)
                    Sv = np.where(ok, Sv + (w * w) * vq, Sv)
            new_col = S / Sw[..., None]
            col = np.where(tap[..., None], new_col, col).astype(F)
            var = np.where(tap, Sv / (Sw * Sw), var).astype(F)
            lum = np.where(tap, _lum(col[..., 0], col[..., 1], col[..., 2]), lum).astype(F)
    return col


# ---- the flux form (spcu_denoise_conserving) -----------------------------------------------------------------------------------
def pair_weights(guides, lum, var_pf, tap, h: int, dx: int, dy: int, sigma_l, sigma_z, sigma_a) -> np.ndarray:
    """w_pq [H, W] of every pixel p and its tap q = p + h (dx, dy), (dx, dy) != (0, 0): 0 where the classes differ, else the
    symmetric weight of spcu_denoise_conserving.  Only meaningful where p and q are taps; 0 where q is outside the image."""
    sigma_l, sigma_z, sigma_a = F(sigma_l), F(sigma_z), F(sigma_a)
    nrm, depth, alb, cls = _guide_fields(guides)
    ox, oy = dx * h, dy * h
    k = B3[dx + 2] * B3[dy + 2]
    with np.errstate(all="ignore"):
        nq = _shift(nrm, ox, oy, F(0))
        dn = (nrm[..., 0] * nq[..., 0] + nrm[..., 1] * nq[..., 1]) + nrm[..., 2] * nq[..., 2]
        wn = np.maximum(F(0), dn)
        for _ in range(7):
            wn = wn * wn
        zq = _shift(depth, ox, oy, F(0))
        az = np.abs(depth - zq) / ((sigma_z * np.minimum(depth, zq)) * F(h * max(abs(dx), abs(dy))))
        aq = _shift(alb, ox, oy, F(0))
        da = np.maximum(np.maximum(np.abs(alb[..., 0] - aq[..., 0]), np.abs(alb[..., 1] - aq[..., 1])), np.abs(alb[..., 2] - aq[..., 2]))
        aa = da / sigma_a
        geo = cls == 0
        wn, az, aa = (np.where(geo, x, d).astype(F) for x, d in ((wn, F(1)), (az, F(0)), (aa, F(0))))
        l_den = sigma_l * np.sqrt(np.maximum(var_pf, _shift(var_pf, ox, oy, F(0)))) + F(1e-4)
        al = np.abs(lum - _shift(lum, ox, oy, F(0))) / l_den
        w = (k * wn) / (((F(1) + al * al) + az * az) + aa * aa)
        same = _shift(cls, ox, oy, -1) == cls
        return np.where(same & _shift(tap, ox, oy, False), w, F(0)).astype(F)


OFFSETS = [(dx, dy) for dy in range(-2, 3) for dx in range(-2, 3)]  # row-major


def flux_terms(guides, col, var, tap, h: int, sigma_l, sigma_z, sigma_a):
    """The pairs of one iteration of the flux form at step h, in row-major tap order: yields (dx, dy, ok, alpha, flux) for
    every offset but the centre, where ok [H, W] = q = p + h (dx, dy) is a tap, alpha [H, W] = alpha_pq and flux [H, W, 3] =
    f_pq = alpha_pq (c_q - c_p).  Only meaningful where p is a tap."""
    lum = _lum(col[..., 0], col[..., 1], col[..., 2])
    var_pf = prefilter(var, tap)
    ws = {o: pair_weights(guides, lum, var_pf, tap, h, *o, sigma_l, sigma_z, sigma_a) for o in OFFSETS if o != (0, 0)}
    W = np.zeros_like(var)
    with np.errstate(all="ignore"):
        for o in OFFSETS:
            ok = _shift(tap, o[0] * h, o[1] * h, False)
            W = np.where(ok, W + (B3[2] * B3[2] if o == (0, 0) else ws[o]), W).astype(F)
        for (dx, dy), w in ws.items():
            ok = _shift(tap, dx * h, dy * h, False)
            alpha = (w / np.maximum(W, _shift(W, dx * h, dy * h, F(0)))).astype(F)
            yield dx, dy, ok, alpha, (alpha[..., None] * (_shift(col, dx * h, dy * h, F(0)) - col)).astype(F)


def conserving_iteration(guides, col, var, tap, h: int, sigma_l, sigma_z, sigma_a):
    """One iteration of spcu_denoise_conserving at step h: (col', var') from (col [H, W, 3], var [H, W]); pixels that are no
    taps pass through."""
    S = np.zeros_like(col)
    A = np.zeros_like(var)
    Sv = np.zeros_like(var)
    with np.errstate(all="ignore"):
        for dx, dy, ok, alpha, flux in flux_terms(guides, col, var, tap, h, sigma_l, sigma_z, sigma_a):
            S = np.where(ok[..., None], S + flux, S)
            A = np.where(ok, A + alpha, A)
            Sv = np.where(ok, Sv + (alpha * alpha) * _shift(var, dx * h, dy * h, F(0)), Sv)
        a0 = F(1) - A
        new_col = np.where(tap[..., None], col + S, col).astype(F)
        new_var = np.where(tap, (a0 * a0) * var + Sv, var).astype(F)
    return new_col, new_var
