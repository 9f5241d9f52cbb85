"""The numpy model of the energy-conserving (flux) form of the denoiser (spcu_denoise_conserving, simplepath_b200/denoise.py):
the consequences its contract in include/spcu.h claims, checked on small random images with mixed classes, empty pixels
and non-finite pixels.  Runs without a GPU; tests/test_gpu_denoise_conserving.py holds the device to this model bit for bit."""
import ctypes as C
import hashlib
import re

import numpy as np
import pytest

from conftest import ROOT
from simplepath_b200 import capi, denoise

F = np.float32
OTHER = dict(sigma_l=2.0, sigma_z=0.05, sigma_a=0.3)
DEFAULTS = {k: capi.DENOISE_DEFAULTS[k] for k in ("sigma_l", "sigma_z", "sigma_a")}


def image(seed, h=19, w=21, spp=6):
    """(guides, rgb_sum, lum_sumsq, counts): gamma-distributed samples with a few 200x fireflies, random normals, depths and
    albedos, about 10 % misses and 10 % light hits, empty pixels, one-sample pixels, one infinite and one NaN sum."""
    rng = np.random.default_rng(seed)
    samples = rng.gamma(2.0, 0.25, size=(spp, h, w, 3)).astype(F)
    samples[rng.random((spp, h, w)) < 0.02] *= F(200)
    rgb = samples.sum(axis=0, dtype=F)
    lum = (F(0.2126) * samples[..., 0] + F(0.7152) * samples[..., 1]) + F(0.0722) * samples[..., 2]
    sq = (lum * lum).sum(axis=0, dtype=F)
    counts = np.full((h, w), spp, dtype=np.uint32)
    counts[rng.random((h, w)) < 0.05] = 0
    counts[rng.random((h, w)) < 0.05] = 1
    rgb[2, 3, 0] = np.inf
    sq[7, 9] = np.nan
    g = np.zeros((h, w), dtype=capi.GUIDE_DTYPE)
    n = rng.normal(size=(h, w, 3)).astype(F)
    n[..., 2] = -np.abs(n[..., 2]) - F(2)
    g["normal"] = (n / np.sqrt((n * n).sum(-1, keepdims=True))).astype(F)
    g["depth"] = rng.uniform(4.0, 6.0, size=(h, w)).astype(F)
    g["albedo"] = rng.uniform(0.2, 0.8, size=(h, w, 3)).astype(F)
    g["id"] = rng.integers(0, 100, size=(h, w))
    g["id"][rng.random((h, w)) < 0.1] = -1
    g["id"][rng.random((h, w)) < 0.1] = -3
    return g, rgb, sq, counts


def iterations_of(g, rgb, sq, counts, iterations, **kw):
    """[(col, var)] before each iteration and after the last, from the model's own steps."""
    col, var, tap = denoise.prepare(rgb, sq, counts)
    out = [(col, var)]
    for i in range(iterations):
        col, var = denoise.conserving_iteration(g, col, var, tap, 1 << i, **{**DEFAULTS, **kw})
        out.append((col, var))
    return out, tap


def in_image(shape, ox, oy):
    """[H, W] bool: p + (ox, oy) lies in the image."""
    h, w = shape
    ys, xs = np.mgrid[0:h, 0:w]
    return (xs + ox >= 0) & (xs + ox < w) & (ys + oy >= 0) & (ys + oy < h)


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("kw", [{}, OTHER], ids=["defaults", "other_sigmas"])
def test_pairs_are_symmetric_bit_for_bit(seed, kw):
    """w_pq from p's end and w_qp from q's end have the same bits; alpha_pq = alpha_qp and f_pq = -f_qp exactly."""
    g, rgb, sq, counts = image(seed)
    states, tap = iterations_of(g, rgb, sq, counts, 3, **kw)
    sig = {**DEFAULTS, **kw}
    checked = 0
    for i, (col, var) in enumerate(states[:-1]):
        h = 1 << i
        lum = (F(0.2126) * col[..., 0] + F(0.7152) * col[..., 1]) + F(0.0722) * col[..., 2]
        pf = denoise.prefilter(var, tap)
        terms = {(dx, dy): (ok, a, f) for dx, dy, ok, a, f in denoise.flux_terms(g, col, var, tap, h, **sig)}
        for (dx, dy), (ok, a, f) in terms.items():
            ox, oy = dx * h, dy * h
            both = tap & ok
            ys, xs = np.nonzero(both)
            if not len(ys):
                continue
            w_pq = denoise.pair_weights(g, lum, pf, tap, h, dx, dy, **sig)[ys, xs]
            w_qp = denoise.pair_weights(g, lum, pf, tap, h, -dx, -dy, **sig)[ys + oy, xs + ox]
            assert w_pq.tobytes() == w_qp.tobytes(), (i, dx, dy)
            ok_b, a_b, f_b = terms[(-dx, -dy)]
            assert ok_b[ys + oy, xs + ox].all()
            assert a[ys, xs].tobytes() == a_b[ys + oy, xs + ox].tobytes()
            assert f[ys, xs].tobytes() == (-f_b[ys + oy, xs + ox]).tobytes()
            checked += len(ys)
            # a pair of different classes exchanges nothing
            cls = np.where(g["id"] >= 0, 0, np.where(g["id"] == -1, 2, 1))
            differ = cls[ys, xs] != cls[ys + oy, xs + ox]
            assert (w_pq[differ] == 0).all() and (a[ys, xs][differ] == 0).all()
    assert checked > 1000


@pytest.mark.parametrize("iterations", [1, 5, 8])
def test_channel_sums_are_conserved(iterations):
    """Summed in float64, the pairs' float32 fluxes cancel: every channel's total over the image is kept to float64 rounding.
    The float32 outputs round once per tap in each pixel's sum; they keep the total within that accumulation's bound."""
    g, rgb, sq, counts = image(3)
    states, tap = iterations_of(g, rgb, sq, counts, iterations)
    eps = float(np.finfo(F).eps) / 2
    for i, ((col, var), (new_col, _)) in enumerate(zip(states[:-1], states[1:])):
        exact = col.astype(np.float64)
        mag = np.abs(col.astype(np.float64))
        for dx, dy, ok, a, f in denoise.flux_terms(g, col, var, tap, 1 << i, **DEFAULTS):
            use = (tap & ok)[..., None]
            exact += np.where(use, f.astype(np.float64), 0)
            mag += np.where(use, np.abs(f.astype(np.float64)), 0)
        exact = np.where(tap[..., None], exact, col.astype(np.float64))
        mag = np.where(tap[..., None], mag, 0)
        before = col[tap].astype(np.float64).sum(axis=0)
        assert np.allclose(exact[tap].sum(axis=0), before, rtol=1e-12, atol=0), i
        drift = np.abs(new_col[tap].astype(np.float64).sum(axis=0) - before)
        bound = 26 * eps * mag[tap].sum(axis=0)
        assert (drift <= bound).all(), (i, drift, bound)
    # the whole filter: the output's channel sums equal the input means' within 1e-5
    col0, _, tap0 = denoise.prepare(rgb, sq, counts)
    out = denoise.denoise(g, rgb, sq, counts, iterations=iterations, conserve_energy=True)
    s0, s1 = col0[tap0].astype(np.float64).sum(axis=0), out[tap0].astype(np.float64).sum(axis=0)
    assert (np.abs(s1 - s0) <= 1e-5 * s0).all()


@pytest.mark.parametrize("iterations", [1, 5, 8])
def test_constant_image_comes_back_bit_for_bit(iterations):
    """Every difference is 0, so every flux is 0, whatever the variances, guides and empty pixels."""
    g, _, _, counts = image(4)
    counts[counts == 1] = 16
    counts[counts == 6] = 16
    c = np.array([0.3, 0.6, 0.9], dtype=F)
    rgb = np.where((counts > 0)[..., None], c * F(16), F(0)).astype(F)
    sq = np.random.default_rng(4).uniform(0.0, 50.0, size=counts.shape).astype(F)
    for kw in ({}, OTHER):
        out = denoise.denoise(g, rgb, sq, counts, iterations=iterations, conserve_energy=True, **kw)
        want = np.where((counts > 0)[..., None], c, F(0)).astype(F)
        assert out.tobytes() == want.tobytes()


def test_outputs_lie_within_their_taps():
    """sum_q alpha_pq <= 1 - (9/64) / W_p: each output is a convex combination of the pixel and its taps, so it lies within their
    range (up to the rounding of the pixel's sum) and non-negative input stays non-negative."""
    g, rgb, sq, counts = image(5)
    states, tap = iterations_of(g, rgb, sq, counts, 4)
    h_, w_ = tap.shape
    tol = 32 * float(np.finfo(F).eps)
    for i, ((col, var), (new_col, _)) in enumerate(zip(states[:-1], states[1:])):
        h = 1 << i
        lo, hi = col.copy(), col.copy()
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                ok = denoise._shift(tap, dx * h, dy * h, False)[..., None]
                cq = denoise._shift(col, dx * h, dy * h, F(0))
                lo = np.where(ok, np.minimum(lo, cq), lo)
                hi = np.where(ok, np.maximum(hi, cq), hi)
        scale = np.maximum(np.abs(lo), np.abs(hi)).astype(np.float64) * tol
        assert (new_col[tap] >= lo[tap] - scale[tap]).all(), i
        assert (new_col[tap] <= hi[tap] + scale[tap]).all(), i
        assert (new_col[tap] >= 0).all()
        A = np.zeros_like(var)
        for dx, dy, ok, a, f in denoise.flux_terms(g, col, var, tap, h, **DEFAULTS):
            A = np.where(ok, A + a, A)
        assert (A[tap] < 1).all()


def test_non_taps_pass_through_and_exchange_nothing():
    g, rgb, sq, counts = image(6)
    col0, _, tap = denoise.prepare(rgb, sq, counts)
    assert (~tap).sum() > 10
    out = denoise.denoise(g, rgb, sq, counts, iterations=4, conserve_energy=True)
    assert out[~tap].tobytes() == col0[~tap].tobytes()
    assert (out[counts == 0] == 0).all()
    # what the non-taps hold reaches nobody: other sums there leave every tap's output as it was
    rgb2, sq2 = rgb.copy(), sq.copy()
    rgb2[counts == 0] = F(1e6)
    sq2[counts == 0] = F(1e9)
    rgb2[2, 3] = (np.inf, 5.0, np.nan)
    rgb2[7, 9] = F(1e6)
    sq2[7, 9] = -np.inf
    assert denoise.prepare(rgb2, sq2, counts)[2].tobytes() == tap.tobytes()
    out2 = denoise.denoise(g, rgb2, sq2, counts, iterations=4, conserve_energy=True)
    assert out2[tap].tobytes() == out[tap].tobytes()


def reference_iteration(g, col, var, tap, h, sigma_l, sigma_z, sigma_a):
    """One iteration of the flux form written per pixel and per pair, straight from the contract (include/spcu.h)."""
    H, W = tap.shape
    lum = lambda c: (F(0.2126) * c[0] + F(0.7152) * c[1]) + F(0.0722) * c[2]  # noqa: E731
    b = (F(1 / 16), F(1 / 4), F(3 / 8), F(1 / 4), F(1 / 16))
    cls = lambda i: 0 if i >= 0 else (2 if i == -1 else 1)  # noqa: E731
    sigma_l, sigma_z, sigma_a = F(sigma_l), F(sigma_z), F(sigma_a)
    pf = np.zeros((H, W), dtype=F)
    for y in range(H):
        for x in range(W):
            pv = pw = F(0)
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    qx, qy = x + dx, y + dy
                    if 0 <= qx < W and 0 <= qy < H and tap[qy, qx]:
                        wt = F(0.5 if dx == 0 else 0.25) * F(0.5 if dy == 0 else 0.25)
                        pv, pw = pv + wt * var[qy, qx], pw + wt
            pf[y, x] = pv / pw if tap[y, x] else F(0)

    def taps(x, y):
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                qx, qy = x + dx * h, y + dy * h
                if 0 <= qx < W and 0 <= qy < H and tap[qy, qx]:
                    yield dx, dy, qx, qy

    def weight(x, y, qx, qy, dx, dy):
        p, q = g[y, x], g[qy, qx]
        if cls(p["id"]) != cls(q["id"]):
            return F(0)
        wn, az, aa = F(1), F(0), F(0)
        if p["id"] >= 0:
            n, m = p["normal"], q["normal"]
            wn = max(F(0), (n[0] * m[0] + n[1] * m[1]) + n[2] * m[2])
            for _ in range(7):
                wn = wn * wn
            az = np.abs(p["depth"] - q["depth"]) / ((sigma_z * min(p["depth"], q["depth"])) * F(h * max(abs(dx), abs(dy))))
            aa = np.abs(p["albedo"] - q["albedo"]).max() / sigma_a
        al = np.abs(lum(col[y, x]) - lum(col[qy, qx])) / (sigma_l * np.sqrt(max(pf[y, x], pf[qy, qx])) + F(1e-4))
        return (b[dx + 2] * b[dy + 2] * wn) / (((F(1) + al * al) + az * az) + aa * aa)

    Wsum = np.zeros((H, W), dtype=F)
    for y in range(H):
        for x in range(W):
            if tap[y, x]:
                s = F(0)
                for dx, dy, qx, qy in taps(x, y):
                    s = s + (F(9 / 64) if dx == 0 and dy == 0 else weight(x, y, qx, qy, dx, dy))
                Wsum[y, x] = s
    out_c, out_v = col.copy(), var.copy()
    for y in range(H):
        for x in range(W):
            if not tap[y, x]:
                continue
            S, A, Sv = np.zeros(3, dtype=F), F(0), F(0)
            for dx, dy, qx, qy in taps(x, y):
                if dx == 0 and dy == 0:
                    continue
                a = weight(x, y, qx, qy, dx, dy) / max(Wsum[y, x], Wsum[qy, qx])
                S = S + a * (col[qy, qx] - col[y, x])
                A = A + a
                Sv = Sv + (a * a) * var[qy, qx]
            out_c[y, x] = col[y, x] + S
            a0 = F(1) - A
            out_v[y, x] = (a0 * a0) * var[y, x] + Sv
    return out_c, out_v


@pytest.mark.parametrize("iterations", [1, 2, 3])
def test_model_equals_the_definition_on_21x19(iterations):
    """The vectorised model against the contract written per pixel and per pair, on an image whose size is no multiple of any
    step, with the other sigma set."""
    g, rgb, sq, counts = image(7)
    got = denoise.denoise(g, rgb, sq, counts, iterations=iterations, conserve_energy=True, **OTHER)
    col, var, tap = denoise.prepare(rgb, sq, counts)
    with np.errstate(all="ignore"):
        for i in range(iterations):
            col, var = reference_iteration(g, col, var, tap, 1 << i, **{**DEFAULTS, **OTHER})
    assert got.tobytes() == col.tobytes()


# sha256 (first 16 hex digits) of the gather form's output on image(seed) as the model computed it before the flux form was
# added: conserve_energy=False must give those bytes.
GATHER_DIGESTS = {
    (1, 1, False): "205764a291c70b1b", (1, 1, True): "5b9a1072aedff74b", (1, 3, False): "f076a91a84e14469",
    (1, 3, True): "46726828aa3a48ec", (1, 8, False): "3788d4795ac716b4", (1, 8, True): "12efd7ec69d8d897",
    (2, 1, False): "97cd101847f41321", (2, 1, True): "cbec02fec32314bc", (2, 3, False): "57a3338008b40cab",
    (2, 3, True): "882e87d37f4f2247", (2, 8, False): "bc06514bd1037145", (2, 8, True): "55f52b623ef994f0",
}


@pytest.mark.parametrize("seed, iterations, other", list(GATHER_DIGESTS))
def test_gather_form_is_unchanged(seed, iterations, other):
    g, rgb, sq, counts = image(seed)
    kw = OTHER if other else {}
    a = denoise.denoise(g, rgb, sq, counts, iterations=iterations, **kw)
    b = denoise.denoise(g, rgb, sq, counts, iterations=iterations, conserve_energy=False, **kw)
    assert a.tobytes() == b.tobytes()
    assert hashlib.sha256(a.tobytes()).hexdigest()[:16] == GATHER_DIGESTS[(seed, iterations, other)]


def header_params(name):
    text = re.sub(r"/\*.*?\*/", "", (ROOT / "include" / "spcu.h").read_text(), flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^)]*)\)\s*;", text)
    assert m, name
    return [re.sub(r"\s+", " ", p.strip()).rsplit(" ", 1)[0].replace(" *", "*") for p in m.group(1).split(",")]


CTYPE_OF = {"spcu_ctx*": C.c_void_p, "const float*": C.c_void_p, "float*": C.c_void_p, "const uint32_t*": C.c_void_p,
            "uint32_t": C.c_uint32, "void*": C.c_void_p, "const spcu_denoise_params*": C.POINTER(capi.DenoiseParams)}


@pytest.mark.parametrize("name, like", [("spcu_denoise_conserving", "spcu_denoise"),
                                        ("spcu_denoise_conserving_device", "spcu_denoise_device")])
def test_prototypes_match_the_header(built, name, like):
    """The new entry points take spcu_denoise(_device)'s arguments, and the ctypes prototypes follow the header."""
    assert name in capi.EXPORTS
    params = header_params(name)
    assert params == header_params(like)
    fn = getattr(capi.load(), name)
    assert list(fn.argtypes) == [CTYPE_OF[p] for p in params]
    assert fn.restype is C.c_int
