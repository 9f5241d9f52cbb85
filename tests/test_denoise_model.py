"""The numpy model of the denoiser (simplepath_b200/denoise.py): properties of the filter and the guides' albedo rule.
Runs without a GPU; tests/test_gpu_denoise.py holds the device to this model bit for bit."""
import numpy as np
import pytest

from conftest import GOLDEN, golden_names
from simplepath_b200 import capi, denoise
from simplepath_b200.flat import FlatSceneData

F = np.float32


def guides(h, w, normal=(0.0, 0.0, -1.0), depth=5.0, albedo=(0.5, 0.5, 0.5), gid=0):
    g = np.zeros((h, w), dtype=capi.GUIDE_DTYPE)
    g["normal"] = normal
    g["depth"] = depth
    g["albedo"] = albedo
    g["id"] = gid
    return g


def noisy_sums(h, w, spp, seed=1):
    rng = np.random.default_rng(seed)
    samples = rng.gamma(2.0, 0.25, size=(spp, h, w, 3)).astype(F)
    rgb = samples.sum(axis=0, dtype=F)
    lum = (F(0.2126) * samples[..., 0] + F(0.7152) * samples[..., 1]) + F(0.0722) * samples[..., 2]
    return rgb, (lum * lum).sum(axis=0, dtype=F)


# The weighted mean of a constant rounds once per tap; iterations filter the previous one's output, so that compounds.
# Measured: 1 / 4 / 5 / 5 / 4 ulp at 1 / 2 / 3 / 5 / 8 iterations.
CONSTANT_ULP = {1: 2, 5: 6, 8: 6}


def test_constant_image_comes_back():
    """A noise-free constant image comes back within CONSTANT_ULP."""
    h, w, spp = 19, 21, 16
    c = np.array([0.3, 0.6, 0.9], dtype=F)
    rgb = np.broadcast_to(c * F(spp), (h, w, 3)).astype(F)
    lum = (F(0.2126) * c[0] + F(0.7152) * c[1]) + F(0.0722) * c[2]
    sq = np.full((h, w), lum * lum * F(spp), dtype=F)
    for it in (1, 5, 8):
        out = denoise.denoise(guides(h, w), rgb, sq, spp, iterations=it)
        ulp = np.abs(out.view(np.int32) - (rgb / F(spp)).view(np.int32))
        assert ulp.max() <= CONSTANT_ULP[it], (it, ulp.max())


# The 3x3 variance prefilter is the one term that looks across an edge.  One sample per pixel makes every variance 0, so
# that the sides of an edge can be compared, bit for bit, with the model run on each side alone.
def test_orthogonal_normals_never_mix():
    h, w, spp = 19, 21, 1
    rgb, sq = noisy_sums(h, w, spp)
    g = guides(h, w)
    g["normal"][:, 11:] = (1.0, 0.0, 0.0)
    out = denoise.denoise(g, rgb, sq, spp, iterations=5)
    left = denoise.denoise(g[:, :11], rgb[:, :11], sq[:, :11], spp, iterations=5)
    right = denoise.denoise(g[:, 11:], rgb[:, 11:], sq[:, 11:], spp, iterations=5)
    # a zero weight adds +0 to the sums: the two sides equal the model run on each side alone, bit for bit
    assert out[:, :11].tobytes() == left.tobytes()
    assert out[:, 11:].tobytes() == right.tobytes()


def test_classes_never_mix():
    h, w, spp = 19, 21, 1
    rgb, sq = noisy_sums(h, w, spp, seed=2)
    g = guides(h, w)
    g["id"][:7] = -1   # miss
    g["id"][7:12] = -2  # light 0
    out = denoise.denoise(g, rgb, sq, spp, iterations=4)
    for rows in (slice(0, 7), slice(7, 12), slice(12, 19)):
        alone = denoise.denoise(g[rows], rgb[rows], sq[rows], spp, iterations=4)
        assert out[rows].tobytes() == alone.tobytes()


def test_empty_pixels_stay_zero_and_are_no_taps():
    h, w, spp = 19, 21, 8
    rgb, sq = noisy_sums(h, w, spp, seed=3)
    counts = np.full((h, w), spp, dtype=np.uint32)
    counts[::3, ::2] = 0
    out = denoise.denoise(guides(h, w), rgb, sq, counts, iterations=3)
    assert (out[counts == 0] == 0).all()
    # the empty pixels' sums do not matter to anyone
    rgb2, sq2 = rgb.copy(), sq.copy()
    rgb2[counts == 0] = 1e6
    sq2[counts == 0] = 1e9
    assert denoise.denoise(guides(h, w), rgb2, sq2, counts, iterations=3).tobytes() == out.tobytes()


def test_non_finite_pixels_pass_through_and_are_no_taps():
    h, w, spp = 19, 21, 8
    rgb, sq = noisy_sums(h, w, spp, seed=4)
    bad = np.zeros((h, w), dtype=bool)
    bad[4, 5] = bad[10, 17] = bad[0, 0] = True
    rgb[4, 5, 1] = np.inf
    rgb[10, 17, 0] = np.nan
    sq[0, 0] = np.inf
    out = denoise.denoise(guides(h, w), rgb, sq, spp, iterations=4)
    with np.errstate(all="ignore"):
        want = rgb[bad] / F(spp)
    assert out[bad].tobytes() == want.tobytes()
    assert np.isfinite(out[~bad]).all()
    # what the bad pixels hold does not reach their neighbours
    rgb2 = rgb.copy()
    rgb2[4, 5] = (np.inf, np.inf, 7.0)
    out2 = denoise.denoise(guides(h, w), rgb2, sq, spp, iterations=4)
    assert out2[~bad].tobytes() == out[~bad].tobytes()


def reference_iteration(g, col, var, tap, h, sigma_l, sigma_z, sigma_a):
    """One iteration written per pixel and per tap, straight from the definition (include/spcu.h)."""
    H, W = tap.shape
    lum = lambda c: (F(0.2126) * c[0] + F(0.7152) * c[1]) + F(0.0722) * c[2]  # noqa: E731
    b = (F(1 / 16), F(1 / 4), F(3 / 8), F(1 / 4), F(1 / 16))
    cls = lambda i: 0 if i >= 0 else (2 if i == -1 else 1)  # noqa: E731
    out_c, out_v = col.copy(), var.copy()
    for y in range(H):
        for x in range(W):
            if not tap[y, x]:
                continue
            pv = pw = F(0)
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    qx, qy = x + dx, y + dy
                    if 0 <= qx < W and 0 <= qy < H and tap[qy, qx]:
                        wt = F(0.5 if dx == 0 else 0.25) * F(0.5 if dy == 0 else 0.25)
                        pv, pw = pv + wt * var[qy, qx], pw + wt
            l_den = F(sigma_l) * np.sqrt(pv / pw) + F(1e-4)
            S, Sw, Sv = np.zeros(3, dtype=F), F(0), F(0)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    qx, qy = x + dx * h, y + dy * h
                    if not (0 <= qx < W and 0 <= qy < H and tap[qy, qx]):
                        continue
                    k = b[dx + 2] * b[dy + 2]
                    p, q = g[y, x], g[qy, qx]
                    if dx == 0 and dy == 0:
                        wt = k
                    elif cls(p["id"]) != cls(q["id"]):
                        wt = F(0)
                    else:
                        wn, az, aa = F(1), F(0), F(0)
                        if p["id"] >= 0:
                            n, m = p["normal"], q["normal"]
                            wn = max(F(0), (n[0] * m[0] + n[1] * m[1]) + n[2] * m[2])
                            for _ in range(7):
                                wn = wn * wn
                            az = np.abs(p["depth"] - q["depth"]) / ((F(sigma_z) * p["depth"]) * F(h * max(abs(dx), abs(dy))))
                            aa = np.abs(p["albedo"] - q["albedo"]).max() / F(sigma_a)
                        al = np.abs(lum(col[y, x]) - lum(col[qy, qx])) / l_den
                        wt = (k * wn) / (((F(1) + al * al) + az * az) + aa * aa)
                    S = S + wt * col[qy, qx]
                    Sw = Sw + wt
                    Sv = Sv + (wt * wt) * var[qy, qx]
            out_c[y, x] = S / Sw
            out_v[y, x] = Sv / (Sw * Sw)
    return out_c, out_v


@pytest.mark.parametrize("iterations", [1, 2, 4])
def test_taps_near_the_border_on_21x19(iterations):
    """The vectorised model against the definition written per pixel, with mixed classes, normals, depths and albedos and
    a few empty pixels, on an image whose size is no multiple of any step."""
    h, w, spp = 19, 21, 6
    rng = np.random.default_rng(5)
    rgb, sq = noisy_sums(h, w, spp, seed=5)
    counts = np.full((h, w), spp, dtype=np.uint32)
    counts[rng.random((h, w)) < 0.05] = 0
    counts[rng.random((h, w)) < 0.05] = 1
    g = guides(h, w)
    n = rng.normal(size=(h, w, 3)).astype(F)
    n[..., 2] = -np.abs(n[..., 2]) - F(2)
    g["normal"] = (n / np.sqrt((n * n).sum(-1, keepdims=True))).astype(F)
    g["depth"] = rng.uniform(4.0, 6.0, size=(h, w)).astype(F)
    g["albedo"] = rng.uniform(0.2, 0.8, size=(h, w, 3)).astype(F)
    g["id"][rng.random((h, w)) < 0.1] = -1
    g["id"][rng.random((h, w)) < 0.1] = -3
    kw = dict(sigma_l=2.0, sigma_z=0.05, sigma_a=0.3)
    got = denoise.denoise(g, rgb, sq, counts, iterations=iterations, **kw)
    col, var, tap = denoise.prepare(rgb, sq, counts)
    for i in range(iterations):
        col, var = reference_iteration(g, col, var, tap, 1 << i, **kw)
    assert got.tobytes() == col.tobytes()


@pytest.mark.parametrize("name", golden_names())
def test_albedo_rule_on_golden_materials(name):
    flat = FlatSceneData.load(GOLDEN / f"{name}.flat.npz")
    alb = denoise.material_albedos(flat)
    mats = flat.arrays["materials"].view(denoise.MATERIAL_DTYPE).reshape(-1)
    bxdfs = flat.arrays["bxdfs"].view(denoise.BXDF_DTYPE).reshape(-1)
    assert alb.shape == (mats.shape[0], 3) and alb.dtype == F
    for i, m in enumerate(mats):
        depth = 0
        while m["kind"] == denoise.MAT_CLEARCOAT:
            m = mats[m["base"]]
            depth += 1
            assert depth <= denoise.MAX_COAT_DEPTH
        want = np.zeros(3, dtype=F)
        for b in bxdfs[m["first_bxdf"]:m["first_bxdf"] + m["n_bxdfs"]]:
            want = want + b["r"] * (denoise.PI if b["kind"] == denoise.BXDF_LAMBERT else F(1))
        assert alb[i].tobytes() == want.tobytes(), (name, i)
        assert np.isfinite(alb[i]).all() and (alb[i] >= 0).all()


def test_albedo_of_example_scene_by_hand():
    """example_scene (scenes.sp_example_scene): material 0 is a Lambert with diffuse (0.1, 0.2, 0.8), which the flattener
    stores as diffuse / pi; material 1 is a clearcoat over it and takes its base's albedo.  Both come back to the scene
    file's diffuse within 1 ulp."""
    alb = denoise.material_albedos(FlatSceneData.load(GOLDEN / "g_example.flat.npz"))
    want = np.array([0.1, 0.2, 0.8], dtype=F)
    for a in alb:
        assert np.abs(a.view(np.int32) - want.view(np.int32)).max() <= 1, a
