"""Converged images at the BASELINE.json configs' REAL resolution against renders of the real reference, by relMSE
(north star: "converged images must match the reference render within a stated relMSE").

Reference side: tests/golden/converged_<cfg>.npz (tests/golden/make_golden_converged.py: libsp_ref.so's own integrator and
mt19937_64 sampler; per-block mean luminance and per-block mean of the per-pixel RunningStats variance; block = 1 pixel
for the 256x256 config, the reference's 8x8 tile for the 1080p ones).  CUDA side: the configured scene at its configured
resolution through the product path (reference parser -> flattener -> spcu_upload_scene -> spcu_render).

    relMSE   = mean over blocks of (lum_cuda - lum_ref)^2 / (lum_ref^2 + EPS)
    expected = mean over blocks of lum_var / B^2 * (1 / N_cuda + 1 / N_ref) / (lum_ref^2 + EPS)      (two unbiased renders)

STATED BOUND (DESIGN.md §6): 0.6 * expected <= relMSE <= 1.5 * expected + 1e-5, i.e. the CUDA image differs from the
reference image by no more than the two renders' own Monte-Carlo noise — no bias visible at that resolution — and is not
suspiciously closer either; and the image's mean luminance agrees within 1 %.
"""
import numpy as np
import pytest

from conftest import GOLDEN
from simplepath_b200 import host, rsequence

pytestmark = pytest.mark.gpu
EPS = 1e-3
# config -> (scene, samples per pixel rendered here)
CONFIGS = {
    "c1": ("c1_material_spheres", 16),      # BASELINE configs[0]: 256x256, 16 spp, the 1024x512 image-based light
    "c1_1024": ("c1_material_spheres", 1024),  # the same config converged as far as the reference render is
    "c2": ("c2_example_scene", 64),         # configs[1]: 1920x1080, 64 spp
    "c3": ("c3_bunny", 256),                # configs[2]: 1920x1080, 256 spp
    "c4": ("c4_elf", 64),                   # configs[3] at a quarter of its 256 spp (the reference render holds 12)
}


def lum(c):
    return 0.2126 * c[..., 0] + 0.7152 * c[..., 1] + 0.0722 * c[..., 2]


def block_mean(a, b):
    h, w = a.shape[:2]
    return a.reshape(h // b, b, w // b, b, *a.shape[2:]).mean(axis=(1, 3))


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_relmse_against_the_reference_render(ctx, cfg):
    scene, spp = CONFIGS[cfg]
    path = GOLDEN / f"converged_{cfg.split('_')[0]}.npz"
    if not path.exists():
        pytest.skip(f"{path.name} not generated")
    if not host.loadable(scene):
        pytest.skip(f"{scene} needs the reference's parser + the flattener (libsphost.so), which is not built")
    gold = np.load(path)
    b, n_ref = int(gold["block"]), int(gold["spp"])
    flat = host.workload(scene)
    assert (flat.width, flat.height) == (int(gold["width"]), int(gold["height"]))
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), rsequence.jitter_table(spp), keepalive=flat)
    rgb, _, st = ctx.render_frame(ctx.partition(spp=spp, integrator="iterative_rrnee", seed=20261018), want_sumsq=False)
    assert st["paths"] == flat.width * flat.height * spp
    mine = block_mean(lum(rgb.astype(np.float64) / spp), b)
    ref, var = gold["lum"].astype(np.float64), gold["lum_var"].astype(np.float64)
    denom = ref ** 2 + EPS
    relmse = float(((mine - ref) ** 2 / denom).mean())
    expected = float((var / (b * b) * (1.0 / spp + 1.0 / n_ref) / denom).mean())
    print(f"\n{cfg}: {flat.width}x{flat.height} {spp} spp vs reference {n_ref} spp, block {b}: relMSE {relmse:.3e}, "
          f"expected from the renders' own variance {expected:.3e} (ratio {relmse / expected:.2f}); "
          f"mean luminance {mine.mean():.5f} vs {ref.mean():.5f}")
    assert 0.6 * expected <= relmse <= 1.5 * expected + 1e-5, f"{cfg}: relMSE {relmse:.3e} vs expected {expected:.3e}"
    assert abs(mine.mean() - ref.mean()) <= 0.01 * ref.mean()
