"""The drop-in with SPCU_DENOISE=conserve: the reference's main.cpp with the INTEGRATION.md hunks writes the image that
Context.denoise(..., conserve_energy=True) gives from the same sums, with a fixed sample count and with SPCU_ADAPTIVE's count
map."""
import os
import subprocess

import numpy as np
import pytest

from simplepath_b200 import capi, host, scenes

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not host.DRIVER.exists() or not host.available(),
                                 reason="host plugin not built (needs the reference sources)")]
SEED = 12


def run_driver(tmp_path, spp=16, **env):
    sp = scenes.ensure("g_bunny", tmp_path)
    proc = subprocess.run([str(host.DRIVER), "--samples", str(spp), "--integrator", "cuda", sp.name], cwd=tmp_path,
                          env=dict(os.environ, SPCU_SEED=str(SEED), **env), stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                          text=True, timeout=120)
    return sp, proc


@pytest.mark.parametrize("spp, adaptive", [(16, None), (64, "0.1")], ids=["fixed", "adaptive"])
def test_driver_writes_the_conserving_image(ctx, tmp_path, spp, adaptive):
    env = {"SPCU_DENOISE": "conserve"}
    if adaptive:  # passes of 16 samples up to the budget of 64
        env["SPCU_ADAPTIVE"] = adaptive
    sp, proc = run_driver(tmp_path, spp, **env)
    assert proc.returncode == 0, proc.stdout[-2000:]
    assert "denoised, energy-conserving form" in proc.stdout
    img = scenes.read_pfm(tmp_path / "image.pfm")

    flat = host.parse(sp)
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_AUTO)
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), host.jitter(spp), keepalive=flat)
    part = ctx.partition(spp=spp, integrator="iterative_rrnee", seed=SEED)
    if adaptive:
        rgb, sq, counts, _ = ctx.render_adaptive(part, float(adaptive), min_spp=16, pass_spp=16)
    else:
        rgb, sq, _ = ctx.render_frame(part)
        counts = spp
    mean = ctx.denoise(rgb, sq, counts, conserve_energy=True)
    want = ctx.pack_image(mean, 1, capi.IMAGE_PFM)[::-1]  # packed rows are bottom-up, read_pfm's top-down
    assert img.tobytes() == np.ascontiguousarray(want).tobytes()


@pytest.mark.parametrize("value", ["conserv", "Conserve", "conserve "])
def test_driver_rejects_bad_values(tmp_path, value):
    _, proc = run_driver(tmp_path, SPCU_DENOISE=value)
    assert proc.returncode != 0 and "SPCU_DENOISE must be 1" in proc.stdout
