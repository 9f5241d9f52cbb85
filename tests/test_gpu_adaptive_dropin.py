"""The drop-in with SPCU_ADAPTIVE=<rel_error>: the reference's main.cpp with the INTEGRATION.md hunks renders adaptively, with
--samples as the budget, and writes the image that render_adaptive followed by pack_image_counts gives."""
import os
import subprocess

import numpy as np
import pytest

from simplepath_b200 import capi, host, scenes

pytestmark = pytest.mark.gpu


@pytest.mark.skipif(not host.DRIVER.exists() or not host.available(), reason="host plugin not built (needs the reference sources)")
def test_driver_with_adaptive_sampling_writes_the_same_image(ctx, tmp_path):
    sp = scenes.ensure("g_bunny", tmp_path)
    spp, rel = 64, 0.1
    env = dict(os.environ, SPCU_SEED="11", SPCU_ADAPTIVE=str(rel))
    proc = subprocess.run([str(host.DRIVER), "--samples", str(spp), "--integrator", "cuda", sp.name], cwd=tmp_path, env=env,
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert proc.returncode == 0, proc.stdout[-2000:]
    assert "adaptive sampling" in proc.stdout
    img = scenes.read_pfm(tmp_path / "image.pfm")

    flat = host.parse(sp)
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_AUTO)
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), host.jitter(spp), keepalive=flat)
    rgb, _, spp_map, _ = ctx.render_adaptive(ctx.partition(spp=spp, integrator="iterative_rrnee", seed=11), rel, min_spp=16,
                                             pass_spp=16, want_sumsq=False)
    want = ctx.pack_image(rgb, spp_map, capi.IMAGE_PFM)[::-1]  # packed rows are bottom-up, read_pfm's top-down
    assert img.tobytes() == np.ascontiguousarray(want).tobytes()


@pytest.mark.skipif(not host.DRIVER.exists() or not host.available(), reason="host plugin not built (needs the reference sources)")
def test_driver_rejects_adaptive_sampling_over_several_devices(tmp_path):
    sp = scenes.ensure("g_bunny", tmp_path)
    env = dict(os.environ, SPCU_ADAPTIVE="0.1", SPCU_DEVICES="2")
    proc = subprocess.run([str(host.DRIVER), "--samples", "16", "--integrator", "cuda", sp.name], cwd=tmp_path, env=env,
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert proc.returncode != 0 and "SPCU_ADAPTIVE renders on one device" in proc.stdout
