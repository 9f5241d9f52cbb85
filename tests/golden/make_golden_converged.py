"""Reference renders of the BASELINE.json configs AT THEIR REAL RESOLUTION, reduced to what the converged-image (relMSE)
tests need (tests/test_gpu_converged.py).  Run in the development container only (needs oracle/_ref/libsp_ref.so):

    python tests/golden/make_golden_converged.py [config ...]

For every config it renders `iterative_rrnee` with the REAL reference (libsp_ref.so, its own integrator, its own
mt19937_64 sampler) at the stated sample count and stores, per block of BxB pixels (B = 1 for the 256x256 config, B = 8 =
the reference's tile size for the 1080p configs, so that the file stays a few hundred KB):

    lum       block mean of the per-pixel mean luminance              [H/B, W/B]
    lum_var   block mean of the per-pixel luminance VARIANCE (RunningStats, base/RunningStats.h:12-69)  [H/B, W/B]
    spp, block, width, height

relMSE of a render R against this reference is  mean over blocks of (lum_R - lum)^2 / (lum^2 + EPS);  its EXPECTED value
when R is an unbiased render with N_R samples per pixel is  mean over blocks of lum_var / B^2 * (1/N_R + 1/spp) / (lum^2 + EPS).
"""
from __future__ import annotations

import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))

from oracle import ref  # noqa: E402
from simplepath_b200 import scenes  # noqa: E402

HERE = Path(__file__).resolve().parent
# config -> (scene, reference samples per pixel, block)
CONFIGS = {
    "c1": ("c1_material_spheres", 1024, 1),
    "c2": ("c2_example_scene", 48, 8),
    "c3": ("c3_bunny", 12, 8),
    "c4": ("c4_elf", 12, 8),
}


def block_mean(a: np.ndarray, b: int) -> np.ndarray:
    h, w = a.shape[:2]
    assert h % b == 0 and w % b == 0
    return a.reshape(h // b, b, w // b, b, *a.shape[2:]).mean(axis=(1, 3)).astype(np.float32)


def main() -> None:
    if not ref.available():
        raise SystemExit("oracle/_ref/libsp_ref.so missing: run `make -C oracle REF=<the reference sources>`")
    import os
    threads = os.cpu_count() or 1
    for cfg in (sys.argv[1:] or list(CONFIGS)):
        scene, spp, b = CONFIGS[cfg]
        t0 = time.time()
        rs = ref.RefScene(scenes.ensure(scene))
        rgb, mean, var, secs = rs.render("iterative_rrnee", spp, threads)
        rs.close()
        # no colour image: the relMSE is taken over luminance, and the image kept converged_c1.npz above 1 MB (files
        # written before this change still hold it as rgb, which nothing reads)
        np.savez_compressed(HERE / f"converged_{cfg}.npz", lum=block_mean(mean, b),
                            lum_var=block_mean(var, b), spp=np.array(spp), block=np.array(b),
                            width=np.array(rgb.shape[1]), height=np.array(rgb.shape[0]))
        print(cfg, scene, f"{spp} spp, render {secs:.1f} s, total {time.time() - t0:.1f} s", flush=True)


if __name__ == "__main__":
    main()
