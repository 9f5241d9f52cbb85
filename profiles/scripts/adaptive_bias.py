#!/usr/bin/env python
"""How far does stopping on an estimated variance move an adaptive render from the reference?  The computation of
tests/test_gpu_adaptive.py::test_relmse_against_the_reference_render (relMSE against the reference's converged render, over
the relMSE two unbiased renders of the same per-pixel sample counts would have) for several target errors and window radii,
printed instead of asserted.    python profiles/scripts/adaptive_bias.py [--radius 0 1 2 7] > profiles/rNN_adaptive_bias.jsonl"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))
from simplepath_b200 import capi, host, rsequence  # noqa: E402

GOLDEN = ROOT / "tests" / "golden"
CONFIGS = {"c2": ("c2_example_scene", 64), "c3": ("c3_bunny", 256), "c4": ("c4_elf", 64)}
ERRORS = [0.1, 0.05, 0.02, 0.01]
EPS = 1e-3


def lum(c):
    return 0.2126 * c[..., 0] + 0.7152 * c[..., 1] + 0.0722 * c[..., 2]


def block_mean(a, b):
    h, w = a.shape[:2]
    return a.reshape(h // b, b, w // b, b, *a.shape[2:]).mean(axis=(1, 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--radius", type=int, nargs="+", default=[0], help="window radii of the stopping rule (0..7)")
    ap.add_argument("--errors", type=float, nargs="+", default=ERRORS)
    ap.add_argument("--configs", nargs="+", default=list(CONFIGS))
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         text=True).stdout.strip().splitlines()[0]
    ctx = capi.Context(0)
    for cfg in args.configs:
        scene, budget = CONFIGS[cfg]
        gold = np.load(GOLDEN / f"converged_{cfg}.npz")
        b, n_ref = int(gold["block"]), int(gold["spp"])
        ref, var = gold["lum"].astype(np.float64), gold["lum_var"].astype(np.float64)
        denom = ref ** 2 + EPS
        flat = host.workload(scene)
        ctx.set_wavefront_size(0)
        ctx.upload_scene(flat.pointer(), rsequence.jitter_table(budget), keepalive=flat)
        for radius, rel in ((r, e) for r in args.radius for e in args.errors):
            rgb, _, spp_map, st = ctx.render_adaptive(ctx.partition(spp=budget, seed=20261018), rel, min_spp=16, pass_spp=16,
                                                      want_sumsq=False, radius=radius)
            n = spp_map.astype(np.float64)
            mine = block_mean(lum(rgb.astype(np.float64) / n[..., None]), b)
            relmse = float(((mine - ref) ** 2 / denom).mean())
            expected = float((var / (b * b) * (block_mean(1.0 / n, b) + 1.0 / n_ref) / denom).mean())
            print(json.dumps({"config": cfg, "scene": scene, "budget": budget, "rel_error": rel, "radius": radius, "min_spp": 16,
                              "pass_spp": 16,
                              "mean_spp": float(n.mean()), "passes": st["passes"], "relmse": relmse, "expected": expected,
                              "ratio": relmse / expected, "mean_lum": float(mine.mean()), "ref_mean_lum": float(ref.mean()),
                              "mean_lum_rel_diff": float(mine.mean() / ref.mean() - 1.0), "gpu": gpu}), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
