#!/usr/bin/env python
"""Adaptive sampling against fixed spp at equal image quality: time, paths and relMSE of fixed renders (16 .. 256 spp) and of
adaptive renders with a budget of 256 at several target errors and window radii, on the 1080p configs, against a 1024 spp "truth" render of
another seed.  relMSE = mean over pixels of (L - L_truth)^2 / (L_truth^2 + 1e-3) (the converged tests' metric, per pixel).
Times: host clock around a call that ends in a synchronise (host-buffer entry points), after a warm-up call of the same
shape; median of --reps calls.  One JSON line per point, then one "equal_relmse" line per adaptive point: the fixed-spp time
at the same relMSE, interpolated log-log between the two fixed points around it (null outside the fixed range).
    python profiles/scripts/adaptive_probe.py [--radius 0 1 2 7] --out profiles/rNN_adaptive_probe.jsonl"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))
from simplepath_b200 import capi, host, rsequence  # noqa: E402

SCENES = ["c2_example_scene", "c3_bunny", "c4_elf"]
FIXED = [16, 32, 64, 128, 256]
ERRORS = [0.1, 0.05, 0.02, 0.01]
BUDGET, TRUTH_SPP, MIN_SPP, PASS_SPP = 256, 1024, 16, 16
ABS_FLOOR = 0.03  # ~ sqrt of the metric's 1e-3: pixels darker than that weigh little in relMSE
SEED, TRUTH_SEED = 20261020, 77


def lum(c):
    return 0.2126 * c[..., 0] + 0.7152 * c[..., 1] + 0.0722 * c[..., 2]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    name, power, clock = (x.strip() for x in q[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(call, reps):
    call()  # warm-up of this shape
    times, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = call()
        times.append(time.perf_counter() - t0)
    return float(np.median(times)), out


def interp_fixed_time(fixed, relmse):
    """log-log interpolation of the fixed renders' time at a given relMSE (fixed: [(relmse, seconds)], relMSE falling)."""
    for (e0, t0), (e1, t1) in zip(fixed, fixed[1:]):
        if e1 <= relmse <= e0:
            a = (np.log(relmse) - np.log(e0)) / (np.log(e1) - np.log(e0))
            return float(np.exp(np.log(t0) + a * (np.log(t1) - np.log(t0))))
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scenes", nargs="*", default=SCENES)
    ap.add_argument("--radius", type=int, nargs="+", default=[0], help="window radii of the stopping rule (0..7)")
    args = ap.parse_args()
    info = gpu_info()
    ctx = capi.Context(0)
    with open(args.out, "w") as f:
        def emit(rec):
            line = json.dumps({**rec, **info})
            print(line, flush=True)
            f.write(line + "\n")

        for scene in args.scenes:
            flat = host.workload(scene)
            ctx.set_wavefront_size(0)
            ctx.upload_scene(flat.pointer(), rsequence.jitter_table(TRUTH_SPP), keepalive=flat)
            pipeline = ctx.resolved_pipeline()
            truth, _, _ = ctx.render_frame(ctx.partition(spp=TRUTH_SPP, seed=TRUTH_SEED), want_sumsq=False)
            lt = lum(truth.astype(np.float64) / TRUTH_SPP)
            denom = lt ** 2 + 1e-3

            def relmse(rgb, n):
                return float(((lum(rgb.astype(np.float64) / n) - lt) ** 2 / denom).mean())

            base = {"scene": scene, "width": flat.width, "height": flat.height, "pipeline": pipeline, "truth_spp": TRUTH_SPP}
            fixed = []
            for spp in FIXED:
                part = ctx.partition(spp=TRUTH_SPP, sample_end=spp, seed=SEED)
                sec, (rgb, _, st) = timed(lambda: ctx.render_frame(part, want_sumsq=False), args.reps)
                e = relmse(rgb, spp)
                fixed.append((e, sec))
                emit({**base, "mode": "fixed", "spp": spp, "seconds": sec, "paths": st["paths"], "mean_spp": float(spp),
                      "passes": 1, "relmse": e, "device_ms": st["device_ms"]})
            for radius, rel in ((r, e) for r in args.radius for e in ERRORS):
                part = ctx.partition(spp=TRUTH_SPP, sample_end=BUDGET, seed=SEED)
                sec, (rgb, _, spp_map, st) = timed(lambda: ctx.render_adaptive(part, rel, min_spp=MIN_SPP, pass_spp=PASS_SPP,
                                                                               abs_floor=ABS_FLOOR, want_sumsq=False,
                                                                               radius=radius), args.reps)
                n = spp_map.astype(np.float64)
                e = relmse(rgb, n[..., None])
                t_fixed = interp_fixed_time(fixed, e)
                emit({**base, "mode": "adaptive", "rel_error": rel, "radius": radius, "abs_floor": ABS_FLOOR, "budget": BUDGET, "min_spp": MIN_SPP,
                      "pass_spp": PASS_SPP, "seconds": sec, "paths": st["paths"], "mean_spp": float(n.mean()),
                      "passes": st["passes"], "stopped_early": float((spp_map < BUDGET).mean()), "relmse": e,
                      "device_ms": st["device_ms"]})
                emit({**base, "mode": "equal_relmse", "rel_error": rel, "radius": radius, "relmse": e, "adaptive_seconds": sec,
                      "fixed_seconds_at_equal_relmse": t_fixed, "speedup": (t_fixed / sec) if t_fixed else None})
    ctx.close()


if __name__ == "__main__":
    main()
