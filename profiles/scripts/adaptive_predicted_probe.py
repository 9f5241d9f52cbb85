#!/usr/bin/env python
"""Adaptive sampling with predicted sample counts (render_adaptive_predicted) against the pass schedule (render_adaptive) and
fixed spp, on the 1080p configs, with the set-up of adaptive_probe.py (budget 256, abs_floor 0.03, min_spp 16, a 1024 spp truth
of another seed, median of --reps calls after a warm-up, host clock around calls that end in a synchronise).

  "pass" lines (--passes): where the pass schedule's time goes.  The schedule's boundaries depend only on min_spp, pass_spp
      and the budget, so a call with budget s_k runs exactly the first k + 1 passes of the call with budget 256: pass k's
      device time, paths and launches are the differences between consecutive budgets (its compaction included), and its
      active pixels are those the full map gives more than s_{k-1} samples.  A least-squares line time = a + b * paths over
      the passes after the first ("pass_fit") separates a per-call cost a from a per-path cost b.
  "fixed" / "passes" / "predicted" lines: time, mean spp, passes or rounds and render calls, relMSE against the truth.
  "equal_relmse" lines: each adaptive point's time against the fixed renders' and the pass schedule's (same radius) at the
      same relMSE, interpolated log-log (null outside their range).
  "bias" lines (--bias): relMSE over the expected and mean luminance against the reference's converged renders, as
      adaptive_bias.py, for both modes.
    python profiles/scripts/adaptive_predicted_probe.py --passes --bias --out profiles/rNN_adaptive_predicted_probe.jsonl"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))
from simplepath_b200 import adaptive, capi, host, rsequence  # noqa: E402

SCENES = ["c2_example_scene", "c3_bunny", "c4_elf"]
FIXED = [16, 32, 64, 128, 256]
ERRORS = [0.1, 0.05, 0.02, 0.01]
STEPS = [1, 2, 4, 8]
BUDGET, TRUTH_SPP, MIN_SPP, PASS_SPP = 256, 1024, 16, 16
ABS_FLOOR = 0.03
SEED, TRUTH_SEED = 20261020, 77
GOLDEN = ROOT / "tests" / "golden"
BIAS = {"c2": ("c2_example_scene", 64), "c3": ("c3_bunny", 256), "c4": ("c4_elf", 64)}  # adaptive_bias.py's configs


def lum(c):
    return 0.2126 * c[..., 0] + 0.7152 * c[..., 1] + 0.0722 * c[..., 2]


def block_mean(a, b):
    h, w = a.shape[:2]
    return a.reshape(h // b, b, w // b, b, *a.shape[2:]).mean(axis=(1, 3))


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


def interp_time(curve, relmse):
    """log-log interpolation of a curve [(relmse, seconds)] at a relMSE (null outside it)."""
    curve = sorted(curve, reverse=True)
    for (e0, t0), (e1, t1) in zip(curve, curve[1:]):
        if e1 <= relmse <= e0 and e0 > e1:
            a = (np.log(relmse) - np.log(e0)) / (np.log(e1) - np.log(e0))
            return float(np.exp(np.log(t0) + a * (np.log(t1) - np.log(t0))))
    return None


def pass_breakdown(ctx, emit, base, rel, reps):
    kw = dict(min_spp=MIN_SPP, pass_spp=PASS_SPP, abs_floor=ABS_FLOOR, want_sumsq=False)
    bounds = adaptive.boundaries(BUDGET, MIN_SPP, PASS_SPP)
    totals, spp_map = [], None
    for s in bounds:  # the call with budget s runs the first passes of the full call exactly
        part = ctx.partition(spp=TRUTH_SPP, sample_end=s, seed=SEED)
        ctx.render_adaptive(part, rel, **kw)  # warm-up
        runs = [ctx.render_adaptive(part, rel, **kw) for _ in range(reps)]
        totals.append(sorted((r[3] for r in runs), key=lambda st: st["device_ms"])[reps // 2])
        spp_map = runs[-1][2]
    recs = []
    for k, (s, st) in enumerate(zip(bounds, totals)):
        prev = totals[k - 1] if k else {"device_ms": 0.0, "paths": 0, "kernel_launches": 0}
        rec = {"pass": k, "begin": bounds[k - 1] if k else 0, "end": s,
               "active_pixels": int((spp_map > bounds[k - 1]).sum()) if k else int(spp_map.size),
               "device_ms": st["device_ms"] - prev["device_ms"], "paths": st["paths"] - prev["paths"],
               "launches": st["kernel_launches"] - prev["kernel_launches"]}
        recs.append(rec)
        emit({**base, "mode": "pass", "rel_error": rel, "radius": 0, **rec})
    tail = [r for r in recs[1:] if r["paths"] > 0]
    if len(tail) >= 2:
        x = np.array([r["paths"] for r in tail], dtype=np.float64)
        y = np.array([r["device_ms"] for r in tail])
        b, a = np.polyfit(x, y, 1)
        emit({**base, "mode": "pass_fit", "rel_error": rel, "passes_fitted": len(tail), "ms_per_call": float(a),
              "ns_per_path": float(b * 1e6), "mean_tail_ms": float(y.mean()), "mean_tail_paths": float(x.mean()),
              "mean_tail_launches": float(np.mean([r["launches"] for r in tail])),
              "pass0_ns_per_path": recs[0]["device_ms"] * 1e6 / recs[0]["paths"]})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scenes", nargs="*", default=SCENES)
    ap.add_argument("--radius", type=int, nargs="+", default=[0, 2])
    ap.add_argument("--steps", type=int, nargs="+", default=STEPS)
    ap.add_argument("--errors", type=float, nargs="+", default=ERRORS)
    ap.add_argument("--passes", action="store_true", help="per-pass breakdown of the pass schedule on elf and example_scene")
    ap.add_argument("--bias", action="store_true", help="the bias table against the converged reference renders")
    args = ap.parse_args()
    info = gpu_info()
    ctx = capi.Context(0)
    with open(args.out, "w") as f:
        def emit(rec):
            line = json.dumps({**rec, **info})
            print(line, flush=True)
            f.write(line + "\n")

        if args.passes:
            for scene in ("c4_elf", "c2_example_scene"):
                flat = host.workload(scene)
                ctx.set_wavefront_size(0)
                ctx.upload_scene(flat.pointer(), rsequence.jitter_table(TRUTH_SPP), keepalive=flat)
                base = {"scene": scene, "width": flat.width, "height": flat.height, "pipeline": ctx.resolved_pipeline(),
                        "budget": BUDGET, "min_spp": MIN_SPP, "pass_spp": PASS_SPP, "abs_floor": ABS_FLOOR}
                for rel in (0.1, 0.05):
                    pass_breakdown(ctx, emit, base, rel, args.reps)

        for scene in args.scenes:
            flat = host.workload(scene)
            ctx.set_wavefront_size(0)
            ctx.upload_scene(flat.pointer(), rsequence.jitter_table(TRUTH_SPP), keepalive=flat)
            truth, _, _ = ctx.render_frame(ctx.partition(spp=TRUTH_SPP, seed=TRUTH_SEED), want_sumsq=False)
            lt = lum(truth.astype(np.float64) / TRUTH_SPP)
            denom = lt ** 2 + 1e-3

            def relmse(rgb, n):
                return float(((lum(rgb.astype(np.float64) / n) - lt) ** 2 / denom).mean())

            base = {"scene": scene, "width": flat.width, "height": flat.height, "pipeline": ctx.resolved_pipeline(),
                    "truth_spp": TRUTH_SPP, "budget": BUDGET, "min_spp": MIN_SPP, "abs_floor": ABS_FLOOR}
            fixed = []
            for spp in FIXED:
                part = ctx.partition(spp=TRUTH_SPP, sample_end=spp, seed=SEED)
                sec, (rgb, _, st) = timed(lambda: ctx.render_frame(part, want_sumsq=False), args.reps)
                e = relmse(rgb, spp)
                fixed.append((e, sec))
                emit({**base, "mode": "fixed", "spp": spp, "seconds": sec, "mean_spp": float(spp), "relmse": e})
            part = ctx.partition(spp=TRUTH_SPP, sample_end=BUDGET, seed=SEED)
            points = []
            for radius in args.radius:
                schedule = []
                for rel in args.errors:
                    sec, (rgb, _, m, st) = timed(lambda: ctx.render_adaptive(part, rel, min_spp=MIN_SPP, pass_spp=PASS_SPP,
                                                                             abs_floor=ABS_FLOOR, want_sumsq=False, radius=radius),
                                                 args.reps)
                    e = relmse(rgb, m.astype(np.float64)[..., None])
                    schedule.append((e, sec))
                    points.append(("passes", radius, None, rel, e, sec))
                    emit({**base, "mode": "passes", "radius": radius, "rel_error": rel, "pass_spp": PASS_SPP, "seconds": sec,
                          "mean_spp": float(m.mean()), "passes": st["passes"], "calls": st["passes"], "relmse": e})
                for step in args.steps:
                    for rel in args.errors:
                        sec, (rgb, _, m, st) = timed(lambda: ctx.render_adaptive_predicted(part, rel, min_spp=MIN_SPP, max_step=step,
                                                                                           abs_floor=ABS_FLOOR, want_sumsq=False,
                                                                                           radius=radius), args.reps)
                        e = relmse(rgb, m.astype(np.float64)[..., None])
                        points.append(("predicted", radius, step, rel, e, sec))
                        emit({**base, "mode": "predicted", "radius": radius, "max_step": step, "rel_error": rel, "seconds": sec,
                              "mean_spp": float(m.mean()), "rounds": st["rounds"], "calls": st["calls"], "relmse": e})
                for mode, r, step, rel, e, sec in points:
                    if r != radius:
                        continue
                    t_fixed, t_sched = interp_time(fixed, e), interp_time(schedule, e)
                    emit({**base, "mode": "equal_relmse", "of": mode, "radius": r, "max_step": step, "rel_error": rel, "relmse": e,
                          "seconds": sec, "fixed_seconds_at_equal_relmse": t_fixed, "speedup_vs_fixed": t_fixed / sec if t_fixed else None,
                          "passes_seconds_at_equal_relmse": t_sched, "speedup_vs_passes": t_sched / sec if t_sched else None})

        if args.bias:
            for cfg, (scene, budget) in BIAS.items():
                gold = np.load(GOLDEN / f"converged_{cfg}.npz")
                b, n_ref = int(gold["block"]), int(gold["spp"])
                ref, var = gold["lum"].astype(np.float64), gold["lum_var"].astype(np.float64)
                denom = ref ** 2 + 1e-3
                flat = host.workload(scene)
                ctx.set_wavefront_size(0)
                ctx.upload_scene(flat.pointer(), rsequence.jitter_table(budget), keepalive=flat)
                part = ctx.partition(spp=budget, seed=20261018)
                for radius, rel in ((r, e) for r in args.radius for e in args.errors):
                    runs = [("passes", None, ctx.render_adaptive(part, rel, min_spp=16, pass_spp=16, want_sumsq=False, radius=radius))]
                    runs += [("predicted", s, ctx.render_adaptive_predicted(part, rel, min_spp=16, max_step=s, want_sumsq=False,
                                                                            radius=radius)) for s in args.steps]
                    for mode, step, (rgb, _, m, st) in runs:
                        n = m.astype(np.float64)
                        mine = block_mean(lum(rgb.astype(np.float64) / n[..., None]), b)
                        e = float(((mine - ref) ** 2 / denom).mean())
                        expected = float((var / (b * b) * (block_mean(1.0 / n, b) + 1.0 / n_ref) / denom).mean())
                        emit({"mode": "bias", "of": mode, "config": cfg, "scene": scene, "budget": budget, "rel_error": rel,
                              "radius": radius, "max_step": step, "min_spp": 16, "mean_spp": float(n.mean()), "relmse": e,
                              "expected": expected, "ratio": e / expected, "mean_lum_rel_diff": float(mine.mean() / ref.mean() - 1.0)})
    ctx.close()


if __name__ == "__main__":
    main()
