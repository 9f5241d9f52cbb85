#!/usr/bin/env python
"""Denoising against more samples at equal image quality, on the 1080p configs.

  - time of the guide kernel and of the filter (CUDA events around spcu_render_guides_device / spcu_denoise_device on device
    buffers, median of --reps after a warm-up call), at the scene's 1920x1080 and at 3840x2160 (the same camera with its
    pixel axes halved);
  - relMSE (adaptive_probe.py's: mean over pixels of (L - L_truth)^2 / (L_truth^2 + 1e-3)) against a TRUTH_SPP render of another
    seed, raw and denoised, at 4, 16 and 64 spp and over adaptive renders (radius 2, budget 64) for every filter setting;
  - the fixed-spp render time (host clock around spcu_render_frame, median of --reps) at which a raw render reaches each
    denoised relMSE, interpolated log-log between the fixed renders around it (null beyond 256 spp), next to the time of the
    denoised frame (render + filter).
With --conserve it compares the gather form (spcu_denoise) with the energy-conserving flux form (spcu_denoise_conserving)
instead: device time of guides + filter for both forms at 1080p and 2160p, 3 and 5 iterations; relMSE raw and denoised and
the mean luminance change at 4 and 16 spp for sigma_l 2 / 4 / 8 and both forms, against the same 512-spp truth.
Every line carries the GPU's name and power limit.
    python profiles/scripts/denoise_probe.py --out profiles/r07a_denoise_probe.jsonl
    python profiles/scripts/denoise_probe.py --conserve --out profiles/r08a_denoise_conserving_probe.jsonl"""
import argparse
import ctypes as C
import json
import sys
import time
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(HERE))
from adaptive_probe import gpu_info, interp_fixed_time, lum, timed  # noqa: E402
from simplepath_b200 import capi, host, rsequence  # noqa: E402
from simplepath_b200.flat import FlatSceneData  # noqa: E402

SCENES = ["c2_example_scene", "c3_bunny", "c4_elf"]
FIXED = [4, 8, 16, 32, 64, 128, 256]
DENOISED_AT = [4, 16, 64]
SETTINGS = [dict(iterations=5, sigma_l=4.0, sigma_z=0.1, sigma_a=0.1), dict(iterations=3, sigma_l=4.0, sigma_z=0.1, sigma_a=0.1),
            dict(iterations=5, sigma_l=2.0, sigma_z=0.1, sigma_a=0.1), dict(iterations=5, sigma_l=8.0, sigma_z=0.1, sigma_a=0.1),
            dict(iterations=5, sigma_l=16.0, sigma_z=0.1, sigma_a=0.1), dict(iterations=5, sigma_l=32.0, sigma_z=0.1, sigma_a=0.1),
            dict(iterations=5, sigma_l=64.0, sigma_z=0.1, sigma_a=0.1)]
ADAPTIVE = dict(budget=64, min_spp=4, pass_spp=4, rel_error=0.05, abs_floor=0.03, radius=2)
TRUTH_SPP, SEED, TRUTH_SEED = 512, 20261020, 77
FORMS = {"gather": "spcu_denoise_device", "conserving": "spcu_denoise_conserving_device"}
CONSERVE_AT = [4, 16]
CONSERVE_SIGMA_L = [2.0, 4.0, 8.0]


def scaled(flat: FlatSceneData, k: int) -> FlatSceneData:
    """The same view at k times the resolution: the camera's pixel axes (columns 0 and 1) divided by k."""
    head = dict(flat.head)
    head["width"], head["height"] = flat.width * k, flat.height * k
    cam = list(head["camera"])
    head["camera"] = [v / k for v in cam[:6]] + cam[6:]
    return FlatSceneData(head, flat.arrays)


def event_ms(call, reps):
    """Median CUDA-event time of call() on the current stream, after one warm-up call."""
    call()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for _ in range(reps):
        a.record()
        call()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out))


def kernel_times(ctx, flat, rgb, sq, spp, reps):
    h, w = flat.height, flat.width
    d_rgb = torch.from_numpy(np.ascontiguousarray(rgb)).cuda()
    d_sq = torch.from_numpy(np.ascontiguousarray(sq)).cuda()
    d_out = torch.empty_like(d_rgb)
    d_g = torch.empty(h * w * 32, dtype=torch.uint8, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    guide_ms = event_ms(lambda: ctx._check(ctx.lib.spcu_render_guides_device(ctx.h, C.c_void_p(d_g.data_ptr()), stream),
                                           "spcu_render_guides_device"), reps)
    res = {"guides_ms": guide_ms}
    for s in SETTINGS:
        p = capi.DenoiseParams(s["iterations"], s["sigma_l"], s["sigma_z"], s["sigma_a"])
        ms = event_ms(lambda: ctx._check(ctx.lib.spcu_denoise_device(ctx.h, C.c_void_p(d_rgb.data_ptr()), C.c_void_p(d_sq.data_ptr()),
                                                                       None, spp, C.byref(p), C.c_void_p(d_out.data_ptr()), stream),
                                         "spcu_denoise_device"), reps)
        res[f"denoise_ms_it{s['iterations']}"] = ms  # guides + filter
    return res


def form_times(ctx, rgb, sq, spp, reps):
    """Guides + filter device time of both forms at 3 and 5 iterations (defaults otherwise)."""
    d_rgb = torch.from_numpy(np.ascontiguousarray(rgb)).cuda()
    d_sq = torch.from_numpy(np.ascontiguousarray(sq)).cuda()
    d_out = torch.empty_like(d_rgb)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    res = {}
    for iterations in (3, 5):
        p = capi.DenoiseParams(iterations, capi.DENOISE_DEFAULTS["sigma_l"], capi.DENOISE_DEFAULTS["sigma_z"],
                               capi.DENOISE_DEFAULTS["sigma_a"])
        for form, fn in FORMS.items():
            call = getattr(ctx.lib, fn)
            res[f"{form}_ms_it{iterations}"] = event_ms(lambda: ctx._check(call(
                ctx.h, C.c_void_p(d_rgb.data_ptr()), C.c_void_p(d_sq.data_ptr()), None, spp, C.byref(p), C.c_void_p(d_out.data_ptr()),
                stream), fn), reps)
    return res


def conserve_probe(ctx, args, emit):
    for scene in args.scenes:
        flat = host.workload(scene)
        base = {"scene": scene}
        for k in (1, 2):  # device times at 1080p and 2160p
            fk = scaled(flat, k) if k > 1 else flat
            ctx.set_wavefront_size(0)
            ctx.upload_scene(fk.pointer(), rsequence.jitter_table(4), keepalive=fk)
            rgb, sq, _ = ctx.render_frame(ctx.partition(spp=4, seed=SEED))
            emit({**base, "mode": "kernel_time", "width": fk.width, "height": fk.height, "spp": 4,
                  **form_times(ctx, rgb, sq, 4, args.reps)})
        ctx.upload_scene(flat.pointer(), rsequence.jitter_table(TRUTH_SPP), keepalive=flat)
        truth, _, _ = ctx.render_frame(ctx.partition(spp=TRUTH_SPP, seed=TRUTH_SEED), want_sumsq=False)
        lt = lum(truth.astype(np.float64) / TRUTH_SPP)
        denom = lt ** 2 + 1e-3
        base.update(width=flat.width, height=flat.height, pipeline=ctx.resolved_pipeline(), truth_spp=TRUTH_SPP)
        for spp in CONSERVE_AT:
            rgb, sq, _ = ctx.render_frame(ctx.partition(spp=TRUTH_SPP, sample_end=spp, seed=SEED))
            raw_l = lum(rgb.astype(np.float64) / spp)
            raw = float(((raw_l - lt) ** 2 / denom).mean())
            for sigma_l in CONSERVE_SIGMA_L:
                for form in FORMS:
                    s = dict(capi.DENOISE_DEFAULTS, sigma_l=sigma_l)
                    out_l = lum(ctx.denoise(rgb, sq, spp, conserve_energy=form == "conserving", **s).astype(np.float64))
                    e = float(((out_l - lt) ** 2 / denom).mean())
                    emit({**base, "mode": "denoised", "form": form, "input": f"fixed_{spp}", **s, "relmse_raw": raw,
                          "relmse_denoised": e, "factor": raw / e, "mean_lum_truth": float(lt.mean()),
                          "mean_lum_raw": float(raw_l.mean()), "mean_lum_denoised": float(out_l.mean()),
                          "mean_lum_change": float(out_l.mean() / raw_l.mean() - 1)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scenes", nargs="*", default=SCENES)
    ap.add_argument("--conserve", action="store_true", help="compare the gather and the energy-conserving form")
    args = ap.parse_args()
    info = gpu_info()
    ctx = capi.Context(0)
    with open(args.out, "w") as f:
        def emit(rec):
            line = json.dumps({**rec, **info})
            print(line, flush=True)
            f.write(line + "\n")

        if args.conserve:
            conserve_probe(ctx, args, emit)
        for scene in ([] if args.conserve else args.scenes):
            flat = host.workload(scene)
            base = {"scene": scene}
            for k in (1, 2):  # kernel times at 1080p and 2160p
                fk = scaled(flat, k) if k > 1 else flat
                ctx.set_wavefront_size(0)
                ctx.upload_scene(fk.pointer(), rsequence.jitter_table(4), keepalive=fk)
                rgb, sq, _ = ctx.render_frame(ctx.partition(spp=4, seed=SEED))
                emit({**base, "mode": "kernel_time", "width": fk.width, "height": fk.height, "spp": 4,
                      **kernel_times(ctx, fk, rgb, sq, 4, args.reps)})
            ctx.upload_scene(flat.pointer(), rsequence.jitter_table(TRUTH_SPP), keepalive=flat)
            truth, _, _ = ctx.render_frame(ctx.partition(spp=TRUTH_SPP, seed=TRUTH_SEED), want_sumsq=False)
            lt = lum(truth.astype(np.float64) / TRUTH_SPP)
            denom = lt ** 2 + 1e-3
            base.update(width=flat.width, height=flat.height, pipeline=ctx.resolved_pipeline(), truth_spp=TRUTH_SPP)

            def relmse(mean):
                return float(((lum(mean.astype(np.float64)) - lt) ** 2 / denom).mean())

            fixed, frames = [], {}
            for spp in FIXED:
                part = ctx.partition(spp=TRUTH_SPP, sample_end=spp, seed=SEED)
                sec, (rgb, sq, st) = timed(lambda: ctx.render_frame(part), args.reps)
                e = relmse(rgb / spp)
                fixed.append((e, sec))
                frames[spp] = (rgb, sq, sec)
                emit({**base, "mode": "fixed", "spp": spp, "seconds": sec, "relmse": e,
                      "mean_lum": float(lum(rgb.astype(np.float64) / spp).mean())})
            inputs = [(f"fixed_{spp}", frames[spp][0], frames[spp][1], spp, frames[spp][2]) for spp in DENOISED_AT]
            part = ctx.partition(spp=TRUTH_SPP, sample_end=ADAPTIVE["budget"], seed=SEED)
            sec, (a_rgb, a_sq, a_map, a_st) = timed(lambda: ctx.render_adaptive(
                part, ADAPTIVE["rel_error"], min_spp=ADAPTIVE["min_spp"], pass_spp=ADAPTIVE["pass_spp"], abs_floor=ADAPTIVE["abs_floor"],
                radius=ADAPTIVE["radius"]), args.reps)
            inputs.append(("adaptive", a_rgb, a_sq, a_map, sec))
            for label, rgb, sq, n, render_sec in inputs:
                nn = n if isinstance(n, int) else np.maximum(n, 1)[..., None]
                raw = relmse(rgb / nn)
                for s in SETTINGS:
                    dsec, out = timed(lambda: ctx.denoise(rgb, sq, n, **s), args.reps)
                    e = relmse(out)
                    t_eq = interp_fixed_time(fixed, e)
                    emit({**base, "mode": "denoised", "input": label, **s, "mean_spp": float(np.mean(n)),
                          "relmse_raw": raw, "relmse_denoised": e, "factor": raw / e,
                          "mean_lum_raw": float(lum(rgb.astype(np.float64) / nn).mean()),
                          "mean_lum_denoised": float(lum(out.astype(np.float64)).mean()),
                          "render_seconds": render_sec, "denoise_call_seconds": dsec,
                          "fixed_seconds_at_equal_relmse": t_eq,
                          "speedup": (t_eq / (render_sec + dsec)) if t_eq else None})
    ctx.close()


if __name__ == "__main__":
    main()
