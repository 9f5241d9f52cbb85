#!/usr/bin/env python
"""Benchmark of the hot path: whole-frame renders of the BASELINE.json workloads through the CUDA backend.

    python bench.py --gpus N --steps K --warmup W            # this repo's CudaIntegrator path (one rank per GPU)
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU implementation, same workload
    python bench.py --steps K --warmup W --dump-outputs DIR  # + the last timed frame's per-pixel sums as DIR/*.npy

A *step* is ONE FRAME of the workload.  The default workload is BASELINE.json configs[2] — bunny.sp, 1920x1080, 256 spp,
iterative_rrnee — the config BASELINE.json quotes "at 1/2/4/8 GPUs".  With N ranks the frame's 256 samples per pixel are
split into N sample ranges (rank r renders global samples [r*256/N, (r+1)*256/N) of every pixel; scene replicated; random
numbers keyed by the global sample index, so the union is exactly the one-GPU frame) and the per-pixel accumulators are
summed into rank 0 by the product library's own NCCL reduction (spcu_reduce_to_root) inside the timed region: total work is
fixed, "scaling": "strong".

value    = Mpaths/s of the whole job, device-timed (CUDA events on the launching stream, max over ranks), scene resident in
           HBM, accumulators on the device
e2e      = the same metric through the host-buffer C-ABI call a plugin makes: spcu_upload_scene + spcu_render_frame at N = 1,
           spcu_upload_scene + spcu_render_frame_reduced at N > 1 (ONE image arrives in rank 0's host buffer): flattened scene
           copied host->device and the frame copied device->host inside the timed region
roofline = the kernel with the largest share of the step.  These kernels are bound by instruction issue at partial SIMD
           occupancy, not by HBM (profiles/ncu_kernels_r02_*.json): `bound` names the resource with the higher fraction,
           `issue_frac` = thread instructions per second (ncu's count per item x the items of the timed launches / their CUDA-
           event duration) over SMs x 4 schedulers x 32 lanes x SM clock, `hbm_frac` = MEASURED DRAM traffic over the same
           duration against MEASURED_PEAKS.json, `algorithmic_gbs` = SURVEY §8(d)'s byte model (what an uncached walk would move)
cpu_baseline = the reference binary (oracle/_ref/SimplePath) on this box's host cores on a bounded sample of the workload
configs  = at N = 1 the other BASELINE configs as short side runs (fewer steps; not the headline): c1 material_spheres with the
           image-based light, c2 example_scene, c4 elf, c5 lucy as a stated spp sample with the BVH built on the device
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import re
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name -> (scene name in simplepath_b200.scenes, spp of the whole frame)
    "material_spheres_256_16spp": ("c1_material_spheres", 16),
    "material_spheres_const_256_16spp": ("c1_material_spheres_const", 16),
    "example_scene_1080p_64spp": ("c2_example_scene", 64),
    "bunny_1080p_256spp": ("c3_bunny", 256),
    "elf_1080p_256spp": ("c4_elf", 256),
    "lucy_4k_256spp": ("c5_lucy", 256),
}
DEFAULT_WORKLOAD = "bunny_1080p_256spp"
INTEGRATOR = "iterative_rrnee"
SM_SCHEDULERS, WARP_LANES = 4, 32

# ---- byte model (DESIGN.md): algorithmic bytes per item of each wavefront stage, excluding traversal ---------------
STAGE_BYTES = {
    # 32-byte records of csrc/device_scene.h: what a stage must read and write per queue entry
    "raygen": 88,               # pixel id in; RayRec, PathRec, RNG counter, queue entry out
    "extend": 72,               # queue, RayRec in; ExtendRec, sorted-queue entry out (+ traversal bytes)
    "shade": 240,               # queue, ExtendRec, RayRec, PathRec, shading record + meta in; VertexRec, SampleRec, queue out
    "nee_light": 108,           # queue, VertexRec, PathRec in; LightRec, counter, queue out
    "shadow": 56,               # queue, VertexRec.p, LightRec in; queue out (+ traversal bytes)
    "nee_bsdf": 188,            # queue, VertexRec, LightRec, PathRec, RayRec.d in; MisRec, counter, queue out
    "mis_trace": 44,            # queue, VertexRec.p, MisRec.d in; light/occluded out (+ traversal bytes)
    "nee_mis_accumulate": 116,  # queue, MisRec, PathRec in; PathRec.L out
    "direct_accumulate": 116,
    "advance": 156,             # queue, SampleRec, VertexRec, PathRec in; PathRec.tp, RayRec, counter, queue out
    "resolve": 20,              # radiance sample in, per-pixel sums amortised
    "paths": 20,  # SM-local wavefront / persistent path kernel: 4 B pixel id in, 16 B radiance sample out; the rest stays on chip
}
NODE_BYTES, TRI_BYTES, XF_BYTES = 64, 48, 96
TRAVERSING = {"extend", "shadow", "mis_trace", "paths"}


def ncu_kernel_summary(stage: str, workload: str, pipeline: str) -> tuple[dict | None, str | None]:
    """What ncu measured for the kernels of one stage on one workload (profiles/ncu_kernels_rNN_*.json, made by
    profiles/traffic_probe.py + traffic_join.py from one capture of the whole render): DRAM bytes, thread and warp
    instructions per item, time-weighted issue-slot utilisation."""
    for path in sorted((ROOT / "profiles").glob("ncu_kernels_r*.json"), reverse=True):
        d = json.loads(path.read_text())
        p = d.get("probe", {})
        if p.get("workload") == workload and p.get("pipeline") in (pipeline, None) and stage in d.get("stages", {}):
            return d["stages"][stage], path.name
    return None, None


def peaks() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# =====================================================================================================================
# scenes
# =====================================================================================================================
def load_scene(ctx, scene_name: str, spp_total: int):
    """Flatten and upload a workload's scene; returns (flat, jitter, reupload) where reupload() repeats the host->device
    copy of the step's inputs (the e2e leg).  c5_lucy never goes through the reference's parser: its 28 M-triangle mesh is
    generated procedurally, ingested and BUILT ON THE DEVICE (spcu_ingest_mesh -> spcu_upload_scene_build), with camera,
    materials, plane and light flattened from the same scene text over a small stand-in mesh."""
    from simplepath_b200 import host
    jitter = host.jitter(spp_total)
    if scene_name != "c5_lucy":
        flat = host.workload(scene_name)

        def reupload():
            ctx.upload_scene(flat.pointer(), jitter, keepalive=flat)
        reupload()
        return flat, jitter, reupload
    from simplepath_b200 import scenes
    from simplepath_b200.flat import unbuilt_scene_with_mesh
    standin = host.workload("c5_lucy_standin")   # lucy.sp's camera / materials / plane / light over a 40 K-triangle stand-in
    v, f = scenes.bumpy_sphere(scenes.LUCY_TRIS, scenes.LUCY_LO, scenes.LUCY_HI)
    # scenes/lucy.sp: rotate 1 0 0 -90, i.e. object (x, y, z) -> world (x, z, -y); columns c0 c1 c2, then the affine part
    rot = [1, 0, 0, 0, 0, -1, 0, 1, 0]
    flat = unbuilt_scene_with_mesh(ctx, standin, v, f, rot + [0, 0, 0], rot)
    built = {}

    def reupload():
        _, built["head"] = ctx.upload_scene_build(flat.pointer(), jitter, keepalive=flat)
    reupload()
    flat.head["geom"].update({k: built["head"][k] for k in ("n_nodes", "max_depth")})   # for the report only
    return flat, jitter, reupload


# =====================================================================================================================
# one workload, measured
# =====================================================================================================================
def measure(ctx, args, workload: str, spp_total: int, steps: int, warmup: int, world: int, rank: int, clocks_index=None,
            e2e_steps: int = 3, keep_outputs: bool = False) -> dict:
    import torch
    import torch.distributed as dist
    from simplepath_b200 import capi, distributed

    scene_name, _ = WORKLOADS[workload]
    if spp_total % world:
        raise SystemExit(f"{spp_total} spp do not split over {world} ranks")
    spp_rank = spp_total // world
    flat, jitter, reupload = load_scene(ctx, scene_name, spp_total)
    w, h = flat.width, flat.height
    part = capi.Partition(0, 1, rank * spp_rank, (rank + 1) * spp_rank, spp_total, capi.INTEGRATORS[INTEGRATOR], args.seed)
    rgb = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
    sq = torch.zeros((h, w), dtype=torch.float32, device="cuda")
    stream = torch.cuda.current_stream()

    def step(want_stats: bool):
        rgb.zero_(); sq.zero_()
        st = ctx.render_device(part, rgb.data_ptr(), sq.data_ptr(), stream.cuda_stream, want_stats=want_stats)
        ctx.reduce_to_root(rgb.data_ptr(), sq.data_ptr(), stream.cuda_stream)   # the library's ncclReduce; no-op at N = 1
        return st

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also: one counting pass on the reference-order walk for the byte model's N_node / N_tri / N_xf) --------
    ctx.set_option(capi.OPT_COUNT_NODES, 1)
    counted = step(True)
    ctx.set_option(capi.OPT_COUNT_NODES, 0)
    for _ in range(max(warmup - 1, 2)):
        step(False)
    barrier()

    # ---- timed region: K steps, device-timed ---------------------------------------------------------------------------
    sampler = ClockSampler(clocks_index) if clocks_index is not None and rank == 0 else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(steps):
        step(False)          # nothing but kernel launches (and the NCCL reduce) between the two events
    e1.record(stream)
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    # what the last timed step handed its caller: rank 0's per-pixel sums after the reduction (the later steps overwrite them)
    outputs = {"rgb_sum": rgb.cpu().numpy(), "lum_sumsq": sq.cpu().numpy()} if keep_outputs and rank == 0 else None

    # ---- per-kernel CUDA-event durations, same workload, directly after the timed steps (one event pair per launch would
    # perturb the headline number in the wavefront pipeline, so they are taken on their own steps) --------------------------
    ctx.set_option(capi.OPT_STAGE_TIMING, 1)
    stage_ms: dict[str, float] = {}
    stage_launches: dict[str, int] = {}
    stage_items: dict[str, int] = {}
    last = None
    stage_steps = max(1, min(steps, 2))
    for _ in range(stage_steps):
        last = step(True)
        for s in ctx.stage_times():
            stage_ms[s["name"]] = stage_ms.get(s["name"], 0.0) + s["ms"]
            stage_launches[s["name"]] = stage_launches.get(s["name"], 0) + s["launches"]
            stage_items[s["name"]] = stage_items.get(s["name"], 0) + s["items"]
    barrier()
    clocks = sampler.stop() if sampler else None
    ctx.set_option(capi.OPT_STAGE_TIMING, 0)

    counts = torch.tensor([last["paths"], last["rays_closest"], last["rays_any"], last["rays_lights"],
                           last["kernel_launches"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(counts)
    paths, rays_closest, rays_any, rays_lights, launches = (float(x) for x in counts.tolist())

    # ---- end to end through the host-buffer C-ABI (what sp::CudaIntegrator::render_frame does) -------------------------
    h_rgb = torch.empty((h, w, 3), dtype=torch.float32, pin_memory=True).numpy() if rank == 0 else None
    h_sq = torch.empty((h, w), dtype=torch.float32, pin_memory=True).numpy() if rank == 0 else None

    def e2e_step():
        reupload()                                   # host -> device: the step's inputs (flattened scene + jitter table)
        if world == 1:
            ctx.render_frame(part, out=(h_rgb, h_sq))    # device -> host: the step's result (overwritten, not accumulated)
        else:                                        # ranks render their sample ranges, NCCL sums them, rank 0 reads ONE frame
            ctx.render_frame_reduced(part, out=(h_rgb, h_sq) if rank == 0 else None, want_stats=False)

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s.item())
    if rank != 0:
        return {}
    scene_bytes = ctx.scene_bytes()
    acc_bytes = h_rgb.nbytes + h_sq.nbytes
    e2e_sanity = float(h_rgb.sum(dtype=np.float64) / (w * h * spp_total))

    # ---- roofline of the dominant kernel ---------------------------------------------------------------------------------
    peak, peak_src = peaks()
    pipeline = ctx.resolved_pipeline()
    dominant = max(stage_ms, key=stage_ms.get)
    n_launch = max(stage_launches[dominant], 1)
    items = stage_items[dominant]
    bytes_total = items * STAGE_BYTES[dominant]
    geom_queries = counted["rays_closest"] + counted["rays_any"]
    per_query = ((counted["nodes_visited"] * NODE_BYTES + counted["prims_tested"] * TRI_BYTES +
                  counted["xf_prims_tested"] * XF_BYTES) / max(geom_queries, 1))
    if dominant == "paths":  # one item = one path = (closest + any-hit) geometry queries
        bytes_total += geom_queries * per_query * (items / max(counted["paths"], 1))
    elif dominant in TRAVERSING:
        bytes_total += items * per_query
    dur_s = stage_ms[dominant] / 1e3 / n_launch          # mean duration of one launch of the dominant stage
    algorithmic_gbs = bytes_total / n_launch / dur_s / 1e9 if dur_s > 0 else 0.0
    kernel_ms = sum(stage_ms.values())
    ncu, ncu_src = ncu_kernel_summary(dominant, workload, pipeline)
    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    sm_ghz = ((clocks or {}).get("sm_max_mhz") or 1965.0) / 1e3
    issue_peak = sm_count * SM_SCHEDULERS * WARP_LANES * sm_ghz          # G thread-instructions / s
    roof = {"kernel": dominant, "share_of_step": stage_ms[dominant] / kernel_ms if kernel_ms else None,
            "launches": n_launch, "items_per_launch": items / n_launch, "launch_ms": dur_s * 1e3,
            "timed": "CUDA events around every launch on extra steps right after the timed ones, ONE batch at a time (the timed "
                     "steps overlap batches on several streams, where a launch has no duration of its own)",
            "algorithmic_gbs": algorithmic_gbs, "algorithmic_frac_of_hbm": algorithmic_gbs / peak,
            "algorithmic_bytes_per_item": bytes_total / max(items, 1), "hbm_peak_gbs": peak, "peak_source": peak_src,
            "ncu_source": ncu_src}
    if ncu is not None and dur_s > 0:
        traffic = ncu["dram_bytes_per_item"] * items / n_launch
        hbm_gbs = traffic / dur_s / 1e9
        issue_g = ncu["thread_inst_per_item"] * items / n_launch / dur_s / 1e9
        hbm_frac, issue_frac = hbm_gbs / peak, issue_g / issue_peak
        roof.update({"traffic": traffic, "hbm_gbs": hbm_gbs, "hbm_frac": hbm_frac,
                     "issue_gthread_inst_per_s": issue_g, "issue_peak": issue_peak, "issue_frac": issue_frac,
                     "lanes_per_instruction": ncu.get("lanes_per_instruction"),
                     "issue_slot_utilisation_ncu": ncu.get("issue_active_pct")})
        if issue_frac >= hbm_frac:
            roof.update({"bound": "issue", "achieved": issue_g, "peak": issue_peak, "unit": "Gthread-inst/s", "frac": issue_frac})
        else:
            roof.update({"bound": "hbm", "achieved": hbm_gbs, "peak": peak, "unit": "GB/s", "frac": hbm_frac})
    else:  # no capture of this kernel on this workload: only the byte model can be stated
        roof.update({"bound": "hbm", "achieved": algorithmic_gbs, "peak": peak, "unit": "GB/s", "frac": algorithmic_gbs / peak,
                     "traffic": None, "note": "no ncu capture for this kernel/workload: frac is the ALGORITHMIC byte model"})

    # ---- the whole frame against the same two peaks: every stage's instructions and DRAM traffic (ncu, per item) x the
    # items it processed, over the frame's device time — the figure that sees what overlapping the batches buys ----------------
    frame_inst = frame_bytes = 0.0
    frame_cover = 0.0
    for st_name, n_items in stage_items.items():
        per, _ = ncu_kernel_summary(st_name, workload, pipeline)
        if per is not None and n_items:
            frame_inst += per["thread_inst_per_item"] * n_items / stage_steps
            frame_bytes += per["dram_bytes_per_item"] * n_items / stage_steps
            frame_cover += stage_ms.get(st_name, 0.0)
    if frame_inst > 0 and total_ms > 0:
        frame_s = total_ms / steps / 1e3
        roof["frame"] = {"thread_inst_per_frame": frame_inst * world, "dram_bytes_per_frame": frame_bytes * world,
                         "issue_frac": frame_inst / frame_s / 1e9 / issue_peak, "hbm_frac": frame_bytes / frame_s / 1e9 / peak,
                         "kernels_covered_by_ncu_summaries": frame_cover / kernel_ms if kernel_ms else None,
                         "what": "all stages' thread instructions / DRAM bytes (ncu per-item figures x this rank's items) over the "
                                 "timed frame's duration, per GPU: with batches overlapping, the frame — not a launch — is what has a duration"}

    steps_s = total_ms / 1e3
    batch_note = ("SM-local wavefront: path state lives in shared memory; every step writes 16 B per path of radiance samples "
                  f"({paths * 16 / 1e9:.1f} GB) and the accumulators, far above the 126 MB L2 — no explicit flush"
                  if pipeline == "smwave" else
                  "no explicit flush: every batch streams its wavefront state (2^24 slots x 256 B = 4.3 GB) and queues through "
                  "HBM, far above the 126 MB L2; up to 4 batches are in flight at once (SPCU_OPT_BATCH_LANES)")
    return {
        "value": paths * steps / steps_s / 1e6, "unit": "Mpaths/s", "ms_per_step": total_ms / steps, "steps": steps,
        "warmup": warmup,
        "config": {"workload": workload, "scene": scene_name, "width": w, "height": h, "spp": spp_total,
                   "spp_per_gpu": spp_rank, "integrator": INTEGRATOR, "pipeline": pipeline,
                   "traversal": "exact" if ctx.traversal_exact else "ordered", "max_depth": flat.head["max_depth"],
                   "rr_depth": flat.head["rr_depth"], "primitives": int(flat.n_prims), "paths_per_step": int(paths),
                   "partition": f"sample ranges x{world} of one frame, scene replicated", "l2": batch_note,
                   "batch_lanes": 1 if pipeline == "smwave" else (args.batch_lanes or "library default (4 batches in flight, event-ordered resolve)")},
        "mrays_per_s": (rays_closest + rays_any) * steps / steps_s / 1e6,
        "rays": {"closest_per_path": rays_closest / paths, "any_hit_per_path": rays_any / paths,
                 "lights_accel_per_path": rays_lights / paths},
        "e2e": {"value": paths * e2e_steps / e2e_s / 1e6, "unit": "Mpaths/s", "h2d_bytes_per_step": scene_bytes,
                "d2h_bytes_per_step": acc_bytes, "steps": e2e_steps, "mean_radiance_of_the_frame": e2e_sanity,
                "call": ("spcu_upload_scene + spcu_render_frame" if world == 1 else
                         "spcu_upload_scene + spcu_render_frame_reduced (NCCL inside the library, ONE frame on rank 0)") +
                        " (host buffers, page-locked result)"},
        "gpu_launches": int(launches / world * steps),
        "clocks": clocks,
        "roofline": roof,
        "stages_ms_per_step": {k: v / stage_steps for k, v in stage_ms.items() if stage_launches.get(k)},
        "_flat": flat,
        **({"_outputs": outputs} if outputs is not None else {}),
    }


def dump_outputs(directory: Path, outputs: dict, limit: int = 64 << 20) -> None:
    """Writes each output as <directory>/<name>.npy.  Outputs larger than `limit` in all (the 4K frames) are written as the
    same seeded sample of pixels for every array, with that sample's flat pixel indices as pixel_index.npy."""
    directory.mkdir(parents=True, exist_ok=True)
    total = sum(a.nbytes for a in outputs.values())
    if total > limit:
        h, w = outputs["lum_sumsq"].shape
        keep = (limit - 4096) // (total // (h * w) + 8)   # bytes per pixel of the outputs and of its float64 index; .npy headers
        pick = np.sort(np.random.default_rng(0).choice(h * w, keep, replace=False))
        n_pix = h * w
        outputs = {k: a.reshape(n_pix, *a.shape[2:])[pick] for k, a in outputs.items()}
        outputs["pixel_index"] = pick.astype(np.float64)
    for name, a in outputs.items():
        np.save(directory / f"{name}.npy", np.ascontiguousarray(a))


def ordered_walk_report(ctx, flat) -> dict:
    """The render's default extend stage walks nearer-child-first; its answers may differ from the reference-order walk on
    epsilon ties only.  Counted here on 2^18 camera rays + 2^18 random rays of the resident scene, both through the renderer's
    own stage kernels (spcu_extend_batch)."""
    from simplepath_b200 import capi
    sys.path.insert(0, str(ROOT / "tests"))
    import raybatches
    n = 1 << 18
    k = np.arange(n, dtype=np.uint64)
    cam = ctx.generate_rays((k * (flat.width * flat.height) // n).astype(np.uint32), np.zeros(n, dtype=np.uint32))
    rays = np.concatenate([cam, raybatches.random_rays(flat, n, seed=12345)])
    exact, _ = ctx.extend_batch(rays, capi.TRAVERSAL_EXACT)
    fast, _ = ctx.extend_batch(rays, capi.TRAVERSAL_ORDERED)
    bad = exact["id"] != fast["id"]
    return {"rays": int(rays.shape[0]), "id_mismatches": int(bad.sum()),
            "t_mismatches_where_ids_agree": int(((exact["t"] != fast["t"]) & ~bad).sum()),
            "what": "spcu_extend_batch EXACT vs ORDERED: 2^18 camera + 2^18 random rays (seed 12345)"}


# =====================================================================================================================
def run_cuda(args) -> None:
    import torch
    import torch.distributed as dist
    from simplepath_b200 import capi, distributed
    if not capi.LIB_PATH.exists() and int(os.environ.get("LOCAL_RANK", "0")) == 0:
        import __graft_entry__   # the library normally travels with the snapshot; build it here if it did not
        __graft_entry__.build()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    ctx = capi.Context(local_rank)
    ctx.traversal_exact = args.traversal == "exact"
    ctx.set_option(capi.OPT_PIPELINE, {"auto": capi.PIPELINE_AUTO, "smwave": capi.PIPELINE_SMWAVE, "paths": capi.PIPELINE_PATHS,
                                       "wavefront": capi.PIPELINE_WAVEFRONT}[args.pipeline])
    ctx.set_option(capi.OPT_TRAVERSAL, capi.TRAVERSAL_EXACT if ctx.traversal_exact else capi.TRAVERSAL_ORDERED)
    ctx.set_option(capi.OPT_BATCH_LANES, args.batch_lanes)
    ctx.set_wavefront_size(args.wavefront_size)
    distributed.init_product_comm(ctx)   # libspcu's own NCCL communicator (torch.distributed only carries the unique id)

    spp_total = args.spp or WORKLOADS[args.workload][1]
    main = measure(ctx, args, args.workload, spp_total, args.steps, args.warmup, world, rank, clocks_index=local_rank,
                   e2e_steps=max(1, min(args.steps, 3)), keep_outputs=args.dump_outputs is not None)
    if rank == 0 and args.dump_outputs is not None:
        dump_outputs(Path(args.dump_outputs), main.pop("_outputs"))
    side: dict[str, dict] = {}
    if world > 1 and args.workload == DEFAULT_WORKLOAD and world == 8 and not args.no_side_configs:
        # BASELINE configs[4]: lucy 3840x2160 256 spp "on 8xB200" — the whole config, two timed frames.  Every rank takes
        # the same branch: a scene that cannot be loaded here must not leave the other ranks waiting in a collective.
        from simplepath_b200 import host
        if host.loadable("c5_lucy_standin"):
            r = measure(ctx, args, "lucy_4k_256spp", 256, 2, 3, world, rank, e2e_steps=1)
            if rank == 0:
                r.pop("_flat")
                side["c5_lucy_4k_256spp_8gpu"] = r
        elif rank == 0:
            side["c5_lucy_4k_256spp_8gpu"] = {"error": "c5_lucy_standin needs the reference's parser (libsphost.so), "
                                                       "which is not built"}
    if rank != 0:
        ctx.close()
        if world > 1:
            dist.destroy_process_group()
        return

    flat = main.pop("_flat")
    scene_name = main["config"]["scene"]
    ordered = ordered_walk_report(ctx, flat) if not ctx.traversal_exact and flat.n_nodes else None
    cpu = cpu_baseline(scene_name) if world == 1 and not args.no_cpu else None

    if world == 1 and args.workload == DEFAULT_WORKLOAD and not args.no_side_configs:
        # the other BASELINE configs, short: (workload, spp of the frame rendered here, timed steps)
        for key, wl, spp, k in (("c1_material_spheres_256_16spp", "material_spheres_256_16spp", 16, 5),
                                ("c2_example_scene_1080p_64spp", "example_scene_1080p_64spp", 64, 5),
                                ("c4_elf_1080p_256spp", "elf_1080p_256spp", 256, 2),
                                ("c5_lucy_4k_8spp_sample_of_256", "lucy_4k_256spp", 8, 2)):
            try:
                gc.collect()   # the previous config's host-side scene (lucy: 2.8 GB) goes before the next one is built
                r = measure(ctx, args, wl, spp, k, 3, 1, 0, e2e_steps=2 if wl == "lucy_4k_256spp" else 1)
                sflat = r.pop("_flat")
                if sflat.n_nodes and not ctx.traversal_exact:
                    r["ordered_walk"] = ordered_walk_report(ctx, sflat)
                del sflat
                if not args.no_cpu and wl != "lucy_4k_256spp":
                    r["cpu_baseline"] = cpu_baseline(WORKLOADS[wl][0], budget_s=8.0)
                side[key] = r
            except Exception as e:  # a side config must never cost the headline line
                side[key] = {"error": f"{type(e).__name__}: {e}"}

    line = {
        "metric": "Mpaths/s", "value": main["value"], "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": main["config"],
        "mrays_per_s": main["mrays_per_s"], "rays": main["rays"], "e2e": main["e2e"], "gpu_launches": main["gpu_launches"],
        "clocks": main["clocks"], "roofline": main["roofline"], "stages_ms_per_step": main["stages_ms_per_step"],
        "ordered_walk": ordered, "cpu_baseline": cpu, "configs": side,
        "construction_side": construction_side(ctx) if world == 1 and not args.no_cpu else None,
    }
    emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def construction_side(ctx) -> dict:
    """Outside the timed region and not part of `value`: the steps either side of the path (SURVEY.md §8(f)) on a bounded
    synthetic input, device-timed — BVHAccelerator::construct (spcu_build_bvh), read_ply's normal passes + Mesh's constructor
    (spcu_ingest_mesh) — and the same inputs through the oracle's sequential restatement on one host core."""
    from oracle import port
    from simplepath_b200 import scenes
    n = 1_000_000
    rng = np.random.default_rng(5)
    c = rng.random((n, 3), dtype=np.float32) * np.float32(100.0)
    h = rng.random((n, 3), dtype=np.float32) * np.float32(0.05)
    boxes = np.concatenate([c - h, c + h], axis=1)
    ctx.build_bvh(boxes)  # warm-up (allocations, kernel load)
    built = ctx.build_bvh(boxes)
    t0 = time.perf_counter()
    want = port.build_bvh(boxes)
    cpu_build_ms = (time.perf_counter() - t0) * 1e3
    v, f = scenes.bumpy_sphere(n, (-0.1, 0.03, -0.06), (0.06, 0.19, 0.06))
    v, f = np.asarray(v, dtype=np.float32), np.asarray(f, dtype=np.uint32)
    xf = np.array([10, 0, 0, 0, 10, 0, 0, 0, 10, 0, 0, 0], dtype=np.float32)
    nxf = np.array([0.1, 0, 0, 0, 0.1, 0, 0, 0, 0.1], dtype=np.float32)
    ctx.ingest_mesh(v, f, xf, nxf)
    ingested = ctx.ingest_mesh(v, f, xf, nxf)
    t0 = time.perf_counter()
    want_mesh = port.ingest_mesh(v, f, xf, nxf)
    cpu_ingest_ms = (time.perf_counter() - t0) * 1e3
    return {
        "bvh_build": {"primitives": n, "device_ms": built["device_ms"], "internal_nodes": built["head"]["n_nodes"],
                      "oracle_port_ms_1_core": cpu_build_ms,
                      "identical_to_oracle": bool(built["nodes"].tobytes() == want["nodes"].tobytes()
                                                  and np.array_equal(built["order"], want["order"]))},
        "mesh_ingest": {"faces": int(len(f)), "vertices": int(len(v)), "device_ms": ingested["device_ms"],
                        "oracle_port_ms_1_core": cpu_ingest_ms,
                        "positions_identical_to_oracle": bool(ingested["prims"].tobytes() == want_mesh["prims"].tobytes())},
    }


# =====================================================================================================================
# the reference's own CPU implementation
# =====================================================================================================================
def ref_binary() -> Path | None:
    p = ROOT / "oracle" / "_ref" / "SimplePath"
    return p if p.exists() else None


def run_reference_binary(scene_path: Path, spp: int, threads: int, timeout: float) -> float:
    """Stock reference executable; render seconds from its own Stopwatch line (main.cpp:138-141).  The process hangs at
    exit (AccumulatedLogger), so it is killed as soon as the line is seen."""
    proc = subprocess.Popen(["stdbuf", "-o0", str(ref_binary()), "--threads", str(threads), "--samples", str(spp),
                             "--integrator", INTEGRATOR, scene_path.name],
                            cwd=scene_path.parent, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    deadline = time.time() + timeout
    secs, buf = None, ""
    try:
        while time.time() < deadline:
            ch = proc.stdout.read(1)
            if not ch:
                break
            buf += ch
            m = re.search(r"Elapsed time:\s*([^\n]+)\n", buf)
            if m:
                secs = parse_elapsed(m.group(1))
                break
    finally:
        proc.kill()
        proc.wait()
    if secs is None:
        raise RuntimeError(f"reference did not finish within {timeout}s: {buf[-300:]}")
    return secs


def parse_elapsed(text: str) -> float:
    """Stopwatch::print (base/Stopwatch.h:47-60) writes HH:MM:SS.cc (centiseconds)."""
    m = re.fullmatch(r"\s*(\d+):(\d+):(\d+)\.(\d+)\s*", text)
    if not m:
        raise ValueError(f"cannot parse elapsed time {text!r}")
    hh, mm, ss, cc = (int(g) for g in m.groups())
    return hh * 3600.0 + mm * 60.0 + ss + cc / 100.0


def reference_sample(scene_name: str, budget_s: float):
    """Bounded sample of the workload for the CPU: same scene and resolution, reduced spp (throughput is spp independent,
    SURVEY.md §8d), sized from a 1 spp probe to about `budget_s` seconds per run."""
    from simplepath_b200 import scenes
    path = scenes.ensure(scene_name)
    w, h, spp_full = scenes.info(scene_name)
    threads = os.cpu_count() or 1
    probe = run_reference_binary(path, 1, threads, 600)
    spp = int(max(1, min(spp_full, budget_s / max(probe, 1e-3))))
    return path, w, h, spp, threads, probe


def cpu_baseline(scene_name: str, budget_s: float = 15.0) -> dict:
    """Reference CPU path on this box's host cores, bounded sample.  kind 'reference' = the compiled reference binary;
    'port' = the oracle's C restatement when that binary is not present."""
    threads = os.cpu_count() or 1
    if ref_binary() is not None:
        path, w, h, spp, threads, probe = reference_sample(scene_name, budget_s)
        secs = run_reference_binary(path, spp, threads, 900) if spp > 1 else probe
        return {"value": w * h * spp / secs / 1e6, "unit": "Mpaths/s", "cores": threads, "kind": "reference",
                "sample": f"{scene_name} {w}x{h} at {spp} spp ({w * h * spp} paths, {secs:.2f} s), stock binary "
                          f"--threads {threads} --integrator {INTEGRATOR}, its own Stopwatch"}
    from oracle import port
    from simplepath_b200 import host
    from simplepath_b200.capi import INTEGRATORS, Partition
    flat = host.workload(scene_name)
    spp = 1
    jitter = host.jitter(spp)
    t0 = time.perf_counter()
    _, _, st = port.render(flat.pointer(), jitter, Partition(0, 1, 0, spp, spp, INTEGRATORS[INTEGRATOR], 0), threads=threads)
    secs = time.perf_counter() - t0
    return {"value": st["paths"] / secs / 1e6, "unit": "Mpaths/s", "cores": threads, "kind": "port",
            "sample": f"{scene_name} at {spp} spp ({st['paths']} paths, {secs:.2f} s), oracle C restatement, OpenMP"}


def run_reference(args) -> None:
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores, on the cuda arm's
    config, metric and unit.  Every one of the K steps (after W warm-up steps) is a bounded SAMPLE of the workload's frame —
    same scene, resolution and integrator, `spp_sample` samples per pixel instead of the frame's, sized from a 1 spp probe so
    that K + W steps end within a few minutes (a whole 256 spp bunny frame takes the reference ~9 minutes on 16 cores).
    Mpaths/s is normalised by the paths actually rendered."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from simplepath_b200 import scenes
    scene_name, spp_full = WORKLOADS[args.workload]
    spp_full = args.spp or spp_full
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    w, h, _ = scenes.info(scene_name)
    n_runs = args.steps + args.warmup
    if ref_binary() is not None:
        path, w, h, spp, threads, _ = reference_sample(scene_name, budget_s=max(1.0, 150.0 / max(n_runs, 1)))
        spp = min(spp, spp_full)
        kind = "reference"

        def one():
            return run_reference_binary(path, spp, threads, 900)
    else:
        from oracle import port
        from simplepath_b200 import host
        from simplepath_b200.capi import INTEGRATORS, Partition
        flat = host.workload(scene_name)
        spp, threads, kind = 1, os.cpu_count() or 1, "port"
        jitter = host.jitter(spp)

        def one():
            t0 = time.perf_counter()
            port.render(flat.pointer(), jitter, Partition(0, 1, 0, spp, spp, INTEGRATORS[INTEGRATOR], 0), threads=threads)
            return time.perf_counter() - t0
    for _ in range(args.warmup):
        one()
    secs = [one() for _ in range(args.steps)]
    paths = w * h * spp
    value = paths * args.steps / sum(secs) / 1e6
    sample = (f"every step = {scene_name} {w}x{h} at {spp} spp ({paths} paths; the workload's frame is {spp_full} spp), "
              f"{'stock reference binary, its own Stopwatch' if kind == 'reference' else 'oracle C restatement'}, {threads} threads")
    emit({
        "impl": "reference", "metric": "Mpaths/s", "value": value, "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(secs) / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "scene": scene_name, "width": w, "height": h, "spp": spp_full,
                   "integrator": INTEGRATOR},
        "cpu_baseline": {"value": value, "unit": "Mpaths/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


_REAL_STDOUT = None


def claim_stdout() -> None:
    """stdout carries exactly ONE JSON line: everything libraries print (NCCL's version banner, torchrun notices)
    goes to stderr instead; emit() writes the line to the real stdout."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict) -> None:
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main() -> None:
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--spp", type=int, default=0, help="override the samples per pixel of the frame (all GPUs together)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / construction_side legs")
    ap.add_argument("--no-side-configs", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--traversal", default="ordered", choices=["exact", "ordered"],
                    help="closest-hit walk of the extend stage (SPCU_OPT_TRAVERSAL; the library's default is ordered)")
    ap.add_argument("--pipeline", default="auto", choices=["auto", "smwave", "paths", "wavefront"],
                    help="kernel organisation (SPCU_OPT_PIPELINE); same estimator and random numbers either way")
    ap.add_argument("--batch-lanes", type=int, default=0,
                    help="wavefront batches in flight at once (SPCU_OPT_BATCH_LANES; 0 = the library's default, 4)")
    ap.add_argument("--wavefront-size", type=int, default=0, help="slots per wavefront batch (spcu_set_wavefront_size; 0 = default 2^24)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline workload's per-pixel sums of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "cuda":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl cuda")
    if args.warmup < 3 and args.impl == "cuda":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
