"""Regenerates the committed golden vectors from the REAL reference (oracle/_ref/libsp_ref.so, compiled from
/root/reference by oracle/Makefile with -ffp-contract=off).  Run in the development container only:

    python tests/golden/make_golden.py

For every tiny scene g_* of simplepath_b200.scenes it writes
    <name>.flat.npz     the flattened scene (product flattener applied to the reference's own Scene object)
    <name>.vectors.npz  ray batches and what the reference answers for them: Scene::intersect (primitive id, t),
                        Scene::intersect_p, Scene::intersect_lights, Intersection records, camera rays, the R-sequence
                        jitter table and the traversal counters of the reference walk
and, for g_spheres / g_example / g_bunny, <name>.render.npz: per-pixel mean RGB, luminance mean and variance of a
reference render (iterative_rrnee and direct_lighting, N samples) for the statistical image tests.
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from oracle import ref  # noqa: E402
from simplepath_b200 import scenes  # noqa: E402
from simplepath_b200.flat import FlatSceneData  # noqa: E402
import raybatches  # noqa: E402

HERE = Path(__file__).resolve().parent
NAMES = ["g_spheres", "g_spheres_ibl", "g_example", "g_bunny", "g_elf", "g_chain", "g_lights"]
RENDERS = {"g_spheres": 1024, "g_spheres_ibl": 1024, "g_example": 1024, "g_bunny": 1024, "g_elf": 1024, "g_chain": 1024,
           "g_lights": 1024}
N_EACH = 4096


def main() -> None:
    if not ref.available():
        raise SystemExit("oracle/_ref/libsp_ref.so missing: run `make -C oracle REF=<the reference sources>`")
    for name in (sys.argv[1:] or NAMES):   # python tests/golden/make_golden.py [scene ...]
        path = scenes.ensure(name)
        w, h, spp = scenes.info(name)
        rs = ref.RefScene(path)
        flat = FlatSceneData.from_struct(rs.flat())
        flat.save(HERE / f"{name}.flat.npz")

        out = {"jitter": rs.jitter(spp)}
        pix = np.repeat(np.arange(w * h, dtype=np.uint32), spp)
        smp = np.tile(np.arange(spp, dtype=np.uint32), w * h)
        out["cam_pix"], out["cam_smp"] = pix, smp
        cam = rs.generate_rays(pix, smp, spp)
        batches = {"camera": cam, **raybatches.all_batches(flat, N_EACH)}
        if name == "g_chain":   # deep-stack rays through the chain BVH (depth 54 > the 24 shared-memory stack levels)
            batches["cone"] = raybatches.cone_rays(N_EACH)
        for bname, rays in batches.items():
            hits, cnt = rs.trace_closest(rays, counters=True)
            out[f"{bname}.rays"] = rays.view(np.float32).reshape(-1, 8)
            out[f"{bname}.closest_id"] = hits["id"]
            out[f"{bname}.closest_t"] = hits["t"]
            out[f"{bname}.counters"] = cnt
            out[f"{bname}.any"] = rs.trace_any(rays)
            lh = rs.trace_lights(rays)
            out[f"{bname}.lights_id"] = lh["id"]
            out[f"{bname}.lights_t"] = lh["t"]
            out[f"{bname}.records"] = rs.hit_records(rays)
        np.savez_compressed(HERE / f"{name}.vectors.npz", **out)
        print(name, flat.n_prims, "prims", flat.n_nodes, "nodes",
              {b: int((out[f'{b}.closest_id'] >= 0).sum()) for b in batches})

        if name in RENDERS:
            n = RENDERS[name]
            rend = {}
            for integ in ("iterative_rrnee", "direct_lighting", "brute_force_iterative_rr", "whitted"):
                rgb, mean, var, secs = rs.render(integ, n, 8)
                rend[f"{integ}.rgb"] = rgb
                rend[f"{integ}.lum_mean"] = mean
                rend[f"{integ}.lum_var"] = var
                rend[f"{integ}.spp"] = np.array(n)
                print("  render", integ, n, "spp", f"{secs:.1f}s")
            np.savez_compressed(HERE / f"{name}.render.npz", **rend)
        rs.close()


if __name__ == "__main__":
    main()
