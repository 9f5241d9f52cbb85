"""Regenerates tests/golden/bvh_build.npz and tests/golden/<scene>.bounds.npz from the REAL reference
(oracle/_ref/libsp_ref.so): for every box set of tests/bvhcases.py the tree the reference's own BVHAccelerator(first, last)
(shapes/BVHAccelerator.h:123-209) builds over it, flattened like the product's flattener does (oracle/ref_harness.cpp
spref_build_bvh); and for the golden mesh scenes Hitable::get_world_bounds() of every primitive.  Development container only:

    python tests/golden/make_golden_bvh.py
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
import bvhcases  # noqa: E402

HERE = Path(__file__).resolve().parent
HEAD_KEYS = ("n_prims", "n_unbounded", "n_nodes", "root", "root_count", "max_depth")


def main() -> None:
    if not ref.available():
        raise SystemExit("oracle/_ref/libsp_ref.so missing: run `make -C oracle REF=<the reference sources>`")
    out = {}
    for name, (bounds, non_tri, first_id) in bvhcases.cases().items():
        r = ref.build_bvh(bounds, non_tri, first_id)
        out[f"{name}.nodes"] = r["nodes"].view(np.uint8).reshape(-1, 64)
        out[f"{name}.order"] = r["order"]
        out[f"{name}.head"] = np.array([r["head"][k] for k in HEAD_KEYS], dtype=np.int64)
        out[f"{name}.root_bounds"] = r["root_bounds"]
        print(name, len(bounds), r["head"])
    np.savez_compressed(HERE / "bvh_build.npz", **out)
    for name in ("g_bunny", "g_elf"):
        rs = ref.RefScene(scenes.ensure(name))
        flat = FlatSceneData.from_struct(rs.flat())
        np.savez_compressed(HERE / f"{name}.bounds.npz", bounds=rs.geom_bounds(flat.n_prims))
        rs.close()


if __name__ == "__main__":
    main()
