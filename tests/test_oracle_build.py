"""BVH construction (BVHAccelerator::construct, reference shapes/BVHAccelerator.h:175-209): the oracle's sequential
restatement against trees the REAL reference built (tests/golden/bvh_build.npz, made by tests/golden/make_golden_bvh.py
with the reference's own BVHAccelerator), against the BVHs inside the golden scenes, and — where the reference libraries
exist — against the live reference on fresh inputs."""
import numpy as np
import pytest

from conftest import GOLDEN
from simplepath_b200.capi import NODE_DTYPE
from simplepath_b200.flat import FlatSceneData
import bvhcases

HEAD_KEYS = ("n_prims", "n_unbounded", "n_nodes", "root", "root_count", "max_depth")


def golden_build(name: str) -> dict:
    with np.load(GOLDEN / "bvh_build.npz") as z:
        return {"nodes": z[f"{name}.nodes"].reshape(-1).view(NODE_DTYPE), "order": z[f"{name}.order"],
                "head": dict(zip(HEAD_KEYS, (int(v) for v in z[f"{name}.head"]))), "root_bounds": z[f"{name}.root_bounds"]}


def scene_bvh(name: str):
    """(bounded triangles' records in leaf order, reference-built nodes, accel head) of a golden mesh scene."""
    flat = FlatSceneData.load(GOLDEN / f"{name}.flat.npz")
    head = flat.head["geom"]
    nu = head["n_unbounded"]
    meta = flat.arrays["geom_meta"].view(np.uint32).reshape(-1)
    assert ((meta[nu:] & 3) == 0).all(), "bounded primitives of this scene are all triangles"
    tris = flat.arrays["geom_prims"].view(np.float32).reshape(-1, 12)[nu:]
    return tris, flat.arrays["geom_nodes"].reshape(-1).view(NODE_DTYPE), head


CASES = bvhcases.cases()


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_build_matches_reference_trees(oracle_port, name):
    bounds, non_tri, first_id = CASES[name]
    want = golden_build(name)
    got = oracle_port.build_bvh(bounds, non_tri, first_id)
    assert not bvhcases.same(got, want), bvhcases.same(got, want)
    assert got["root_bounds"].tobytes() == want["root_bounds"].tobytes()
    assert sorted(got["order"].tolist()) == list(range(len(bounds)))


@pytest.mark.parametrize("name", ["g_bunny", "g_elf"])
def test_oracle_triangle_bounds_match_reference(oracle_port, name):
    tris, _, head = scene_bvh(name)
    want = np.load(GOLDEN / f"{name}.bounds.npz")["bounds"][head["n_unbounded"]:]
    assert oracle_port.triangle_bounds(tris).tobytes() == want.tobytes()


@pytest.mark.parametrize("name", ["g_bunny", "g_elf"])
def test_oracle_rebuilds_the_scene_bvh(oracle_port, name):
    """Hoare's partition does not move an already partitioned range, so construction from the leaf order is a fixed point:
    it must give back, bit for bit, the nodes the reference built when it parsed the scene."""
    tris, nodes, head = scene_bvh(name)
    got = oracle_port.build_bvh(oracle_port.triangle_bounds(tris), None, head["n_unbounded"])
    assert got["head"] == head
    assert got["nodes"].tobytes() == nodes.tobytes()
    assert np.array_equal(got["order"], np.arange(len(tris)))


def test_oracle_build_on_live_reference(oracle_port):
    from oracle import ref
    if not ref.available():
        pytest.skip("reference library not built (needs the reference sources: SP_REFERENCE, or a checkout named reference beside the repository)")
    rng = np.random.default_rng(77)
    for n in (7, 100, 4097, 60000):
        b = bvhcases.boxes(rng, n, spread=float(rng.uniform(0.1, 100)), size=float(rng.uniform(1e-4, 1.0)))
        nt = (rng.random(n) < 0.1).astype(np.uint8)
        want, got = ref.build_bvh(b, nt, 5), oracle_port.build_bvh(b, nt, 5)
        assert not bvhcases.same(got, want), (n, bvhcases.same(got, want))
