"""Mesh ingest (read_ply's face / vertex-normal passes + Mesh's constructor, reference base/PlyReader.cpp:487-531,
shapes/Triangle.h:25-51): the oracle's restatement against what the reference's own read_ply produced for the committed mesh
(tests/golden/mesh_ingest.npz, made by tests/golden/make_golden_mesh.py) — bit for bit on x86, normals included."""
import numpy as np
import pytest

from conftest import GOLDEN
import meshcases


def golden():
    return np.load(GOLDEN / "mesh_ingest.npz")


def test_golden_inputs_are_the_generated_mesh():
    z = golden()
    v, f = meshcases.mesh()
    assert np.array_equal(z["in_vertices"], v) and np.array_equal(z["in_faces"], f)
    assert z["object_to_world"].tobytes() == meshcases.transform().tobytes()
    assert len(z["indices"]) < len(f), "the case must contain zero-area faces"


def test_oracle_ingest_matches_reference_mesh(oracle_port):
    z = golden()
    r = oracle_port.ingest_mesh(z["in_vertices"], z["in_faces"], z["object_to_world"], z["normal_xf"], material=3)
    assert r["world_vertices"].tobytes() == z["vertices"].tobytes()
    assert r["world_normals"].tobytes() == z["normals"].tobytes()
    idx = z["indices"]
    assert len(r["prims"]) == len(idx)
    assert np.array_equal(r["prims"].reshape(-1, 3, 4)[:, :, :3], z["vertices"][idx])
    assert np.array_equal(r["shade"].reshape(-1, 3, 4)[:, :, :3], z["normals"][idx])
    assert (r["prims"].reshape(-1, 3, 4)[:, :, 3] == 0).all() and (r["meta"] == (3 << 2)).all()


def test_oracle_ingest_on_live_reference(oracle_port, tmp_path):
    from oracle import ref
    from simplepath_b200 import scenes
    if not ref.available():
        pytest.skip("reference library not built (needs the reference sources: SP_REFERENCE, or a checkout named reference beside the repository)")
    v, f = meshcases.mesh(n_tris=20000, seed=8)
    xf = meshcases.transform(seed=12)
    scenes.write_ply(tmp_path / "m.ply", v, f)
    want = ref.read_ply(tmp_path / "m.ply", xf, len(v), len(f))
    r = oracle_port.ingest_mesh(v, f, xf, want["normal_xf"])
    assert r["world_vertices"].tobytes() == want["vertices"].tobytes()
    assert r["world_normals"].tobytes() == want["normals"].tobytes()
    assert np.array_equal(r["prims"].reshape(-1, 3, 4)[:, :, :3], want["vertices"][want["indices"]])


ACCEL_CASES = ("plane_first", "planes_around", "planes_inside", "no_plane")
HEAD_KEYS = ("n_prims", "n_unbounded", "n_nodes", "root", "root_count", "max_depth")


def golden_accel(name):
    from simplepath_b200.capi import NODE_DTYPE
    z = np.load(GOLDEN / "scene_accel.npz")
    return {"unbounded": z[f"{name}.unbounded"], "order": z[f"{name}.order"], "nodes": z[f"{name}.nodes"].reshape(-1).view(NODE_DTYPE),
            "head": dict(zip(HEAD_KEYS, (int(x) for x in z[f"{name}.head"])))}


def list_order(ingested, unbounded):
    """Parser-order list [unbounded stand-ins | the mesh's triangles in face order] -> (bounded list positions in
    pre-construction order, unbounded list positions, triangle records in pre-construction order)."""
    from simplepath_b200.flat import pre_construction_order
    bounded, unb = pre_construction_order(unbounded == 0)
    triangle_of_position = np.cumsum(unbounded == 0) - 1
    return bounded, unb, {k: ingested[k][triangle_of_position[bounded]] for k in ("prims", "shade", "meta")}


@pytest.mark.parametrize("name", ACCEL_CASES)
def test_cpu_pipeline_reproduces_the_reference_scene_accelerator(oracle_port, name):
    """vertex / face lists -> oracle ingest -> std::partition(is_bounded) order -> oracle bounds + construction, against what
    the reference's own create_acceleration_structure (base/Scene.h:27-45) built over the triangles of the mesh IT read:
    the same primitive behind every ID, the same nodes, the same header."""
    z, g = golden(), golden_accel(name)
    ing = oracle_port.ingest_mesh(z["in_vertices"], z["in_faces"], z["object_to_world"], z["normal_xf"])
    bounded, unb, rec = list_order(ing, g["unbounded"])
    built = oracle_port.build_bvh(oracle_port.triangle_bounds(rec["prims"]), None, len(unb))
    assert built["head"] == g["head"]
    assert np.array_equal(np.concatenate([unb, bounded[built["order"]]]), g["order"])
    assert built["nodes"].tobytes() == g["nodes"].tobytes()


def golden_stl():
    z = np.load(GOLDEN / "mesh_ingest_stl.npz")
    v, f = meshcases.stl_index(z["corners"])
    return z, v, f


def test_stl_vertex_indexer_matches_reference():
    z, v, f = golden_stl()
    corners, stored = meshcases.stl_soup()
    assert np.array_equal(z["corners"], corners) and np.array_equal(z["stored_normals"], stored)
    assert np.array_equal(f, z["indices"]) and len(v) == len(z["vertices"])


def test_oracle_stl_ingest_matches_reference_mesh(oracle_port):
    """read_binary_stl (base/STLReader.cpp:60-137): stored normals, zero normals replaced by the cross product, faces whose
    normal is_zero by the 1e-5 epsilon kept in the mesh without a contribution."""
    z, v, f = golden_stl()
    r = oracle_port.ingest_mesh_stl(v, f, z["stored_normals"], z["object_to_world"], z["normal_xf"], material=2)
    assert len(r["prims"]) == len(f) == len(z["indices"])            # nothing is dropped on the STL path
    assert r["world_vertices"].tobytes() == z["vertices"].tobytes()
    assert r["world_normals"].tobytes() == z["normals"].tobytes()
    assert np.array_equal(r["shade"].reshape(-1, 3, 4)[:, :, :3], z["normals"][z["indices"]])
    # the case exercises the epsilon: some faces contribute nothing although their area is not exactly zero
    tri = z["corners"].astype(np.float64)
    cross = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    silent = (np.abs(z["stored_normals"]) <= 1e-5).all(axis=1) & (np.abs(cross) <= 1e-5).all(axis=1)
    assert silent.sum() > 20 and (np.linalg.norm(cross[silent], axis=1) > 0).any()


def test_small_degenerate_meshes_on_live_reference(oracle_port, tmp_path):
    """Vertex coordinates from a handful of values: collinear, coincident and repeated corners in most meshes, vertices
    whose face normals cancel exactly, vertices no face uses — PLY and STL readers of the live reference against the oracle."""
    from oracle import ref
    from simplepath_b200 import scenes
    if not ref.available():
        pytest.skip("reference library not built (needs the reference sources: SP_REFERENCE, or a checkout named reference beside the repository)")
    rng = np.random.default_rng(123)
    values = np.array([0.0, 1.0, -1.0, 0.5, 2.0], dtype=np.float32)
    xf = meshcases.transform(seed=21)
    for trial in range(60):
        nv, nf = int(rng.integers(3, 12)), int(rng.integers(1, 30))
        v = values[rng.integers(0, len(values), (nv, 3))]
        f = rng.integers(0, nv, (nf, 3)).astype(np.uint32)
        scenes.write_ply(tmp_path / "m.ply", v, f)
        want = ref.read_ply(tmp_path / "m.ply", xf, nv, nf)
        got = oracle_port.ingest_mesh(v, f, xf, want["normal_xf"])
        assert len(got["prims"]) == len(want["indices"]), trial
        assert got["world_vertices"].tobytes() == want["vertices"].tobytes(), trial
        assert got["world_normals"].tobytes() == want["normals"].tobytes(), trial
        assert np.array_equal(got["prims"].reshape(-1, 3, 4)[:, :, :3], want["vertices"][want["indices"]]), trial
        # the same triangles as an STL: soup + stored normals (a third of them zero)
        corners = v[f.astype(np.int64)]
        stored = rng.normal(size=(nf, 3)).astype(np.float32)
        stored[rng.random(nf) < 0.34] = 0.0
        meshcases.write_stl(tmp_path / "m.stl", corners, stored)
        want = ref.read_ply(tmp_path / "m.stl", xf, 3 * nf, nf)
        sv, sf = meshcases.stl_index(corners)
        assert np.array_equal(sf, want["indices"]), trial
        got = oracle_port.ingest_mesh_stl(sv, sf, stored, xf, want["normal_xf"])
        assert got["world_vertices"].tobytes() == want["vertices"].tobytes(), trial
        assert got["world_normals"].tobytes() == want["normals"].tobytes(), trial
