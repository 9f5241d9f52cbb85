"""Host-side pieces that need no GPU: the jitter table, flattened-scene containers, scene generators."""
import numpy as np
import pytest

from conftest import GOLDEN
from simplepath_b200 import host, rsequence, scenes
from simplepath_b200.flat import FlatSceneData


def test_jitter_table_is_the_reference_sequence_bitwise():
    want = np.load(GOLDEN / "jitter.npz")["jitter4096"]
    for spp in (1, 4, 16, 64, 256, 4096):
        got = rsequence.jitter_table(spp)
        assert got.dtype == np.float32 and got.shape == (spp, 2)
        assert got.tobytes() == want[:spp].tobytes()
    assert ((want >= 0) & (want < 1)).all()


def test_flat_scene_round_trip(tmp_path):
    flat = FlatSceneData.load(GOLDEN / "g_bunny.flat.npz")
    flat.save(tmp_path / "copy.npz")
    again = FlatSceneData.load(tmp_path / "copy.npz")
    assert again.head == flat.head
    for k in FlatSceneData.ARRAYS:
        assert again.arrays[k].tobytes() == flat.arrays[k].tobytes()
    s = again.struct()
    assert s.geom.n_prims == flat.n_prims and s.n_lights == 1


def test_flat_scene_invariants():
    """Reference-order IDs: unbounded prims first, leaves cover [n_unbounded, n_prims) exactly once, left to right."""
    for name in ("g_bunny", "g_elf"):
        flat = FlatSceneData.load(GOLDEN / f"{name}.flat.npz")
        g = flat.head["geom"]
        nodes = flat.arrays["geom_nodes"].view(np.int32).reshape(-1, 16)
        child = nodes[:, 12:14]
        count = nodes[:, 14:16].view(np.uint32) & 0x7FFFFFFF
        leaves = []

        def walk(link, cnt):
            if link < 0:
                leaves.append((~link, cnt))
                return
            for k in range(2):
                walk(int(child[link, k]), int(count[link, k]))

        walk(g["root"], g["root_count"] & 0x7FFFFFFF)
        pos = g["n_unbounded"]
        for first, cnt in leaves:
            assert first == pos
            pos += cnt
        assert pos == g["n_prims"]


@pytest.mark.parametrize("name", ["g_bunny", "g_elf"])
def test_assembled_scene_is_the_flattened_scene_bitwise(oracle_port, name):
    """host.assemble (the mesh workloads without the reference's parser) rebuilds the shells' own scenes byte for byte."""
    want = FlatSceneData.load(GOLDEN / f"{name}.flat.npz")
    got = host.assemble(name)
    assert got.head == want.head
    for k in FlatSceneData.ARRAYS:
        assert got.arrays[k].tobytes() == want.arrays[k].tobytes(), k


def test_raster_camera_across_resolutions():
    """The same camera flattened at 48x27 and at 1920x1080 (example_scene): rescaled, within 2 ulp of the parser's."""
    small = FlatSceneData.load(GOLDEN / "g_example.flat.npz")
    big = FlatSceneData.load(host.FLAT_DIR / "c2_example_scene.flat.npz")
    for a, b in ((small, big), (big, small)):
        got = np.array(host.raster_camera(a.head["camera"], a.width, a.height, b.width, b.height), dtype=np.float32)
        want = np.array(b.head["camera"], dtype=np.float32)
        assert np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32)).max() <= 2


def _fov(camera, w, h):
    """(vertical, horizontal) angle spanned by the frame's edges, and the direction through its centre."""
    c = np.asarray(camera, dtype=np.float64)
    d = lambda x, y: c[6:9] + c[0:3] * x + c[3:6] * y  # noqa: E731
    angle = lambda a, b: np.arccos(a @ b / np.linalg.norm(a) / np.linalg.norm(b))  # noqa: E731
    centre = d(w / 2, h / 2)
    return angle(d(w / 2, 0), d(w / 2, h)), angle(d(0, h / 2), d(w, h / 2)), centre / np.linalg.norm(centre)


def test_raster_camera_keeps_the_vertical_field_of_view_across_aspect_ratios():
    """The parser's cameras span the .sp fov vertically at every aspect ratio (1:1, 4:3, 16:9, 256x256 and 1080p); the
    rescaled camera of a 4:3 shell at 16:9 (c4_elf from g_elf) keeps that angle and the centre direction and widens the
    horizontal one as the aspect ratio says."""
    for path, fov in ((GOLDEN / "g_spheres.flat.npz", 45), (GOLDEN / "g_elf.flat.npz", 45), (GOLDEN / "g_bunny.flat.npz", 45),
                      (GOLDEN / "g_chain.flat.npz", 30), (host.FLAT_DIR / "c1_material_spheres_const.flat.npz", 45),
                      (host.FLAT_DIR / "c2_example_scene.flat.npz", 45)):
        s = FlatSceneData.load(path)
        assert abs(np.degrees(_fov(s.head["camera"], s.width, s.height)[0]) - fov) < 1e-4, path.name
    shell = FlatSceneData.load(GOLDEN / "g_elf.flat.npz")
    w, h, _ = scenes.info("c4_elf")
    v0, _, c0 = _fov(shell.head["camera"], shell.width, shell.height)
    v1, h1, c1 = _fov(host.raster_camera(shell.head["camera"], shell.width, shell.height, w, h), w, h)
    assert abs(v1 - v0) < 1e-6 and np.abs(c1 - c0).max() < 1e-6
    assert abs(np.tan(h1 / 2) / np.tan(v1 / 2) - w / h) < 1e-5


def test_generated_scenes_are_deterministic(tmp_path):
    a = scenes.ensure("g_bunny", tmp_path / "a")
    b = scenes.ensure("g_bunny", tmp_path / "b")
    assert a.read_text() == b.read_text()
    pa = next((tmp_path / "a").glob("*.ply")).read_bytes()
    pb = next((tmp_path / "b").glob("*.ply")).read_bytes()
    assert pa == pb
    v, f = scenes.bumpy_sphere(scenes.BUNNY_TRIS, scenes.BUNNY_LO, scenes.BUNNY_HI)
    assert f.shape == (scenes.BUNNY_TRIS, 3)


def test_scene_assets_can_be_generated_by_concurrent_ranks(tmp_path):
    """Every rank of a torchrun job calls scenes.ensure() on a fresh box: writers must not trip over each other's files."""
    import multiprocessing as mp
    with mp.get_context("spawn").Pool(6) as pool:
        texts = pool.starmap(_ensure_text, [("g_bunny", str(tmp_path))] * 6)
    assert len(set(texts)) == 1
    assert not [p for p in tmp_path.iterdir() if p.name.endswith(".tmp")]


def _ensure_text(name, out):
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
    from simplepath_b200 import scenes
    return scenes.ensure(name, out).read_text()
