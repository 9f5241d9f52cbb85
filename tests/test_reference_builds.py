"""Against the LIVE reference (oracle/_ref/libsp_ref*.so, compiled from /root/reference by oracle/Makefile; skipped where
those libraries are absent): the oracle's restatement on a larger scene than the golden ones, and the noise floor between
the canonical build (-ffp-contract=off) and GCC's default contraction, which the reference's CMake flags would produce
(SURVEY.md §0.6, §8c)."""
import numpy as np
import pytest

from oracle import ref
from simplepath_b200 import scenes
from simplepath_b200.flat import FlatSceneData
import raybatches

pytestmark = pytest.mark.skipif(not (ref.available(ref.STRICT) and ref.available(ref.FAST)),
                                reason="reference libraries not built (needs the reference sources: SP_REFERENCE, or a checkout named reference beside the repository)")


@pytest.fixture(scope="module")
def bunny():
    path = scenes.ensure("t_bunny")
    strict = ref.RefScene(path, ref.STRICT)
    fast = ref.RefScene(path, ref.FAST)
    yield strict, fast
    strict.close()
    fast.close()


def test_oracle_restatement_on_live_reference(oracle_port, bunny):
    strict, _ = bunny
    flat = FlatSceneData.from_struct(strict.flat())
    for name, rays in raybatches.all_batches(flat, 1 << 14).items():
        want, cnt = strict.trace_closest(rays, counters=True)   # asserts walk == Scene::intersect internally
        got, got_cnt = oracle_port.trace_closest(flat.pointer(), rays, counters=True)
        assert np.array_equal(got["id"], want["id"]), name
        assert got["t"].tobytes() == want["t"].tobytes(), name
        assert np.array_equal(cnt, got_cnt), name
        assert np.array_equal(oracle_port.trace_any(flat.pointer(), rays), strict.trace_any(rays)), name


@pytest.mark.parametrize("scene_name", ["t_bunny", "t_spheres_const", "t_example"])
def test_noise_floor_between_reference_builds(scene_name):
    """How much the reference disagrees WITH ITSELF across compiler contraction settings: the floor below which a
    mismatch says nothing about an implementation.  Printed; bounded loosely.  Triangles use explicit madd/msub and do
    not move; the sphere's `b*b - 4ac` (shapes/Sphere.h:88) is what GCC contracts."""
    path = scenes.ensure(scene_name)
    strict, fast = ref.RefScene(path, ref.STRICT), ref.RefScene(path, ref.FAST)
    flat = FlatSceneData.from_struct(strict.flat())
    total = ids = ts = 0
    for name, rays in raybatches.all_batches(flat, 1 << 14).items():
        a = strict.trace_closest(rays)
        b = fast.trace_closest(rays)
        total += rays.shape[0]
        ids += int((a["id"] != b["id"]).sum())
        ts += int((a["t"].view(np.uint32) != b["t"].view(np.uint32)).sum())
    strict.close()
    fast.close()
    print(f"\n{scene_name}: reference strict vs default-contraction build: {ids} ID mismatches, {ts} distance-bit mismatches of {total} rays")
    assert ids <= total // 500
