"""Hit-ID parity AT BASELINE SCALE (SURVEY.md §8d: "first 2^20 camera rays per scene + 2^20 random rays, seed 12345"):
the bunny scene of BASELINE.json configs[2] (277,805 primitives, BVH depth 27) and a million-triangle statue at the
lucy framing (depth > 30: past the 24 traversal-stack levels kept in shared memory), against the oracle's restatement
of the reference walk (all host cores).  Both the one-thread-per-ray query kernels (spcu_trace_*) and the renderer's
own traversal stages (spcu_extend_batch / spcu_shadow_batch: begin + persistent walk, lane refill, warp-wide leaf
steps) must return the reference's primitive IDs and distances bit for bit; the ordered walk — the render default — is
held to "epsilon ties only", counted and printed."""
import numpy as np
import pytest

from simplepath_b200 import host, rsequence
from simplepath_b200.capi import RAY_DTYPE, TRAVERSAL_EXACT, TRAVERSAL_ORDERED
import raybatches
from test_gpu_trace import extend_reference, ulp_diff

pytestmark = pytest.mark.gpu
N_RAYS = 1 << 20
SCENES = ["c3_bunny", "t_lucy_1m"]


@pytest.fixture(scope="module", params=SCENES)
def big_scene(request, ctx):
    if not host.loadable(request.param):
        pytest.skip(f"{request.param} needs the reference's parser + the flattener (libsphost.so), which is not built")
    flat = host.workload(request.param)
    jitter = rsequence.jitter_table(4)
    ctx.upload_scene(flat.pointer(), jitter, keepalive=flat)
    n_pix = flat.width * flat.height
    # camera rays spread evenly over the whole image (sample 0..3 in turn), then uniformly random rays in the scene's bounds
    k = np.arange(N_RAYS, dtype=np.uint64)
    pix = (k * n_pix // N_RAYS).astype(np.uint32)
    smp = (k % 4).astype(np.uint32)
    camera = ctx.generate_rays(pix, smp)
    rand = raybatches.random_rays(flat, N_RAYS, seed=12345)
    return request.param, flat, {"camera": camera, "random": rand}


@pytest.mark.parametrize("batch", ["camera", "random"])
def test_hit_ids_bit_exact_at_scale(ctx, oracle_port, big_scene, batch):
    name, flat, batches = big_scene
    assert flat.head["geom"]["max_depth"] > 24, "the scene must exercise the thread-local overflow stack"
    rays = batches[batch]
    want = oracle_port.trace_closest(flat.pointer(), rays)
    got = ctx.trace_closest(rays)
    assert int((got["id"] != want["id"]).sum()) == 0, f"{name}/{batch}: per-ray kernel"
    assert got["t"].tobytes() == want["t"].tobytes()
    assert (want["id"] >= flat.head["geom"]["n_unbounded"]).mean() > 0.02, "the batch must actually hit the mesh"

    # the renderer's extend stage (exact walk): lights first, then geometry under the shrunk limit
    wl = oracle_port.trace_lights(flat.pointer(), rays)
    hits, lights = ctx.extend_batch(rays, TRAVERSAL_EXACT)
    assert np.array_equal(lights["id"], wl["id"]) and lights["t"].tobytes() == wl["t"].tobytes()
    want_ext = extend_reference(flat, rays, wl["id"], wl["t"], oracle_port)
    assert int((hits["id"] != want_ext["id"]).sum()) == 0, f"{name}/{batch}: extend stage"
    assert hits["t"].tobytes() == want_ext["t"].tobytes()

    # the renderer's shadow stage = Scene::intersect_p
    assert np.array_equal(ctx.shadow_batch(rays), oracle_port.trace_any(flat.pointer(), rays)), f"{name}/{batch}: shadow stage"

    # the render default: ordered walk.  Epsilon ties only, counted.
    fast, _ = ctx.extend_batch(rays, TRAVERSAL_ORDERED)
    bad = fast["id"] != want_ext["id"]
    tied = bad & (fast["id"] >= 0) & (want_ext["id"] >= 0)
    assert ulp_diff(fast["t"][tied], want_ext["t"][tied]).max(initial=0) <= 4
    one_sided = bad & ~tied   # one walk accepts a grazing hit at the limit that the other culls with its box
    print(f"\n{name}/{batch}: ordered walk differs from the reference on {int(bad.sum())} of {rays.shape[0]} rays "
          f"({int(tied.sum())} equal-distance ties, {int(one_sided.sum())} one-sided)")
    assert bad.sum() <= rays.shape[0] // 5_000
