"""The render entry points against each other, and the context's shared scratch across calls.

spcu_render_device (on the legacy default stream and on a stream of its own), spcu_render_frame_reduced without a
communicator and spcu_render_adaptive_device compute, bit for bit, what their host-buffer counterparts compute.  Every call
borrows the context's wavefront state, queues and counters: a render on a side stream followed at once by one on the
context's stream, and ray batches through the render's stages between renders of other batch shapes and lane counts, must
each give what they give alone.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from simplepath_b200 import capi, rsequence
from simplepath_b200.flat import FlatSceneData

pytestmark = pytest.mark.gpu
PIPELINES = {"smwave": capi.PIPELINE_SMWAVE, "paths": capi.PIPELINE_PATHS, "wavefront": capi.PIPELINE_WAVEFRONT}
SPP = 32
STATS = ("paths", "rays_closest", "rays_any", "rays_lights")


@pytest.fixture
def clean(ctx):
    """The session context, with the options these tests change restored afterwards."""
    yield ctx
    ctx.set_option(capi.OPT_PIPELINE, capi.PIPELINE_AUTO)
    ctx.set_option(capi.OPT_BATCH_LANES, 0)
    ctx.set_wavefront_size(0)


def upload(ctx, name, pipeline=capi.PIPELINE_WAVEFRONT):
    flat = FlatSceneData.load(GOLDEN / f"{name}.flat.npz")
    ctx.set_option(capi.OPT_PIPELINE, pipeline)
    ctx.set_wavefront_size(0)
    ctx.upload_scene(flat.pointer(), rsequence.jitter_table(SPP), keepalive=flat)


def device_buffers(ctx):
    rgb = torch.zeros((ctx.height, ctx.width, 3), dtype=torch.float32, device="cuda")
    sq = torch.zeros((ctx.height, ctx.width), dtype=torch.float32, device="cuda")
    return rgb, sq


@pytest.mark.parametrize("where", ["legacy_default_stream", "side_stream"])
@pytest.mark.parametrize("pipeline", PIPELINES)
def test_render_device_equals_render(clean, pipeline, where):
    ctx = clean
    upload(ctx, "g_bunny", PIPELINES[pipeline])
    part = ctx.partition(seed=41, rank=1, world=3)
    want, want_sq, st_w = ctx.render(part)
    rgb, sq = device_buffers(ctx)
    stream = None
    if where == "side_stream":
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())  # (the buffers were zeroed there)
    st_g = ctx.render_device(part, rgb.data_ptr(), sq.data_ptr(), stream.cuda_stream if stream else None)
    torch.cuda.synchronize()
    assert rgb.cpu().numpy().tobytes() == want.tobytes() and sq.cpu().numpy().tobytes() == want_sq.tobytes()
    assert all(st_g[k] == st_w[k] for k in STATS), (st_g, st_w)


def test_render_device_then_host_render_without_sync(clean):
    """A render enqueued on a side stream still holds the context's scratch when a host-buffer render starts on the context's
    own stream: the second must wait for the first (and rebuild the pixel list of its partition only after it)."""
    ctx = clean
    upload(ctx, "g_bunny")
    ctx.set_wavefront_size(777)  # a long chain of batches over the lanes
    a, b = ctx.partition(seed=1), ctx.partition(seed=2, rank=1, world=2)
    want_a, want_a_sq, _ = ctx.render(a)
    want_b, want_b_sq, _ = ctx.render(b)
    rgb, sq = device_buffers(ctx)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        torch.cuda._sleep(100_000_000)  # the device render is still queued when the host-buffer render is issued
    ctx.render_device(a, rgb.data_ptr(), sq.data_ptr(), side.cuda_stream, want_stats=False)  # enqueue only
    got_b, got_b_sq, _ = ctx.render(b)
    torch.cuda.synchronize()
    assert rgb.cpu().numpy().tobytes() == want_a.tobytes() and sq.cpu().numpy().tobytes() == want_a_sq.tobytes()
    assert got_b.tobytes() == want_b.tobytes() and got_b_sq.tobytes() == want_b_sq.tobytes()


@pytest.mark.parametrize("with_sumsq", [True, False])
def test_frame_reduced_without_communicator_equals_frame(clean, with_sumsq):
    ctx = clean
    upload(ctx, "g_bunny")
    part = ctx.partition(seed=9)
    want, want_sq, st_w = ctx.render_frame(part, want_sumsq=with_sumsq)
    got, got_sq, st_g = ctx.render_frame_reduced(part, want_sumsq=with_sumsq)
    assert got.tobytes() == want.tobytes()
    assert (got_sq is None and want_sq is None) if not with_sumsq else got_sq.tobytes() == want_sq.tobytes()
    assert all(st_g[k] == st_w[k] for k in STATS), (st_g, st_w)


@pytest.mark.parametrize("pipeline", PIPELINES)
def test_render_adaptive_device_equals_render_adaptive(clean, pipeline):
    ctx = clean
    upload(ctx, "g_bunny", PIPELINES[pipeline])
    part = ctx.partition(seed=17)
    kw = dict(min_spp=4, pass_spp=4, abs_floor=1e-3)
    # the target error whose map holds the most distinct sample counts: pixels stop in several passes
    runs = [(e, ctx.render_adaptive(part, e, **kw)) for e in (1.0, 0.5, 0.3, 0.2, 0.1, 0.05, 0.02, 0.01)]
    rel, (want, want_sq, want_map, st_w) = max(runs, key=lambda r: len(np.unique(r[1][2])))
    assert len(np.unique(want_map)) >= 3, np.unique(want_map)

    rgb, sq = device_buffers(ctx)
    spp_map = torch.zeros((ctx.height, ctx.width), dtype=torch.int32, device="cuda")
    ad, passes, st = capi.Adaptive(kw["min_spp"], kw["pass_spp"], rel, kw["abs_floor"]), C.c_uint32(), capi.Stats()
    ctx._check(ctx.lib.spcu_render_adaptive_device(ctx.h, C.byref(part), C.byref(ad), C.c_void_p(rgb.data_ptr()),
                                                   C.c_void_p(sq.data_ptr()), C.c_void_p(spp_map.data_ptr()), C.byref(passes),
                                                   C.byref(st), None), "spcu_render_adaptive_device")
    torch.cuda.synchronize()
    assert rgb.cpu().numpy().tobytes() == want.tobytes() and sq.cpu().numpy().tobytes() == want_sq.tobytes()
    assert np.array_equal(spp_map.cpu().numpy().view(np.uint32), want_map)
    assert passes.value == st_w["passes"] and all(getattr(st, k) == st_w[k] for k in STATS)


@pytest.mark.parametrize("lanes", [1, 4])
@pytest.mark.parametrize("name", ["g_bunny", "g_lights"])
def test_stage_batches_between_renders(clean, name, lanes):
    """spcu_extend_batch / spcu_shadow_batch borrow lane 0 of the render's wavefront state, laid out for their own batch
    size: between renders of the default batch shape and of 777-slot batches, everything equals its run on a fresh context."""
    ctx = clean
    vec = np.load(GOLDEN / f"{name}.vectors.npz")
    rays = np.ascontiguousarray(vec["random.rays"]).view(capi.RAY_DTYPE).reshape(-1)

    def render(c, size):
        c.set_wavefront_size(size)
        rgb, sq, st = c.render(c.partition(seed=13))
        return rgb.tobytes(), sq.tobytes(), [st[k] for k in STATS]

    def stage_batches(c):
        hits, lights = c.extend_batch(rays)
        return hits.tobytes(), lights.tobytes(), c.shadow_batch(rays).tobytes()

    def alone(run):
        fresh = capi.Context(0)
        try:
            upload(fresh, name)
            fresh.set_option(capi.OPT_BATCH_LANES, lanes)
            return run(fresh)
        finally:
            fresh.close()

    want = {0: alone(lambda c: render(c, 0)), 777: alone(lambda c: render(c, 777)), "batches": alone(stage_batches)}
    upload(ctx, name)
    ctx.set_option(capi.OPT_BATCH_LANES, lanes)
    for step, size in enumerate([0, 0, 777, 0, 777]):
        assert render(ctx, size) == want[size], f"render {step} (wavefront size {size})"
        assert stage_batches(ctx) == want["batches"], f"stage batches after render {step}"
