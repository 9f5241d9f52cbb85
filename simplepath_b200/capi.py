"""ctypes mirror of include/spcu.h and loader of the CUDA backend `libspcu.so`.

There is no CPU fallback: if the shared library (built by `__graft_entry__.build()` /
`make -C simplepath_b200/csrc`) is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent
import os
LIB_PATH = Path(os.environ.get("SPCU_LIB", PKG / "csrc" / "libspcu.so"))  # SPCU_LIB: experiments with another build

ABI_VERSION = 2
INTEGRATORS = {"iterative_rrnee": 0, "brute_force_iterative_rr": 1, "direct_lighting": 2, "whitted": 3}


class Ray(C.Structure):
    _fields_ = [("ox", C.c_float), ("oy", C.c_float), ("oz", C.c_float), ("t_min", C.c_float),
                ("dx", C.c_float), ("dy", C.c_float), ("dz", C.c_float), ("t_max", C.c_float)]


class Hit(C.Structure):
    _fields_ = [("id", C.c_int32), ("t", C.c_float)]


RAY_DTYPE = np.dtype([("o", "<f4", 3), ("t_min", "<f4"), ("d", "<f4", 3), ("t_max", "<f4")])
HIT_DTYPE = np.dtype([("id", "<i4"), ("t", "<f4")])
NODE_DTYPE = np.dtype([("box", "<f4", 12), ("child", "<i4", 2), ("count", "<u4", 2)])
BOUNDS_DTYPE = np.dtype([("lo", "<f4", 3), ("hi", "<f4", 3)])
PRIM_DTYPE = np.dtype([("v", "<f4", 12)])
assert RAY_DTYPE.itemsize == 32 and HIT_DTYPE.itemsize == 8 and NODE_DTYPE.itemsize == 64


class BvhNode(C.Structure):
    _fields_ = [("box", C.c_float * 12), ("child", C.c_int32 * 2), ("count", C.c_uint32 * 2)]


class PrimGeom(C.Structure):
    _fields_ = [("v", C.c_float * 12)]


class PrimShade(C.Structure):
    _fields_ = [("v", C.c_float * 12)]


class Accel(C.Structure):
    _fields_ = [("n_prims", C.c_uint32), ("n_unbounded", C.c_uint32), ("n_nodes", C.c_uint32),
                ("root", C.c_int32), ("root_count", C.c_uint32), ("max_depth", C.c_uint32),
                ("nodes", C.POINTER(BvhNode))]


class Bxdf(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("r", C.c_float * 3), ("alpha_x", C.c_float), ("alpha_y", C.c_float),
                ("ior", C.c_float), ("sample_visible", C.c_uint32)]


class Material(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("n_bxdfs", C.c_uint32), ("first_bxdf", C.c_uint32), ("base", C.c_uint32),
                ("ior", C.c_float), ("specular", C.c_float * 3)]


class Light(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("radiance", C.c_float * 3),
                ("world_to_object", C.c_float * 12), ("object_to_world", C.c_float * 12), ("normal_xf", C.c_float * 9),
                ("light_to_world", C.c_float * 9), ("world_to_light", C.c_float * 9),
                ("img_w", C.c_uint32), ("img_h", C.c_uint32), ("nu", C.c_uint32), ("nv", C.c_uint32),
                ("marg_integral", C.c_float), ("_pad", C.c_uint32),
                ("img_off", C.c_uint64), ("cond_func_off", C.c_uint64), ("cond_cdf_off", C.c_uint64),
                ("cond_int_off", C.c_uint64), ("marg_func_off", C.c_uint64), ("marg_cdf_off", C.c_uint64)]


class FlatScene(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32),
                ("rr_depth", C.c_uint32), ("max_depth", C.c_uint32), ("camera", C.c_float * 12),
                ("geom", Accel), ("geom_prims", C.POINTER(PrimGeom)), ("geom_shade", C.POINTER(PrimShade)),
                ("geom_meta", C.POINTER(C.c_uint32)),
                ("lights_accel", Accel), ("n_lights", C.c_uint32), ("_pad0", C.c_uint32),
                ("lights", C.POINTER(Light)), ("light_order", C.POINTER(C.c_uint32)),
                ("n_materials", C.c_uint32), ("n_bxdfs", C.c_uint32),
                ("materials", C.POINTER(Material)), ("bxdfs", C.POINTER(Bxdf)),
                ("n_pool", C.c_uint64), ("float_pool", C.POINTER(C.c_float))]


class Partition(C.Structure):
    _fields_ = [("tile_offset", C.c_uint32), ("tile_stride", C.c_uint32), ("sample_begin", C.c_uint32),
                ("sample_end", C.c_uint32), ("spp_total", C.c_uint32), ("integrator", C.c_uint32),
                ("seed", C.c_uint64)]


class Stats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("rays_closest", C.c_uint64), ("rays_any", C.c_uint64),
                ("rays_lights", C.c_uint64), ("nodes_visited", C.c_uint64), ("prims_tested", C.c_uint64),
                ("xf_prims_tested", C.c_uint64), ("shade_calls", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("device_ms", C.c_float), ("trace_ms", C.c_float), ("shade_ms", C.c_float), ("_pad", C.c_float)]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_ if not n.startswith("_")}


class Adaptive(C.Structure):
    """spcu_adaptive: parameters of spcu_render_adaptive (include/spcu.h)."""
    _fields_ = [("min_spp", C.c_uint32), ("pass_spp", C.c_uint32), ("rel_error", C.c_float), ("abs_floor", C.c_float),
                ("radius", C.c_uint32)]


class Guide(C.Structure):
    """spcu_guide: first-hit guide record of a pixel (include/spcu.h)."""
    _fields_ = [("normal", C.c_float * 3), ("depth", C.c_float), ("albedo", C.c_float * 3), ("id", C.c_int32)]


class DenoiseParams(C.Structure):
    """spcu_denoise_params: parameters of spcu_denoise (include/spcu.h)."""
    _fields_ = [("iterations", C.c_uint32), ("sigma_l", C.c_float), ("sigma_z", C.c_float), ("sigma_a", C.c_float)]


GUIDE_DTYPE = np.dtype([("normal", "<f4", 3), ("depth", "<f4"), ("albedo", "<f4", 3), ("id", "<i4")])
assert GUIDE_DTYPE.itemsize == C.sizeof(Guide) == 32
DENOISE_DEFAULTS = {"iterations": 5, "sigma_l": 8.0, "sigma_z": 0.1, "sigma_a": 0.1}  # DESIGN.md §12, profiles/r07a


class StageTime(C.Structure):
    _fields_ = [("name", C.c_char * 24), ("launches", C.c_uint64), ("items", C.c_uint64), ("ms", C.c_float),
                ("traverses", C.c_uint32)]


EXPORTS = [
    "spcu_create", "spcu_destroy", "spcu_last_error", "spcu_abi_version", "spcu_upload_scene",
    "spcu_trace_closest", "spcu_trace_any", "spcu_trace_lights", "spcu_trace_closest_fast",
    "spcu_generate_rays", "spcu_render", "spcu_render_frame", "spcu_render_device", "spcu_set_wavefront_size", "spcu_set_option",
    "spcu_scene_bytes", "spcu_trace_closest_counted", "spcu_stage_times", "spcu_resolved_pipeline",
    "spcu_build_bvh", "spcu_triangle_bounds", "spcu_upload_scene_build", "spcu_pack_image", "spcu_render_image", "spcu_ingest_mesh", "spcu_ingest_mesh_stl",
    "spcu_extend_batch", "spcu_shadow_batch",
    "spcu_comm_unique_id", "spcu_comm_init_rank", "spcu_comm_init_all", "spcu_comm_destroy", "spcu_comm_rank", "spcu_comm_size",
    "spcu_reduce_to_root", "spcu_render_frame_reduced",
    "spcu_render_adaptive", "spcu_render_adaptive_device", "spcu_pack_image_counts",
    "spcu_render_guides", "spcu_render_guides_device", "spcu_denoise", "spcu_denoise_device",
]
NCCL_ID_BYTES = 128
OPT_COUNT_NODES, OPT_STAGE_TIMING, OPT_PIPELINE, OPT_TRAVERSAL, OPT_GENERIC_KERNELS, OPT_BATCH_LANES = 0, 1, 2, 3, 4, 5
TRAVERSAL_EXACT, TRAVERSAL_ORDERED = 0, 1
PIPELINE_WAVEFRONT, PIPELINE_PATHS, PIPELINE_SMWAVE, PIPELINE_AUTO = 0, 1, 2, 3
IMAGE_PFM, IMAGE_PPM = 0, 1
IMAGE_DTYPES = {IMAGE_PFM: np.float32, IMAGE_PPM: np.uint16}


class SpcuError(RuntimeError):
    pass


_lib = None


def load(path: Path | str | None = None) -> C.CDLL:
    """dlopen libspcu.so and declare prototypes.  Raises if the library is absent (no fallback)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path else LIB_PATH
    if not p.exists():
        raise SpcuError(f"CUDA backend {p} is not built; run `python -c 'import __graft_entry__ as g; g.build()'`. "
                        "There is no CPU fallback.")
    lib = C.CDLL(str(p))
    vp = C.c_void_p
    lib.spcu_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.spcu_create.restype = C.c_int
    lib.spcu_destroy.argtypes = [vp]
    lib.spcu_destroy.restype = None
    lib.spcu_last_error.argtypes = [vp]
    lib.spcu_last_error.restype = C.c_char_p
    lib.spcu_abi_version.argtypes = []
    lib.spcu_abi_version.restype = C.c_int
    lib.spcu_upload_scene.argtypes = [vp, C.POINTER(FlatScene), C.POINTER(C.c_float), C.c_uint32]
    lib.spcu_upload_scene.restype = C.c_int
    for fn in (lib.spcu_trace_closest, lib.spcu_trace_lights):
        fn.argtypes = [vp, vp, C.c_uint64, vp]
        fn.restype = C.c_int
    lib.spcu_trace_closest_fast.argtypes = [vp, vp, C.c_uint64, vp, vp]
    lib.spcu_trace_closest_fast.restype = C.c_int
    lib.spcu_trace_any.argtypes = [vp, vp, C.c_uint64, vp]
    lib.spcu_trace_any.restype = C.c_int
    lib.spcu_comm_unique_id.argtypes = [vp]
    lib.spcu_comm_unique_id.restype = C.c_int
    lib.spcu_comm_init_rank.argtypes = [vp, C.c_int, C.c_int, vp]
    lib.spcu_comm_init_rank.restype = C.c_int
    lib.spcu_comm_destroy.argtypes = [vp]
    lib.spcu_comm_destroy.restype = None
    lib.spcu_comm_rank.argtypes = [vp]
    lib.spcu_comm_size.argtypes = [vp]
    lib.spcu_reduce_to_root.argtypes = [vp, vp, vp, vp]
    lib.spcu_reduce_to_root.restype = C.c_int
    lib.spcu_render_frame_reduced.argtypes = [vp, C.POINTER(Partition), C.c_int, vp, vp, C.POINTER(Stats)]
    lib.spcu_render_frame_reduced.restype = C.c_int
    lib.spcu_extend_batch.argtypes = [vp, vp, C.c_uint64, C.c_uint32, vp, vp]
    lib.spcu_extend_batch.restype = C.c_int
    lib.spcu_shadow_batch.argtypes = [vp, vp, C.c_uint64, vp]
    lib.spcu_shadow_batch.restype = C.c_int
    lib.spcu_generate_rays.argtypes = [vp, vp, vp, C.c_uint64, vp]
    lib.spcu_generate_rays.restype = C.c_int
    lib.spcu_render.argtypes = [vp, C.POINTER(Partition), vp, vp, C.POINTER(Stats)]
    lib.spcu_render.restype = C.c_int
    lib.spcu_render_frame.argtypes = [vp, C.POINTER(Partition), vp, vp, C.POINTER(Stats)]
    lib.spcu_render_frame.restype = C.c_int
    lib.spcu_render_device.argtypes = [vp, C.POINTER(Partition), vp, vp, C.POINTER(Stats), vp]
    lib.spcu_render_device.restype = C.c_int
    lib.spcu_set_wavefront_size.argtypes = [vp, C.c_uint64]
    lib.spcu_set_wavefront_size.restype = C.c_int
    lib.spcu_set_option.argtypes = [vp, C.c_uint32, C.c_uint32]
    lib.spcu_set_option.restype = C.c_int
    lib.spcu_scene_bytes.argtypes = [vp]
    lib.spcu_scene_bytes.restype = C.c_uint64
    lib.spcu_trace_closest_counted.argtypes = [vp, vp, C.c_uint64, vp, vp]
    lib.spcu_trace_closest_counted.restype = C.c_int
    lib.spcu_stage_times.argtypes = [vp, C.POINTER(StageTime), C.c_uint32, C.POINTER(C.c_uint32)]
    lib.spcu_stage_times.restype = C.c_int
    lib.spcu_build_bvh.argtypes = [vp, vp, C.c_uint32, vp, C.c_uint32, vp, vp, C.c_uint32, C.POINTER(Accel),
                                   C.POINTER(C.c_float)]
    lib.spcu_build_bvh.restype = C.c_int
    lib.spcu_upload_scene_build.argtypes = [vp, C.POINTER(FlatScene), C.POINTER(C.c_float), C.c_uint32, vp, vp, C.POINTER(Accel)]
    lib.spcu_upload_scene_build.restype = C.c_int
    lib.spcu_ingest_mesh.argtypes = [vp, vp, C.c_uint32, vp, C.c_uint32, vp, vp, C.c_uint32, vp, vp, vp, C.POINTER(C.c_uint32), vp, vp,
                                     C.POINTER(C.c_float)]
    lib.spcu_ingest_mesh.restype = C.c_int
    lib.spcu_ingest_mesh_stl.argtypes = [vp, vp, C.c_uint32, vp, C.c_uint32, vp, vp, vp, C.c_uint32, vp, vp, vp, C.POINTER(C.c_uint32),
                                         vp, vp, C.POINTER(C.c_float)]
    lib.spcu_ingest_mesh_stl.restype = C.c_int
    lib.spcu_pack_image.argtypes = [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp]
    lib.spcu_pack_image.restype = C.c_int
    lib.spcu_pack_image_counts.argtypes = [vp, vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, vp]
    lib.spcu_pack_image_counts.restype = C.c_int
    lib.spcu_render_adaptive.argtypes = [vp, C.POINTER(Partition), C.POINTER(Adaptive), vp, vp, vp, C.POINTER(C.c_uint32),
                                         C.POINTER(Stats)]
    lib.spcu_render_adaptive.restype = C.c_int
    lib.spcu_render_adaptive_device.argtypes = [vp, C.POINTER(Partition), C.POINTER(Adaptive), vp, vp, vp, C.POINTER(C.c_uint32),
                                                C.POINTER(Stats), vp]
    lib.spcu_render_adaptive_device.restype = C.c_int
    lib.spcu_render_guides.argtypes = [vp, vp]
    lib.spcu_render_guides.restype = C.c_int
    lib.spcu_render_guides_device.argtypes = [vp, vp, vp]
    lib.spcu_render_guides_device.restype = C.c_int
    lib.spcu_denoise.argtypes = [vp, vp, vp, vp, C.c_uint32, C.POINTER(DenoiseParams), vp]
    lib.spcu_denoise.restype = C.c_int
    lib.spcu_denoise_device.argtypes = [vp, vp, vp, vp, C.c_uint32, C.POINTER(DenoiseParams), vp, vp]
    lib.spcu_denoise_device.restype = C.c_int
    lib.spcu_render_image.argtypes = [vp, C.POINTER(Partition), C.c_uint32, vp, C.POINTER(Stats)]
    lib.spcu_render_image.restype = C.c_int
    lib.spcu_triangle_bounds.argtypes = [vp, vp, C.c_uint32, vp]
    lib.spcu_triangle_bounds.restype = C.c_int
    if lib.spcu_abi_version() != ABI_VERSION:
        raise SpcuError("libspcu.so ABI version mismatch")
    if path is None:
        _lib = lib
    return lib


def _ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)


class Context:
    """One CUDA device context (spcu_ctx).  Mirrors what sp::CudaIntegrator owns on the C++ side."""

    def __init__(self, device: int = 0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.spcu_create(device, C.byref(h))
        if rc != 0:
            raise SpcuError(f"spcu_create({device}) failed: {self.lib.spcu_last_error(None).decode()}")
        self.h = h
        self.device = device
        self._scene_keepalive = None
        self.width = self.height = 0

    def close(self) -> None:
        if getattr(self, "h", None):
            self.lib.spcu_destroy(self.h)
            self.h = None

    __del__ = close

    def _check(self, rc: int, what: str) -> None:
        if rc != 0:
            raise SpcuError(f"{what} failed ({rc}): {self.lib.spcu_last_error(self.h).decode()}")

    def upload_scene(self, flat: "C.POINTER(FlatScene) | FlatScene", jitter: np.ndarray, keepalive=None) -> None:
        jitter = np.ascontiguousarray(jitter, dtype=np.float32).reshape(-1, 2)
        fp = flat if isinstance(flat, C.POINTER(FlatScene)) else C.pointer(flat)
        self._check(self.lib.spcu_upload_scene(self.h, fp, jitter.ctypes.data_as(C.POINTER(C.c_float)),
                                               jitter.shape[0]), "spcu_upload_scene")
        self.width, self.height = fp.contents.width, fp.contents.height
        self.spp = jitter.shape[0]
        self._scene_keepalive = keepalive

    def upload_scene_build(self, flat, jitter: np.ndarray, bounds=None, keepalive=None):
        """spcu_upload_scene_build: geometry in pre-construction order, BVH built on the device.  Returns (order, accel head)."""
        jitter = np.ascontiguousarray(jitter, dtype=np.float32).reshape(-1, 2)
        fp = flat if isinstance(flat, C.POINTER(FlatScene)) else C.pointer(flat)
        g = fp.contents.geom
        order = np.zeros(max(g.n_prims - g.n_unbounded, 1), dtype=np.uint32)
        b = None if bounds is None else np.ascontiguousarray(bounds, dtype=np.float32).reshape(-1, 6)
        accel = Accel()
        self._check(self.lib.spcu_upload_scene_build(self.h, fp, jitter.ctypes.data_as(C.POINTER(C.c_float)), jitter.shape[0],
                                                     _ptr(b) if b is not None else None, _ptr(order), C.byref(accel)),
                    "spcu_upload_scene_build")
        self.width, self.height = fp.contents.width, fp.contents.height
        self.spp = jitter.shape[0]
        self._scene_keepalive = keepalive
        head = {k: int(getattr(accel, k)) for k in ("n_prims", "n_unbounded", "n_nodes", "root", "root_count", "max_depth")}
        return order[:g.n_prims - g.n_unbounded].copy(), head

    def _trace(self, fn, rays: np.ndarray, what: str) -> np.ndarray:
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        self._check(fn(self.h, _ptr(rays), rays.shape[0], _ptr(hits)), what)
        return hits

    def trace_closest(self, rays):
        return self._trace(self.lib.spcu_trace_closest, rays, "spcu_trace_closest")

    def trace_closest_counted(self, rays):
        """(hits, [internal nodes visited, triangle tests, sphere/plane tests])"""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        cnt = np.zeros(3, dtype=np.uint64)
        self._check(self.lib.spcu_trace_closest_counted(self.h, _ptr(rays), rays.shape[0], _ptr(hits), _ptr(cnt)),
                    "spcu_trace_closest_counted")
        return hits, cnt

    def set_option(self, option: int, value: int) -> None:
        self._check(self.lib.spcu_set_option(self.h, option, value), "spcu_set_option")

    def stage_times(self) -> list[dict]:
        """Per-kernel breakdown of the last render call that asked for stats."""
        arr = (StageTime * 16)()
        n = C.c_uint32()
        self._check(self.lib.spcu_stage_times(self.h, arr, 16, C.byref(n)), "spcu_stage_times")
        return [{"name": arr[i].name.decode(), "launches": arr[i].launches, "items": arr[i].items, "ms": arr[i].ms,
                 "traverses": bool(arr[i].traverses)} for i in range(n.value)]

    def scene_bytes(self) -> int:
        return int(self.lib.spcu_scene_bytes(self.h))

    def trace_closest_fast(self, rays):
        """Ordered walk: (hits, [internal nodes visited, triangle tests, sphere/plane tests])"""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        cnt = np.zeros(3, dtype=np.uint64)
        self._check(self.lib.spcu_trace_closest_fast(self.h, _ptr(rays), rays.shape[0], _ptr(hits), _ptr(cnt)),
                    "spcu_trace_closest_fast")
        return hits, cnt

    def trace_lights(self, rays):
        return self._trace(self.lib.spcu_trace_lights, rays, "spcu_trace_lights")

    def trace_any(self, rays) -> np.ndarray:
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        out = np.empty(rays.shape[0], dtype=np.uint8)
        self._check(self.lib.spcu_trace_any(self.h, _ptr(rays), rays.shape[0], _ptr(out)), "spcu_trace_any")
        return out

    def extend_batch(self, rays, traversal: int = TRAVERSAL_EXACT):
        """The render's extend stage on a ray batch (Integrator.cpp:558-563): (geometry hits under the light-shrunk limit,
        light hits)."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        lights = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        self._check(self.lib.spcu_extend_batch(self.h, _ptr(rays), rays.shape[0], traversal, _ptr(hits), _ptr(lights)),
                    "spcu_extend_batch")
        return hits, lights

    def shadow_batch(self, rays) -> np.ndarray:
        """The render's shadow stage on a ray batch (Scene::intersect_p): uint8 occlusion flags."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        out = np.empty(rays.shape[0], dtype=np.uint8)
        self._check(self.lib.spcu_shadow_batch(self.h, _ptr(rays), rays.shape[0], _ptr(out)), "spcu_shadow_batch")
        return out

    def generate_rays(self, pix, smp) -> np.ndarray:
        pix = np.ascontiguousarray(pix, dtype=np.uint32)
        smp = np.ascontiguousarray(smp, dtype=np.uint32)
        rays = np.empty(pix.shape[0], dtype=RAY_DTYPE)
        self._check(self.lib.spcu_generate_rays(self.h, _ptr(pix), _ptr(smp), pix.shape[0], _ptr(rays)),
                    "spcu_generate_rays")
        return rays

    def partition(self, spp: int | None = None, integrator: str = "iterative_rrnee", rank: int = 0, world: int = 1,
                  sample_begin: int = 0, sample_end: int | None = None, seed: int = 0) -> Partition:
        spp = self.spp if spp is None else spp
        return Partition(rank, world, sample_begin, spp if sample_end is None else sample_end, spp,
                         INTEGRATORS[integrator], seed)

    def render(self, part: Partition, want_sumsq: bool = True, into=None):
        """Host-buffer render: returns (rgb_sum [H,W,3], lum_sumsq [H,W] | None, stats dict).  `into` = (rgb, sq) of
        an earlier call to keep accumulating into."""
        if into is not None:
            rgb, sq = into
            want_sumsq = sq is not None
        else:
            rgb = np.zeros((self.height, self.width, 3), dtype=np.float32)
            sq = np.zeros((self.height, self.width), dtype=np.float32) if want_sumsq else None
        st = Stats()
        self._check(self.lib.spcu_render(self.h, C.byref(part), _ptr(rgb), _ptr(sq) if want_sumsq else None,
                                         C.byref(st)), "spcu_render")
        return rgb, sq, st.as_dict()

    def render_passes(self, passes: int, spp: int | None = None, integrator: str = "iterative_rrnee", seed: int = 0,
                      rank: int = 0, world: int = 1):
        """Progressive rendering — the multi-pass mode the reference's TileScheduler provides for (`pass` of a ScheduledTile,
        base/TileScheduler.h:58-86; main.cpp:111 runs it with num_passes = 1): pass p adds samples [p*k, (p+1)*k) of the
        frame's spp to the same accumulators.  Yields (samples_so_far, rgb_sum, lum_sumsq, stats) after every pass; the
        arrays are the running SUMS (divide by samples_so_far for the preview), and after the last pass they are, bit for
        bit, what one spcu_render call of the whole frame returns (sample ranges accumulate in sample order)."""
        spp = self.spp if spp is None else spp
        passes = max(1, min(passes, spp))
        acc = None
        for p in range(passes):
            lo, hi = spp * p // passes, spp * (p + 1) // passes
            part = Partition(rank, world, lo, hi, spp, INTEGRATORS[integrator], seed)
            rgb, sq, st = self.render(part, into=acc)
            acc = (rgb, sq)
            yield hi, rgb, sq, st

    def render_frame(self, part: Partition, out=None, want_sumsq: bool = True):
        """Host-buffer render that OVERWRITES its outputs (no accumulator upload, nothing to zero): returns
        (rgb_sum, lum_sumsq | None, stats).  `out` = (rgb, sq) preallocated, e.g. page-locked, arrays to write into."""
        if out is not None:
            rgb, sq = out
            want_sumsq = sq is not None
        else:
            rgb = np.empty((self.height, self.width, 3), dtype=np.float32)
            sq = np.empty((self.height, self.width), dtype=np.float32) if want_sumsq else None
        st = Stats()
        self._check(self.lib.spcu_render_frame(self.h, C.byref(part), _ptr(rgb), _ptr(sq) if want_sumsq else None,
                                               C.byref(st)), "spcu_render_frame")
        return rgb, sq, st.as_dict()

    def render_device(self, part: Partition, d_rgb_sum: int, d_lum_sumsq: int | None, stream: int | None = None,
                      want_stats: bool = True) -> dict | None:
        """Accumulate into DEVICE buffers on `stream`.  Without stats the call only enqueues work (no host sync)."""
        st = Stats()
        self._check(self.lib.spcu_render_device(self.h, C.byref(part), C.c_void_p(d_rgb_sum),
                                                C.c_void_p(d_lum_sumsq) if d_lum_sumsq else None,
                                                C.byref(st) if want_stats else None,
                                                C.c_void_p(stream) if stream else None), "spcu_render_device")
        return st.as_dict() if want_stats else None

    # ---- multi-GPU (one process per GPU): NCCL communicator of the product library ------------------------------------------
    def comm_unique_id(self) -> bytes:
        """ncclGetUniqueId (rank 0 calls; the launcher hands the bytes to every rank)."""
        buf = (C.c_uint8 * NCCL_ID_BYTES)()
        self._check(self.lib.spcu_comm_unique_id(buf), "spcu_comm_unique_id")
        return bytes(buf)

    def comm_init_rank(self, nranks: int, rank: int, unique_id: bytes) -> None:
        assert len(unique_id) == NCCL_ID_BYTES
        buf = (C.c_uint8 * NCCL_ID_BYTES).from_buffer_copy(unique_id)
        self._check(self.lib.spcu_comm_init_rank(self.h, nranks, rank, buf), "spcu_comm_init_rank")

    def reduce_to_root(self, d_rgb_sum: int, d_lum_sumsq: int | None, stream: int | None = None) -> None:
        """ncclReduce(sum, root 0) of the device accumulators, in place, on `stream` (enqueue only)."""
        self._check(self.lib.spcu_reduce_to_root(self.h, C.c_void_p(d_rgb_sum), C.c_void_p(d_lum_sumsq) if d_lum_sumsq else None,
                                                 C.c_void_p(stream) if stream else None), "spcu_reduce_to_root")

    def render_frame_reduced(self, part: Partition, out=None, want_sumsq: bool = True, want_stats: bool = True):
        """This rank's partition + NCCL reduction + (rank 0 only) the device->host copy: (rgb_sum, lum_sumsq, stats) on rank 0,
        (None, None, stats) elsewhere."""
        root = self.lib.spcu_comm_rank(self.h) == 0
        rgb = sq = None
        if root:
            if out is not None:
                rgb, sq = out
            else:
                rgb = np.empty((self.height, self.width, 3), dtype=np.float32)
                sq = np.empty((self.height, self.width), dtype=np.float32) if want_sumsq else None
        st = Stats()
        self._check(self.lib.spcu_render_frame_reduced(self.h, C.byref(part), 1 if want_sumsq else 0,
                                                       _ptr(rgb) if root else None, _ptr(sq) if root and want_sumsq else None,
                                                       C.byref(st) if want_stats else None), "spcu_render_frame_reduced")
        return rgb, sq, (st.as_dict() if want_stats else None)

    def resolved_pipeline(self) -> str:
        """The kernel organisation the next render runs (PIPELINE_AUTO resolved for the uploaded scene)."""
        self.lib.spcu_resolved_pipeline.argtypes = [C.c_void_p]
        self.lib.spcu_resolved_pipeline.restype = C.c_int
        code = self.lib.spcu_resolved_pipeline(self.h)
        return {PIPELINE_WAVEFRONT: "wavefront", PIPELINE_PATHS: "paths", PIPELINE_SMWAVE: "smwave"}.get(code, "none")

    def build_bvh(self, bounds, non_triangle=None, first_id: int = 0, capacity: int | None = None) -> dict:
        """BVHAccelerator::construct on the device (spcu_build_bvh): {nodes, order, head (accel fields), device_ms}."""
        bounds = np.ascontiguousarray(bounds, dtype=np.float32).reshape(-1, 6)
        return run_build(lambda *a: self._check(self.lib.spcu_build_bvh(self.h, *a), "spcu_build_bvh"),
                         bounds, non_triangle, first_id, capacity, with_ms=True)

    def triangle_bounds(self, tris) -> np.ndarray:
        """Triangle::get_world_bounds for spcu_prim_geom records [n, 12] -> [n, 6]."""
        tris = np.ascontiguousarray(tris, dtype=np.float32).reshape(-1, 12)
        out = np.empty((tris.shape[0], 6), dtype=np.float32)
        self._check(self.lib.spcu_triangle_bounds(self.h, _ptr(tris), tris.shape[0], _ptr(out)), "spcu_triangle_bounds")
        return out

    def ingest_mesh(self, vertices, faces, object_to_world, normal_xf, material: int = 0) -> dict:
        """spcu_ingest_mesh: {prims [k,12], shade [k,12], meta [k], world_vertices, world_normals, device_ms}."""
        return run_ingest(lambda *a: self._check(self.lib.spcu_ingest_mesh(self.h, *a), "spcu_ingest_mesh"),
                          vertices, faces, object_to_world, normal_xf, material, with_ms=True)

    def ingest_mesh_stl(self, vertices, faces, face_normals, object_to_world, normal_xf, material: int = 0) -> dict:
        """spcu_ingest_mesh_stl: as ingest_mesh, with the normals stored in the STL file."""
        return run_ingest(lambda *a: self._check(self.lib.spcu_ingest_mesh_stl(self.h, *a), "spcu_ingest_mesh_stl"),
                          vertices, faces, object_to_world, normal_xf, material, with_ms=True, face_normals=face_normals)

    def pack_image(self, rgb_sum, spp, fmt: int) -> np.ndarray:
        """Host sums [H, W, 3] -> write_pfm payload (float32) / write_ppm numbers (uint16), rows bottom-up.  spp: the samples
        of every pixel (int), or the per-pixel counts [H, W] of render_adaptive (spcu_pack_image_counts)."""
        rgb_sum = np.ascontiguousarray(rgb_sum, dtype=np.float32)
        h, w = rgb_sum.shape[:2]
        out = np.empty((h, w, 3), dtype=IMAGE_DTYPES[fmt])
        if isinstance(spp, np.ndarray):
            counts = np.ascontiguousarray(spp, dtype=np.uint32)
            if counts.shape != (h, w):
                raise ValueError(f"spp map of shape {counts.shape} for a {h}x{w} image")
            self._check(self.lib.spcu_pack_image_counts(self.h, _ptr(rgb_sum), _ptr(counts), w, h, fmt, _ptr(out)),
                        "spcu_pack_image_counts")
            return out
        self._check(self.lib.spcu_pack_image(self.h, _ptr(rgb_sum), w, h, spp, fmt, _ptr(out)), "spcu_pack_image")
        return out

    def render_adaptive(self, part: Partition, rel_error: float, min_spp: int = 16, pass_spp: int = 16, abs_floor: float = 0.0,
                        want_sumsq: bool = True, radius: int = 0):
        """Adaptive sampling (spcu_render_adaptive): each pixel of the partition gets samples [0, n_p) until the standard error of
        its mean luminance is at most rel_error * (mean + abs_floor), n_p <= part.sample_end (the budget).  radius > 0: a pixel
        stops only when every pixel within `radius` of it in its 8x8 tile meets the target too.  Outputs are overwritten:
        (rgb_sum [H,W,3], lum_sumsq [H,W] | None, spp_map [H,W] uint32 = n_p, stats dict with "passes")."""
        rgb = np.empty((self.height, self.width, 3), dtype=np.float32)
        sq = np.empty((self.height, self.width), dtype=np.float32) if want_sumsq else None
        spp_map = np.empty((self.height, self.width), dtype=np.uint32)
        ad = Adaptive(min_spp, pass_spp, rel_error, abs_floor, radius)
        passes = C.c_uint32()
        st = Stats()
        self._check(self.lib.spcu_render_adaptive(self.h, C.byref(part), C.byref(ad), _ptr(rgb), _ptr(sq) if want_sumsq else None,
                                                  _ptr(spp_map), C.byref(passes), C.byref(st)), "spcu_render_adaptive")
        stats = st.as_dict()
        stats["passes"] = passes.value
        return rgb, sq, spp_map, stats

    def render_guides(self) -> np.ndarray:
        """First-hit guide records of sample 0's camera rays (spcu_render_guides): structured array [H, W] of GUIDE_DTYPE."""
        out = np.empty((self.height, self.width), dtype=GUIDE_DTYPE)
        self._check(self.lib.spcu_render_guides(self.h, _ptr(out)), "spcu_render_guides")
        return out

    def denoise(self, rgb_sum, lum_sumsq, spp, iterations: int = DENOISE_DEFAULTS["iterations"],
                sigma_l: float = DENOISE_DEFAULTS["sigma_l"], sigma_z: float = DENOISE_DEFAULTS["sigma_z"],
                sigma_a: float = DENOISE_DEFAULTS["sigma_a"]) -> np.ndarray:
        """Denoised mean colour [H, W, 3] of a frame's sums (spcu_denoise).  spp: the samples of every pixel (int), or the
        per-pixel counts [H, W] of render_adaptive.  pack_image(result, 1, fmt) packs it."""
        rgb_sum = np.ascontiguousarray(rgb_sum, dtype=np.float32)
        sq = None if lum_sumsq is None else np.ascontiguousarray(lum_sumsq, dtype=np.float32)
        h, w = rgb_sum.shape[:2]
        if (h, w) != (self.height, self.width) or (sq is not None and sq.shape != (h, w)):
            raise ValueError(f"sums of shape {rgb_sum.shape} for a {self.height}x{self.width} scene")
        counts = None
        if isinstance(spp, np.ndarray):
            counts = np.ascontiguousarray(spp, dtype=np.uint32)
            if counts.shape != (h, w):
                raise ValueError(f"spp map of shape {counts.shape} for a {h}x{w} image")
            spp = 0
        out = np.empty((h, w, 3), dtype=np.float32)
        p = DenoiseParams(iterations, sigma_l, sigma_z, sigma_a)
        self._check(self.lib.spcu_denoise(self.h, _ptr(rgb_sum), _ptr(sq) if sq is not None else None,
                                          _ptr(counts) if counts is not None else None, spp, C.byref(p), _ptr(out)),
                    "spcu_denoise")
        return out

    def render_image(self, part: Partition, fmt: int):
        """Render + pack on the device: (packed image [H, W, 3], stats)."""
        out = np.empty((self.height, self.width, 3), dtype=IMAGE_DTYPES[fmt])
        st = Stats()
        self._check(self.lib.spcu_render_image(self.h, C.byref(part), fmt, _ptr(out), C.byref(st)), "spcu_render_image")
        return out, st.as_dict()

    def set_wavefront_size(self, n: int) -> None:
        self._check(self.lib.spcu_set_wavefront_size(self.h, n), "spcu_set_wavefront_size")


def run_build(call, bounds: np.ndarray, non_triangle, first_id: int, capacity: int | None, with_ms: bool, extra=()) -> dict:
    """Shared argument marshalling of the three BVH builders (CUDA, oracle restatement, reference harness):
    call(bounds, n, non_triangle, first_id, order, nodes, capacity, accel, [ms | root_bounds], *extra)."""
    n = bounds.shape[0]
    nt = None if non_triangle is None else np.ascontiguousarray(non_triangle, dtype=np.uint8)
    cap = max(n, 1) - 1 if capacity is None else capacity
    nodes = np.zeros(max(cap, 1), dtype=NODE_DTYPE)
    order = np.zeros(max(n, 1), dtype=np.uint32)
    accel = Accel()
    if with_ms:
        tail = C.c_float()
        call(_ptr(bounds), n, _ptr(nt) if nt is not None else None, first_id, _ptr(order), _ptr(nodes), cap,
             C.byref(accel), C.byref(tail), *extra)
        tail_out = {"device_ms": float(tail.value)}
    else:
        root = np.zeros(6, dtype=np.float32)
        call(_ptr(bounds), n, _ptr(nt) if nt is not None else None, first_id, _ptr(order), _ptr(nodes), cap,
             C.byref(accel), _ptr(root), *extra)
        tail_out = {"root_bounds": root}
    head = {k: int(getattr(accel, k)) for k in ("n_prims", "n_unbounded", "n_nodes", "root", "root_count", "max_depth")}
    return {"nodes": nodes[:head["n_nodes"]].copy(), "order": order[:n].copy(), "head": head, **tail_out}


def run_ingest(call, vertices, faces, object_to_world, normal_xf, material: int, with_ms: bool, face_normals=None) -> dict:
    """Shared marshalling of the mesh-ingest entry points (CUDA, oracle): call(vertices, nv, faces, nf, xf, nxf, material,
    prims, shade, meta, n_kept, world_vertices, world_normals[, device_ms])."""
    v = np.ascontiguousarray(vertices, dtype=np.float32).reshape(-1, 3)
    f = np.ascontiguousarray(faces, dtype=np.uint32).reshape(-1, 3)
    xf = np.ascontiguousarray(object_to_world, dtype=np.float32).reshape(12)
    nxf = np.ascontiguousarray(normal_xf, dtype=np.float32).reshape(9)
    nv, nf = v.shape[0], f.shape[0]
    prims = np.zeros((max(nf, 1), 12), dtype=np.float32)
    shade = np.zeros((max(nf, 1), 12), dtype=np.float32)
    meta = np.zeros(max(nf, 1), dtype=np.uint32)
    wv = np.zeros((max(nv, 1), 3), dtype=np.float32)
    wn = np.zeros((max(nv, 1), 3), dtype=np.float32)
    kept = C.c_uint32()
    args = [_ptr(v), nv, _ptr(f), nf]
    if face_normals is not None:  # the STL flavour takes the file's normals after the faces
        fn = np.ascontiguousarray(face_normals, dtype=np.float32).reshape(-1, 3)
        assert fn.shape[0] == nf
        args.append(_ptr(fn))
    args += [_ptr(xf), _ptr(nxf), material, _ptr(prims), _ptr(shade), _ptr(meta), C.byref(kept), _ptr(wv), _ptr(wn)]
    ms = C.c_float()
    if with_ms:
        args.append(C.byref(ms))
    call(*args)
    k = kept.value
    return {"prims": prims[:k].copy(), "shade": shade[:k].copy(), "meta": meta[:k].copy(), "world_vertices": wv[:nv].copy(),
            "world_normals": wn[:nv].copy(), "device_ms": float(ms.value)}
