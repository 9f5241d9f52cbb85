"""Python mirror of the host side of the drop-in: loads `.sp` scenes through the reference's own parser
(libsphost.so = reference objects + the scene flattener, built by simplepath_b200/host/Makefile where the reference
sources exist) and hands out flattened scenes for the C-ABI.  Mirrors what sp::CudaIntegrator does in C++."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from . import rsequence, scenes
from .capi import BvhNode, FlatScene
from .flat import FlatSceneData

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "host" / "libsphost.so"
DRIVER = PKG / "host" / "SimplePathCuda"
FLAT_DIR = PKG.parent / "scenes" / "flat"   # committed flattened scenes of the small workloads
SHELL_DIR = PKG.parent / "tests" / "golden"  # committed flattened scenes of the tiny versions (scenes.ASSEMBLED)

_lib = None


def available() -> bool:
    return LIB_PATH.exists()


def loadable(name: str) -> bool:
    """Whether workload(name) can produce the scene here."""
    return available() or (FLAT_DIR / f"{name}.flat.npz").exists() or name in scenes.ASSEMBLED


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        from . import capi
        capi.load()  # libsphost.so links against libspcu.so
        l = C.CDLL(str(LIB_PATH))
        l.sphost_load.argtypes = [C.c_char_p, C.c_char_p, C.c_size_t]
        l.sphost_load.restype = C.c_void_p
        l.sphost_free.argtypes = [C.c_void_p]
        l.sphost_free.restype = None
        l.sphost_flat.argtypes = [C.c_void_p]
        l.sphost_flat.restype = C.POINTER(FlatScene)
        l.sphost_output_file_name.argtypes = [C.c_void_p]
        l.sphost_output_file_name.restype = C.c_char_p
        l.sphost_jitter.argtypes = [C.c_uint, C.c_void_p]
        l.sphost_jitter.restype = None
        _lib = l
    return _lib


def parse(sp_path: Path | str) -> FlatSceneData:
    """FileParser -> Scene -> flattener, then copied into numpy arrays (the C++ objects are freed)."""
    l = lib()
    err = C.create_string_buffer(512)
    h = l.sphost_load(str(sp_path).encode(), err, 512)
    if not h:
        raise RuntimeError(f"{sp_path}: {err.value.decode()}")
    try:
        return FlatSceneData.from_struct(l.sphost_flat(h))
    finally:
        l.sphost_free(h)


def jitter(spp: int) -> np.ndarray:
    """Pixel jitter table; the pure-Python restatement is bitwise equal to the reference's (tests/test_host_logic.py)."""
    return rsequence.jitter_table(spp)


def workload(name: str) -> FlatSceneData:
    """A named scene of simplepath_b200.scenes, flattened.  Uses the parser library when it is present (it is built only
    where the reference sources are), else the committed flattened copy, else a scene put together from a committed
    shell and generated meshes (assemble)."""
    if available():
        return parse(scenes.ensure(name))
    path = FLAT_DIR / f"{name}.flat.npz"
    if path.exists():
        return FlatSceneData.load(path)
    if name in scenes.ASSEMBLED:
        return assemble(name)
    raise RuntimeError(f"cannot load workload {name}: {LIB_PATH} is not built, {path} does not exist and the scene "
                       "has no shell to be assembled from")


def assemble(name: str) -> FlatSceneData:
    """What the parser + flattener make of a mesh scene, without them: the shell (the tiny flattened scene of the same
    .sp text: materials, lights, unbounded primitives, camera) at the scene's resolution, the generated meshes ingested
    by the oracle's restatement of read_ply + Mesh, and BVHAccelerator::construct over their triangles by the oracle's
    restatement.  Both restatements are bit-exact with the reference on x86 (tests/test_oracle_mesh.py,
    tests/test_oracle_build.py), so geometry, normals and tree are the parser's; tests/test_host_logic.py rebuilds the
    shells' own scenes this way and compares every byte.  The camera is rescaled from the shell's resolution in float64
    (raster_camera)."""
    from oracle import port
    shell_name, meshes = scenes.ASSEMBLED[name]
    shell = FlatSceneData.load(SHELL_DIR / f"{shell_name}.flat.npz")
    w, h, _ = scenes.info(name)
    nu = shell.head["geom"]["n_unbounded"]
    recs = []
    for n_tris, lo, hi, translate, scale, material in meshes:
        xf = np.array([scale, 0, 0, 0, scale, 0, 0, 0, scale, *translate], dtype=np.float32)
        nxf = np.float32(1.0 / scale) * np.eye(3, dtype=np.float32).reshape(9)
        v, f = scenes.bumpy_sphere(n_tris, lo, hi)
        recs.append(port.ingest_mesh(v, f, xf, nxf, material))
    prims, shade, meta = (np.concatenate([r[k] for r in recs]) for k in ("prims", "shade", "meta"))
    built = port.build_bvh(port.triangle_bounds(prims), None, nu)
    order = built["order"]
    arrays = dict(shell.arrays)
    for key, new, width in (("geom_prims", prims, 48), ("geom_shade", shade, 48), ("geom_meta", meta, 4)):
        arrays[key] = np.concatenate([shell.arrays[key][:nu], np.ascontiguousarray(new[order]).view(np.uint8).reshape(-1, width)])
    arrays["geom_nodes"] = built["nodes"].view(np.uint8).reshape(-1, C.sizeof(BvhNode)).copy()
    head = dict(shell.head, width=w, height=h, camera=raster_camera(shell.head["camera"], shell.width, shell.height, w, h),
                geom=built["head"])
    return FlatSceneData(head, arrays)


def raster_camera(camera, w0: int, h0: int, w: int, h: int) -> list[float]:
    """The flattened camera (raster x / y steps, direction to pixel (0, 0), origin) of a w0 x h0 frame, for a w x h frame
    with the same vertical field of view (the parser keeps the .sp fov vertical whatever the aspect ratio): the steps stay,
    the direction to the corner moves.  Within 2 ulp of the parser's own camera (tests/test_host_logic.py)."""
    c = np.asarray(camera, dtype=np.float64)
    dx, dy = c[0:3], c[3:6]
    forward = (c[6:9] + dx * (w0 / 2) + dy * (h0 / 2)) * (h / h0)
    out = np.asarray(camera, dtype=np.float32).copy()
    out[6:9] = forward - dx * (w / 2) - dy * (h / 2)
    return [float(x) for x in out]
