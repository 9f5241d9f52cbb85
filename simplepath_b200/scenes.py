"""Deterministic scene / asset generators for the BASELINE.json configs.

None of the reference's five configured scenes runs as shipped (SURVEY.md §0.5): the PLY/STL/PFM assets
are not in the repository, `example_scene.sp` uses block types the parser rejects
(base/FileParser.cpp:871-873) and `scenes/elf.sp:11` has commas the vector reader cannot parse.  This module
writes `.sp` files the *stock* reference parser accepts, with

  * geometry / materials / lights / cameras copied in meaning from the reference scenes
    (scenes/material_spheres.sp:15-88, scenes/bunny.sp, scenes/elf.sp, scenes/lucy.sp, example_scene.sp),
  * procedural binary little-endian PLY meshes with the named triangle counts (closed-form displacement of a
    sphere, no RNG) in exactly the dialect base/PlyReader.cpp:326-531 reads,
  * a synthetic lat-long PFM environment map (analytic sky + one bright lobe) for Image/Image.cpp:78-119.

Everything is a pure function of its arguments, so a GPU box regenerates identical bytes.
CLI:  python -m simplepath_b200.scenes [--out DIR] [names...]
"""
from __future__ import annotations

import argparse
import os
import struct
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent.parent
DEFAULT_OUT = REPO / "scenes" / "_gen"

BUNNY_TRIS = 69_451        # bun_zipper.ply (public Stanford figure)
LUCY_TRIS = 28_055_742     # lucy.ply (public Stanford figure)
ELF_TRIS = 750_000         # stand-in for stl_files/elf/nude-body.stl (count not published; stated in reports)


# --------------------------------------------------------------------------------------------------
# assets
# --------------------------------------------------------------------------------------------------
def _grid_for(n_tris: int) -> tuple[int, int]:
    """Smallest near-square (nu, nv) with 2*nu*nv >= n_tris."""
    nv = int(np.floor(np.sqrt(n_tris / 2.0)))
    nu = nv
    while 2 * nu * nv < n_tris:
        nu += 1
    return nu, nv


def bumpy_sphere(n_tris: int, lo, hi) -> tuple[np.ndarray, np.ndarray]:
    """Displaced sphere with exactly n_tris triangles, fitted to the box [lo, hi].

    Latitude runs over (eps, pi-eps) so no triangle is degenerate (the reader drops zero-area faces,
    base/PlyReader.cpp:489-493); the face list of the full grid is truncated to n_tris."""
    nu, nv = _grid_for(n_tris)
    eps = 0.02
    theta = np.linspace(eps, np.pi - eps, nv + 1, dtype=np.float64)[:, None]      # rows
    phi = (np.arange(nu, dtype=np.float64) * (2.0 * np.pi / nu))[None, :]          # columns (wrapping)
    r = (1.0 + 0.18 * np.sin(3.0 * theta) * np.sin(5.0 * phi)
         + 0.07 * np.sin(13.0 * theta + 0.5) * np.sin(17.0 * phi + 1.0)
         + 0.02 * np.sin(41.0 * theta) * np.cos(37.0 * phi))
    x = r * np.sin(theta) * np.cos(phi)
    y = r * np.cos(theta) * np.ones_like(phi)
    z = r * np.sin(theta) * np.sin(phi)
    v = np.stack([x, y, z], axis=-1).reshape(-1, 3)
    vmin, vmax = v.min(0), v.max(0)
    lo = np.asarray(lo, np.float64)
    hi = np.asarray(hi, np.float64)
    v = (v - vmin) / (vmax - vmin) * (hi - lo) + lo

    i = np.arange(nv, dtype=np.int64)[:, None]
    j = np.arange(nu, dtype=np.int64)[None, :]
    a = i * nu + j
    b = i * nu + (j + 1) % nu
    c = (i + 1) * nu + j
    d = (i + 1) * nu + (j + 1) % nu
    # counter-clockwise seen from outside (y up, theta from +y)
    t0 = np.stack([a, b, c], axis=-1)
    t1 = np.stack([b, d, c], axis=-1)
    faces = np.stack([t0, t1], axis=2).reshape(-1, 3)[:n_tris]
    assert faces.shape[0] == n_tris
    return v.astype("<f4"), faces.astype("<i4")


def chain_mesh(n_tris: int = 58) -> tuple[np.ndarray, np.ndarray]:
    """A mesh whose spatial-median BVH is a CHAIN: triangle i lies in the plane x = 1e10 * 0.45^i (object space; the scene
    scales it by 1e-10) with a size proportional to its distance from the origin (a self-similar cone).
    BVHAccelerator::construct (shapes/BVHAccelerator.h:175-209) splits at the centre of the node's bounds along x, which
    peels ONE triangle off per level: depth = n_tris - 4, far beyond the 24 traversal-stack levels the kernels keep in shared
    memory.  A ray aimed at the apex crosses every triangle, so the reference-order walk leaves a pending right child at
    every level.  (The object-space scale keeps sqr_length(face normal) of the smallest triangle above float underflow:
    read_ply drops faces where it is exactly 0, base/PlyReader.cpp:497.)"""
    x = 1e10 * 0.45 ** np.arange(n_tris, dtype=np.float64)
    s = 0.2 * x
    v = np.stack([np.stack([x, -s, -s], 1), np.stack([x, s, -s], 1), np.stack([x, 0 * s, s], 1)], axis=1).reshape(-1, 3)
    f = np.arange(3 * n_tris, dtype=np.int64).reshape(-1, 3)
    return v.astype("<f4"), f.astype("<i4")


def write_ply(path: Path, verts: np.ndarray, faces: np.ndarray) -> None:
    header = (
        "ply\n"
        "format binary_little_endian 1.0\n"
        f"element vertex {len(verts)}\n"
        "property float x\nproperty float y\nproperty float z\n"
        f"element face {len(faces)}\n"
        "property list uchar int vertex_indices\n"
        "end_header\n"
    ).encode("ascii")
    rec = np.empty(len(faces), dtype=[("n", "u1"), ("i", "<i4", (3,))])
    rec["n"] = 3
    rec["i"] = faces
    tmp = path.with_suffix(path.suffix + f".{os.getpid()}.tmp")  # one per process: ranks of a torchrun job generate concurrently
    with open(tmp, "wb") as f:
        f.write(header)
        f.write(np.ascontiguousarray(verts, dtype="<f4").tobytes())
        f.write(rec.tobytes())
    os.replace(tmp, path)


def sky_image(w: int, h: int) -> np.ndarray:
    """[h, w, 3] radiance, row 0 = top of the lat-long map (theta = 0)."""
    v = (np.arange(h, dtype=np.float64) + 0.5)[:, None] / h        # theta / pi
    u = (np.arange(w, dtype=np.float64) + 0.5)[None, :] / w        # phi / 2pi
    up = np.clip(1.0 - 2.0 * v, -1.0, 1.0)                         # cos(theta)-ish
    horizon = np.exp(-8.0 * np.abs(up))
    base_r = 0.15 + 0.35 * horizon + 0.10 * np.maximum(up, 0.0)
    base_g = 0.20 + 0.40 * horizon + 0.25 * np.maximum(up, 0.0)
    base_b = 0.35 + 0.45 * horizon + 0.60 * np.maximum(up, 0.0)
    ground = (up < 0.0) * 0.6
    lobe = 60.0 * np.exp(-((u - 0.30) ** 2 / (2 * 0.012 ** 2) + (v - 0.28) ** 2 / (2 * 0.02 ** 2)))
    img = np.stack([
        base_r * (1.0 - ground) + 0.08 * ground + lobe * 1.00 + 0.0 * u,
        base_g * (1.0 - ground) + 0.07 * ground + lobe * 0.90 + 0.0 * u,
        base_b * (1.0 - ground) + 0.06 * ground + lobe * 0.70 + 0.0 * u,
    ], axis=-1)
    return img.astype("<f4")


def write_pfm(path: Path, img: np.ndarray) -> None:
    """Image(x, y) = img[y, x]; the file stores rows j = ny-1 .. 0 (Image/Image.cpp:40-55)."""
    h, w, _ = img.shape
    tmp = path.with_suffix(path.suffix + f".{os.getpid()}.tmp")
    with open(tmp, "wb") as f:
        f.write(f"PF\n{w} {h}\n-1\n".encode("ascii"))
        f.write(np.ascontiguousarray(img[::-1], dtype="<f4").tobytes())
    os.replace(tmp, path)


def read_pfm(path: Path) -> np.ndarray:
    with open(path, "rb") as f:
        assert f.readline().strip() == b"PF"
        w, h = map(int, f.readline().split())
        f.readline()
        data = np.frombuffer(f.read(w * h * 12), dtype="<f4").reshape(h, w, 3)
    return data[::-1].copy()


# --------------------------------------------------------------------------------------------------
# .sp text
# --------------------------------------------------------------------------------------------------
_MATERIALS_SPHERES = """\
material_lambertian {
    name: "material_lambertian"
    diffuse: 0.1 0.8 0.8
}

material_lambertian {
    name: "material_lambertian_base"
    diffuse: 0.1 0.2 0.8
}

material_glossy {
    name: "material_glossy_base"
    diffuse: 0.8 0.2 0.8
    ior: 1.8
    roughness: 0.25
}

material_glossy {
    name: "material_glossy"
    diffuse: 0.8 0.2 0.2
    ior: 1.8
    roughness: 0.75
}

material_glossy {
    name: "material_glossy_plane"
    diffuse: 0.6 0.6 0.6
    ior: 1.8
    roughness: 0.01
}

material_clearcoat {
    name: "material_lambertian_clearcoat"
    base: "material_lambertian_base"
    ior: 1.5
    color: 1.0 0.8 0.8
}

material_clearcoat {
    name: "material_glossy_clearcoat"
    base: "material_glossy_base"
    ior: 1.3
    color: 1.0 1.0 1.0
}
"""

_MATERIALS_STATUE = """\
material_glossy {
    name: "material_glossy_base"
    diffuse: 0.7 0.7 0.7
    ior: 1.3
    roughness: 0.75
}

material_glossy {
    name: "material_glossy_plane"
    diffuse: 0.4 0.1 0.1
    ior: 1.8
    roughness: 0.01
}

material_clearcoat {
    name: "material_glossy_clearcoat"
    base: "material_glossy_base"
    ior: 1.5
    color: 1.0 1.0 1.0
}
"""


def _head(w: int, h: int, extra: str = "") -> str:
    return f"version: 1\n\nscene_parameters {{\n    output_file_name: \"image.pfm\"\n    width: {w}\n    height: {h}\n{extra}}}\n\n"


def sp_material_spheres(w: int, h: int, env: str) -> str:
    """scenes/material_spheres.sp:15-88 verbatim; env = 'const' or a PFM path (scenes/material_spheres.sp:90-95)."""
    light = ("environment_light {\n    rotate: 0.0 1.0 0.0 45.0\n    radiance: 1.0 1.0 1.0\n}\n" if env == "const" else
             f"environment_light {{\n    rotate: 0.0 1.0 0.0 45.0\n    radiance: 1.0 1.0 1.0\n    max_radiance: 100\n    image: \"{env}\"\n}}\n")
    return (_head(w, h) +
            "perspective_camera {\n    origin: 0.0 0.0 10.0\n    look_at: 0.0 0.0 0.0\n    fov: 45\n}\n\n" +
            _MATERIALS_SPHERES + "\n" +
            "sphere {\n    translate: 0.0 3.0 0.0\n    material: \"material_glossy_clearcoat\"\n}\n\n"
            "sphere {\n    translate: 0.0 1.0 0.0\n    material: \"material_lambertian_clearcoat\"\n}\n\n"
            "sphere {\n    translate: 0.0 -1.0 0.0\n    material: \"material_lambertian\"\n}\n\n"
            "sphere {\n    translate: 0.0 -3.0 0.0\n    material: \"material_glossy\"\n}\n\n"
            "plane {\n    material: \"material_glossy_plane\"\n    rotate: 1 0 0 90\n    translate: 0.0 0.0 -1.0\n}\n\n" +
            light)


def sp_example_scene(w: int, h: int) -> str:
    """Parseable restatement of example_scene.sp (SURVEY.md §8d C2): clearcoat(ior 1.3) over Lambert (0.1,0.2,0.8)
    sphere scaled 10 at (10,0.5,0) rotated 45 deg about y; y=0 plane; sphere light; constant environment."""
    return (_head(w, h) +
            "perspective_camera {\n    origin: 0.0 2.0 5.0\n    look_at: 0.0 1.0 0.0\n    fov: 45\n}\n\n"
            "material_lambertian {\n    name: \"base\"\n    diffuse: 0.1 0.2 0.8\n}\n\n"
            "material_clearcoat {\n    name: \"material0\"\n    base: \"base\"\n    ior: 1.3\n}\n\n"
            "sphere {\n    translate: 10.0 0.5 0.0\n    rotate: 0.0 1.0 0.0 45.0\n    scale: 10.0 10.0 10.0\n    material: \"material0\"\n}\n\n"
            "plane {\n    material: \"base\"\n}\n\n"
            "sphere_light {\n    translate: 10.0 15.0 0.0\n    radiance: 10.0 10.0 15.0\n}\n\n"
            "environment_light {\n    rotate: 0.0 1.0 0.0 45.0\n    radiance: 1.0 1.0 1.3\n}\n")


def sp_bunny(w: int, h: int, ply: str) -> str:
    """scenes/bunny.sp with the PLY path replaced."""
    meshes = ""
    for tx, mat in ((2.25, "material_glossy_clearcoat"), (0.75, "material_lambertian_clearcoat"),
                    (-0.75, "material_lambertian"), (-2.25, "material_glossy")):
        meshes += (f"mesh {{\n    file: \"{ply}\"\n    translate: {tx} 0.0 0.0\n    scale: 10.0 10.0 10.0\n"
                   f"    material: \"{mat}\"\n}}\n\n")
    return (_head(w, h) +
            "perspective_camera {\n    origin: 0.0 2.0 5.0\n    look_at: -0.25 1.0 0.0\n    fov: 45\n}\n\n" +
            _MATERIALS_SPHERES + "\n" + meshes +
            "plane {\n    material: \"material_glossy_plane\"\n    translate: 0.0 0.329874 0.0\n}\n\n"
            "sphere_light {\n    translate: 0.0 3.0 0.0\n    scale: 0.5 0.5 0.5\n    radiance: 10.0 10.0 10.0\n}\n")


def sp_elf(w: int, h: int, ply: str) -> str:
    """scenes/elf.sp with the commas of :11 removed and the STL replaced by a procedural PLY."""
    return (_head(w, h) +
            "perspective_camera {\n    origin: -1.79536 -0.0338669 130.0\n    look_at: -1.79536 -0.0338669 13.8378\n    fov: 45\n}\n\n" +
            _MATERIALS_STATUE + "\n" +
            f"mesh {{\n    file: \"{ply}\"\n    material: \"material_glossy_clearcoat\"\n}}\n\n"
            "plane {\n    material: \"material_glossy_plane\"\n    translate: 0.0 -42.7188 0.0\n}\n\n"
            "environment_light {\n    rotate: 0.0 1.0 0.0 45.0\n    radiance: 0.75 0.75 0.75\n}\n")


def sp_lucy(w: int, h: int, ply: str) -> str:
    """scenes/lucy.sp with the PLY path replaced."""
    return (_head(w, h) +
            "perspective_camera {\n    origin: 690.756 500.0 -2000.0\n    look_at: 690.756 200.0 192.627\n    fov: 45\n}\n\n" +
            _MATERIALS_STATUE + "\n" +
            f"mesh {{\n    file: \"{ply}\"\n    rotate: 1.0 0.0 0.0 -90.0\n    material: \"material_glossy_clearcoat\"\n}}\n\n"
            "plane {\n    material: \"material_glossy_plane\"\n    translate: 0.0 -605.893 0.0\n}\n\n"
            "environment_light {\n    rotate: 0.0 1.0 0.0 45.0\n    radiance: 1.0 1.0 1.3\n}\n")


def sp_chain(w: int, h: int, ply: str) -> str:
    """The chain mesh (deep BVH) seen from outside the cone, on a plane, under one sphere light."""
    return (_head(w, h) +
            "perspective_camera {\n    origin: 3.0 0.12 0.06\n    look_at: 0.0 0.0 0.0\n    fov: 30\n}\n\n" +
            _MATERIALS_SPHERES + "\n" +
            f"mesh {{\n    file: \"{ply}\"\n    scale: 1e-10 1e-10 1e-10\n    material: \"material_glossy\"\n}}\n\n"
            "plane {\n    material: \"material_lambertian\"\n    translate: 0.0 -0.25 0.0\n}\n\n"
            "sphere_light {\n    translate: 1.0 2.0 1.0\n    scale: 0.3 0.3 0.3\n    radiance: 10.0 10.0 10.0\n}\n")


def sp_many_lights(w: int, h: int) -> str:
    """Seven sphere lights + a constant environment: Scene's lights accelerator (base/Scene.h:29-45) becomes
    [environment, BVH(7 sphere lights)] with INTERNAL nodes (k_max_leaf_elements = 4), so Scene::intersect_lights walks
    NodeInternal::intersect_lights (shapes/BVHAccelerator.h:45-60).  Geometry: three spheres on a plane."""
    lights = ""
    for i, (x, y, z, r) in enumerate(((-3.0, 3.0, 1.0, 0.35), (-2.0, 4.0, -1.0, 0.25), (-0.8, 3.5, 2.0, 0.3), (0.5, 4.5, 0.0, 0.4),
                                      (1.6, 3.2, -2.0, 0.3), (2.6, 3.8, 1.5, 0.25), (3.4, 2.8, -0.5, 0.35))):
        c = (6.0 + 2.0 * (i % 3), 6.0 + 1.5 * ((i + 1) % 3), 6.0 + 2.5 * ((i + 2) % 3))
        lights += (f"sphere_light {{\n    translate: {x} {y} {z}\n    scale: {r} {r} {r}\n"
                   f"    radiance: {c[0]} {c[1]} {c[2]}\n}}\n\n")
    return (_head(w, h) +
            "perspective_camera {\n    origin: 0.0 2.5 9.0\n    look_at: 0.0 1.5 0.0\n    fov: 45\n}\n\n" +
            _MATERIALS_SPHERES + "\n" +
            "sphere {\n    translate: -2.0 1.0 0.0\n    material: \"material_glossy_clearcoat\"\n}\n\n"
            "sphere {\n    translate: 0.0 1.0 0.0\n    material: \"material_lambertian\"\n}\n\n"
            "sphere {\n    translate: 2.0 1.0 0.0\n    material: \"material_glossy\"\n}\n\n"
            "plane {\n    material: \"material_glossy_plane\"\n}\n\n" + lights +
            "environment_light {\n    rotate: 0.0 1.0 0.0 45.0\n    radiance: 0.2 0.2 0.25\n}\n")


# Stanford-bunny object-space bounds (public figures; consistent with the plane at y = 0.329874 after x10).
BUNNY_LO, BUNNY_HI = (-0.0947, 0.0329874, -0.0619), (0.0610, 0.1873, 0.0588)
# elf: stands on the plane at y = -42.7188, centred on the camera axis x = -1.795, z ~ 13.8
ELF_LO, ELF_HI = (-22.0, -42.7188, -4.0), (18.4, 42.6, 31.7)
# lucy is modelled z-up and rotated -90 deg about x by the scene; after rotation it should stand on
# y = -605.893 around (690.8, *, 192.6).  Object space: (x, y, z) -> world (x, z, -y).
LUCY_LO, LUCY_HI = (290.0, -420.0, -605.893), (1090.0, 35.0, 994.0)


# name -> (width, height, spp, builder)
def _specs():
    return {
        # BASELINE.json configs
        "c1_material_spheres": (256, 256, 16, lambda o: sp_material_spheres(256, 256, _pfm(o, 1024, 512))),
        "c1_material_spheres_const": (256, 256, 16, lambda o: sp_material_spheres(256, 256, "const")),
        "c2_example_scene": (1920, 1080, 64, lambda o: sp_example_scene(1920, 1080)),
        "c3_bunny": (1920, 1080, 256, lambda o: sp_bunny(1920, 1080, _ply(o, "bunny", BUNNY_TRIS, BUNNY_LO, BUNNY_HI))),
        "c4_elf": (1920, 1080, 256, lambda o: sp_elf(1920, 1080, _ply(o, "elf", ELF_TRIS, ELF_LO, ELF_HI))),
        "c5_lucy": (3840, 2160, 256, lambda o: sp_lucy(3840, 2160, _ply(o, "lucy", LUCY_TRIS, LUCY_LO, LUCY_HI))),
        # lucy.sp's camera / materials / plane / light at the config's resolution over a 40 K-triangle stand-in: what bench.py
        # flattens through the reference's parser before it swaps in the 28 M-triangle mesh built on the device
        "c5_lucy_standin": (3840, 2160, 256, lambda o: sp_lucy(3840, 2160, _ply(o, "lucy_small", 40_002, LUCY_LO, LUCY_HI))),
        # reduced sizes of the same scenes for parity tests (oracle finishes in seconds)
        "t_spheres_const": (96, 96, 8, lambda o: sp_material_spheres(96, 96, "const")),
        "t_spheres_ibl": (96, 96, 8, lambda o: sp_material_spheres(96, 96, _pfm(o, 128, 64))),
        "t_example": (160, 90, 8, lambda o: sp_example_scene(160, 90)),
        "t_bunny": (160, 90, 4, lambda o: sp_bunny(160, 90, _ply(o, "bunny_small", 5_001, BUNNY_LO, BUNNY_HI))),
        "t_bunny_full": (480, 270, 4, lambda o: sp_bunny(480, 270, _ply(o, "bunny", BUNNY_TRIS, BUNNY_LO, BUNNY_HI))),
        "t_elf": (120, 90, 4, lambda o: sp_elf(120, 90, _ply(o, "elf_small", 20_000, ELF_LO, ELF_HI))),
        "t_lucy": (128, 72, 4, lambda o: sp_lucy(128, 72, _ply(o, "lucy_small", 40_002, LUCY_LO, LUCY_HI))),
        # a million-triangle statue at the lucy framing: the >= 10^6-primitive parity case (tests/test_gpu_scale.py)
        "t_lucy_1m": (256, 144, 4, lambda o: sp_lucy(256, 144, _ply(o, "lucy_1m", 1_000_002, LUCY_LO, LUCY_HI))),
        # tiny versions whose flattened form is committed under tests/golden/ (tests/golden/make_golden.py)
        "g_spheres": (32, 32, 4, lambda o: sp_material_spheres(32, 32, "const")),
        "g_spheres_ibl": (32, 32, 4, lambda o: sp_material_spheres(32, 32, _pfm(o, 32, 16))),
        "g_example": (48, 27, 4, lambda o: sp_example_scene(48, 27)),
        "g_bunny": (48, 27, 4, lambda o: sp_bunny(48, 27, _ply(o, "bunny_tiny", 420, BUNNY_LO, BUNNY_HI))),
        "g_elf": (32, 24, 4, lambda o: sp_elf(32, 24, _ply(o, "elf_tiny", 1_500, ELF_LO, ELF_HI))),
        "g_chain": (32, 24, 4, lambda o: sp_chain(32, 24, _chain_ply(o, 58))),
        "g_lights": (32, 24, 4, lambda o: sp_many_lights(32, 24)),
    }


# Mesh scenes that host.assemble() puts together without the reference's parser: name -> (tiny scene of the same .sp text
# whose flattened form is committed, meshes in .sp order as (triangles, lo, hi, translate, uniform scale, material)).
# material = the flattener's index of the mesh's material: sp_bunny's four meshes use material_glossy_clearcoat,
# material_lambertian_clearcoat, material_lambertian and material_glossy; sp_elf's mesh material_glossy_clearcoat.
_BUNNY_MESHES = ((2.25, 6), (0.75, 4), (-0.75, 2), (-2.25, 1))
ASSEMBLED = {
    "c3_bunny": ("g_bunny", [(BUNNY_TRIS, BUNNY_LO, BUNNY_HI, (tx, 0.0, 0.0), 10.0, m) for tx, m in _BUNNY_MESHES]),
    "c4_elf": ("g_elf", [(ELF_TRIS, ELF_LO, ELF_HI, (0.0, 0.0, 0.0), 1.0, 2)]),
    "g_bunny": ("g_bunny", [(420, BUNNY_LO, BUNNY_HI, (tx, 0.0, 0.0), 10.0, m) for tx, m in _BUNNY_MESHES]),
    "g_elf": ("g_elf", [(1_500, ELF_LO, ELF_HI, (0.0, 0.0, 0.0), 1.0, 2)]),
}


def _ply(out: Path, stem: str, n_tris: int, lo, hi) -> str:
    path = out / f"{stem}_{n_tris}.ply"
    if not path.exists():
        v, f = bumpy_sphere(n_tris, lo, hi)
        write_ply(path, v, f)
    return path.name


def _chain_ply(out: Path, n_tris: int) -> str:
    path = out / f"chain_{n_tris}.ply"
    if not path.exists():
        v, f = chain_mesh(n_tris)
        write_ply(path, v, f)
    return path.name


def _pfm(out: Path, w: int, h: int) -> str:
    path = out / f"sky_{w}x{h}.pfm"
    if not path.exists():
        write_pfm(path, sky_image(w, h))
    return path.name


def names() -> list[str]:
    return list(_specs().keys())


def info(name: str) -> tuple[int, int, int]:
    w, h, spp, _ = _specs()[name]
    return w, h, spp


def ensure(name: str, out: Path | str = DEFAULT_OUT) -> Path:
    """Write <out>/<name>.sp (and the assets it references, beside it) if missing; return its path."""
    out = Path(out)
    out.mkdir(parents=True, exist_ok=True)
    w, h, spp, build = _specs()[name]
    path = out / f"{name}.sp"
    text = build(out)
    if not path.exists() or path.read_text() != text:
        tmp = out / f"{name}.sp.{os.getpid()}.tmp"
        tmp.write_text(text)
        os.replace(tmp, path)  # atomic: a concurrent rank never reads a half-written file
    return path


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=str(DEFAULT_OUT))
    ap.add_argument("names", nargs="*", default=[n for n in names() if n != "c5_lucy"])
    args = ap.parse_args()
    for n in args.names:
        print(ensure(n, args.out))


if __name__ == "__main__":
    main()
