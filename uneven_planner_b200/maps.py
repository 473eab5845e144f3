"""UnevenMap inputs: .pcd reader, map construction (host threads via libualm), own binary map file,
and analytic synthetic terrains for tests.

The reference builds the SE(2)->(z, sigma, z_b) grid once per terrain and caches it as CSV
(uneven_map/src/uneven_map.cpp:270-315, 400-412; 6 significant digits).  This repo caches a binary
`.umap` file instead: 64-byte header + float32 cells [X][Y][Yaw][4] in the reference address order
(uneven_map.h:427-435).  float32 (7 significant digits) is what BOTH the CPU oracle and the GPU path
consume, so cached and freshly built runs are identical (the reference's are not: SURVEY Q9).
"""
import ctypes as C
import os
import struct

import numpy as np

from . import _lib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BUILT_DIR = os.path.join(ROOT, "maps_built")          # git-ignored, travels with gpurun snapshots
REF_MAPS = "/root/reference/src/uneven_planner/uneven_map/maps"   # only present in the build container
MAGIC = b"UMAP0001"

# per-terrain cloud files and occupancy thresholds live in configs.TERRAINS (one table, derived from the reference's yaml files)
from .configs import TERRAINS  # noqa: E402


class UnevenMapData:
    """Geometry + float32 cells [X,Y,Yaw,4] = (z, sigma, zbx, zby)."""

    def __init__(self, geom, cells, name="map", cells64=None):
        self.geom = geom
        self.cells = np.ascontiguousarray(cells, dtype=np.float32)
        # optional: the reference's own grid (RXS2 = 4 doubles per cell, uneven_map.h:36-64) for maps built in-process by the
        # reference; consumers that can (ualm_set_map_f64, the oracle) read it instead of the float32 copy
        self.cells64 = None if cells64 is None else np.ascontiguousarray(cells64, dtype=np.float64)
        self.name = name
        X, Y, W = geom.voxel_num
        assert self.cells.shape == (X, Y, W, 4), self.cells.shape
        self._occ = {}

    @property
    def shape(self):
        return tuple(self.geom.voxel_num)

    def occupancy(self, min_cnormal=0.8, max_rho=0.05):
        key = (min_cnormal, max_rho)
        if key not in self._occ:
            X, Y, W = self.shape
            occ3 = np.zeros((X, Y, W), np.uint8)
            occ2 = np.zeros((X, Y), np.uint8)
            rc = _lib.lib().ualm_map_occupancy(self.cells.ctypes.data_as(C.POINTER(C.c_float)), C.byref(self.geom),
                                               min_cnormal, max_rho, occ3.ctypes.data_as(C.POINTER(C.c_uint8)),
                                               occ2.ctypes.data_as(C.POINTER(C.c_uint8)))
            assert rc == 0
            self._occ[key] = (occ3, occ2)
        return self._occ[key]

    def save(self, path):
        g = self.geom
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path + ".tmp", "wb") as f:
            hdr = MAGIC + struct.pack("<3i", *g.voxel_num) + struct.pack("<4d", abs(g.origin[0]) * 2, abs(g.origin[1]) * 2,
                                                                       g.xy_resolution, g.yaw_resolution)
            f.write(hdr.ljust(64, b"\0"))
            f.write(self.cells.tobytes())
        os.replace(path + ".tmp", path)

    @staticmethod
    def load(path, name=None):
        with open(path, "rb") as f:
            hdr = f.read(64)
            assert hdr[:8] == MAGIC, "not a .umap file"
            X, Y, W = struct.unpack("<3i", hdr[8:20])
            sx, sy, rx, ry = struct.unpack("<4d", hdr[20:52])
            geom = _lib.map_geometry(sx, sy, rx, ry)
            assert tuple(geom.voxel_num) == (X, Y, W)
            cells = np.frombuffer(f.read(), dtype=np.float32).reshape(X, Y, W, 4)
        return UnevenMapData(geom, cells, name or os.path.basename(path))


def read_pcd_xyz(path):
    """Minimal PCD reader (ASCII header, DATA binary, float32 fields; only x,y,z are used like
    pcl::PointXYZ in uneven_map.cpp:127-131)."""
    with open(path, "rb") as f:
        raw = f.read()
    hdr_end = raw.index(b"DATA")
    hdr_end = raw.index(b"\n", hdr_end) + 1
    hdr = raw[:hdr_end].decode("ascii", "replace").splitlines()
    kv = {l.split()[0]: l.split()[1:] for l in hdr if l and not l.startswith("#")}
    assert kv["DATA"] == ["binary"], kv["DATA"]
    fields, sizes, counts = kv["FIELDS"], list(map(int, kv["SIZE"])), list(map(int, kv["COUNT"]))
    assert all(s == 4 for s in sizes) and all(c == 1 for c in counts) and set(kv["TYPE"]) == {"F"}
    n = int(kv["POINTS"][0])
    arr = np.frombuffer(raw, dtype=np.float32, count=n * len(fields), offset=hdr_end).reshape(n, len(fields))
    ix = [fields.index(k) for k in ("x", "y", "z")]
    return np.ascontiguousarray(arr[:, ix])


def build_from_cloud(pts, geom=None, ellipsoid=(0.2, 0.1, 0.1), iter_num=2, nthreads=0, name="map"):
    geom = geom or _lib.map_geometry()
    X, Y, W = geom.voxel_num
    cells = np.zeros((X, Y, W, 4), np.float32)
    pts = np.ascontiguousarray(pts, dtype=np.float32)
    rc = _lib.lib().ualm_map_build(pts.ctypes.data_as(C.POINTER(C.c_float)), pts.shape[0], C.byref(geom),
                                   ellipsoid[0], ellipsoid[1], ellipsoid[2], iter_num, nthreads,
                                   cells.ctypes.data_as(C.POINTER(C.c_float)))
    if rc != 0:
        raise RuntimeError(f"ualm_map_build failed: {rc}")
    return UnevenMapData(geom, cells, name)


def terrain_path(name):
    return os.path.join(BUILT_DIR, f"{name}.umap")


def get_terrain(name, build_if_missing=True):
    """Load maps_built/<name>.umap; in the build container (reference present) build it from the
    reference's .pcd cloud on first use.  Returns None when neither exists (GPU box without the file)."""
    p = terrain_path(name)
    if os.path.exists(p):
        return UnevenMapData.load(p, name)
    pcd = os.path.join(REF_MAPS, TERRAINS[name]["pcd"])
    if build_if_missing and os.path.exists(pcd):
        m = build_from_cloud(read_pcd_xyz(pcd), name=name)
        m.save(p)
        return m
    return None


# Seeded synthetic stand-ins of the reference's terrains, for tests where maps_built/<name>.umap cannot be had (the reference's
# point clouds are not part of this repository).  hill's stand-in is the terrain bench.py falls back to.
STANDIN_SEED = {"hill": 0, "desert": 1, "volcano": 2, "forest": 4}


def terrain_or_standin(name):
    """The reference terrain `name` when its .umap exists (or can be built), else its seeded synthetic stand-in.  A stand-in is
    NOT the reference terrain: results on it compare implementations with each other, not with the reference's maps."""
    return get_terrain(name) or synthetic_terrain("bumps", seed=STANDIN_SEED[name])


def synthetic_terrain(kind="bumps", seed=0, size=(200, 200, 64)):
    """Analytic terrain z = h(x,y) turned into the same grid the builder produces (normal of the surface
    at the 0.12 m forward-shifted footprint centre, sigma from curvature).  Used by tests and as a clearly
    labelled fallback when no .umap file is available; NOT one of the reference's terrains."""
    geom = _lib.map_geometry()
    X, Y, W = geom.voxel_num
    xs = (np.arange(X) + 0.5) * geom.xy_resolution + geom.origin[0]
    ys = (np.arange(Y) + 0.5) * geom.xy_resolution + geom.origin[1]
    yaws = (np.arange(W) + 0.5) * geom.yaw_resolution + geom.origin[2]
    gx, gy, gw = np.meshgrid(xs, ys, yaws, indexing="ij")
    px = gx + 0.12 * np.cos(gw)
    py = gy + 0.12 * np.sin(gw)
    rng = np.random.default_rng(seed)
    if kind == "flat":
        z = np.zeros_like(px); hx = np.zeros_like(px); hy = np.zeros_like(px); lap = np.zeros_like(px)
    elif kind == "tilt":
        a, b = 0.2, -0.1
        z = a * px + b * py; hx = np.full_like(px, a); hy = np.full_like(px, b); lap = np.zeros_like(px)
    else:
        z = np.zeros_like(px); hx = np.zeros_like(px); hy = np.zeros_like(px); lap = np.zeros_like(px)
        for _ in range(6):
            cx, cy = rng.uniform(-4, 4, 2)
            amp = rng.uniform(0.2, 0.8) * rng.choice([-1, 1])
            s = rng.uniform(0.9, 2.0)
            e = amp * np.exp(-((px - cx) ** 2 + (py - cy) ** 2) / (2 * s * s))
            z += e
            hx += -e * (px - cx) / (s * s)
            hy += -e * (py - cy) / (s * s)
            lap += e * (((px - cx) ** 2 + (py - cy) ** 2) / s ** 4 - 2 / s ** 2)
    nrm = np.sqrt(hx * hx + hy * hy + 1.0)
    cells = np.stack([z, 0.01 * np.abs(lap) / (1 + np.abs(lap)), -hx / nrm, -hy / nrm], axis=-1).astype(np.float32)
    return UnevenMapData(geom, cells, f"synthetic-{kind}")
