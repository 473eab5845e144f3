"""Generates tests/golden/kino_search_golden.npz: polylines and closed-node counts of the host KinoAstar search (ualm_kino_astar_plan) on
the four seeded stand-in terrains and on the edge cases below.  Each polyline is stored as its point count and the SHA-256 of its float64
bytes (fingerprint()), which pins it bit for bit at 40 bytes per pair instead of kilobytes of raw doubles; the pairs themselves are
pinned by one SHA-256 per case.  It was run on the search as it stood before the search moved into
csrc/kino_search.h, so the golden pins the header-based host search (and, through it, the device search's host twin) to the original
std::priority_queue / std::unordered_map implementation.

cases() is imported by the tests, which rebuild the same maps and pairs from it:
  * <terrain>: 256 random pairs on maps.synthetic_terrain("bumps", STANDIN_SEED[terrain]) with the terrain's occupancy thresholds (about
    half of them have an occupied start or goal);
  * edges (hill's stand-in at max_rho 0.003, 9 % occupied): explicitly occupied starts and goals, starts and goals at yaw +-pi, a start walled in by an obstacle ring (the open set runs
    empty) and a goal walled in (the one-shot never clears, the pool fills);
  * small: a 40 x 40 crop of hill's stand-in; every other goal is walled in, so those searches end when the 1600-node pool fills;
  * altered: hill's stand-in at max_rho 0.003 with every A* parameter moved off its default (more primitives, finer yaw bins, other weights)."""
import ctypes as C
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "kino_search_golden.npz")
TERRAINS = ("hill", "desert", "volcano", "forest")


def with_occupancy(view, occ3, occ2):
    """view with its occupancy grids replaced (keeps the arrays alive)"""
    from uneven_planner_b200 import _lib
    u8 = C.POINTER(C.c_uint8)
    view.occ3 = np.ascontiguousarray(occ3, np.uint8); view.occ2 = np.ascontiguousarray(occ2, np.uint8)
    view.c = _lib.AstarMap(view.c.geom, view.c.cells, view.c.cells64, view.occ3.ctypes.data_as(u8), view.occ2.ctypes.data_as(u8))
    return view


def altered_params():
    from uneven_planner_b200 import front_end
    p = front_end.default_params()
    p.yaw_resolution = 0.4; p.lambda_heu = 1.3; p.weight_so2 = 0.8; p.weight_v_change = 0.3; p.weight_delta_change = 0.2
    p.weight_sigma = 25.0; p.time_interval = 0.25; p.collision_interval = 0.05; p.oneshot_range = 1.5; p.max_steer = 0.45
    p.max_vel = 0.7
    return p


def _pairs(rng, B, lo=-4.3, hi=4.3):
    s = np.column_stack([rng.uniform(lo, hi, B), rng.uniform(lo, hi, B), rng.uniform(-np.pi, np.pi, B)])
    e = np.column_stack([rng.uniform(lo, hi, B), rng.uniform(lo, hi, B), rng.uniform(-np.pi, np.pi, B)])
    return s, e


def _disc(g, shape, centre, r):
    cx = (np.arange(shape[0]) + 0.5) * g.xy_resolution + g.origin[0]
    cy = (np.arange(shape[1]) + 0.5) * g.xy_resolution + g.origin[1]
    return np.hypot(cx[:, None] - centre[0], cy[None, :] - centre[1]) < r


def _cell_centre(g, ix, iy):
    return [g.origin[0] + (ix + 0.5) * g.xy_resolution, g.origin[1] + (iy + 0.5) * g.xy_resolution]


def cases():
    """[(name, view, params, starts, goals)] -- deterministic; the views hold their maps"""
    from uneven_planner_b200 import _lib, configs, front_end, maps
    out = []
    for t in TERRAINS:
        m = maps.synthetic_terrain("bumps", seed=maps.STANDIN_SEED[t])
        view = front_end.MapView(m, configs.TERRAINS[t]["min_cnormal"], configs.TERRAINS[t]["max_rho"])
        s, e = _pairs(np.random.default_rng(1000 + maps.STANDIN_SEED[t]), 256)
        out.append((t, view, front_end.default_params(), s, e))

    hill = maps.synthetic_terrain("bumps", seed=maps.STANDIN_SEED["hill"])
    g = hill.geom
    base = front_end.MapView(hill, 0.8, 0.003)
    occ3, occ2 = base.occ3.copy(), base.occ2.copy()
    rng = np.random.default_rng(5)
    s, e = _pairs(rng, 48)
    free = np.argwhere(occ2 == 0)
    free = free[rng.permutation(len(free))]
    for k in range(8):                                   # starts on cells occupied in 3-D, goals on cells occupied in 2-D
        x3, y3, w3 = np.argwhere(occ3)[rng.integers(0, int(occ3.sum()))]
        s[k] = _cell_centre(g, x3, y3) + [g.origin[2] + (w3 + 0.5) * g.yaw_resolution]
        x2, y2 = np.argwhere(occ2)[rng.integers(0, int(occ2.sum()))]
        e[8 + k, :2] = _cell_centre(g, x2, y2)
    for k in range(16, 32):                              # yaw exactly +-pi on free cells
        fs, fg = free[2 * k], free[2 * k + 1]
        s[k] = _cell_centre(g, *fs) + [np.pi if k % 2 else -np.pi]
        e[k] = _cell_centre(g, *fg) + [-np.pi if k % 4 < 2 else np.pi]
    # a start walled in (open set runs empty) and a goal walled in (one-shot never clears: the 40000-node pool fills)
    for c in ((-3.0, -3.0), (3.0, 3.0)):
        wall = _disc(g, occ2.shape, c, 0.5) & ~_disc(g, occ2.shape, c, 0.35)
        inside = _disc(g, occ2.shape, c, 0.35)
        occ2[wall] = 1; occ3[wall] = 1
        occ2[inside] = 0; occ3[inside] = 0
    s[32:36] = [[-3.0, -3.0, 0.3], [-2.95, -3.05, -2.0], [-3.0, -3.0, np.pi], [-3.05, -2.9, 1.0]]
    e[32:36] = [[2.0, -1.0, 0.0], [1.0, 2.0, 1.0], [-1.0, 0.5, 2.0], [0.0, 0.0, 0.0]]
    s[36:38] = [[1.2, 1.6, 0.0], [0.8, 2.5, 2.0]]
    e[36:38] = [[3.0, 3.0, 0.5], [3.05, 2.95, -1.0]]
    out.append(("edges", with_occupancy(front_end.MapView(hill, 0.8, 0.003), occ3, occ2), front_end.default_params(), s, e))

    # every other goal walled in: those searches end when the pool fills
    sg = _lib.map_geometry(2.0, 2.0, 0.05, g.yaw_resolution)
    small = front_end.MapView(maps.UnevenMapData(sg, hill.cells[80:120, 80:120], "hill-standin-crop40"), 0.8, 0.003)
    occ3, occ2 = small.occ3.copy(), small.occ2.copy()
    wall = _disc(sg, occ2.shape, (0.5, 0.5), 0.35) & ~_disc(sg, occ2.shape, (0.5, 0.5), 0.25)
    occ2[wall] = 1; occ3[wall] = 1
    s, e = _pairs(np.random.default_rng(6), 64, -0.95, 0.95)
    e[::2, :2] = 0.5
    out.append(("small", with_occupancy(small, occ3, occ2), front_end.default_params(), s, e))

    s, e = _pairs(np.random.default_rng(7), 128)
    out.append(("altered", front_end.MapView(hill, 0.8, 0.003), altered_params(), s, e))
    return out


def run(plan, cs):
    """{key: array} of every case: the planner `plan(view, start, goal, params) -> (path, n_expanded)` over the case's pairs"""
    from concurrent.futures import ThreadPoolExecutor
    res = {}
    with ThreadPoolExecutor(os.cpu_count()) as ex:
        for name, view, p, s, e in cs:
            got = list(ex.map(lambda b: plan(view, s[b], e[b], p), range(len(s))))
            res[name + "/starts"] = s; res[name + "/goals"] = e
            res[name + "/lens"] = np.array([len(x[0]) for x in got])
            res[name + "/n_expanded"] = np.array([x[1] for x in got])
            res[name + "/paths"] = np.concatenate([x[0] for x in got]) if res[name + "/lens"].sum() else np.zeros((0, 3))
    return res


def _sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a, dtype="<f8").tobytes()).digest(), np.uint8)


def fingerprint(res):
    """run()'s output as the golden stores it: per case the SHA-256 of the pairs, the point counts, the closed-node counts and one
    SHA-256 per polyline"""
    out = {}
    for k in res:
        if not k.endswith("/lens"):
            continue
        n = k[:-5]
        off = np.concatenate([[0], np.cumsum(res[k])])
        out[n + "/pairs_sha256"] = _sha(np.concatenate([res[n + "/starts"], res[n + "/goals"]]))
        out[n + "/lens"] = res[k].astype(np.int32)
        out[n + "/n_expanded"] = res[n + "/n_expanded"].astype(np.int32)
        out[n + "/path_sha256"] = np.stack([_sha(res[n + "/paths"][off[b]:off[b + 1]]) for b in range(len(res[k]))])
    return out


if __name__ == "__main__":
    from uneven_planner_b200 import front_end
    res = run(front_end.plan, cases())
    np.savez_compressed(OUT, **fingerprint(res))
    for k in res:
        if k.endswith("/lens"):
            n = k[:-5]
            print(n, "pairs", len(res[k]), "with a path", int((res[k] > 0).sum()), "max closed", int(res[n + "/n_expanded"].max()))
