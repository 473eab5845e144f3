"""Host side of the boundary: input contract (PlanManager resampler), initial path generator, map geometry/builder,
and the C ABI surface (every symbol of include/ualm.h is exported; compute calls fail loudly without a GPU)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from uneven_planner_b200 import _lib, maps, problems

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_every_declared_symbol_is_exported(built):
    hdr = open(os.path.join(ROOT, "include", "ualm.h")).read()
    names = sorted(set(re.findall(r"\b(ualm_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 20
    L = C.CDLL(_lib.LIB_PATH)
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing


def test_compute_calls_fail_loudly_without_gpu(built):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = _lib.lib()
    h = C.c_void_p()
    rc = L.ualm_create(C.byref(h), 0, 64)
    assert rc == _lib.UALM_ENOCUDA
    assert b"CUDA" in L.ualm_last_error()


def test_unsupported_precision_is_rejected(built):
    L = _lib.lib()
    h = C.c_void_p()
    assert L.ualm_create(C.byref(h), 0, 16) == _lib.UALM_EINVAL


def test_map_geometry_matches_reference_rule(built):
    g = _lib.map_geometry()  # run_hill.yaml: 10 x 10 m, 0.05 m, 0.1 rad
    assert tuple(g.voxel_num) == (200, 200, 64)  # SURVEY 8a a8 / uneven_map.cpp:108-110
    assert g.origin[0] == -5.0 and abs(g.origin[2] + (np.pi + 0.025)) < 1e-15


def py_resample(path, piece_len=0.3, ypt=2.0, mean_vel=0.5, itt=1.2, isv=0.05):
    """independent Python restatement of plan_manager.cpp:62-122"""
    p = np.array(path, dtype=np.float64)
    for i in range(len(p) - 1):
        while p[i + 1, 2] - p[i, 2] >= np.pi / 2: p[i + 1, 2] -= 2 * np.pi
        while p[i + 1, 2] - p[i, 2] <= -np.pi / 2: p[i + 1, 2] += 2 * np.pi
    tly = tlp = tot = 0.0
    ply = piece_len / ypt
    xy, yaw = [], []
    for k in range(len(p) - 1):
        seg = np.hypot(*(p[k + 1, :2] - p[k, :2]))
        tly += seg; tlp += seg; tot += seg
        while tly > ply:
            yaw.append(p[k, 2] + (1.0 - (tly - ply) / seg) * (p[k + 1, 2] - p[k, 2])); tly -= ply
        while tlp > piece_len:
            xy.append(p[k, :2] + (1.0 - (tlp - piece_len) / seg) * (p[k + 1, :2] - p[k, :2])); tlp -= piece_len
    return len(xy) + 1, len(yaw) + 1, np.array(xy).ravel(), np.array(yaw), tot / mean_vel * itt, p


def test_resampler_matches_python_restatement(built):
    rng = np.random.default_rng(0)
    for trial in range(20):
        s = np.array([rng.uniform(-4, 4), rng.uniform(-4, 4), rng.uniform(-np.pi, np.pi)])
        e = np.array([rng.uniform(-4, 4), rng.uniform(-4, 4), rng.uniform(-np.pi, np.pi)])
        path = problems.dubins(s, e)
        N, M, bnd, T, ixy, iyaw = problems.resample(path)
        N2, M2, ixy2, iyaw2, T2, p = py_resample(path)
        assert (N, M) == (N2, M2)
        assert np.allclose(ixy, ixy2, atol=1e-14) and np.allclose(iyaw, iyaw2, atol=1e-14) and abs(T - T2) < 1e-12
        # boundary states: 0.05 m/s along the heading, zero acceleration (pm.cpp:80-94)
        assert np.allclose(bnd[:6], [p[0, 0], p[0, 1], 0.05 * np.cos(p[0, 2]), 0.05 * np.sin(p[0, 2]), 0, 0])
        assert np.allclose(bnd[12:15], [p[0, 2], 0, 0]) and np.allclose(bnd[15:18], [p[-1, 2], 0, 0])
        # derived sizes of SURVEY section 3.1
        L = np.hypot(np.diff(path[:, 0]), np.diff(path[:, 1])).sum()
        assert abs(N - (int(L / 0.3) + 1)) <= 1 and abs(M - (int(L / 0.15) + 1)) <= 1


def test_dubins_reaches_goal_with_bounded_curvature(built):
    rng = np.random.default_rng(3)
    for trial in range(50):
        s = np.array([rng.uniform(-4, 4), rng.uniform(-4, 4), rng.uniform(-np.pi, np.pi)])
        e = np.array([rng.uniform(-4, 4), rng.uniform(-4, 4), rng.uniform(-np.pi, np.pi)])
        path = problems.dubins(s, e, radius=0.6, ds=0.02)
        assert np.allclose(path[0, :2], s[:2]) and np.allclose(path[-1, :2], e[:2], atol=1e-9)
        d = np.hypot(np.diff(path[:-1, 0]), np.diff(path[:-1, 1]))
        assert np.all(d < 0.0201)
        dyaw = np.abs(np.angle(np.exp(1j * np.diff(path[:-1, 2]))))
        assert np.all(dyaw <= 0.02 / 0.6 + 1e-9)  # |kappa| <= 1/radius
        # heading is the path tangent (forward motion)
        mid = len(path) // 2
        tang = np.arctan2(path[mid + 1, 1] - path[mid, 1], path[mid + 1, 0] - path[mid, 0])
        assert abs(np.angle(np.exp(1j * (tang - path[mid, 2])))) < 0.03
        # the last sampled heading meets the goal heading
        assert abs(np.angle(np.exp(1j * (path[-2, 2] - e[2])))) < 0.05


def test_map_builder_on_analytic_cloud(built):
    """constructMap restatement: a cloud sampled from a tilted plane must give its normal, sigma ~ 0 and z on the plane."""
    rng = np.random.default_rng(0)
    a, b = 0.15, -0.1
    xy = rng.uniform(-5, 5, (300000, 2))
    pts = np.column_stack([xy, 1.0 + a * xy[:, 0] + b * xy[:, 1]]).astype(np.float32)
    m = maps.build_from_cloud(pts, nthreads=8)
    nrm = np.array([-a, -b, 1.0]) / np.sqrt(1 + a * a + b * b)
    inner = m.cells[20:180, 20:180]
    assert np.abs(inner[..., 2] - nrm[0]).max() < 2e-3 and np.abs(inner[..., 3] - nrm[1]).max() < 2e-3
    assert inner[..., 1].max() < 1e-6  # surface variation of an exact plane (float32 cloud -> ~1e-9)
    g = m.geom
    xs = (np.arange(200) + 0.5) * g.xy_resolution + g.origin[0]
    yaws = (np.arange(64) + 0.5) * g.yaw_resolution + g.origin[2]
    # z is the mean height of the points in the ellipsoid centred 0.12 m ahead of the cell (uneven_map.cpp:341-342)
    X, Y, W = np.meshgrid(xs, xs, yaws, indexing="ij")
    zexp = 1.0 + a * (X + 0.12 * np.cos(W)) + b * (Y + 0.12 * np.sin(W))
    err = np.abs(m.cells[20:180, 20:180, :, 0] - zexp[20:180, 20:180])  # sample mean of ~190 random points per footprint
    assert err.mean() < 2e-3 and err.max() < 3e-2
    occ3, occ2 = m.occupancy()
    assert occ2[20:180, 20:180].sum() == 0


def test_umap_file_roundtrip(built, tmp_path):
    m = maps.synthetic_terrain("bumps", seed=1)
    p = str(tmp_path / "t.umap")
    m.save(p)
    m2 = maps.UnevenMapData.load(p)
    assert np.array_equal(m.cells, m2.cells) and tuple(m2.geom.voxel_num) == (200, 200, 64)


def test_problem_generator_is_deterministic_and_valid(bumps_map):
    a = problems.generate(bumps_map, 16, seed=7)
    b = problems.generate(bumps_map, 16, seed=7)
    assert np.array_equal(a.N, b.N) and np.array_equal(a.inner_xy, b.inner_xy) and np.array_equal(a.bnd, b.bnd)
    assert a.N.min() >= 5 and a.N.max() <= 56 and np.all(a.M >= a.N)
    assert np.all(np.hypot(*(a.starts[:, :2] - a.goals[:, :2]).T) >= 1.5)
    sub = a.select([3, 5])
    assert np.array_equal(sub.x0(1), a.x0(5))


REF_PARAMS = "/root/reference/src/uneven_planner/plan_manager/params"


def test_config_table_matches_reference_yaml(built):
    """uneven_planner_b200/configs.py is the one table of per-terrain parameter deltas: re-derive it from the reference's own yaml
    files where they exist (this container; the GPU box has no /root/reference)."""
    if not os.path.isdir(REF_PARAMS):
        pytest.skip("the reference project's plan_manager/params/run_*.yaml are not part of this repository and not recorded under tests/golden/")
    import yaml
    from uneven_planner_b200 import configs
    keys = [n for n, _ in _lib.Params._fields_ if n != "gravity"]
    for name, fname in configs.YAML.items():
        y = yaml.safe_load(open(os.path.join(REF_PARAMS, fname)))
        node = y["manager_node"]
        alm, um = node["alm_traj_opt"], node["uneven_map"]
        p = configs.params_for(name, overrides=False)
        for k in keys:
            want = alm[k]
            want = (1 if want else 0) if isinstance(want, bool) else float(want)
            assert float(getattr(p, k)) == float(want), (name, k, getattr(p, k), want)
        assert p.gravity == float(um["gravity"])
        g = configs.gen_kwargs(name)
        assert g["max_rho"] == float(um["max_rho"]) and g["min_cnormal"] == float(um["min_cnormal"]), name
    # BASELINE config 4's overrides stay explicit, on top of run_vocano.yaml
    p4 = configs.params_for("volcano")
    assert p4.max_kap == 0.3 and p4.int_K == 64 and p4.max_sig == 0.08 and p4.use_scaling == 1
    pf = configs.params_for("forest")
    assert pf.use_scaling == 0 and pf.rho_T == 500.0 and pf.max_sig == 0.001


def test_snapshot_to_the_gpu_box_includes_every_map():
    """maps_built/*.umap travel with the gpurun snapshot (they cannot be rebuilt on the GPU box, which has no reference clouds): a
    development-time exclusion left in .gpurunignore would silently turn configs 3-5 into the synthetic fallback"""
    import os
    p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), ".gpurunignore")
    if os.path.exists(p):
        lines = [l.strip() for l in open(p) if l.strip() and not l.startswith("#")]
        assert not [l for l in lines if "maps_built" in l or "umap" in l or "libualm" in l or "_ref" in l], lines


def test_dubins_curves_reach_the_goal_with_every_word(built):
    """csrc/dubins.h through ualm_kino_astar_plan's one-shot is exercised by the A* pins; here the curve family itself: whatever word
    wins, walking it ends at the goal pose, it is at least as long as the straight line, and all six words occur"""
    import ctypes as C
    from uneven_planner_b200 import _lib, problems
    rng = np.random.default_rng(5)
    radius = 0.26 / np.tan(0.5)
    turns = set()
    for _ in range(300):
        s = np.array([rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(-np.pi, np.pi)])
        e = np.array([rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(-np.pi, np.pi)])
        p = problems.dubins(s, e, radius=radius, ds=0.01)
        seg = np.hypot(np.diff(p[:, 0]), np.diff(p[:, 1])).sum()
        assert seg >= np.hypot(*(e[:2] - s[:2])) - 1e-9
        assert np.hypot(*(p[-1, :2] - e[:2])) < 1e-9 and abs(np.angle(np.exp(1j * (p[-1, 2] - e[2])))) < 1e-6
        assert np.hypot(*(p[-2, :2] - e[:2])) <= 0.01 + 1e-9          # the sampled curve itself arrives there, not only the appended goal
        dyaw = np.diff(np.unwrap(p[:-1, 2]))
        sign = np.sign(np.round(dyaw, 9))
        runs = [int(v) for k, v in enumerate(sign) if v != 0 and (k == 0 or sign[k - 1] != v)]
        turns.add(tuple(runs[:3]))
        # the front-end's own curve (csrc/dubins.h, the restatement of OMPL's DubinsStateSpace) describes the same shortest curve
        buf = np.zeros((4096, 3)); ln = C.c_double()
        dp = C.POINTER(C.c_double)
        n = _lib.lib().ualm_dubins_shot(s.ctypes.data_as(dp), e.ctypes.data_as(dp), radius, 0.01, buf.ctypes.data_as(dp), 4096, C.byref(ln))
        assert n >= 1 and abs(ln.value - (len(p) - 2) * 0.01) <= 0.01 + 1e-9 and np.allclose(buf[0], [s[0], s[1], np.angle(np.exp(1j * s[2]))], atol=1e-12)
        m_ = min(n, len(p) - 1)
        assert np.abs(buf[:m_, :2] - p[:m_, :2]).max() < 1e-8
    assert {(1,), (-1,), (1, -1), (-1, 1)} <= turns or len(turns) >= 4


def test_front_end_batch_equals_the_sequential_front_end(built, bumps_map):
    """ualm_front_end_batch = KinoAstar::plan + PlanManager's resampler per pair, whatever the number of host threads; pairs without a
    path are left out and reported"""
    from uneven_planner_b200 import front_end, problems
    view = front_end.MapView(bumps_map, 0.8, 0.003)
    rng = np.random.default_rng(2)
    B = 24
    starts = np.column_stack([rng.uniform(-4.3, 4.3, B), rng.uniform(-4.3, 4.3, B), rng.uniform(-np.pi, np.pi, B)])
    goals = np.column_stack([rng.uniform(-4.3, 4.3, B), rng.uniform(-4.3, 4.3, B), rng.uniform(-np.pi, np.pi, B)])
    ox, oy = np.argwhere(view.occ2)[7]
    g = bumps_map.geom
    goals[5, :2] = [g.origin[0] + (ox + 0.5) * g.xy_resolution, g.origin[1] + (oy + 0.5) * g.xy_resolution]      # goal inside an obstacle
    pb1, packed1, nexp1 = front_end.plan_batch(view, starts, goals, nthreads=1)
    pb4, packed4, nexp4 = front_end.plan_batch(view, starts, goals, nthreads=4)
    assert np.array_equal(packed1, packed4) and np.array_equal(nexp1, nexp4)
    for a, b in zip((pb1.N, pb1.M, pb1.bnd, pb1.total_time, pb1.inner_xy, pb1.inner_yaw), (pb4.N, pb4.M, pb4.bnd, pb4.total_time, pb4.inner_xy, pb4.inner_yaw)):
        assert np.array_equal(a, b)
    assert packed1[5] == -1 and (packed1 >= 0).sum() == pb1.B >= B // 2
    oxy, oyaw, _, _ = pb1.offsets()
    for b in range(B):
        path, nexp = front_end.plan(view, starts[b], goals[b])
        assert nexp == nexp1[b]
        k = packed1[b]
        if k < 0:
            assert len(path) < 2 or problems.resample(path)[0] > 64 or problems.resample(path)[1] > 128
            continue
        N, M, bnd, T, ixy, iyaw = problems.resample(path)
        assert (N, M, T) == (pb1.N[k], pb1.M[k], pb1.total_time[k]) and np.array_equal(bnd, pb1.bnd[k])
        assert np.array_equal(ixy, pb1.inner_xy[oxy[k]:oxy[k + 1]]) and np.array_equal(iyaw, pb1.inner_yaw[oyaw[k]:oyaw[k + 1]])


def test_astar_workload_generator_is_deterministic(built, bumps_map):
    """problems.generate_astar: same (map, B, seed) -> same batch whatever the thread count; every problem within the optimizer's limits"""
    from uneven_planner_b200 import problems
    a = problems.generate_astar(bumps_map, 24, seed=4, max_rho=0.003, nthreads=1)
    b = problems.generate_astar(bumps_map, 24, seed=4, max_rho=0.003, nthreads=3)
    assert a.B == b.B == 24
    for x, y in zip((a.N, a.M, a.bnd, a.total_time, a.inner_xy, a.inner_yaw, a.starts, a.goals), (b.N, b.M, b.bnd, b.total_time, b.inner_xy, b.inner_yaw, b.starts, b.goals)):
        assert np.array_equal(x, y)
    assert a.N.max() <= 64 and a.M.max() <= 128 and a.N.min() >= 1


def test_kino_astar_reproduces_the_reference_golden_paths(built, bumps_map):
    """tests/golden/kino_astar_golden.npz holds the polylines of the reference's own KinoAstar::plan (kino_astar.cpp compiled unmodified, see
    tests/golden/make_kino_golden.py) on the synthetic terrain: ualm_kino_astar_plan returns them bit for bit -- also where /root/reference and the
    reference build are absent"""
    import os
    from uneven_planner_b200 import front_end
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kino_astar_golden.npz"))
    view = front_end.MapView(bumps_map, float(gold["min_cnormal"]), float(gold["max_rho"]))
    off = np.concatenate([[0], np.cumsum(gold["lens"])])
    nonempty = 0
    for b in range(len(gold["lens"])):
        path, _ = front_end.plan(view, gold["starts"][b], gold["goals"][b])
        want = gold["paths"][off[b]:off[b + 1]]
        assert path.shape == want.shape and np.array_equal(path, want), b
        nonempty += len(want) > 0
    assert nonempty >= 6
