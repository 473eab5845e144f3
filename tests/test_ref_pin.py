"""Pins of the oracle against the REFERENCE'S OWN SOURCE TEXT.

oracle/_ref/libref.so is back_end/include/utils/{se2traj,banded_system,lbfgs}.hpp compiled unmodified from /root/reference
against oracle/shim (a minimal Eigen stand-in; Eigen and ROS are absent from this image) by `make -C oracle ref`
(oracle/ref_driver.cpp).  These tests feed identical seeded inputs to that build and to the oracle's restatement
(oracle/oracle.cpp) and require BIT-IDENTICAL outputs for MinJerkOpt<1|2>::generate / getTrajJerkCost / calJerkGradCT /
calGradCTtoQT (SURVEY 8a rows a4-a6, a9, through BandedSystem a5) and for lbfgs_optimize + line_search_lewisoverton with the
reference's local modifications (row a2, quirk Q8).  The shim fixes what the reference leaves to Eigen: dot()/norm() in the
oracle's canonical 32-lane order, sum() in element order (oracle/shim/Eigen/Eigen header comment).

Every test here needs oracle/_ref/, which only `make -C oracle ref` builds from a checkout of the reference project; that project is
not part of this repository, so on a checkout without that build each of them skips and says so.  Their reference outputs are not
stored under tests/golden/ yet: recording them needs that build.  tests/golden/make_kino_golden.py is the pattern, and so far only
KinoAstar's paths are recorded (tests/test_host_tools.py::test_kino_astar_reproduces_the_reference_golden_paths)."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "libref.so")
NO_REF = ("oracle/_ref/%s not built: it is compiled from the reference project's sources (make -C oracle ref), which are not part of "
          "this repository, and its outputs are not recorded under tests/golden/")
dp = C.POINTER(C.c_double)


def P(a):
    return None if a is None else a.ctypes.data_as(dp)


@pytest.fixture(scope="module")
def ref(built):
    if os.path.isdir("/root/reference/src/uneven_planner/back_end/include"):
        import subprocess
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "-s", "ref"], check=True)
    if not os.path.exists(REF):
        pytest.skip(NO_REF % "libref.so")
    L = C.CDLL(REF)
    L.ref_minco.restype = C.c_int
    L.ref_minco.argtypes = [C.c_int, C.c_int, dp, dp, dp, dp, dp, dp, dp, dp, dp, dp, dp]
    L.ref_banded.argtypes = [C.c_int, C.c_int, C.c_int, dp, dp, C.c_int, C.c_int]
    L.ref_lbfgs_rosenbrock.argtypes = [C.c_int, dp, dp, C.c_int, C.c_double, C.c_int, C.c_double, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    return L


@pytest.fixture(scope="module")
def orc(built):
    import pyoracle as po
    L = po.lib()
    L.orc_minco_generate.argtypes = [C.c_int, C.c_int, dp, dp, dp, dp, dp]
    L.orc_minco_jerk.restype = C.c_double
    L.orc_minco_jerk.argtypes = [C.c_int, C.c_int, dp, dp, dp, dp]
    L.orc_minco_grad_ct_to_qt.argtypes = [C.c_int, C.c_int, dp, dp, dp, dp, dp, dp, dp]
    L.orc_lbfgs_rosenbrock.argtypes = [C.c_int, dp, dp, C.c_int, C.c_double, C.c_int, C.c_double, C.POINTER(C.c_int)]
    return L


@pytest.mark.parametrize("Dim", [1, 2])
@pytest.mark.parametrize("N,uniform", [(1, True), (2, False), (5, True), (21, True), (21, False), (64, True)])
def test_minco_headers_match_oracle_bitwise(ref, orc, Dim, N, uniform):
    rng = np.random.default_rng(100 * N + Dim)
    inPs = rng.normal(0, 2.0, Dim * max(N - 1, 1))[:Dim * (N - 1)].copy()
    ts = np.full(N, rng.uniform(0.3, 1.2)) if uniform else rng.uniform(0.3, 1.2, N)
    head = rng.normal(0, 1.0, Dim * 3); tail = rng.normal(0, 1.0, Dim * 3)
    gdC_in = rng.normal(0, 1.0, 6 * N * Dim); gdT0 = rng.normal(0, 1.0, N)
    # reference headers
    c_r = np.zeros(6 * N * Dim); jerk_r = np.zeros(1); gC_r = np.zeros(6 * N * Dim); gT_r = np.zeros(N)
    gdT_r = gdT0.copy(); gdP_r = np.zeros(max(Dim * (N - 1), 1))
    assert ref.ref_minco(Dim, N, P(inPs) if N > 1 else P(np.zeros(1)), P(ts), P(head), P(tail), P(c_r), P(jerk_r), P(gC_r), P(gT_r),
                         P(gdC_in), P(gdT_r), P(gdP_r)) == 0
    # oracle restatement
    c_o = np.zeros(6 * N * Dim)
    orc.orc_minco_generate(Dim, N, P(inPs) if N > 1 else P(np.zeros(1)), P(ts), P(head), P(tail), P(c_o))
    gC_o = np.zeros(6 * N * Dim); gT_o = np.zeros(N)
    jerk_o = orc.orc_minco_jerk(Dim, N, P(c_o), P(ts), P(gC_o), P(gT_o))
    gdT_o = gdT0.copy(); gdP_o = np.zeros(max(Dim * (N - 1), 1))
    orc.orc_minco_grad_ct_to_qt(Dim, N, P(inPs) if N > 1 else P(np.zeros(1)), P(ts), P(head), P(tail), P(gdC_in), P(gdT_o), P(gdP_o))
    assert np.array_equal(c_r, c_o)                        # generate: banded fill, factorizeLU, solve
    assert jerk_r[0] == jerk_o                             # getTrajJerkCost
    assert np.array_equal(gC_r, gC_o) and np.array_equal(gT_r, gT_o)     # calJerkGradCT
    assert np.array_equal(gdT_r, gdT_o) and np.array_equal(gdP_r[:Dim * (N - 1)], gdP_o[:Dim * (N - 1)])   # calGradCTtoQT (solveAdj)
    # and the solution is a solution: waypoints interpolated, boundary states met
    cm = c_r.reshape(Dim, 6 * N)
    assert np.allclose(cm[:, 0], head[:Dim]) and np.allclose(cm[:, 1], head[Dim:2 * Dim])


def test_banded_system_header_solves(ref):
    """BandedSystem (banded_system.hpp:25-145) of the reference build on a random diagonally dominant band matrix: solve and
    adjoint solve against numpy."""
    rng = np.random.default_rng(7)
    n, lo, up, m = 30, 6, 6, 2
    A = np.zeros((n, n))
    for i in range(n):
        for j in range(max(0, i - lo), min(n, i + up + 1)):
            A[i, j] = rng.normal()
        A[i, i] += 20.0
    b = rng.normal(size=(n, m))
    for adj in (0, 1):
        x = np.asfortranarray(b.copy())
        ref.ref_banded(n, lo, up, P(np.ascontiguousarray(A)), P(x), m, adj)
        want = np.linalg.solve(A.T if adj else A, b)
        assert np.allclose(x, want, rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("n,mem,past", [(2, 8, 3), (10, 8, 3), (20, 256, 3), (6, 4, 0)])
def test_lbfgs_header_matches_oracle_bitwise(ref, orc, n, mem, past):
    """lbfgs_optimize + line_search_lewisoverton of lbfgs.hpp (with the reference's own modifications, lbfgs.hpp:327-330) against
    the oracle's restatement on the Rosenbrock function: same return code, iteration count, final point and value, bit for bit."""
    x0 = np.tile([-1.2, 1.0], n // 2).astype(np.float64)
    xr = x0.copy(); fr = np.zeros(1); ir = C.c_int(); er = C.c_int()
    rr = ref.ref_lbfgs_rosenbrock(n, P(xr), P(fr), mem, 1e-6, past, 1e-6, C.byref(ir), C.byref(er))
    xo = x0.copy(); fo = np.zeros(1); io = C.c_int()
    ro = orc.orc_lbfgs_rosenbrock(n, P(xo), P(fo), mem, 1e-6, past, 1e-6, C.byref(io))
    assert rr == ro and ir.value == io.value
    assert fr[0] == fo[0] and np.array_equal(xr, xo)
    assert fr[0] < 1e-6 and np.allclose(xr, 1.0, atol=1e-2)


# ---------------------------------------------------------------------------------------------------------------------
# the whole path: ALMTrajOpt::optimizeSE2Traj of back_end/src/alm_traj_opt.cpp (unmodified) vs the oracle
# ---------------------------------------------------------------------------------------------------------------------
class RefParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("rho_T", "rho_ter", "max_vel", "max_acc_lon", "max_acc_lat", "max_kap", "min_cxi", "max_sig")] + \
               [("use_scaling", C.c_int)] + \
               [(n, C.c_double) for n in ("rho", "beta", "gamma", "epsilon_con", "max_iter", "g_epsilon", "min_step", "inner_max_iter", "delta")] + \
               [("mem_size", C.c_int), ("past", C.c_int), ("int_K", C.c_int), ("gravity", C.c_double)]


def _ref_solve(L, params, mapdata, pb, i):
    g = mapdata.geom
    rp = RefParams()
    for n, _ in RefParams._fields_:
        setattr(rp, n, getattr(params, n))
    cells = np.ascontiguousarray(mapdata.cells, dtype=np.float64)
    N, M = int(pb.N[i]), int(pb.M[i])
    S = N * (params.int_K + 1)
    oxy, oyaw, _, _ = pb.offsets()
    ixy = np.ascontiguousarray(pb.inner_xy[oxy[i]:oxy[i + 1]]); iyaw = np.ascontiguousarray(pb.inner_yaw[oyaw[i]:oyaw[i + 1]])
    out = dict(c_xy=np.zeros(12 * N), c_yaw=np.zeros(6 * M), piece_T=np.zeros(2), lam=np.zeros(S), mu=np.zeros(6 * S), hx=np.zeros(S),
               gx=np.zeros(6 * S), sfx=np.zeros(1), scx=np.zeros(7 * S), rho=np.zeros(1), feas=np.zeros(7))
    vn = (C.c_int * 3)(*g.voxel_num); org = (C.c_double * 3)(*g.origin); mxb = (C.c_double * 3)(*g.max_boundary)
    L.ref_alm_solve.restype = C.c_int
    ret = L.ref_alm_solve(C.byref(rp), P(cells), vn, org, mxb, C.c_double(g.xy_resolution), C.c_double(g.yaw_resolution), N, M,
                          P(np.ascontiguousarray(pb.bnd[i])), C.c_double(float(pb.total_time[i])), P(ixy if ixy.size else np.zeros(1)),
                          P(iyaw if iyaw.size else np.zeros(1)), 0, P(out["c_xy"]), P(out["c_yaw"]), P(out["piece_T"]), P(out["lam"]), P(out["mu"]),
                          P(out["hx"]), P(out["gx"]), P(out["sfx"]), P(out["scx"]), P(out["rho"]), P(out["feas"]))
    return ret, out


@pytest.mark.parametrize("which,use_scaling", [("bumps", 1), ("bumps", 0), ("hill", 1), ("volcano", 1), ("forest", 0)])
def test_reference_optimizeSE2Traj_matches_oracle_bitwise(ref, built, request, which, use_scaling):
    """ALMTrajOpt::optimizeSE2Traj compiled from the reference's alm_traj_opt.cpp (innerCallback, calConstrainCostGrad, initScaling,
    earlyExit, dual update, UnevenMap::getAllWithGrad, MINCO, L-BFGS) against oracle.cpp on the same problems: return code,
    coefficients, piece durations, multipliers, constraint values, scales and the final rho, all bit-identical."""
    import pyoracle as po
    from uneven_planner_b200 import _lib, maps, problems
    from uneven_planner_b200 import configs
    m = request.getfixturevalue("bumps_map") if which == "bumps" else maps.get_terrain(which)
    if m is None:
        pytest.skip(which + ".umap not present")
    if which in ("volcano", "forest"):
        # BASELINE config 4: run_vocano.yaml (max_sig 0.08) + max_kap 0.3 + 64 samples per piece on the volcano terrain;
        # config 5: run_forest.yaml (no scaling, rho_T 500, max_sig 0.001) on the forest terrain
        params = configs.params_for(which)
        assert params.use_scaling == use_scaling
        pb = problems.generate(m, 2 if which == "volcano" else 3, seed=11, **configs.gen_kwargs(which))
    else:
        params = _lib.default_params()
        params.use_scaling = use_scaling
        if not use_scaling:
            params.rho_T = 500.0
        pb = problems.generate(m, 6, seed=11)
    om = po.OracleMap(m)
    op = po.params_from(params)
    for i in range(pb.B):
        ret, out = _ref_solve(ref, params, m, pb, i)
        r, ocxy, ocyaw, _, olam, omu, oscx = po.solve_one(op, om, pb, i, want_duals=True)
        assert ret == r.ret_code, i
        assert np.array_equal(out["c_xy"], ocxy) and np.array_equal(out["c_yaw"], ocyaw), i
        tt = 0.0
        for _ in range(int(pb.N[i])):
            tt += out["piece_T"][0]
        assert tt == r.total_T and out["rho"][0] == r.rho_final and out["sfx"][0] == r.scale_fx, i
        assert np.array_equal(out["lam"], olam) and np.array_equal(out["mu"], omu) and np.array_equal(out["scx"], oscx), i
        assert max(np.abs(out["hx"]).max(), 0.0) == r.res_h, i      # judgeConvergence's first norm, from the reference's own hx
        # the reference's own post-solve report (getMaxVxAxAyCurAttSig + getNonHolError) against orc_feasibility on its trajectory
        of = po.feasibility(om, params.gravity, int(pb.N[i]), int(pb.M[i]), out["c_xy"], out["c_yaw"], out["piece_T"][0], out["piece_T"][1], 0.01)
        assert np.array_equal(out["feas"], of[:7]), (i, out["feas"], of)


# ---------------------------------------------------------------------------------------------------------------------
# the caller of the path: PlanManager::rcvWpsCallBack of plan_manager/src/plan_manager.cpp (unmodified)
# ---------------------------------------------------------------------------------------------------------------------
def _poly(c, t):
    """Piece::getValue (se2traj.hpp:106-118) on coefficients low -> high."""
    v, tn = 0.0, 1.0
    for k in range(6):
        v += tn * c[k]
        tn *= t
    return v


def _end_value(c, P, dur):
    """PolyTrajectory::getValue(getTotalDuration()) (se2traj.hpp:291-300, 343-367) of a P-piece spline with uniform durations."""
    total = 0.0
    for _ in range(P):
        total += dur
    t, idx = total, 0
    while idx < P and t > dur:
        t -= dur
        idx += 1
    if idx == P:
        idx -= 1
        t += dur
    return _poly(c[6 * idx:6 * idx + 6], t)


@pytest.mark.parametrize("seed", [3, 4])
def test_reference_plan_manager_callback_matches_host_tools_and_oracle(ref, built, bumps_map, seed):
    """PlanManager::rcvWpsCallBack of the reference (yaw unwrapping + arc-length resampling pm.cpp:62-122, optimizeSE2Traj, SE2Traj
    message pm.cpp:151-185) fed with a front-end polyline, against ualm_resample_path + the oracle solve + the message layout of
    include/ualm_traj_opt.hpp::toSE2TrajMsg: piece start points, end points and durations of both splines, bit for bit."""
    import pyoracle as po
    from uneven_planner_b200 import _lib, problems
    params = _lib.default_params()
    pb = problems.generate(bumps_map, 3, seed=seed)
    op = po.params_from(params)
    om = po.OracleMap(bumps_map)
    g = bumps_map.geom
    rp = RefParams()
    for n, _ in RefParams._fields_:
        setattr(rp, n, getattr(params, n))
    cells = np.ascontiguousarray(bumps_map.cells, dtype=np.float64)
    vn = (C.c_int * 3)(*g.voxel_num); org = (C.c_double * 3)(*g.origin); mxb = (C.c_double * 3)(*g.max_boundary)
    mgr = np.array([0.3, 2.0, 0.5, 1.2, 0.05])                      # run_hill.yaml manager/* (problems.resample defaults)
    for i in range(pb.B):
        path = np.ascontiguousarray(problems.dubins(pb.starts[i], pb.goals[i]))
        N, M = int(pb.N[i]), int(pb.M[i])
        counts = (C.c_int * 2)()
        pos = np.zeros(2 * (N + 8)); posT = np.zeros(N + 8); ang = np.zeros(M + 8); angT = np.zeros(M + 8)
        rc = ref.ref_pm_plan(C.byref(rp), P(cells), vn, org, mxb, C.c_double(g.xy_resolution), C.c_double(g.yaw_resolution), P(mgr), P(path),
                             int(path.shape[0]), counts, P(pos), P(posT), P(ang), P(angT))
        assert rc == 0
        assert (counts[0], counts[1]) == (N + 1, M + 1), i          # the reference's resampler produced the same piece counts
        r, cxy, cyaw, _, _, _, _ = po.solve_one(op, om, pb, i, want_duals=True)
        feas = np.zeros(1)
        # durations: N * Tx == total_T with Tx the last evaluation's piece duration; recover Tx, Ty from the reference message itself and
        # check them against the oracle's total
        Tx, Ty = posT[0], angT[0]
        tt = 0.0
        for _ in range(N):
            tt += Tx
        assert tt == r.total_T and np.all(posT[:N] == Tx) and np.all(angT[:M] == Ty), i
        want_pos = np.zeros(2 * (N + 1))
        for k in range(N):
            want_pos[2 * k] = cxy[6 * k]; want_pos[2 * k + 1] = cxy[6 * N + 6 * k]           # pos_traj[k].getValue(0)
        want_pos[2 * N] = _end_value(cxy[:6 * N], N, Tx); want_pos[2 * N + 1] = _end_value(cxy[6 * N:], N, Tx)
        want_ang = np.array([cyaw[6 * k] for k in range(M)] + [_end_value(cyaw, M, Ty)])
        assert np.array_equal(pos[:2 * (N + 1)], want_pos), i
        assert np.array_equal(ang[:M + 1], want_ang), i


def test_mpc_side_minco_resolve_matches_oracle_bitwise(ref, orc, built, bumps_map):
    """SURVEY 8f-3: the MPC rebuilds the trajectory it tracks from the SE2Traj message with its own MINCO copy
    (mpc_controller/include/utils/minco_traj.hpp:336-460; TrajAnalyzer::setTraj, traj_anal.hpp:125-181: piece start points as
    waypoints, zero boundary velocity / acceleration).  That re-solve, done by the unmodified reference header, equals the oracle's
    MINCO on the same message bit for bit -- and differs from the back-end's own spline only by the boundary speed the back-end
    uses (init_sig_vel, plan_manager.cpp:93-94)."""
    import pyoracle as po
    from uneven_planner_b200 import _lib, problems
    ref.ref_mpc_minco.argtypes = [C.c_int, C.c_int, dp, dp, dp, dp, dp]
    params = _lib.default_params()
    pb = problems.generate(bumps_map, 3, seed=8)
    op, om = po.params_from(params), po.OracleMap(bumps_map)
    for i in range(pb.B):
        N, M = int(pb.N[i]), int(pb.M[i])
        r, cxy, cyaw, _ = po.solve_one(op, om, pb, i)
        Tx = r.total_T / N
        for Dim, P_, c, dur in ((2, N, cxy, Tx), (1, M, cyaw, r.total_T / M)):
            cm = c.reshape(Dim, 6 * P_)
            start = cm[:, 0::6]                                  # piece start points = the message's pos_pts / angle_pts
            end = np.array([_end_value(cm[d], P_, dur) for d in range(Dim)])
            head = np.zeros((3, Dim)); tail = np.zeros((3, Dim))
            head[0] = start[:, 0]; tail[0] = end                 # init_v = init_a = 0 in the message (plan_manager.cpp:153-158)
            inPs = np.ascontiguousarray(start[:, 1:].T).ravel()  # Dim x (P-1) column-major
            ts = np.full(P_, dur)
            c_mpc = np.zeros(6 * P_ * Dim); c_orc = np.zeros(6 * P_ * Dim)
            assert ref.ref_mpc_minco(Dim, P_, P(inPs if inPs.size else np.zeros(1)), P(ts), P(np.ascontiguousarray(head).ravel()),
                                     P(np.ascontiguousarray(tail).ravel()), P(c_mpc)) == 0
            orc.orc_minco_generate(Dim, P_, P(inPs if inPs.size else np.zeros(1)), P(ts), P(np.ascontiguousarray(head).ravel()),
                                   P(np.ascontiguousarray(tail).ravel()), P(c_orc))
            assert np.array_equal(c_mpc, c_orc)
            # the re-solved spline interpolates the same waypoints; it deviates from the back-end spline near the ends only
            assert np.allclose(c_mpc.reshape(Dim, 6 * P_)[:, 0::6], start, atol=1e-9)


@pytest.mark.parametrize("use_scaling", [1, 0])
def test_reference_calConstrainCostGrad_matches_oracle_bitwise(ref, built, bumps_map, use_scaling):
    """Kernel-level pin: ONE ALMTrajOpt::calConstrainCostGrad call of the reference (alm_traj_opt.cpp:663-991) at random multipliers,
    scales and rho -- so both branches of every inequality (active / inactive) are taken -- against orc_eval: penalty cost, hx, gx and
    the coefficient / time gradients before the adjoint, bit for bit."""
    import pyoracle as po
    from uneven_planner_b200 import _lib, problems
    params = _lib.default_params()
    params.use_scaling = use_scaling
    pb = problems.generate(bumps_map, 4, seed=31)
    op, om = po.params_from(params), po.OracleMap(bumps_map)
    g = bumps_map.geom
    rp = RefParams()
    for n, _ in RefParams._fields_:
        setattr(rp, n, getattr(params, n))
    cells = np.ascontiguousarray(bumps_map.cells, dtype=np.float64)
    vn = (C.c_int * 3)(*g.voxel_num); org = (C.c_double * 3)(*g.origin); mxb = (C.c_double * 3)(*g.max_boundary)
    ref.ref_map_create.restype = C.c_void_p
    ref.ref_map_destroy.argtypes = [C.c_void_p]
    h = C.c_void_p(ref.ref_map_create(P(cells), vn, org, mxb, C.c_double(g.xy_resolution), C.c_double(g.yaw_resolution), C.c_double(params.gravity)))
    rng = np.random.default_rng(5)
    try:
        for i in range(pb.B):
            N, M = int(pb.N[i]), int(pb.M[i])
            S = N * (params.int_K + 1)
            x = pb.x0(i) + rng.normal(0, 0.02, 1 + 2 * (N - 1) + (M - 1))
            lam = rng.normal(0, 1.0, S)
            mu = np.maximum(rng.normal(0, 20.0, 6 * S), 0.0)                    # about half of the multipliers exactly zero, the rest large enough to activate
            scx = rng.uniform(0.05, 1.0, 7 * S)
            sfx, rho = float(rng.uniform(1e-6, 1.0)), float(rng.choice([1.0, 8.0, 1000.0]))
            o = po.eval_one(op, om, pb, i, x, lam, mu, scx, sfx, rho)
            cost = np.zeros(1); hx = np.zeros(S); gx = np.zeros(6 * S); gCxy = np.zeros(12 * N); gTxy = np.zeros(N); gCyaw = np.zeros(6 * M); gTyaw = np.zeros(M)
            rc = ref.ref_alm_constrain(C.byref(rp), h, N, M, P(np.ascontiguousarray(pb.bnd[i])), P(np.ascontiguousarray(x)), P(lam), P(mu), P(scx),
                                       C.c_double(sfx), C.c_double(rho), P(cost), P(hx), P(gx), P(gCxy), P(gTxy), P(gCyaw), P(gTyaw))
            assert rc == 0
            assert cost[0] == o["parts"][1], i
            assert np.array_equal(hx, o["hx"]) and np.array_equal(gx, o["gx"]), i
            assert np.array_equal(gCxy, o["gdCxy"]) and np.array_equal(gTxy, o["gdTxy"]), i
            assert np.array_equal(gCyaw, o["gdCyaw"]) and np.array_equal(gTyaw, o["gdTyaw"]), i
            active = (rho * gx + mu > 0)
            assert 0.01 < active.mean() < 0.99                                   # both branches exercised
    finally:
        ref.ref_map_destroy(h)


def test_reference_map_query_matches_oracle_bitwise(ref, built, request):
    """UnevenMap::getAllWithGrad of the reference (trilinear SE(2) interpolation with analytic gradients, yaw seam, out-of-map
    zeros; uneven_map.h:258-377) against orc_map_query at seeded positions, including the map border and the yaw wrap."""
    import pyoracle as po
    from uneven_planner_b200 import maps
    for m in (request.getfixturevalue("bumps_map"), maps.get_terrain("hill")):
        if m is None:
            continue
        g = m.geom
        om = po.OracleMap(m)
        cells = np.ascontiguousarray(m.cells, dtype=np.float64)
        vn = (C.c_int * 3)(*g.voxel_num); org = (C.c_double * 3)(*g.origin); mxb = (C.c_double * 3)(*g.max_boundary)
        ref.ref_map_create.restype = C.c_void_p
        ref.ref_map_destroy.argtypes = [C.c_void_p]
        ref.ref_map_query.argtypes = [C.c_void_p, dp, dp, dp]
        po.lib().orc_map_query.argtypes = [C.c_void_p, dp, dp, dp]
        h = C.c_void_p(ref.ref_map_create(P(cells), vn, org, mxb, C.c_double(g.xy_resolution), C.c_double(g.yaw_resolution), C.c_double(9.81)))
        rng = np.random.default_rng(17)
        pts = np.column_stack([rng.uniform(-5.2, 5.2, 400), rng.uniform(-5.2, 5.2, 400), rng.uniform(-np.pi, np.pi, 400)])
        pts = np.vstack([pts, [[0.0, 0.0, np.pi - 1e-6], [0.0, 0.0, -np.pi + 1e-6], [4.99, -4.99, 3.1], [-5.0, 0.0, 0.0], [2.5, 2.5, 3.14159]]])
        try:
            for pnt in pts:
                pnt = np.ascontiguousarray(pnt)
                vr = np.zeros(7); gr = np.zeros(21); vo = np.zeros(7); go = np.zeros(21)
                ref.ref_map_query(h, P(pnt), P(vr), P(gr))
                po.lib().orc_map_query(C.addressof(om.c), P(pnt), P(vo), P(go))
                assert np.array_equal(vr, vo) and np.array_equal(gr, go), pnt
        finally:
            ref.ref_map_destroy(h)


# ---------------------------------------------------------------- UnevenMap construction (SURVEY 8f-1)
REFMAP = os.path.join(ROOT, "oracle", "_ref", "librefmap.so")


def reference_construct_map(cloud, size, iter_num=2, ellipsoid=(0.2, 0.1, 0.1)):
    """UnevenMap::constructMap + filter of the reference's uneven_map.cpp (compiled unmodified, oracle/ref_map_driver.cpp) on an already
    preprocessed cloud: cells [X, Y, Yaw, 4] in double."""
    from uneven_planner_b200 import _lib
    if not os.path.exists(REFMAP):
        pytest.skip(NO_REF % "librefmap.so")
    R = C.CDLL(REFMAP)
    geom = _lib.map_geometry(size, size, 0.05, 0.1)
    X, Y, W = geom.voxel_num
    cells = np.zeros((X * Y * W, 4))
    vn = (C.c_int * 3)()
    cloud = np.ascontiguousarray(cloud, dtype=np.float32)
    R.ref_map_construct(cloud.ctypes.data_as(C.POINTER(C.c_float)), int(cloud.shape[0]), C.c_double(size), C.c_double(size), C.c_double(0.05), C.c_double(0.1),
                        C.c_double(ellipsoid[0]), C.c_double(ellipsoid[1]), C.c_double(ellipsoid[2]), int(iter_num), cells.ctypes.data_as(C.POINTER(C.c_double)), vn)
    assert tuple(vn) == (X, Y, W)
    return geom, cells.reshape(X, Y, W, 4)


def analytic_cloud(half, n, seed, hole=None):
    """jittered grid on an analytic surface with noise (and an optional empty patch)"""
    rng = np.random.default_rng(seed)
    gx, gy = np.meshgrid(np.linspace(-half, half, n), np.linspace(-half, half, n), indexing="ij")
    px = (gx + rng.uniform(-0.008, 0.008, gx.shape)).ravel(); py = (gy + rng.uniform(-0.008, 0.008, gy.shape)).ravel()
    pz = 0.5 + 0.3 * np.sin(1.3 * px) * np.cos(0.9 * py) + 0.15 * np.exp(-((px - 0.5) ** 2 + (py + 0.3) ** 2) / 0.18) + rng.normal(0, 0.003, px.shape)
    pts = np.column_stack([px, py, pz]).astype(np.float32)
    if hole is not None:
        pts = pts[~((np.abs(pts[:, 0] - hole[0]) < hole[2]) & (np.abs(pts[:, 1] - hole[1]) < hole[2]))]
    return pts


def preprocessed(pts, ellipsoid=(0.2, 0.1, 0.1)):
    """the cloud the builders work on (UnevenMap::init's CropBox + VoxelGrid, through the host tool)"""
    from uneven_planner_b200 import _lib
    L = _lib.lib()
    fp = C.POINTER(C.c_float)
    out = np.zeros((pts.shape[0], 3), np.float32)
    k = L.ualm_map_preprocess_cloud(pts.ctypes.data_as(fp), pts.shape[0], ellipsoid[0], ellipsoid[1], ellipsoid[2], out.ctypes.data_as(fp), pts.shape[0])
    assert k > 0
    return np.ascontiguousarray(out[:k])


def test_reference_constructMap_matches_host_builder(built):
    """SURVEY 8f-1 pinned: the repo's UnevenMap builder (csrc/map_cell.h: bin-grid neighbour search, cyclic Jacobi) against the reference's own
    constructMap + filter (uneven_map.cpp:317-398, 5-43, compiled unmodified; kd-tree and EigenSolver are shim stand-ins with the same
    results up to rounding) on the same preprocessed cloud: every cell (z, sigma, z_b) of the float32 grid is the reference's double value
    rounded to float, up to 2 float ulps -- 1.6 x 1.6 m, 32 x 32 x 64 cells, including cells with an empty footprint.  At the rim of the empty
    patch a handful of cells see two or three (collinear) points: there the smallest eigenvector is not unique, and a point on the
    ellipsoid's surface can fall on either side -- those cells (<= 0.02 %) may differ, every other cell must not."""
    from uneven_planner_b200 import maps
    pts = analytic_cloud(1.1, 100, seed=1, hole=(0.35, -0.3, 0.14))
    cloud = preprocessed(pts)
    geom, ref = reference_construct_map(cloud, 1.6)
    mine = maps.build_from_cloud(pts, geom=geom, nthreads=8)
    assert mine.cells.shape == ref.shape
    d = np.abs(mine.cells.astype(np.float64) - ref)
    scale = np.maximum(np.abs(ref), 1e-3)
    rel = (d / scale).max(axis=-1)
    off = rel > 3e-7
    assert off.mean() <= 2e-4, (int(off.sum()), np.argwhere(off)[:10])
    # the exceptions sit at the rim of the empty patch (0.35, -0.3) +- 0.14 m, nowhere else
    xs = (np.argwhere(off)[:, 0] + 0.5) * 0.05 - 0.8; ys = (np.argwhere(off)[:, 1] + 0.5) * 0.05 - 0.8
    assert np.all((np.abs(xs - 0.35) < 0.14 + 0.35) & (np.abs(ys + 0.3) < 0.14 + 0.35))
    # the empty-footprint branch (uneven_map.cpp:379-386) is exercised: cells over the hole keep the default normal and sigma
    flat = (ref[..., 1] == 0.0) & (ref[..., 2] == 0.0) & (ref[..., 3] == 0.0)
    assert flat.any() and not flat.all()


# ---------------------------------------------------------------------------------------------------------------------------------
# SURVEY 8f-2: KinoAstar::plan (front_end/src/kino_astar.cpp:67-236) compiled UNMODIFIED against the shim (oracle/_ref/librefkino.so,
# oracle/ref_kino_driver.cpp) versus the product's restatement (uneven_planner_b200/csrc/kino_astar.cpp).  OMPL is absent: both sides get
# their Dubins curves from csrc/dubins.h (through oracle/shim/ompl on the reference side), so the pin covers the search itself -- motion
# primitives, NaN states of the v = 0 primitives, costs incl. getTerrainSig, collision checks, the in-place update of OPEN nodes without
# re-sorting, the one-shot trigger and the path assembly -- and the UnevenMap helpers it calls, not OMPL's arithmetic.
# ---------------------------------------------------------------------------------------------------------------------------------
REFKINO = os.path.join(ROOT, "oracle", "_ref", "librefkino.so")


@pytest.fixture(scope="module")
def refkino(ref):
    if not os.path.exists(REFKINO):
        pytest.skip(NO_REF % "librefkino.so")
    L = C.CDLL(REFKINO)
    u8 = C.POINTER(C.c_uint8)
    L.ref_kino_plan.argtypes = [dp, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, dp, dp, dp, dp, C.c_int, u8, u8]
    return L


def _ref_plan(refkino, m, cells64, min_cnormal, max_rho, ap, s, e):
    from uneven_planner_b200 import _lib
    g = m.geom
    X, Y, W = m.shape
    kp = np.array([getattr(ap, n) for n, _ in _lib.AstarParams._fields_])
    out = np.zeros((1 << 15, 3)); o3 = np.zeros((X, Y, W), np.uint8); o2 = np.zeros((X, Y), np.uint8)
    u8 = C.POINTER(C.c_uint8)
    s = np.ascontiguousarray(s, dtype=np.float64); e = np.ascontiguousarray(e, dtype=np.float64)
    n = refkino.ref_kino_plan(P(cells64), -2 * g.origin[0], -2 * g.origin[1], g.xy_resolution, g.yaw_resolution, min_cnormal, max_rho, P(kp), P(s), P(e), P(out),
                              out.shape[0], o3.ctypes.data_as(u8), o2.ctypes.data_as(u8))
    assert n >= 0
    return out[:n].copy(), o3, o2


@pytest.mark.parametrize("which", ["bumps", "hill", "desert", "volcano", "forest"])
def test_kino_astar_matches_reference_bitwise(refkino, built, which, request):
    from uneven_planner_b200 import configs, front_end, maps
    if which == "bumps":
        m0 = request.getfixturevalue("bumps_map"); min_cnormal, max_rho = 0.8, 0.003      # ~10 % of the synthetic terrain becomes obstacle
    else:
        m0 = request.getfixturevalue("terrain")(which)                                    # occupancy thresholds of the terrain's own yaml file
        gk = configs.gen_kwargs(which); min_cnormal, max_rho = gk["min_cnormal"], gk["max_rho"]
    cells64 = np.ascontiguousarray(m0.cells, dtype=np.float64)
    m = maps.UnevenMapData(m0.geom, m0.cells, which, cells64=cells64)
    view = front_end.MapView(m, min_cnormal, max_rho)
    ap = front_end.default_params()
    rng = np.random.default_rng(11)
    X, Y, W = m.shape
    frac = view.occ2.mean()
    assert 0.005 < frac < 0.8, frac
    npath = nlong = 0
    cases = [(rng.uniform(-4.3, 4.3, 2), rng.uniform(-np.pi, np.pi), rng.uniform(-4.3, 4.3, 2), rng.uniform(-np.pi, np.pi)) for _ in range(10)]
    for k, (sp, sy, ep, ey) in enumerate(cases):
        s = np.array([sp[0], sp[1], sy]); e = np.array([ep[0], ep[1], ey])
        want, o3, o2 = _ref_plan(refkino, m, cells64, min_cnormal, max_rho, ap, s, e)
        if k == 0:
            assert np.array_equal(o3, view.occ3) and np.array_equal(o2, view.occ2)      # ualm_map_occupancy == uneven_map.cpp:169-179
        got, nexp = front_end.plan(view, s, e, ap)
        assert got.shape == want.shape and np.array_equal(got, want), (k, got.shape, want.shape)
        npath += len(got) > 0
        nlong += nexp > 500
    assert npath >= 3 and (nlong >= 1 or which in ("desert",))
    # entry checks (kino_astar.cpp:85-95): an occupied start (3-D grid) or goal (2-D grid) gives an empty path on both sides
    ox, oy = np.argwhere(view.occ2)[len(np.argwhere(view.occ2)) // 2]
    g = m.geom
    bad = np.array([g.origin[0] + (ox + 0.5) * g.xy_resolution, g.origin[1] + (oy + 0.5) * g.xy_resolution, 0.2])
    free = np.array([cases[0][0][0], cases[0][0][1], cases[0][1]])
    for s, e in ((free, bad),):
        want, _, _ = _ref_plan(refkino, m, cells64, min_cnormal, max_rho, ap, s, e)
        got, _ = front_end.plan(view, s, e, ap)
        assert len(want) == 0 and len(got) == 0
    # other parameters: finer yaw bins, no terrain term, a different primitive duration
    ap2 = front_end.default_params()
    ap2.yaw_resolution = 0.8; ap2.weight_sigma = 0.0; ap2.time_interval = 0.4; ap2.weight_v_change = 0.3; ap2.weight_delta_change = 0.2
    for sp, sy, ep, ey in cases[:3]:
        s = np.array([sp[0], sp[1], sy]); e = np.array([ep[0], ep[1], ey])
        want, _, _ = _ref_plan(refkino, m, cells64, min_cnormal, max_rho, ap2, s, e)
        got, _ = front_end.plan(view, s, e, ap2)
        assert got.shape == want.shape and np.array_equal(got, want)
