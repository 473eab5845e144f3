"""Pins of the CPU oracle (oracle/oracle.cpp).

The reference ships no tests or golden vectors for this path (SURVEY.md section 4, 8c), so the oracle is
pinned by analytic invariants, dense re-solves and finite differences -- the list of SURVEY 8c "pins the new repo
must create".  Tolerances are stated per test.
"""
import ctypes as C

import numpy as np
import pytest

import pyoracle as po
from uneven_planner_b200 import _lib, maps, problems

dp = C.POINTER(C.c_double)
P = po.P


# ---------------------------------------------------------------- (1) tau <-> T  (alm_traj_opt.h:232-253)
def test_expC2_logC2_inverse_and_derivative():
    L = po.lib()
    for T in [0.05, 0.3, 0.999, 1.0, 1.001, 3.0, 16.8, 250.0]:
        assert abs(L.orc_expC2(L.orc_logC2(T)) - T) <= 4e-15 * T
    for tau in [-3.0, -0.5, -1e-9, 1e-9, 0.4, 5.0]:
        h = 1e-6
        fd = (L.orc_expC2(tau + h) - L.orc_expC2(tau - h)) / (2 * h)
        assert abs(fd - L.orc_dTdtau(tau)) < 1e-8 * max(1.0, abs(fd))
    # C2 at tau = 0: both branches give T=1, T'=1
    assert L.orc_expC2(0.0) == 1.0 and L.orc_dTdtau(0.0) == 1.0


# ---------------------------------------------------------------- (2) MINCO  (se2traj.hpp:595-680)
def dense_A_b(N, ts, inPs, head, tail, Dim):
    """Row-by-row restatement of the linear system the reference assembles, as a dense matrix."""
    n = 6 * N
    A = np.zeros((n, n)); b = np.zeros((n, Dim))
    beta = lambda t, d: np.array([0.0 if k < d else np.prod(np.arange(k, k - d, -1)) * t ** (k - d) for k in range(6)])
    A[0, :6] = beta(0, 0); A[1, :6] = beta(0, 1); A[2, :6] = beta(0, 2)
    b[0] = head[:, 0]; b[1] = head[:, 1]; b[2] = head[:, 2]
    for i in range(N - 1):
        T = ts[i]
        r = 6 * i
        A[r + 3, r:r + 6] = beta(T, 3); A[r + 3, r + 6:r + 12] = -beta(0, 3)
        A[r + 4, r:r + 6] = beta(T, 4); A[r + 4, r + 6:r + 12] = -beta(0, 4)
        A[r + 5, r:r + 6] = beta(T, 0); b[r + 5] = inPs[:, i]
        A[r + 6, r:r + 6] = beta(T, 0); A[r + 6, r + 6:r + 12] = -beta(0, 0)
        A[r + 7, r:r + 6] = beta(T, 1); A[r + 7, r + 6:r + 12] = -beta(0, 1)
        A[r + 8, r:r + 6] = beta(T, 2); A[r + 8, r + 6:r + 12] = -beta(0, 2)
    T = ts[N - 1]
    A[n - 3, n - 6:] = beta(T, 0); A[n - 2, n - 6:] = beta(T, 1); A[n - 1, n - 6:] = beta(T, 2)
    b[n - 3] = tail[:, 0]; b[n - 2] = tail[:, 1]; b[n - 1] = tail[:, 2]
    return A, b


def minco(Dim, N, inPs, ts, head, tail):
    c = np.zeros(6 * N * Dim)
    po.lib().orc_minco_generate(Dim, N, P(np.asfortranarray(inPs).ravel(order="F")), P(np.ascontiguousarray(ts)),
                                P(np.asfortranarray(head).ravel(order="F")), P(np.asfortranarray(tail).ravel(order="F")), P(c))
    return c.reshape(Dim, 6 * N).T  # (6N, Dim)


@pytest.mark.parametrize("N,Dim", [(1, 1), (1, 2), (2, 2), (7, 2), (21, 2), (41, 1), (64, 2)])
def test_minco_matches_dense_pivoted_solve(N, Dim):
    rng = np.random.default_rng(N * 10 + Dim)
    ts = rng.uniform(0.3, 1.5, N)
    inPs = rng.standard_normal((Dim, max(N - 1, 0))).cumsum(axis=1) * 0.3
    head = rng.standard_normal((Dim, 3)) * 0.2; tail = rng.standard_normal((Dim, 3)) * 0.2
    c = minco(Dim, N, inPs, ts, head, tail)
    A, b = dense_A_b(N, ts, inPs, head, tail, Dim)
    ref = np.linalg.solve(A, b)
    assert np.abs(c - ref).max() <= 1e-9 * max(1.0, np.abs(ref).max())
    # the spline interpolates, is C4 at the knots and meets the boundary states: residual of all 6N rows
    assert np.abs(A @ c - b).max() < 1e-9 * max(1.0, np.abs(b).max())


def test_minco_figure_eight_instance():
    """The only fixed MINCO inputs in the reference tree: mpc_controller's figure-eight (traj_anal.hpp:447-462),
    a NON-uniform-duration instance with zero boundary velocity/acceleration."""
    eight = np.array([[2.34191, -0.382897], [3.09871, 0.936706], [1.99125, 2.68782], [0.394621, 3.877], [-0.0799935, 5.86051],
                      [1.90338, 6.56037], [3.17197, 5.21122], [2.12699, 3.42104], [0.48492, 2.23846], [-0.00904252, 0.365258]]).T
    ts = np.array([3.0] + [1.5] * 9 + [1.0]) * 1.5 / 0.8
    head = np.zeros((2, 3)); tail = np.zeros((2, 3))
    c = minco(2, 11, eight, ts, head, tail)
    A, b = dense_A_b(11, ts, eight, head, tail, 2)
    assert np.abs(A @ c - b).max() < 1e-10
    for i in range(10):  # waypoint i is the start of piece i+1
        assert np.allclose(c[6 * (i + 1)], eight[:, i], atol=1e-12)


def test_minco_single_piece_closed_form():
    T = 0.9
    head = np.array([[0.3, -0.1, 0.05]]); tail = np.array([[1.2, 0.2, -0.3]])
    c = minco(1, 1, np.zeros((1, 0)), np.array([T]), head, tail)[:, 0]
    assert c[0] == 0.3 and c[1] == -0.1 and abs(c[2] - 0.025) < 1e-16
    t = T
    assert abs(np.polyval(c[::-1], t) - 1.2) < 1e-12
    assert abs(np.polyval(np.polyder(c[::-1]), t) - 0.2) < 1e-12
    assert abs(np.polyval(np.polyder(c[::-1], 2), t) + 0.3) < 1e-12


# ---------------------------------------------------------------- (3) jerk cost  (se2traj.hpp:697-747)
def jerk(Dim, N, c, ts):
    gdC = np.zeros(6 * N * Dim); gdT = np.zeros(N)
    J = po.lib().orc_minco_jerk(Dim, N, P(np.ascontiguousarray(c.T).ravel()), P(np.ascontiguousarray(ts)), P(gdC), P(gdT))
    return J, gdC.reshape(Dim, 6 * N).T, gdT


def test_jerk_cost_is_integral_of_squared_jerk():
    rng = np.random.default_rng(5)
    N, Dim = 5, 2
    ts = rng.uniform(0.4, 1.2, N); c = rng.standard_normal((6 * N, Dim))
    J, gdC, gdT = jerk(Dim, N, c, ts)
    xs, ws = np.polynomial.legendre.leggauss(4)  # exact for degree <= 7
    num = 0.0
    for i in range(N):
        t = 0.5 * ts[i] * (xs + 1)
        for d in range(Dim):
            p = c[6 * i:6 * i + 6, d][::-1]
            num += 0.5 * ts[i] * np.sum(ws * np.polyval(np.polyder(p, 3), t) ** 2)
    assert abs(J - num) < 1e-10 * abs(num)
    # closed-form gradients vs central differences
    h = 1e-6
    for (r, d) in [(3, 0), (10, 1), (17, 0), (29, 1)]:
        cp = c.copy(); cp[r, d] += h; cm = c.copy(); cm[r, d] -= h
        fd = (jerk(Dim, N, cp, ts)[0] - jerk(Dim, N, cm, ts)[0]) / (2 * h)
        assert abs(fd - gdC[r, d]) < 1e-6 * max(1.0, abs(fd))
    for i in range(N):
        tp = ts.copy(); tp[i] += h; tm = ts.copy(); tm[i] -= h
        fd = (jerk(Dim, N, c, tp)[0] - jerk(Dim, N, c, tm)[0]) / (2 * h)
        assert abs(fd - gdT[i]) < 1e-6 * max(1.0, abs(fd))


# ---------------------------------------------------------------- (4) adjoint (se2traj.hpp:751-816)
def test_grad_ct_to_qt_matches_finite_differences():
    rng = np.random.default_rng(8)
    N, Dim = 6, 2
    ts = rng.uniform(0.5, 1.1, N)
    inPs = rng.standard_normal((Dim, N - 1)).cumsum(axis=1) * 0.3
    head = rng.standard_normal((Dim, 3)) * 0.2; tail = rng.standard_normal((Dim, 3)) * 0.2

    def W(inPs_, ts_):
        return jerk(Dim, N, minco(Dim, N, inPs_, ts_, head, tail), ts_)[0]

    c = minco(Dim, N, inPs, ts, head, tail)
    _, gdC, gdT = jerk(Dim, N, c, ts)
    gdT = gdT.copy(); gdP = np.zeros(Dim * (N - 1))
    po.lib().orc_minco_grad_ct_to_qt(Dim, N, P(np.asfortranarray(inPs).ravel(order="F")), P(ts), P(np.asfortranarray(head).ravel(order="F")),
                                     P(np.asfortranarray(tail).ravel(order="F")), P(np.ascontiguousarray(gdC.T).ravel()), P(gdT), P(gdP))
    gdP = gdP.reshape(N - 1, Dim).T
    h = 1e-6
    for d in range(Dim):
        for i in range(N - 1):
            a = inPs.copy(); a[d, i] += h; b_ = inPs.copy(); b_[d, i] -= h
            fd = (W(a, ts) - W(b_, ts)) / (2 * h)
            assert abs(fd - gdP[d, i]) < 2e-6 * max(1.0, abs(fd))
    for i in range(N):
        a = ts.copy(); a[i] += h; b_ = ts.copy(); b_[i] -= h
        fd = (W(inPs, a) - W(inPs, b_)) / (2 * h)
        assert abs(fd - gdT[i]) < 2e-6 * max(1.0, abs(fd))


# ---------------------------------------------------------------- (5) map query (uneven_map.h:258-377)
def test_map_flat_is_neutral(built):
    om = po.OracleMap(maps.synthetic_terrain("flat"))
    v, g = om.query([0.33, -1.2, 0.7])
    assert np.allclose(v, [1, 0, 1, 0, 1, 1, 0], atol=0) and np.all(g == 0)
    v, g = om.query([7.0, 0.0, 0.0])  # outside the map: zero RXS2 + zero gradient (uneven_map.h:260-265, Q5)
    assert np.allclose(v, [1, 0, 1, 0, 1, 1, 0]) and np.all(g == 0)


def test_map_constant_tilt_closed_form(built):
    m = maps.synthetic_terrain("tilt")
    om = po.OracleMap(m)
    a, b = float(m.cells[0, 0, 0, 2]), float(m.cells[0, 0, 0, 3])
    c = np.sqrt(1 - a * a - b * b)
    for yaw in [-2.0, 0.0, 0.9, 3.0]:
        v, g = om.query([0.7, -0.4, yaw])
        t = np.cos(yaw) * a + np.sin(yaw) * b
        s = np.sin(yaw) * a - np.cos(yaw) * b
        r = 1 / np.sqrt(1 - t * t)
        assert np.allclose(v, [r, -c * t * r, 1 / (r * c), s * r, c, 1 / c, 0.0], rtol=1e-12, atol=1e-15)
        assert np.abs(g[:, :2]).max() < 1e-9  # constant plane: no x/y dependence


def test_map_values_at_cell_centres_and_gradients_fd(bumps_map):
    m = bumps_map; om = po.OracleMap(m); g = m.geom
    ix, iy, iw = 57, 120, 20
    pos = [(ix + 0.5) * g.xy_resolution + g.origin[0], (iy + 0.5) * g.xy_resolution + g.origin[1], (iw + 0.5) * g.yaw_resolution + g.origin[2]]
    v, _ = om.query(pos)
    cell = m.cells[ix, iy, iw].astype(np.float64)
    assert abs(v[6] - cell[1]) < 1e-15 and abs(v[4] - np.sqrt(1 - cell[2] ** 2 - cell[3] ** 2)) < 1e-15
    rng = np.random.default_rng(4)
    h = 1e-7
    worst = 0.0
    for _ in range(40):
        p = np.array([rng.uniform(-4, 4), rng.uniform(-4, 4), rng.uniform(-3, 3)])
        # keep the FD stencil inside one trilinear cell
        fr = [((p[0] - g.origin[0]) / g.xy_resolution - 0.5) % 1, ((p[1] - g.origin[1]) / g.xy_resolution - 0.5) % 1,
              ((p[2] - g.origin[2]) / g.yaw_resolution - 0.5) % 1]
        if min(fr) < 0.01 or max(fr) > 0.99:
            continue
        v0, g0 = om.query(p)
        for k in range(3):
            pp = p.copy(); pp[k] += h; pm = p.copy(); pm[k] -= h
            fd = (om.query(pp)[0] - om.query(pm)[0]) / (2 * h)
            worst = max(worst, np.abs(fd - g0[:, k]).max() / max(1.0, np.abs(g0[:, k]).max()))
    assert worst < 1e-6


# ---------------------------------------------------------------- (6) L-BFGS (lbfgs.hpp:439-722)
def test_lbfgs_rosenbrock():
    n = 10
    x = np.tile([-1.2, 1.0], n // 2).astype(np.float64)
    f = C.c_double(); it = C.c_int()
    # past=0 disables both the delta stop and the reference's early-exit modification (lbfgs.hpp:327: param.past > 0)
    r = po.lib().orc_lbfgs_rosenbrock(n, P(x), C.byref(f), 8, 1e-8, 0, 1e-6, C.byref(it))
    assert r == 0 and f.value < 1e-12 and np.abs(x - 1).max() < 1e-6
    # with m >= iterations the limited-memory recursion is full BFGS: same minimiser
    x2 = np.tile([-1.2, 1.0], n // 2).astype(np.float64)
    r2 = po.lib().orc_lbfgs_rosenbrock(n, P(x2), C.byref(f), 256, 1e-8, 0, 1e-6, C.byref(it))
    assert r2 == 0 and np.abs(x2 - 1).max() < 1e-6


# ---------------------------------------------------------------- (7) innerCallback gradient (alm_traj_opt.cpp:280-347)
def test_inner_callback_gradient_fd(bumps_map, oparams):
    pb = problems.generate(bumps_map, 3, seed=11)
    om = po.OracleMap(bumps_map)
    prm = po.params_from(_lib.default_params())
    rng = np.random.default_rng(0)
    for i in range(pb.B):
        N = int(pb.N[i]); S = N * (prm.int_K + 1)
        lam = rng.standard_normal(S) * 0.05; mu = np.abs(rng.standard_normal(6 * S)) * 0.05; scx = rng.uniform(0.2, 1.0, 7 * S)
        x = pb.x0(i) * (1 + 1e-3 * rng.standard_normal(pb.nvar()[i]))
        base = po.eval_one(prm, om, pb, i, x, lam, mu, scx, 1e-3, 4.0)
        h = 1e-6
        idx = rng.choice(np.arange(1, len(x)), 12, replace=False)
        for k in idx:
            xp = x.copy(); xp[k] += h; xm = x.copy(); xm[k] -= h
            fd = (po.eval_one(prm, om, pb, i, xp, lam, mu, scx, 1e-3, 4.0)["f"] - po.eval_one(prm, om, pb, i, xm, lam, mu, scx, 1e-3, 4.0)["f"]) / (2 * h)
            # the cost is only C0 across map cells (trilinear): allow a loose bound, typical agreement is 1e-7
            assert abs(fd - base["grad"][k]) < 2e-4 * max(1.0, abs(fd)), (i, k, fd, base["grad"][k])
    # tau component: exact only without the sigma^2 running cost, whose time-gradient the reference writes as
    # user_cost/int_K instead of user_cost/T_i (alm_traj_opt.cpp:827; SURVEY Q3) -- so test with rho_ter = 0
    prm0 = po.params_from(_lib.default_params()); prm0.rho_ter = 0.0
    for i in range(pb.B):
        x = pb.x0(i)
        base = po.eval_one(prm0, om, pb, i, x, None, None, None, 1e-3, 1.0)
        h = 1e-6
        xp = x.copy(); xp[0] += h; xm = x.copy(); xm[0] -= h
        fd = (po.eval_one(prm0, om, pb, i, xp, None, None, None, 1e-3, 1.0)["f"] - po.eval_one(prm0, om, pb, i, xm, None, None, None, 1e-3, 1.0)["f"]) / (2 * h)
        assert abs(fd - base["grad"][0]) < 2e-4 * max(1.0, abs(fd))


def test_init_scaling_definition(bumps_map):
    """scale_cx(i) = 1 / max(1, |grad_x c_i|_inf)  (alm_traj_opt.cpp:654-660): check a few constraints by FD of hx/gx."""
    pb = problems.generate(bumps_map, 1, seed=5)
    om = po.OracleMap(bumps_map)
    prm = po.params_from(_lib.default_params())
    sfx, scx = po.init_scaling(prm, om, pb, 0)
    assert 0 < sfx <= 1 and np.all(scx > 0) and np.all(scx <= 1)
    x = pb.x0(0); h = 1e-6
    base = po.eval_one(prm, om, pb, 0, x)
    J = np.zeros((7 * len(base["hx"]), len(x)))
    for k in range(len(x)):
        xp = x.copy(); xp[k] += h; xm = x.copy(); xm[k] -= h
        a = po.eval_one(prm, om, pb, 0, xp); b = po.eval_one(prm, om, pb, 0, xm)
        S = len(a["hx"])
        J[0::7, k] = (a["hx"] - b["hx"]) / (2 * h)
        for t in range(6):
            J[1 + t::7, k] = (a["gx"][t::6] - b["gx"][t::6]) / (2 * h)
    pred = 1.0 / np.maximum(1.0, np.abs(J[:, 1:]).max(axis=1))  # q-components (tau component carries Q3-free terms only)
    rel = np.abs(pred - scx) / scx
    assert np.median(rel) < 1e-5 and np.mean(rel < 1e-3) > 0.9


# ---------------------------------------------------------------- (8) frozen outputs
@pytest.mark.parametrize("name", ["hill", "desert", "volcano", "forest"])
def test_oracle_matches_golden_fixture(terrain, golden, name):
    """frozen oracle outputs per terrain / BASELINE config parameter set (tests/golden/make_golden.py)"""
    from uneven_planner_b200 import configs
    m = terrain(name)
    gold = golden(name, m)
    pb = problems.generate(m, int(gold["B"]), seed=int(gold["seed"]), **configs.gen_kwargs(name))
    prm = po.params_from(configs.params_for(name))
    out = po.solve_batch(prm, po.OracleMap(m), pb, threads=4)
    assert np.array_equal(np.array([r[0].ret_code for r in out]), gold["ret_code"])
    assert np.array_equal(np.array([r[0].n_evals for r in out]), gold["n_evals"])
    assert np.array_equal(np.array([r[0].inner_cost for r in out]), gold["inner_cost"])
    assert np.array_equal(np.concatenate([r[1] for r in out]), gold["c_xy"])
    assert np.array_equal(np.concatenate([r[2] for r in out]), gold["c_yaw"])


# ---------------------------------------------------------------- (9) post-solve scan (SURVEY 8f-4)
def test_feasibility_scan_closed_forms():
    """orc_feasibility on a flat map: a straight constant-speed run and a constant-rate turn have closed-form maxima
    (alm_traj_opt.h:170-229, se2traj.hpp:551-561)."""
    from uneven_planner_b200 import maps
    flat = maps.synthetic_terrain("flat")
    om = po.OracleMap(flat)
    N, M, Tx, Ty = 2, 4, 1.0, 0.5
    v, yaw0 = 0.4, 0.3
    cxy = np.zeros(12 * N); cyaw = np.zeros(6 * M)
    for i in range(N):           # x = v cos(yaw0) t, y = v sin(yaw0) t, piece-local coefficients low -> high
        cxy[6 * i] = v * np.cos(yaw0) * Tx * i; cxy[6 * i + 1] = v * np.cos(yaw0)
        cxy[6 * N + 6 * i] = v * np.sin(yaw0) * Tx * i; cxy[6 * N + 6 * i + 1] = v * np.sin(yaw0)
    for i in range(M):
        cyaw[6 * i] = yaw0
    out = po.feasibility(om, 9.81, N, M, cxy, cyaw, Tx, Ty)
    n = int(out[7])
    assert n in (200, 201)                                    # t = 0, 0.01, ... < 2.0 by repeated addition
    assert abs(out[0] - v) < 1e-12 and abs(out[1]) < 1e-12 and abs(out[2]) < 1e-12 and out[3] == 0.0
    assert out[4] == -1.0 and out[5] == 0.0 and out[6] < 1e-12 * n
    # heading off by 90 degrees: the non-holonomic error integrates |v| per sample; a yaw rate w gives curvature w / sqrt(v^2 + 0.01)
    w = 0.2
    for i in range(M):
        cyaw[6 * i] = yaw0 + np.pi / 2 + w * Ty * i; cyaw[6 * i + 1] = w
    out2 = po.feasibility(om, 9.81, N, M, cxy, cyaw, Tx, Ty)
    assert abs(out2[3] - w / np.sqrt(v * v + 0.01)) < 1e-12
    assert out2[6] > 0.9 * v * int(out2[7]) * np.cos(w * 2.0)


# ---------------------------------------------------------------- (10) the population does not depend on the shared deterministic trig
def test_population_is_unchanged_by_the_detmath_choice(hill_map, tmp_path):
    """The oracle, the reference build and the CUDA path all use include/ualm_detmath.h for sin / cos / atan2 (<= 2 ulp from libm) so that
    they can be compared bit for bit.  That choice must not shape the results: the same oracle built with glibc's libm (-DORC_LIBM=1) is a
    second valid double implementation of the reference.  Per trajectory the two differ chaotically (DESIGN.md section 2); as populations
    (256 hill problems, run_hill.yaml) they must agree: converged fraction, evaluations, cost distribution, duration."""
    import os
    import subprocess
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    so = str(tmp_path / "liboracle_libm.so")
    subprocess.run(["g++", "-O3", "-std=c++14", "-ffp-contract=off", "-fPIC", "-shared", "-DORC_LIBM=1", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "oracle", "oracle.cpp"), "-o", so], check=True)
    params = _lib.default_params()
    pb = problems.generate(hill_map, 256, seed=0)
    op, om = po.params_from(params), po.OracleMap(hill_map)
    a = po.solve_batch(op, om, pb, threads=8)
    keep_lib, keep_path = po._lib, po.LIB
    po._lib, po.LIB = None, so
    try:
        b = po.solve_batch(op, om, pb, threads=8)
    finally:
        po._lib, po.LIB = keep_lib, keep_path
    rca = np.array([r[0].ret_code for r in a]); rcb = np.array([r[0].ret_code for r in b])
    eva = np.array([r[0].n_evals for r in a]); evb = np.array([r[0].n_evals for r in b])
    assert any(r[0].inner_cost != s[0].inner_cost for r, s in zip(a, b))          # it IS a different arithmetic
    assert abs((rca == 0).mean() - (rcb == 0).mean()) <= 0.05
    assert abs(np.median(eva) - np.median(evb)) <= 0.08 * np.median(eva) and abs(eva.mean() - evb.mean()) <= 0.08 * eva.mean()
    both = (rca == 0) & (rcb == 0)
    assert both.mean() >= 0.7
    ca = np.array([r[0].inner_cost for r in a]); cb = np.array([r[0].inner_cost for r in b])
    rel = np.abs(cb[both] - ca[both]) / np.abs(ca[both])
    assert np.median(rel) < 5e-3 and np.percentile(rel, 90) < 5e-2
    Ta = np.array([r[0].total_T for r in a]); Tb = np.array([r[0].total_T for r in b])
    assert abs(np.median(Ta[both]) - np.median(Tb[both])) <= 0.01 * np.median(Ta[both])
