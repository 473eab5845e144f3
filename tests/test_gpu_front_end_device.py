"""The front-end on the GPU (ualm_front_end_batch_device, csrc/ualm_front_end.cu: one warp per KinoAstar search) against its host twin
ualm_kino_astar_plan_det + PlanManager's resampler, pair by pair and bit for bit: polylines, closed-node counts, which pairs are packed and
every field of the packed problems.  Then the searched problems through the parity-path solve against the oracle."""
import importlib.util
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
TERRAINS = ("hill", "desert", "volcano", "forest")


@pytest.fixture(scope="module")
def gpu(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from uneven_planner_b200 import api
    opt = api.BatchALMTrajOpt()
    yield opt
    opt.close()


@pytest.fixture(scope="module")
def gold_mod(built):
    spec = importlib.util.spec_from_file_location("make_kino_search_golden", os.path.join(HERE, "golden", "make_kino_search_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _host_twin(view, starts, goals, p):
    from uneven_planner_b200 import front_end
    with ThreadPoolExecutor(os.cpu_count()) as ex:
        return list(ex.map(lambda b: front_end.plan_det(view, starts[b], goals[b], p), range(len(starts))))


def _check_against_host(opt, view, starts, goals, p):
    """device batch == plan_det + the resampler for every pair; returns the device outputs"""
    import ctypes as C
    from uneven_planner_b200 import _lib, front_end, problems
    rp = front_end.resample_params()
    pb, packed, nexp, paths = front_end.plan_batch_device(opt, view, starts, goals, p, rp, return_paths=True)
    cap = _lib.lib().ualm_front_end_path_cap(C.byref(p), C.byref(rp))
    want = _host_twin(view, starts, goals, p)
    oxy, oyaw, _, _ = pb.offsets()
    k = 0
    for b, (path, ne) in enumerate(want):
        assert nexp[b] == ne, b
        if len(path) <= cap:
            assert paths[b].shape == path.shape and np.array_equal(paths[b], path), b
        else:
            assert len(paths[b]) == 0 and packed[b] == -1, b
        ok = 2 <= len(path) <= cap
        if ok:
            N, M, bnd, T, ixy, iyaw = problems.resample(path)
            ok = N <= 64 and M <= 128
        if not ok:
            assert packed[b] == -1, b
            continue
        assert packed[b] == k, b
        assert (N, M, T) == (pb.N[k], pb.M[k], pb.total_time[k]) and np.array_equal(bnd, pb.bnd[k]), b
        assert np.array_equal(ixy, pb.inner_xy[oxy[k]:oxy[k + 1]]) and np.array_equal(iyaw, pb.inner_yaw[oyaw[k]:oyaw[k + 1]]), b
        k += 1
    assert pb.B == k
    return pb, packed, nexp, paths


@pytest.mark.parametrize("altered", [False, True], ids=["default", "altered"])
@pytest.mark.parametrize("name", TERRAINS)
def test_device_search_equals_the_host_twin_on_the_terrains(gpu, gold_mod, name, altered):
    from uneven_planner_b200 import configs, front_end, maps
    m = maps.terrain_or_standin(name)
    view = front_end.MapView(m, configs.TERRAINS[name]["min_cnormal"], configs.TERRAINS[name]["max_rho"])
    p = gold_mod.altered_params() if altered else front_end.default_params()
    rng = np.random.default_rng(300 + 10 * TERRAINS.index(name) + altered)
    B = 512
    starts = np.column_stack([rng.uniform(-4.3, 4.3, B), rng.uniform(-4.3, 4.3, B), rng.uniform(-np.pi, np.pi, B)])
    goals = np.column_stack([rng.uniform(-4.3, 4.3, B), rng.uniform(-4.3, 4.3, B), rng.uniform(-np.pi, np.pi, B)])
    pb, packed, nexp, _ = _check_against_host(gpu, view, starts, goals, p)
    assert pb.B >= (B // 20 if name == "forest" else B // 2)


def test_device_search_equals_the_host_twin_on_the_edge_cases(gpu, gold_mod):
    """occupied and walled-in starts and goals, yaw +-pi, the 40 x 40 map whose pool fills, the altered parameters (the golden's cases)"""
    for name, view, p, s, e in gold_mod.cases():
        if name in gold_mod.TERRAINS:
            continue
        _, _, nexp, paths = _check_against_host(gpu, view, s, e, p)
        if name == "edges":
            assert (nexp[:16] == 0).all() and (nexp[36:38] > 30000).all() and all(len(paths[b]) == 0 for b in range(32, 38))
        if name == "small":
            assert all(len(paths[b]) == 0 for b in range(0, len(s), 2))


def test_device_batch_sizes_and_independence(gpu, gold_mod):
    """B = 0 and B = 1 work, and a search gives the same result alone as inside a batch"""
    from uneven_planner_b200 import front_end
    name, view, p, s, e = gold_mod.cases()[0]
    pb0, packed0, nexp0 = front_end.plan_batch_device(gpu, view, s[:0], e[:0], p)
    assert pb0.B == 0 and len(packed0) == 0 and len(nexp0) == 0
    _, _, nexp, paths = front_end.plan_batch_device(gpu, view, s[:96], e[:96], p, return_paths=True)
    for b in (0, 1, 17, 95):
        _, _, ne1, p1 = front_end.plan_batch_device(gpu, view, s[b:b + 1], e[b:b + 1], p, return_paths=True)
        assert ne1[0] == nexp[b] and np.array_equal(p1[0], paths[b]), b


def test_start_goal_batch_through_the_device_front_end_matches_oracle(gpu, hill_map):
    """(start, goal) -> device front-end -> parity-path solve, bit-identical to the oracle solving the same problems"""
    import pyoracle as po
    from uneven_planner_b200 import _lib, api, front_end
    params = _lib.default_params()
    view = front_end.MapView(hill_map, 0.8, 0.05)
    rng = np.random.default_rng(21)
    B = 64
    starts = np.column_stack([rng.uniform(-4.3, 4.3, B), rng.uniform(-4.3, 4.3, B), rng.uniform(-np.pi, np.pi, B)])
    goals = np.column_stack([rng.uniform(-4.3, 4.3, B), rng.uniform(-4.3, 4.3, B), rng.uniform(-np.pi, np.pi, B)])
    opt = api.BatchALMTrajOpt().init(params).set_environment(hill_map)
    pb, packed, _ = front_end.plan_batch_device(opt, view, starts, goals)
    assert pb.B >= B // 4 and (packed >= 0).sum() == pb.B
    res, cxy, cyaw = opt.optimize(pb)
    opt.close()
    ores = po.solve_batch(po.params_from(params), po.OracleMap(hill_map), pb, threads=8)
    _, _, ocx, ocy = pb.offsets()
    for i in range(pb.B):
        o, oxy, oyaw, _ = ores[i]
        assert (res[i].ret_code, res[i].n_evals, res[i].inner_cost, res[i].total_T) == (o.ret_code, o.n_evals, o.inner_cost, o.total_T), i
        assert np.array_equal(cxy[ocx[i]:ocx[i + 1]], oxy) and np.array_equal(cyaw[ocy[i]:ocy[i + 1]], oyaw), i
    assert np.mean([r.ret_code == 0 for r in res]) > 0.5
