// kino_astar.cpp -- the front-end of the hot path's callers (SURVEY 8f-2): a host-side restatement of KinoAstar::plan
// (front_end/src/kino_astar.cpp:67-236; helpers front_end/include/front_end/kino_astar.h:177-291) over the UnevenMap occupancy grids,
// and the batch form that turns (start, goal) pairs into the optimizer's inputs:
//     KinoAstar::plan -> PlanManager's resampler (ualm_resample_path, plan_manager.cpp:62-122) -> ualm_solve_batch / ualm_submit_batch.
// The search itself is csrc/kino_search.h (shared with the device front-end, csrc/ualm_front_end.cu); here it runs with the C library's
// trigonometry (TrigLibm), one search per host thread.  Pinned bit for bit against kino_astar.cpp compiled unmodified
// (tests/test_ref_pin.py::test_kino_astar_*), with csrc/dubins.h standing in for OMPL on both sides.
#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>

#include "kino_search.h"
#include "ualm.h"
#include "ualm_front_end.h"

namespace {

using ualm_kino::MapView;

bool params_ok(const ualm_astar_params_t *p)
{
    return p && p->yaw_resolution > 0 && p->max_vel > 0 && p->max_steer > 0 && p->collision_interval > 0 && p->time_interval > 0 && p->wheel_base > 0;
}

// one host thread's search state: the node pool (X * Y nodes), OPEN, the expanded-node table, the inputs and the one-shot's samples
template <class T> struct Planner {
    ualm_kino::Search<T> s;
    std::vector<ualm_kino::Node> pool;
    std::vector<int> heap, table;
    std::vector<double> inputs, shot;
    int nin, shot_cap;

    Planner(const MapView &m, const ualm_astar_params_t &p) : pool((size_t)m.g.voxel_num[0] * m.g.voxel_num[1]), heap(pool.size()),
                                                            table(ualm_kino::table_capacity((long long)pool.size()))
    {
        s.map = m; s.p = p; s.yaw_inv = 1.0 / p.yaw_resolution;
        s.rho = p.wheel_base / T::tan(p.max_steer);
        s.pool = pool.data(); s.pool_size = (int)pool.size();
        s.open.h = heap.data(); s.open.n = 0;
        s.closed.slot = table.data(); s.closed.mask = (unsigned)table.size() - 1;
        nin = ualm_kino::build_inputs(p, nullptr, 0);
        inputs.resize(2 * (size_t)nin);
        ualm_kino::build_inputs(p, inputs.data(), nin);
        shot_cap = std::max(ualm_kino::shot_capacity(p, s.rho), 1);
        shot.resize(3 * (size_t)shot_cap);
    }
    // path: (x, y, yaw) triples, empty without a path; expanded: nodes closed.  UALM_OK, or UALM_ELIMIT if the one-shot had more
    // samples than shot_capacity allows for (it cannot)
    int plan(const double start[3], const double goal[3], std::vector<double> &path, int *expanded)
    {
        path.clear();
        std::fill(table.begin(), table.end(), -1);
        int node = -1, nshot = 0;
        const int st = s.plan(start, goal, inputs.data(), nin, shot.data(), shot_cap, &node, &nshot);
        if (expanded) *expanded = s.iter_num;
        if (st == ualm_kino::KS_SHOT_OVERFLOW) return UALM_ELIMIT;
        if (st == ualm_kino::KS_FOUND) {
            const int chain = s.chain_length(node);
            path.resize(3 * (size_t)(chain + nshot));
            s.retrieve(node, chain, shot.data(), nshot, path.data());
        }
        return UALM_OK;
    }
};

template <class T> int plan_one(const ualm_astar_map_t *map, const ualm_astar_params_t *p, const double start[3], const double goal[3], double *path_xyyaw,
                                int max_pts, int *n_expanded)
{
    MapView v;
    if (!ualm_kino::view_of(map, v) || !params_ok(p) || !start || !goal || !path_xyyaw || max_pts < 0) return UALM_EINVAL;
    Planner<T> pl(v, *p);
    std::vector<double> path;
    const int rc = pl.plan(start, goal, path, n_expanded);
    if (rc != UALM_OK) return rc;
    const int n = (int)(path.size() / 3);
    if (n > max_pts) return UALM_ELIMIT;
    std::memcpy(path_xyyaw, path.data(), sizeof(double) * path.size());
    return n;
}

} // namespace

// run_hill.yaml:16-30 (identical in every run_*.yaml)
extern "C" void ualm_astar_default_params(ualm_astar_params_t *p)
{
    p->yaw_resolution = 3.15; p->lambda_heu = 1.0; p->weight_r2 = 1.0; p->weight_so2 = 0.5; p->weight_v_change = 0.0; p->weight_delta_change = 0.0;
    p->weight_sigma = 10.0; p->time_interval = 0.3; p->collision_interval = 0.06; p->oneshot_range = 1.0; p->wheel_base = 0.26; p->max_steer = 0.5;
    p->max_vel = 0.5;
}

extern "C" int ualm_kino_astar_plan(const ualm_astar_map_t *map, const ualm_astar_params_t *p, const double start[3], const double goal[3], double *path_xyyaw,
                                    int max_pts, int *n_expanded)
{
    return plan_one<TrigLibm>(map, p, start, goal, path_xyyaw, max_pts, n_expanded);
}

// the same search with include/ualm_detmath.h's trigonometry: the host twin of ualm_front_end_batch_device, for tests
extern "C" int ualm_kino_astar_plan_det(const ualm_astar_map_t *map, const ualm_astar_params_t *p, const double start[3], const double goal[3],
                                        double *path_xyyaw, int max_pts, int *n_expanded)
{
    return plan_one<TrigDet>(map, p, start, goal, path_xyyaw, max_pts, n_expanded);
}

// the one-shot curve alone (kino_astar.h:246-258 without the occupancy test): samples every `interval` metres of the shortest Dubins
// curve of turning radius `radius`; *length (optional) = its length.  Returns the number of samples
extern "C" int ualm_dubins_shot(const double start[3], const double goal[3], double radius, double interval, double *path_xyyaw, int max_pts, double *length)
{
    if (!start || !goal || !path_xyyaw || !(radius > 0) || !(interval > 0) || max_pts < 1) return UALM_EINVAL;
    const ualm_dubins::Path path = ualm_dubins::shortest<TrigLibm>(start, goal, radius);
    const double len = radius * path.length();
    if (length) *length = len;
    int n = 0;
    for (double l = 0.0; l <= len; l += interval) {
        if (n >= max_pts) return UALM_ELIMIT;
        ualm_dubins::interpolate<TrigLibm>(start, path, radius, l / len, path_xyyaw + 3 * n);
        n++;
    }
    return n;
}

// (start, goal) pairs -> the optimizer's ragged inputs: KinoAstar::plan, then PlanManager's resampler, one search per host thread.
// Problems without a path (start / goal occupied, search exhausted) or over the optimizer's limits are left out: packed[b] = index of
// problem b in the packed outputs or -1.  Returns the number of packed problems.
extern "C" int ualm_front_end_batch(const ualm_astar_map_t *map, const ualm_astar_params_t *ap, const ualm_resample_params_t *rp, int B, const double *starts,
                                    const double *goals, int nthreads, int32_t *N, int32_t *M, double *bnd, double *total_time, double *inner_xy,
                                    long long cap_xy, double *inner_yaw, long long cap_yaw, int32_t *packed, int32_t *n_expanded)
{
    MapView v;
    if (!ualm_kino::view_of(map, v) || !ap || !rp || B < 0 || (B > 0 && (!starts || !goals || !N || !M || !bnd || !total_time || !inner_xy || !inner_yaw || !packed))) return UALM_EINVAL;
    std::vector<ualm_fe::Resampled> res(B);
    std::vector<int> expanded(B, 0), rcs(B, UALM_OK);
    std::atomic<int> next(0);
    if (nthreads <= 0) nthreads = (int)std::max(1u, std::thread::hardware_concurrency());
    nthreads = std::min(nthreads, std::max(B, 1));
    auto worker = [&]() {
        Planner<TrigLibm> pl(v, *ap);
        std::vector<double> path;
        for (;;) {
            const int b = next.fetch_add(1);
            if (b >= B) break;
            rcs[b] = pl.plan(starts + 3 * b, goals + 3 * b, path, &expanded[b]);
            ualm_fe::resample(path.data(), (int)(path.size() / 3), rp, res[b]);
        }
    };
    std::vector<std::thread> th;
    for (int t = 0; t < nthreads; t++) th.emplace_back(worker);
    for (auto &t : th) t.join();
    for (int b = 0; b < B; b++)
        if (rcs[b] != UALM_OK) return rcs[b];
    if (n_expanded) std::copy(expanded.begin(), expanded.end(), n_expanded);
    return ualm_fe::pack(res, N, M, bnd, total_time, inner_xy, cap_xy, inner_yaw, cap_yaw, packed);
}

void ualm_fe::resample(const double *path, int npts, const ualm_resample_params_t *rp, Resampled &o)
{
    o.ok = 0;
    if (npts < 2) return;
    o.ixy.assign(2 * 64, 0.0); o.iyaw.assign(128, 0.0);
    const int rc = ualm_resample_path(path, npts, rp->piece_len, rp->yaw_piece_times, rp->mean_vel, rp->init_time_times, rp->init_sig_vel, o.bnd,
                                      o.ixy.data(), 63, o.iyaw.data(), 127, &o.N, &o.M, &o.T);      // N <= 64, M <= 128: the optimizer's limits
    o.ok = rc == UALM_OK;
}

int ualm_fe::pack(const std::vector<Resampled> &res, int32_t *N, int32_t *M, double *bnd, double *total_time, double *inner_xy, long long cap_xy,
                  double *inner_yaw, long long cap_yaw, int32_t *packed)
{
    int k = 0;
    long long oxy = 0, oyaw = 0;
    for (size_t b = 0; b < res.size(); b++) {
        const Resampled &o = res[b];
        packed[b] = -1;
        if (!o.ok) continue;
        if (oxy + 2LL * (o.N - 1) > cap_xy || oyaw + (o.M - 1) > cap_yaw) return UALM_ELIMIT;
        N[k] = o.N; M[k] = o.M; total_time[k] = o.T;
        std::memcpy(bnd + 18 * (size_t)k, o.bnd, sizeof(o.bnd));
        std::memcpy(inner_xy + oxy, o.ixy.data(), sizeof(double) * 2 * (o.N - 1));
        std::memcpy(inner_yaw + oyaw, o.iyaw.data(), sizeof(double) * (o.M - 1));
        oxy += 2LL * (o.N - 1); oyaw += o.M - 1;
        packed[b] = k++;
    }
    return k;
}
