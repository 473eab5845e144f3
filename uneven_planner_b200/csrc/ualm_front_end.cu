// ualm_front_end.cu -- KinoAstar::plan on the GPU for a batch of (start, goal) pairs: csrc/kino_search.h with the detmath trigonometry
// (TrigDet), one warp per search.  Compiled with -fmad=false like the host side, so each search is bit-identical to the host's
// ualm_kino_astar_plan_det.  PlanManager's resampler stays on the host (ualm_resample_path on the downloaded polylines).
//
// Execution: persistent warps take search indices from an atomic counter.  Each resident warp owns a workspace (node pool of X * Y
// nodes, OPEN heap, expanded-node table, the primitives of one expansion, the one-shot's samples), so memory grows with the number of
// resident warps, not with B.  Per expansion the lanes compute the primitives (state_transit, collision samples, terrainSig, g, f)
// in parallel; none of that reads the expanded-node table.  Lane 0 then applies them in primitive order (lookup, skip if CLOSE, insert
// or rewrite in place, push), so the lookup of primitive i sees the nodes primitives < i inserted, as on the host.  The one-shot test
// on the queue top spreads its Dubins samples over the lanes; each lane walks the running sum l += collision_interval itself, so
// sample k sits at the k-fold sum exactly as on the host.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "kino_search.h"
#include "ualm_front_end.h"

namespace ualm_fe {

using ualm_kino::Node;
using ualm_kino::Prim;
using Search = ualm_kino::Search<TrigDet>;

constexpr int kWarpsPerBlock = 4;
constexpr int kMaxPathCap = 1 << 16;

struct Args {
    Search s;                       // map, parameters, turning radius; the workspace pointers are set per warp
    const double *inputs;           // build_inputs' list
    int nin;
    const double *starts, *goals;
    int B;
    int *next;                      // the atomic search counter
    char *ws;                       // workspaces, ws_stride bytes per warp
    size_t ws_stride, off_heap, off_table, off_prim, off_shot;
    unsigned table_mask;
    int shot_cap, path_cap;
    int *npts;                      // per search: polyline points (0 = no path, -1 = longer than path_cap), -2 = shot overflow
    int *nexp;                      // nodes closed
    double *paths;                  // path_cap (x, y, yaw) per search
};

__global__ void __launch_bounds__(32 * kWarpsPerBlock) kino_search_kernel(Args a)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    char *ws = a.ws + a.ws_stride * (size_t)warp;
    Search s = a.s;
    s.pool = (Node *)ws;
    s.open.h = (int *)(ws + a.off_heap);
    s.closed.slot = (int *)(ws + a.off_table);
    s.closed.mask = a.table_mask;
    Prim *prims = (Prim *)(ws + a.off_prim);
    double *shot = (double *)(ws + a.off_shot);
    for (;;) {
        int b = 0;
        if (lane == 0) b = atomicAdd(a.next, 1);
        b = __shfl_sync(full, b, 0);
        if (b >= a.B) break;
        const double start[3] = {a.starts[3 * b], a.starts[3 * b + 1], a.starts[3 * b + 2]};
        const double goal[3] = {a.goals[3 * b], a.goals[3 * b + 1], a.goals[3 * b + 2]};
        for (unsigned i = lane; i <= a.table_mask; i += 32) s.closed.slot[i] = -1;
        __syncwarp();
        // lane 0 owns the search state (OPEN, the table, the node counters); the other lanes read the nodes after each __syncwarp
        int status = 0;
        if (lane == 0) status = s.begin(start, goal) ? ualm_kino::KS_SEARCHING : ualm_kino::KS_NO_PATH;
        status = __shfl_sync(full, status, 0);
        int node = -1, nshot = 0;
        // every pass closes one node and at most pool_size nodes exist: the loop ends after at most pool_size passes
        for (int pass = 0; status == ualm_kino::KS_SEARCHING && pass <= s.pool_size; pass++) {
            __syncwarp();
            if (__shfl_sync(full, s.open.n, 0) == 0) { status = ualm_kino::KS_NO_PATH; break; }
            const int cur = s.open.h[0];
            const Node cn = s.pool[cur];
            if (s.near_goal(cn, goal)) {
                bool hit = false;
                const int ns = s.shot_samples(cn.state, goal, shot, a.shot_cap, lane, 32, &hit);
                hit = __any_sync(full, hit);
                if (ns > a.shot_cap) { status = ualm_kino::KS_SHOT_OVERFLOW; break; }
                if (!hit) { status = ualm_kino::KS_FOUND; node = cur; nshot = ns; break; }
            }
            if (lane == 0) {
                s.open.pop(s.pool);
                s.pool[cur].node_state = ualm_kino::ST_CLOSE;
                s.iter_num += 1;
            }
            for (int i = lane; i < a.nin; i += 32) s.primitive(cn, a.inputs + 2 * i, goal, prims[i]);
            __syncwarp();
            int filled = 0;
            if (lane == 0)
                for (int i = 0; i < a.nin; i++)
                    if (!s.apply(cur, prims[i])) { filled = 1; break; }
            if (__shfl_sync(full, filled, 0)) status = ualm_kino::KS_POOL_FULL;
        }
        __syncwarp();
        if (lane == 0) {
            int n = 0;
            if (status == ualm_kino::KS_FOUND) {
                const int chain = s.chain_length(node);
                if (chain + nshot > a.path_cap) n = -1;
                else { s.retrieve(node, chain, shot, nshot, a.paths + 3 * (size_t)a.path_cap * b); n = chain + nshot; }
            } else if (status == ualm_kino::KS_SHOT_OVERFLOW) {
                n = -2;
            }
            a.npts[b] = n;
            a.nexp[b] = s.iter_num;
        }
    }
}

template <class T> struct Buf {
    T *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t n)
    {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        const cudaError_t e = cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct FrontEnd {
    ualm_map_geom_t g;
    Buf<uint8_t> occ3, occ2;
    Buf<float> cells;
    Buf<double> cells64;
    Buf<char> ws;
    Buf<double> io, paths, inputs;
    Buf<int> ints;
    cudaStream_t stream = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
};

#define FE_CK(call)                                                                           \
    do {                                                                                      \
        const cudaError_t e_ = (call);                                                        \
        if (e_ != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(e_); return UALM_ENOCUDA; } \
    } while (0)

void release(FrontEnd *fe)
{
    if (!fe) return;
    if (fe->stream) cudaStreamSynchronize(fe->stream);
    fe->occ3.release(); fe->occ2.release(); fe->cells.release(); fe->cells64.release(); fe->ws.release();
    fe->io.release(); fe->paths.release(); fe->inputs.release(); fe->ints.release();
    if (fe->e0) cudaEventDestroy(fe->e0);
    if (fe->e1) cudaEventDestroy(fe->e1);
    if (fe->stream) cudaStreamDestroy(fe->stream);
    delete fe;
}

int set_map(FrontEnd **pfe, const ualm_astar_map_t *m, std::string &err)
{
    ualm_kino::MapView v;
    if (!ualm_kino::view_of(m, v)) { err = "incomplete front-end map"; return UALM_EINVAL; }
    const ualm_map_geom_t &g = *m->geom;
    if (g.voxel_num[0] < 1 || g.voxel_num[1] < 1 || g.voxel_num[2] < 1) { err = "empty map"; return UALM_EINVAL; }
    if (!*pfe) *pfe = new FrontEnd();
    FrontEnd *fe = *pfe;
    if (!fe->stream) FE_CK(cudaStreamCreateWithFlags(&fe->stream, cudaStreamNonBlocking));
    if (!fe->e0) FE_CK(cudaEventCreate(&fe->e0));
    if (!fe->e1) FE_CK(cudaEventCreate(&fe->e1));
    FE_CK(cudaStreamSynchronize(fe->stream));
    const size_t xy = (size_t)g.voxel_num[0] * g.voxel_num[1], cells = xy * g.voxel_num[2];
    FE_CK(fe->occ3.ensure(cells));
    FE_CK(fe->occ2.ensure(xy));
    FE_CK(cudaMemcpy(fe->occ3.p, m->occ3, cells, cudaMemcpyHostToDevice));
    FE_CK(cudaMemcpy(fe->occ2.p, m->occ2, xy, cudaMemcpyHostToDevice));
    // the cell grid as given (sigma_at reads the doubles when cells64 is set, the floats otherwise)
    fe->cells.release(); fe->cells64.release();
    if (m->cells64) {
        FE_CK(fe->cells64.ensure(4 * cells));
        FE_CK(cudaMemcpy(fe->cells64.p, m->cells64, sizeof(double) * 4 * cells, cudaMemcpyHostToDevice));
    } else {
        FE_CK(fe->cells.ensure(4 * cells));
        FE_CK(cudaMemcpy(fe->cells.p, m->cells, sizeof(float) * 4 * cells, cudaMemcpyHostToDevice));
    }
    fe->g = g;
    return UALM_OK;
}

// the one-shot's turning radius, with the search's own tan
static double shot_radius(const ualm_astar_params_t &p) { return p.wheel_base / TrigDet::tan(p.max_steer); }

int path_cap(const ualm_astar_params_t *ap, const ualm_resample_params_t *rp)
{
    // A polyline the resampler accepts (N <= 64, M <= 128) is at most L = piece_len * (min(64, 128 / yaw_piece_times) + 1) long.
    // Consecutive points are at least one step apart -- the chord of the shortest motion primitive, or of one collision_interval
    // of the one-shot -- except the one-shot's first sample, which repeats the node it leaves from.  So such a path has at most
    // L / step + 2 points; +1 for rounding.
    const ualm_astar_params_t &p = *ap;
    const double rho = shot_radius(p);
    double step = 2.0 * rho * std::sin(p.collision_interval / (2.0 * rho));
    if (!(step > 0) || p.collision_interval >= M_PI * rho) step = 0;
    const int nin = ualm_kino::build_inputs(p, nullptr, 0);
    std::vector<double> in(2 * (size_t)nin);
    ualm_kino::build_inputs(p, in.data(), nin);
    for (int i = 0; i < nin; i++) {
        const double s = in[2 * i] * p.time_interval;
        if (!(s > 0)) continue;
        double chord = s;
        if (std::fabs(in[2 * i + 1]) > 1e-4) {
            const double y = s * std::tan(in[2 * i + 1]) / p.wheel_base;
            chord = std::fabs(2.0 * (s / y) * std::sin(0.5 * y));
        }
        step = std::min(step, chord);
    }
    const double L = rp->piece_len * (std::min(64.0, 128.0 / rp->yaw_piece_times) + 1.0);
    if (!(step > 0) || !(L > 0)) return kMaxPathCap;
    const double cap = std::ceil(L / step) + 3.0;
    return cap < kMaxPathCap ? (int)cap : kMaxPathCap;
}

static bool finite_params(const ualm_astar_params_t &p)
{
    const double *v = &p.yaw_resolution;
    for (size_t i = 0; i < sizeof(p) / sizeof(double); i++) if (!std::isfinite(v[i])) return false;
    if (!(p.yaw_resolution > 0 && p.max_vel > 0 && p.max_steer > 0 && p.collision_interval > 0 && p.time_interval > 0 && p.wheel_base > 0))
        return false;
    return p.max_vel * p.time_interval * std::fabs(std::tan(p.max_steer)) / p.wheel_base <= 1e4;      // one primitive's turn (rad)
}

int batch(FrontEnd *fe, const ualm_astar_params_t *ap, const ualm_resample_params_t *rp, int B, const double *starts, const double *goals,
          int32_t *N, int32_t *M, double *bnd, double *total_time, double *inner_xy, long long cap_xy, double *inner_yaw, long long cap_yaw,
          int32_t *packed, int32_t *n_expanded, double *path_xyyaw, long long cap_path, int64_t *path_off, float *search_ms, std::string &err)
{
    if (!fe) { err = "no front-end map (ualm_set_front_end_map)"; return UALM_ESTATE; }
    if (!ap || !rp || B < 0 || (B > 0 && (!starts || !goals || !N || !M || !bnd || !total_time || !inner_xy || !inner_yaw || !packed)) ||
        (path_xyyaw && !path_off)) { err = "bad argument"; return UALM_EINVAL; }
    // finite parameters and poses keep every loop of the search bounded (norm_angle's turns, the primitives' running sums)
    if (!finite_params(*ap)) { err = "A* parameters must be finite and positive, one primitive's turn <= 1e4 rad"; return UALM_EINVAL; }
    for (long long i = 0; i < 3LL * B; i++)
        if (!std::isfinite(starts[i]) || !std::isfinite(goals[i]) || (i % 3 == 2 && (std::fabs(starts[i]) > 1e4 || std::fabs(goals[i]) > 1e4))) {
            err = "start / goal poses must be finite, |yaw| <= 1e4"; return UALM_EINVAL;
        }
    if (search_ms) *search_ms = 0.f;
    if (path_off) path_off[0] = 0;
    if (B == 0) return 0;

    Args a;
    std::memset((void *)&a, 0, sizeof(a));
    Search &s = a.s;
    s.map.g = fe->g;
    s.map.cells = fe->cells.p; s.map.cells64 = fe->cells64.p; s.map.occ3 = fe->occ3.p; s.map.occ2 = fe->occ2.p;
    s.map.xy_inv = 1.0 / fe->g.xy_resolution; s.map.yaw_inv = 1.0 / fe->g.yaw_resolution;
    s.p = *ap;
    s.yaw_inv = 1.0 / ap->yaw_resolution;
    s.rho = shot_radius(*ap);
    s.pool_size = fe->g.voxel_num[0] * fe->g.voxel_num[1];
    const int nin = ualm_kino::build_inputs(*ap, nullptr, 0);
    std::vector<double> inputs(2 * (size_t)nin);
    ualm_kino::build_inputs(*ap, inputs.data(), nin);
    a.nin = nin;
    a.shot_cap = ualm_kino::shot_capacity(*ap, s.rho);
    if (a.shot_cap < 1) { err = "one-shot sample count out of range"; return UALM_EINVAL; }
    a.path_cap = path_cap(ap, rp);
    const unsigned tcap = ualm_kino::table_capacity(s.pool_size);
    a.table_mask = tcap - 1;
    auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
    a.off_heap = align(sizeof(Node) * (size_t)s.pool_size);
    a.off_table = a.off_heap + align(sizeof(int) * (size_t)s.pool_size);
    a.off_prim = a.off_table + align(sizeof(int) * (size_t)tcap);
    a.off_shot = a.off_prim + align(sizeof(Prim) * (size_t)std::max(nin, 1));
    a.ws_stride = a.off_shot + align(sizeof(double) * 3 * (size_t)a.shot_cap);

    // resident warps: what the SMs hold at once, no more than the searches need, and the workspaces within half the free memory
    int dev = 0, sms = 0, per_sm = 0;
    FE_CK(cudaGetDevice(&dev));
    FE_CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    FE_CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kino_search_kernel, 32 * kWarpsPerBlock, 0));
    size_t free_b = 0, total_b = 0;
    FE_CK(cudaMemGetInfo(&free_b, &total_b));
    const size_t out_bytes = (size_t)B * (sizeof(double) * (6 + 3 * (size_t)a.path_cap) + 2 * sizeof(int));
    const size_t avail = (free_b + fe->ws.cap) / 2;
    const long long by_mem = avail > out_bytes ? (long long)((avail - out_bytes) / (a.ws_stride * kWarpsPerBlock)) : 0;
    const long long by_sm = (long long)std::max(per_sm, 1) * sms, by_b = (B + kWarpsPerBlock - 1) / kWarpsPerBlock;
    const int nblocks = (int)std::min(std::min(by_sm, by_b), by_mem);
    if (nblocks < 1) { err = "not enough device memory for the search workspaces"; return UALM_ENOCUDA; }

    FE_CK(fe->ws.ensure((size_t)nblocks * kWarpsPerBlock * a.ws_stride));
    FE_CK(fe->io.ensure(6 * (size_t)B));
    FE_CK(fe->paths.ensure(3 * (size_t)a.path_cap * B));
    FE_CK(fe->inputs.ensure(2 * (size_t)std::max(nin, 1)));
    FE_CK(fe->ints.ensure(2 * (size_t)B + 1));
    FE_CK(cudaMemcpyAsync(fe->io.p, starts, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, fe->stream));
    FE_CK(cudaMemcpyAsync(fe->io.p + 3 * (size_t)B, goals, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, fe->stream));
    FE_CK(cudaMemcpyAsync(fe->inputs.p, inputs.data(), sizeof(double) * 2 * nin, cudaMemcpyHostToDevice, fe->stream));
    FE_CK(cudaMemsetAsync(fe->ints.p + 2 * (size_t)B, 0, sizeof(int), fe->stream));
    a.inputs = fe->inputs.p;
    a.starts = fe->io.p; a.goals = fe->io.p + 3 * (size_t)B;
    a.B = B;
    a.next = fe->ints.p + 2 * (size_t)B;
    a.ws = fe->ws.p;
    a.npts = fe->ints.p; a.nexp = fe->ints.p + B;
    a.paths = fe->paths.p;
    FE_CK(cudaEventRecord(fe->e0, fe->stream));
    kino_search_kernel<<<nblocks, 32 * kWarpsPerBlock, 0, fe->stream>>>(a);
    FE_CK(cudaGetLastError());
    FE_CK(cudaEventRecord(fe->e1, fe->stream));
    std::vector<int> h(2 * (size_t)B);
    std::vector<double> paths(3 * (size_t)a.path_cap * B);
    FE_CK(cudaMemcpyAsync(h.data(), fe->ints.p, sizeof(int) * 2 * B, cudaMemcpyDeviceToHost, fe->stream));
    FE_CK(cudaMemcpyAsync(paths.data(), fe->paths.p, sizeof(double) * paths.size(), cudaMemcpyDeviceToHost, fe->stream));
    FE_CK(cudaStreamSynchronize(fe->stream));
    if (search_ms) FE_CK(cudaEventElapsedTime(search_ms, fe->e0, fe->e1));

    std::vector<Resampled> res(B);
    long long off = 0;
    for (int b = 0; b < B; b++) {
        const int n = h[b];
        if (n == -2) { err = "one-shot sample buffer overflow"; return UALM_ELIMIT; }
        if (n_expanded) n_expanded[b] = h[B + b];
        const double *pth = paths.data() + 3 * (size_t)a.path_cap * b;
        if (n > 0) resample(pth, n, rp, res[b]);
        if (path_xyyaw) {
            const int k = std::max(n, 0);
            if (off + k > cap_path) { err = "cap_path too small for the polylines"; return UALM_ELIMIT; }
            std::memcpy(path_xyyaw + 3 * off, pth, sizeof(double) * 3 * k);
            off += k;
            path_off[b + 1] = off;
        }
    }
    const int k = pack(res, N, M, bnd, total_time, inner_xy, cap_xy, inner_yaw, cap_yaw, packed);
    if (k < 0) err = "cap_xy / cap_yaw too small";
    return k;
}

}  // namespace ualm_fe
