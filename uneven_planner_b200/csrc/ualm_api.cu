// ualm_api.cu -- the extern "C" layer declared in include/ualm.h: context, uploads, kernel launches.
// Host code is thin: it packs descriptors, sizes shared memory from the batch maxima and launches the
// per-trajectory kernels of ualm_kernels.cuh.  There is NO CPU fallback: every compute entry point needs a CUDA
// device and returns UALM_ENOCUDA otherwise.
#include "ualm_kernels.cuh"
#include "map_prep.h"
#include "ualm_tp_host.h"
#include "ualm_front_end.h"

#include <algorithm>
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

using namespace ualm;

static thread_local std::string g_err;
static int fail(int code, const std::string &msg)
{
    g_err = msg;
    return code;
}
#define CK(call)                                                                                             \
    do {                                                                                                     \
        cudaError_t e_ = (call);                                                                             \
        if (e_ != cudaSuccess) return fail(UALM_ENOCUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t n)
    {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// One in-flight batch ("lane"): its own device buffers, launch plan, streams and events.  A context owns up to UALM_MAX_LANES of
// them so that several batches can be resident and running at once (the stragglers of batch k drain while batch k+1 fills the
// SMs they left: ualm_submit_batch / ualm_wait_batch, or ualm_select_lane + the three-step calls).
#define UALM_MAX_LANES 16
struct Lane {
    bool made = false;
    cudaStream_t stream = nullptr, own_stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool have_batch = false, solved = false, in_flight = false;
    int B = 0, Nmax = 0, Mmax = 0, nmax = 0, Smax = 0, n_active = 0;
    std::vector<ProbDesc> desc;
    std::vector<int> order;              // launch order over the ACTIVE problems (largest first)
    std::vector<unsigned char> skip;     // problems over the compiled limits: not solved, ret_code = UALM_ELIMIT in their record
    long long tot_x = 0, tot_s = 0, tot_cxy = 0, tot_cyaw = 0, tot_hist = 0, tot_scr = 0, tot_fac = 0, tot_ws = 0;
    DevBuf<ProbDesc> d_desc;
    DevBuf<int> d_order;
    DevBuf<int4> d_wdesc;
    std::vector<int4> wdesc;
    std::vector<int> group;      // warps per problem (1, 2 or 4)
    struct GClass { int G = 1, n_ctas = 0, r0 = 0, r1 = 0, occ = 1; size_t wd_off = 0, smem = 0; SmemLayout L; };
    std::vector<GClass> cls;
    enum { NAUX = 7 };
    cudaStream_t aux[NAUX] = {};
    cudaEvent_t evs[NAUX + 1] = {};
    DevBuf<double> d_x0, d_x, d_lambda, d_mu, d_scale_cx, d_hx, d_gx, d_lm_s, d_lm_y, d_lm_aux, d_fac, d_scr, d_ws, d_cxy, d_cyaw, d_f, d_grad, d_sfx;
    DevBuf<ualm_result_t> d_res;
    DevBuf<long long> d_prof;
    DevBuf<double> d_pieceT, d_feas;
    float last_ms = 0.f;
    int last_launches = 0;
    SmemLayout L;
    size_t smem_bytes = 0;
    void release()
    {
        d_desc.release(); d_order.release(); d_wdesc.release();
        DevBuf<double> *bufs[] = {&d_x0, &d_x, &d_lambda, &d_mu, &d_scale_cx, &d_hx, &d_gx, &d_lm_s, &d_lm_y, &d_lm_aux, &d_fac,
                                  &d_scr, &d_ws, &d_cxy, &d_cyaw, &d_f, &d_grad, &d_sfx};
        for (auto *b : bufs) b->release();
        d_res.release(); d_prof.release(); d_pieceT.release(); d_feas.release();
        if (!made) return;
        for (int q = 0; q < NAUX; q++) if (aux[q]) cudaStreamDestroy(aux[q]);
        for (int q = 0; q < NAUX + 1; q++) if (evs[q]) cudaEventDestroy(evs[q]);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (own_stream) cudaStreamDestroy(own_stream);
        made = false;
    }
};

struct ualm_ctx {
    int device = 0, precision = 64;
    ualm_tp::TpEngine *tp = nullptr;     // precision 32 / 65: the throughput engine (ualm_tp.cu) behind the same entry points
    bool have_params = false, have_map = false;
    ualm_params_t hp;
    DevParams dp;
    DevMap dm;
    DevBuf<float4> cells;
    DevBuf<double> cells64;
    Lane lanes[UALM_MAX_LANES];
    Lane *b = nullptr;            // the selected lane (ualm_select_lane; lane 0 by default)
    int cur = 0, next_submit = 0;
    int group_mode = 1;
    bool profile = false;
    // pipeline timing (ualm_mark_begin / ualm_mark_end): events on the lanes' own streams, joined on `join`
    cudaStream_t join = nullptr;
    cudaEvent_t evA = nullptr, evB = nullptr;
    ualm_fe::FrontEnd *fe = nullptr;     // the device front-end's map and workspaces (ualm_set_front_end_map)
};

static int lane_make(ualm_ctx *c, Lane &l)
{
    if (l.made) return UALM_OK;
    l.made = true;     // release() cleans up whatever was created if one of the calls below fails
    CK(cudaStreamCreateWithFlags(&l.own_stream, cudaStreamNonBlocking));
    l.stream = l.own_stream;
    for (int q = 0; q < Lane::NAUX; q++) CK(cudaStreamCreateWithFlags(&l.aux[q], cudaStreamNonBlocking));
    for (int q = 0; q < Lane::NAUX + 1; q++) CK(cudaEventCreateWithFlags(&l.evs[q], cudaEventDisableTiming));
    CK(cudaEventCreate(&l.ev0));
    CK(cudaEventCreate(&l.ev1));
    (void)c;
    return UALM_OK;
}

extern "C" const char *ualm_last_error(void) { return g_err.c_str(); }

// throughput contexts forward to the engine; its error text lands in the same thread-local message
#define TP_CALL(expr)                                  \
    do {                                               \
        std::string em_;                               \
        std::string *err = &em_;                       \
        const int rc_ = (expr);                        \
        if (rc_ != UALM_OK) g_err = em_;               \
        return rc_;                                    \
    } while (0)
#define TP_UNSUPPORTED(name) return fail(UALM_EINVAL, name " is an entry point of the parity path (precision 64) only")

extern "C" int ualm_create(ualm_ctx_t **out, int device, int precision)
{
    if (!out) return fail(UALM_EINVAL, "ctx out pointer is NULL");
    if (precision != 64 && precision != 65 && precision != 32)
        return fail(UALM_EINVAL, "precision must be 64 (bit-reproducible double), 65 (throughput path in double) or 32 (throughput path in float)");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0) return fail(UALM_ENOCUDA, std::string("no CUDA device: ") + cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(UALM_EINVAL, "device ordinal out of range");
    CK(cudaSetDevice(device));
    ualm_ctx *c = new ualm_ctx();
    c->device = device; c->precision = precision;
    if (const char *e = getenv("UALM_GROUPS")) c->group_mode = atoi(e);   // 0 = one warp per trajectory everywhere (developer switch)
    c->b = &c->lanes[0];
    if (precision != 64) {
        std::string em;
        const int rc = ualm_tp::tp_create(&c->tp, device, precision, &em);
        if (rc != UALM_OK) { delete c; return fail(rc, em); }
        *out = c;
        return UALM_OK;
    }
    int rc = lane_make(c, c->lanes[0]);
    if (rc == UALM_OK) {
        cudaError_t e1 = cudaStreamCreateWithFlags(&c->join, cudaStreamNonBlocking);
        if (e1 == cudaSuccess) e1 = cudaEventCreate(&c->evA);
        if (e1 == cudaSuccess) e1 = cudaEventCreate(&c->evB);
        if (e1 != cudaSuccess) rc = fail(UALM_ENOCUDA, std::string("context streams/events: ") + cudaGetErrorString(e1));
    }
    if (rc != UALM_OK) { const std::string keep = g_err; ualm_destroy(c); g_err = keep; return rc; }   // no leak on a failed create
    *out = c;
    return UALM_OK;
}

extern "C" int ualm_destroy(ualm_ctx_t *c)
{
    if (!c) return UALM_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    if (c->tp) { ualm_tp::tp_destroy(c->tp); c->tp = nullptr; }
    ualm_fe::release(c->fe); c->fe = nullptr;
    c->cells.release(); c->cells64.release();
    for (auto &l : c->lanes) l.release();
    if (c->join) cudaStreamDestroy(c->join);
    if (c->evA) cudaEventDestroy(c->evA);
    if (c->evB) cudaEventDestroy(c->evB);
    delete c;
    return UALM_OK;
}

extern "C" int ualm_select_lane(ualm_ctx_t *c, int lane)
{
    if (!c) return fail(UALM_EINVAL, "null ctx");
    if (lane < 0 || lane >= UALM_MAX_LANES) return fail(UALM_EINVAL, "lane out of range [0, UALM_MAX_LANES)");
    CK(cudaSetDevice(c->device));
    if (!c->tp) {
        int rc = lane_make(c, c->lanes[lane]);
        if (rc) return rc;
    }
    c->cur = lane; c->b = &c->lanes[lane];
    return UALM_OK;
}

extern "C" int ualm_max_lanes(void) { return UALM_MAX_LANES; }

// all work of the selected lane on a caller-owned stream.  The handle is taken literally: NULL is the legacy default stream
// (what torch.cuda.current_stream().cuda_stream is when torch runs on its default stream); ualm_reset_stream restores the
// lane's own non-blocking stream.
extern "C" int ualm_set_stream(ualm_ctx_t *c, void *s)
{
    if (!c) return fail(UALM_EINVAL, "null ctx");
    if (c->tp) TP_UNSUPPORTED("ualm_set_stream");
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->b->stream));
    c->b->stream = (cudaStream_t)s;
    return UALM_OK;
}
extern "C" int ualm_reset_stream(ualm_ctx_t *c)
{
    if (!c) return fail(UALM_EINVAL, "null ctx");
    if (c->tp) return UALM_OK;
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->b->stream));
    c->b->stream = c->b->own_stream;
    return UALM_OK;
}

extern "C" int ualm_set_params(ualm_ctx_t *c, const ualm_params_t *p)
{
    if (!c || !p) return fail(UALM_EINVAL, "null argument");
    if (p->int_K < 1 || p->int_K > 128) return fail(UALM_ELIMIT, "int_K out of range [1,128]");
    if (p->mem_size < 1 || p->mem_size > 1024) return fail(UALM_ELIMIT, "mem_size out of range [1,1024]");
    if (p->past < 0 || p->past > 16) return fail(UALM_ELIMIT, "past out of range [0,16]");
    for (auto &l : c->lanes)
        if (l.in_flight) return fail(UALM_ESTATE, "ualm_set_params while a submitted batch is in flight (ualm_wait_batch first)");
    // int_K, mem_size and past are baked into the resident batches' descriptors, buffer sizes and shared-memory layouts: a
    // parameter change invalidates every uploaded batch (it must be uploaded again before the next solve / eval call)
    for (auto &l : c->lanes) { l.have_batch = false; l.solved = false; }
    c->hp = *p;
    DevParams &d = c->dp;
    d.rho_T = p->rho_T; d.rho_ter = p->rho_ter; d.max_vel = p->max_vel; d.max_acc_lon = p->max_acc_lon; d.max_acc_lat = p->max_acc_lat;
    d.max_kap = p->max_kap; d.min_cxi = p->min_cxi; d.max_sig = p->max_sig; d.use_scaling = p->use_scaling; d.rho = p->rho;
    d.beta = p->beta; d.gamma = p->gamma; d.epsilon_con = p->epsilon_con; d.max_iter = p->max_iter; d.g_epsilon = p->g_epsilon;
    d.min_step = p->min_step; d.delta = p->delta; d.inner_max_iter = (int)p->inner_max_iter; d.mem_size = p->mem_size; d.past = p->past;
    d.int_K = p->int_K; d.gravity = p->gravity;
    c->have_params = true;
    if (c->tp) TP_CALL(ualm_tp::tp_set_params(c->tp, p, err));
    return UALM_OK;
}

static int map_geometry_set(ualm_ctx *c, const ualm_map_geom_t *g)
{
    DevMap &m = c->dm;
    for (int k = 0; k < 3; k++) { m.vn[k] = g->voxel_num[k]; m.origin[k] = g->origin[k]; m.maxb[k] = g->max_boundary[k]; }
    m.xy_res = g->xy_resolution; m.yaw_res = g->yaw_resolution;
    m.xy_inv = 1.0 / g->xy_resolution; m.yaw_inv = 1.0 / g->yaw_resolution; // uneven_map.cpp:104-105
    c->have_map = true;
    return UALM_OK;
}
static int lanes_idle(ualm_ctx *c, const char *what)
{
    for (auto &l : c->lanes)
        if (l.in_flight) return fail(UALM_ESTATE, std::string(what) + " while a submitted batch is in flight (ualm_wait_batch first)");
    return UALM_OK;
}

extern "C" int ualm_set_map(ualm_ctx_t *c, const ualm_map_geom_t *g, const float *cells)
{
    if (!c || !g || !cells) return fail(UALM_EINVAL, "null argument");
    if (int rc = lanes_idle(c, "ualm_set_map")) return rc;
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    const size_t ncell = (size_t)g->voxel_num[0] * g->voxel_num[1] * g->voxel_num[2];
    CK(c->cells.ensure(ncell));
    CK(cudaMemcpy(c->cells.p, cells, ncell * sizeof(float4), cudaMemcpyHostToDevice));
    c->cells64.release();
    c->dm.cells = c->cells.p; c->dm.cells64 = nullptr;
    map_geometry_set(c, g);
    if (c->tp) TP_CALL(ualm_tp::tp_set_map(c->tp, g, cells, err));      // (the context's own copy serves the post-solve scan)
    return UALM_OK;
}

// the reference's own grid: UnevenMap::map_buffer is RXS2 {double z, sigma; Vector2d zb} = 4 doubles per cell (uneven_map.h:36-64)
extern "C" int ualm_set_map_f64(ualm_ctx_t *c, const ualm_map_geom_t *g, const double *cells, int repack_to_float)
{
    if (!c || !g || !cells) return fail(UALM_EINVAL, "null argument");
    if (int rc = lanes_idle(c, "ualm_set_map_f64")) return rc;
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    const size_t ncell = (size_t)g->voxel_num[0] * g->voxel_num[1] * g->voxel_num[2];
    if (repack_to_float || c->tp) {      // the throughput path always reads the float4 grid
        std::vector<float> f(4 * ncell);
        for (size_t q = 0; q < 4 * ncell; q++) f[q] = (float)cells[q];
        return ualm_set_map(c, g, f.data());
    }
    CK(c->cells64.ensure(4 * ncell));
    CK(cudaMemcpy(c->cells64.p, cells, 4 * ncell * sizeof(double), cudaMemcpyHostToDevice));
    c->cells.release();
    c->dm.cells = nullptr; c->dm.cells64 = c->cells64.p;
    return map_geometry_set(c, g);
}

static int prepare_launch(ualm_ctx *c)
{
    Lane *b = c->b;
    b->L = make_layout(b->Nmax, b->Mmax, b->nmax, c->dp.mem_size, c->dp.past, c->dp.int_K, b->Smax);
    b->smem_bytes = (size_t)b->L.total_doubles * sizeof(double) * UALM_WPB;
    if (b->smem_bytes > 227 * 1024) return fail(UALM_ELIMIT, "problem too large for shared memory (N/M/int_K too big)");
    // the attribute is per function, not per lane: only ever raise it (another lane's kernels may be in flight with a larger size)
    static size_t smem_max = 0;
    if (b->smem_bytes > smem_max) {
        smem_max = b->smem_bytes;
        CK(cudaFuncSetAttribute(solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
        CK(cudaFuncSetAttribute(eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
        CK(cudaFuncSetAttribute(scaling_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
        CK(cudaFuncSetAttribute(penalty_only_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    }
    return UALM_OK;
}

static BatchPtrs batch_ptrs(ualm_ctx *c)
{
    Lane *l = c->b;
    BatchPtrs b;
    b.B = l->B;
    b.n_active = l->n_active;
    b.wdesc = l->d_wdesc.p;
    b.n_leader_slots = 4;
    b.adopt = getenv("UALM_NOADOPT") ? 0 : 1;
    b.desc = l->d_desc.p; b.order = l->d_order.p; b.x0 = l->d_x0.p; b.x = l->d_x.p;
    b.lambda = l->d_lambda.p; b.mu = l->d_mu.p; b.scale_cx = l->d_scale_cx.p; b.hx = l->d_hx.p; b.gx = l->d_gx.p;
    b.lm_s = l->d_lm_s.p; b.lm_y = l->d_lm_y.p; b.lm_aux = l->d_lm_aux.p; b.fac = l->d_fac.p; b.scratch = l->d_scr.p; b.ws_scaling = l->d_ws.p;
    b.c_xy = l->d_cxy.p; b.c_yaw = l->d_cyaw.p; b.results = l->d_res.p; b.piece_T = l->d_pieceT.p; b.f_out = l->d_f.p; b.grad_out = l->d_grad.p;
    b.scale_fx_io = l->d_sfx.p;
    b.prof = c->profile ? l->d_prof.p : nullptr;
    return b;
}

extern "C" int ualm_upload(ualm_ctx_t *c, int B, const int32_t *N, const int32_t *M, const double *bnd, const double *total_time,
                           const double *inner_xy, const double *inner_yaw)
{
    if (!c || B < 0 || (B > 0 && (!N || !M || !bnd || !total_time))) return fail(UALM_EINVAL, "bad argument");
    if (c->tp) TP_CALL(ualm_tp::tp_upload(c->tp, c->cur, B, N, M, bnd, total_time, inner_xy, inner_yaw, err));
    if (!c->have_params) return fail(UALM_ESTATE, "ualm_set_params must be called before ualm_upload");
    Lane *l = c->b;
    if (l->in_flight) return fail(UALM_ESTATE, "ualm_upload into a lane whose submitted batch is still in flight");
    // validate everything before touching the lane; the lane holds no batch until this call has fully succeeded
    long long need_xy = 0, need_yaw = 0;
    for (int b = 0; b < B; b++) {
        if (N[b] < 1 || M[b] < 1) return fail(UALM_EINVAL, "piece counts must be >= 1");
        if (!(total_time[b] > 0.0) || !std::isfinite(total_time[b])) return fail(UALM_EINVAL, "total_time must be finite and > 0");
        need_xy += 2LL * (N[b] - 1); need_yaw += M[b] - 1;
    }
    if ((need_xy > 0 && !inner_xy) || (need_yaw > 0 && !inner_yaw)) return fail(UALM_EINVAL, "inner waypoint arrays are NULL but N > 1 or M > 1");
    l->have_batch = false; l->solved = false;
    CK(cudaSetDevice(c->device));
    const int K = c->dp.int_K, m = c->dp.mem_size;
    l->B = B; l->desc.assign(B, ProbDesc()); l->order.clear(); l->group.assign(B, 1); l->skip.assign(B, 0);
    l->Nmax = l->Mmax = l->nmax = l->Smax = 1;
    for (int b = 0; b < B; b++) {
        ProbDesc &d = l->desc[b];
        d.N = N[b]; d.M = M[b];
        // compiled limits (n <= 256: the L-BFGS register tile, UALM_NREG in ualm_kernels.cuh): such a problem is not solved, its
        // record says UALM_ELIMIT, and the rest of the batch runs
        if (N[b] > UALM_NMAX || M[b] > UALM_MMAX) { l->skip[b] = 1; d.n = 0; d.S = 0; continue; }
        d.n = 1 + 2 * (N[b] - 1) + (M[b] - 1); d.S = N[b] * (K + 1);
        l->Nmax = std::max(l->Nmax, d.N); l->Mmax = std::max(l->Mmax, d.M); l->nmax = std::max(l->nmax, d.n); l->Smax = std::max(l->Smax, d.S);
        l->order.push_back(b);
    }
    l->n_active = (int)l->order.size();
    const int BA = l->n_active;
    // launch order: most samples first (longest-processing-time-first keeps the tail short)
    std::stable_sort(l->order.begin(), l->order.end(), [&](int a, int b2) { return l->desc[a].S > l->desc[b2].S; });
    int rc0 = prepare_launch(c);
    if (rc0) return rc0;
    // Warp groups and size classes.  Problems are sorted by size; the largest get 4 or 2 warps (helpers for the parallel
    // phases) as far as the whole batch still fits on the device at once.  Every (group size, size bucket) class is its own
    // launch with its own shared-memory layout sized by the class maxima: a G=4 CTA holds one trajectory slot + 3 helper
    // rings, a G=2 CTA two slots + 2 rings, a G=1 CTA four slots.  The classes run concurrently on separate streams.
    {
        int dev_sms = 0;
        CK(cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, c->device));
        const int RINGD = 2 * UALM_RINGB * 6 * UALM_FW;
        int occ0 = 1;   // CTAs per SM the register file allows (shared memory is checked per class below)
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ0, solve_kernel, UALM_THREADS * UALM_WPB, 16 * 1024));
        if (getenv("UALM_DEBUG")) {
            cudaFuncAttributes fa;
            CK(cudaFuncGetAttributes(&fa, solve_kernel));
            fprintf(stderr, "[ualm] solve_kernel: %d regs/thread, %zu B local, %zu B static smem, %d CTAs/SM by registers\n", fa.numRegs, fa.localSizeBytes,
                    fa.sharedSizeBytes, occ0);
        }
        const long long W = 4LL * occ0 * dev_sms;   // warp slots on the device
        std::vector<Lane::GClass> best;
        for (int attempt = 0; attempt < 32; attempt++) {
            // Policy (measured on B200, tools/gpu_policy_dev.py): helpers shorten the latency of a trajectory without adding to the
            // L2-resident working set, while more resident trajectories than ~600 thrash the 126 MB L2.  So: everything that fits
            // gets 4 warps; beyond that 2 warps per trajectory with the largest tenth at 4, run in waves.
            long long K4 = 0, K2 = 0;
            if (c->group_mode) {
                if (4LL * BA <= W) K4 = BA;
                else if (2LL * BA <= W) { K4 = std::min<long long>(BA, (W - 2LL * BA) / 2); K2 = (BA - K4) & ~1LL; }
                else { K4 = BA / 10; K2 = (BA - K4) & ~1LL; }
                if (attempt > 0) { K4 = (long long)(K4 * std::pow(0.8, attempt)); K2 = std::min<long long>(BA - K4, K2) & ~1LL; }
            }
            const bool forced = getenv("UALM_F4") || getenv("UALM_F2");   // developer override: fractions of the batch
            if (forced) {
                K4 = (long long)(BA * (getenv("UALM_F4") ? atof(getenv("UALM_F4")) : 0.0));
                K2 = std::min<long long>(BA - K4, (long long)(BA * (getenv("UALM_F2") ? atof(getenv("UALM_F2")) : 0.0))) & ~1LL;
            }
            // rank ranges per group size, each split into size buckets (the order is by descending size)
            std::vector<Lane::GClass> cls;
            const long long lim[4] = {0, K4, K4 + K2, BA};
            for (int gi = 0; gi < 3; gi++) {
                const int G = gi == 0 ? 4 : gi == 1 ? 2 : 1;
                const long long a = lim[gi], b2 = lim[gi + 1];
                if (b2 <= a) continue;
                const int nsplit = (b2 - a) >= 96 ? (gi == 2 ? 3 : 2) : 1;
                for (int sp = 0; sp < nsplit; sp++) {
                    Lane::GClass cl;
                    cl.G = G;
                    long long s0 = a + (b2 - a) * sp / nsplit, s1 = a + (b2 - a) * (sp + 1) / nsplit;
                    const int per = 4 / G;                         // problems per CTA
                    if (sp > 0) s0 = a + ((s0 - a + per - 1) / per) * per;
                    if (sp + 1 < nsplit) s1 = a + ((s1 - a + per - 1) / per) * per;
                    if (s1 <= s0) continue;
                    cl.r0 = (int)s0; cl.r1 = (int)s1;
                    int Nm = 1, Mm = 1, nm = 1, Sm = 1;
                    for (long long r = s0; r < s1; r++) {
                        const ProbDesc &d = l->desc[l->order[r]];
                        Nm = std::max(Nm, d.N); Mm = std::max(Mm, d.M); nm = std::max(nm, d.n); Sm = std::max(Sm, d.S);
                    }
                    cl.L = make_layout(Nm, Mm, nm, c->dp.mem_size, c->dp.past, c->dp.int_K, Sm);
                    cl.smem = ((size_t)per * cl.L.total_doubles + (size_t)(4 - per) * RINGD) * sizeof(double);
                    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cl.occ, solve_kernel, UALM_THREADS * UALM_WPB, cl.smem));
                    cl.n_ctas = (int)((s1 - s0 + per - 1) / per);
                    cls.push_back(cl);
                }
            }
            double sm_need = 0.0;
            for (auto &cl : cls) sm_need += (double)cl.n_ctas / std::max(cl.occ, 1);
            best = cls;
            // multi-wave batches need not fit at once; batches meant to be fully resident must
            if (forced || 2LL * BA > W || sm_need <= 0.98 * dev_sms || attempt >= 12) break;
        }
        l->cls = best;
        l->wdesc.clear();
        for (auto &cl : l->cls) {
            cl.wd_off = l->wdesc.size();
            for (int r = cl.r0; r < cl.r1; r++) l->group[l->order[r]] = cl.G;
            int q = cl.r0;
            while (q < cl.r1) {
                if (cl.G == 4) {
                    for (int w = 0; w < 4; w++) l->wdesc.push_back(make_int4(l->order[q], 0, 4, w | ((w ? w - 1 : 0) << 8)));
                    q += 1;
                } else if (cl.G == 2) {
                    // CTA j of the class pairs its j-th largest with its j-th smallest problem: the small one ends early and its
                    // two warps then help the large one (adoption, ualm_kernels.cuh)
                    const int j = (q - cl.r0) / 2;
                    const int pa = cl.r0 + j, pb = cl.r1 - 1 - j;
                    const int pr[2] = {l->order[pa], pb > pa ? l->order[pb] : -1};
                    for (int h = 0; h < 2; h++) {
                        if (pr[h] >= 0) {
                            l->wdesc.push_back(make_int4(pr[h], h, 2, 0));
                            l->wdesc.push_back(make_int4(pr[h], h, 2, 1 | (h << 8)));
                        } else { l->wdesc.push_back(make_int4(-1, 0, 1, 0)); l->wdesc.push_back(make_int4(-1, 0, 1, 0)); }
                    }
                    q += 2;
                } else {
                    for (int w = 0; w < 4; w++) {
                        if (q < cl.r1) { l->wdesc.push_back(make_int4(l->order[q], w, 1, 0)); q += 1; }
                        else l->wdesc.push_back(make_int4(-1, 0, 1, 0));
                    }
                }
            }
            if ((int)((l->wdesc.size() - cl.wd_off) / 4) != cl.n_ctas) return fail(UALM_EINVAL, "internal: class CTA count mismatch");
            if (getenv("UALM_DEBUG"))
                fprintf(stderr, "[ualm] class G=%d: problems [%d,%d) %d CTAs, smem %zu B, %d CTAs/SM\n", cl.G, cl.r0, cl.r1, cl.n_ctas, cl.smem, cl.occ);
        }
    }
    long long ox = 0, os = 0, ocx = 0, ocy = 0, oh = 0, oscr = 0, oixy = 0, oiyaw = 0, ofac = 0, ows = 0;
    std::vector<double> x0;
    std::vector<ualm_result_t> res0(B);
    for (int b = 0; b < B; b++) {
        ProbDesc &d = l->desc[b];
        d.off_x = ox; d.off_s = os; d.off_cxy = ocx; d.off_cyaw = ocy; d.off_hist = oh; d.off_scr = oscr; d.off_fac = ofac; d.off_ws = ows;
        for (int k = 0; k < 18; k++) d.bnd[k] = bnd[(size_t)b * 18 + k];
        d.total_time = total_time[b];
        memset(&res0[b], 0, sizeof(ualm_result_t));
        ocx += 12 * d.N; ocy += 6 * d.M;
        const long long nxy = 2LL * (d.N - 1), nyw = d.M - 1;
        if (l->skip[b]) { res0[b].ret_code = UALM_ELIMIT; oixy += nxy; oiyaw += nyw; continue; }
        // x = [tau | Pxy | Pyaw]  (alm_traj_opt.cpp:205-216); logC2 (alm_traj_opt.h:238-241) is two IEEE ops + sqrt
        const double T = total_time[b];
        x0.push_back(T > 1.0 ? (std::sqrt(2.0 * T - 1.0) - 1.0) : (1.0 - std::sqrt(2.0 / T - 1.0)));
        for (long long q = 0; q < nxy; q++) x0.push_back(inner_xy[oixy + q]);
        for (long long q = 0; q < nyw; q++) x0.push_back(inner_yaw[oiyaw + q]);
        oixy += nxy; oiyaw += nyw;
        ox += d.n; os += d.S; oh += (long long)m * d.n; oscr += (long long)UALM_NFIELD * d.S;
        ofac += 1LL * UALM_FW * ((6 * d.N + 2 * UALM_FPAD) + (6 * d.M + 2 * UALM_FPAD));
        ows += (long long)(12 * d.N + 6 * d.M) * 32 * l->group[b];
    }
    l->tot_x = ox; l->tot_s = os; l->tot_cxy = ocx; l->tot_cyaw = ocy; l->tot_hist = oh; l->tot_scr = oscr; l->tot_fac = ofac; l->tot_ws = ows;
    CK(l->d_desc.ensure(B)); CK(l->d_order.ensure(BA)); CK(l->d_wdesc.ensure(l->wdesc.size())); CK(l->d_x0.ensure(ox)); CK(l->d_x.ensure(ox)); CK(l->d_grad.ensure(ox));
    CK(l->d_lambda.ensure(os)); CK(l->d_hx.ensure(os)); CK(l->d_mu.ensure(6 * os)); CK(l->d_gx.ensure(6 * os)); CK(l->d_scale_cx.ensure(7 * os));
    CK(l->d_lm_s.ensure(oh)); CK(l->d_lm_y.ensure(oh)); CK(l->d_scr.ensure(oscr));
    CK(l->d_ws.ensure(ows)); CK(l->d_fac.ensure(ofac)); CK(l->d_lm_aux.ensure((size_t)std::max(B, 1) * 3 * m));
    // factor arrays: entries outside the band-in-matrix positions (and the pad rows) are never written and must read 0
    if (ofac > 0) CK(cudaMemsetAsync(l->d_fac.p, 0, sizeof(double) * ofac, l->stream));
    CK(l->d_prof.ensure((size_t)std::max(B, 1) * UALM_NPROF));
    CK(l->d_pieceT.ensure((size_t)std::max(B, 1) * 2)); CK(l->d_feas.ensure((size_t)std::max(B, 1) * 10));
    CK(l->d_cxy.ensure(ocx)); CK(l->d_cyaw.ensure(ocy)); CK(l->d_res.ensure(B)); CK(l->d_f.ensure(B)); CK(l->d_sfx.ensure(B));
    if (B > 0) {
        CK(cudaMemcpyAsync(l->d_desc.p, l->desc.data(), sizeof(ProbDesc) * B, cudaMemcpyHostToDevice, l->stream));
        if (BA > 0) CK(cudaMemcpyAsync(l->d_order.p, l->order.data(), sizeof(int) * BA, cudaMemcpyHostToDevice, l->stream));
        if (!l->wdesc.empty()) CK(cudaMemcpyAsync(l->d_wdesc.p, l->wdesc.data(), sizeof(int4) * l->wdesc.size(), cudaMemcpyHostToDevice, l->stream));
        if (ox > 0) CK(cudaMemcpyAsync(l->d_x0.p, x0.data(), sizeof(double) * ox, cudaMemcpyHostToDevice, l->stream));
        // records of skipped problems (the kernels overwrite the others), zero coefficients and durations for them
        CK(cudaMemcpyAsync(l->d_res.p, res0.data(), sizeof(ualm_result_t) * B, cudaMemcpyHostToDevice, l->stream));
        if (BA < B) {
            CK(cudaMemsetAsync(l->d_cxy.p, 0, sizeof(double) * ocx, l->stream));
            CK(cudaMemsetAsync(l->d_cyaw.p, 0, sizeof(double) * ocy, l->stream));
            CK(cudaMemsetAsync(l->d_pieceT.p, 0, sizeof(double) * 2 * B, l->stream));
        }
        CK(cudaStreamSynchronize(l->stream)); // x0 / res0 are stack-local staging vectors
    }
    l->have_batch = true; l->solved = false;
    return UALM_OK;
}

extern "C" int ualm_solve_resident(ualm_ctx_t *c)
{
    if (!c) return fail(UALM_EINVAL, "null ctx");
    if (c->tp) TP_CALL(ualm_tp::tp_admit(c->tp, c->cur, err));      // joins the pool of running trajectories; ualm_sync / download drive the rounds
    Lane *l = c->b;
    if (!c->have_map || !c->have_params || !l->have_batch) return fail(UALM_ESTATE, "set_params, set_map and upload must precede solve");
    CK(cudaSetDevice(c->device));
    l->last_launches = 0;
    CK(cudaEventRecord(l->ev0, l->stream));
    if (l->n_active > 0) {
        // the classes run concurrently: class 0 on the lane stream, the others on auxiliary streams
        const int last = Lane::NAUX;
        CK(cudaEventRecord(l->evs[last], l->stream));
        for (size_t ci = 0; ci < l->cls.size(); ci++) {
            auto &cl = l->cls[ci];
            if (cl.n_ctas == 0) continue;
            const int ai = (int)((ci - 1) % Lane::NAUX);
            cudaStream_t st = ci == 0 ? l->stream : l->aux[ai];
            if (ci > 0) CK(cudaStreamWaitEvent(st, l->evs[last], 0));
            BatchPtrs bp = batch_ptrs(c);
            bp.wdesc = l->d_wdesc.p + cl.wd_off;
            bp.n_leader_slots = 4 / cl.G;
            solve_kernel<<<cl.n_ctas, UALM_THREADS * UALM_WPB, cl.smem, st>>>(bp, c->dp, c->dm, cl.L);
            CK(cudaGetLastError());
            l->last_launches++;
            if (ci > 0) { CK(cudaEventRecord(l->evs[ai], st)); CK(cudaStreamWaitEvent(l->stream, l->evs[ai], 0)); }
        }
    }
    CK(cudaEventRecord(l->ev1, l->stream));
    l->solved = true;
    return UALM_OK;
}

extern "C" int ualm_sync(ualm_ctx_t *c)
{
    if (!c) return fail(UALM_EINVAL, "null ctx");
    if (c->tp) {
        if (!ualm_tp::tp_lane_in_flight(c->tp, c->cur)) return UALM_OK;
        TP_CALL(ualm_tp::tp_collect(c->tp, c->cur, err));
    }
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->b->stream));
    return UALM_OK;
}

extern "C" int ualm_last_solve_ms(ualm_ctx_t *c, float *ms, int *launches)
{
    if (c && c->tp) return ualm_tp::tp_last_solve(c->tp, c->cur, ms, launches) == UALM_OK ? UALM_OK : fail(UALM_ESTATE, "no collected solve to time");
    if (!c || !c->b->solved) return fail(UALM_ESTATE, "no solve to time");
    Lane *l = c->b;
    CK(cudaEventSynchronize(l->ev1));
    CK(cudaEventElapsedTime(&l->last_ms, l->ev0, l->ev1));
    if (ms) *ms = l->last_ms;
    if (launches) *launches = l->last_launches;
    return UALM_OK;
}

// pipeline timing over several lanes: begin = an event on the selected lane's stream (record it before the first launch of the
// timed region); end = an event on a join stream that waits for the last solve of every lane
extern "C" int ualm_mark_begin(ualm_ctx_t *c)
{
    if (!c) return fail(UALM_EINVAL, "null ctx");
    if (c->tp) TP_CALL(ualm_tp::tp_mark_begin(c->tp, err));
    CK(cudaSetDevice(c->device));
    CK(cudaEventRecord(c->evA, c->b->stream));
    return UALM_OK;
}
extern "C" int ualm_mark_end(ualm_ctx_t *c, float *ms)
{
    if (!c || !ms) return fail(UALM_EINVAL, "null argument");
    if (c->tp) TP_CALL(ualm_tp::tp_mark_end(c->tp, ms, err));
    CK(cudaSetDevice(c->device));
    for (auto &l : c->lanes)
        if (l.made && l.solved) CK(cudaStreamWaitEvent(c->join, l.ev1, 0));
    CK(cudaEventRecord(c->evB, c->join));
    CK(cudaEventSynchronize(c->evB));
    CK(cudaEventElapsedTime(ms, c->evA, c->evB));
    return UALM_OK;
}

extern "C" int ualm_download(ualm_ctx_t *c, ualm_result_t *results, double *c_xy, double *c_yaw)
{
    if (c && c->tp) {
        if (!ualm_tp::tp_lane_in_flight(c->tp, c->cur) && !ualm_tp::tp_lane_collected(c->tp, c->cur)) return fail(UALM_ESTATE, "nothing solved");
        TP_CALL(ualm_tp::tp_download(c->tp, c->cur, results, c_xy, c_yaw, err));
    }
    if (!c || !c->b->solved) return fail(UALM_ESTATE, "nothing solved");
    Lane *l = c->b;
    CK(cudaSetDevice(c->device));
    if (l->B > 0) {
        if (results) CK(cudaMemcpyAsync(results, l->d_res.p, sizeof(ualm_result_t) * l->B, cudaMemcpyDeviceToHost, l->stream));
        if (c_xy) CK(cudaMemcpyAsync(c_xy, l->d_cxy.p, sizeof(double) * l->tot_cxy, cudaMemcpyDeviceToHost, l->stream));
        if (c_yaw) CK(cudaMemcpyAsync(c_yaw, l->d_cyaw.p, sizeof(double) * l->tot_cyaw, cudaMemcpyDeviceToHost, l->stream));
    }
    CK(cudaStreamSynchronize(l->stream));
    return UALM_OK;
}

extern "C" int ualm_solve_batch(ualm_ctx_t *c, int B, const int32_t *N, const int32_t *M, const double *bnd, const double *total_time,
                                const double *inner_xy, const double *inner_yaw, ualm_result_t *results, double *c_xy, double *c_yaw)
{
    int rc = ualm_upload(c, B, N, M, bnd, total_time, inner_xy, inner_yaw);
    if (rc) return rc;
    rc = ualm_solve_resident(c);
    if (rc) return rc;
    return ualm_download(c, results, c_xy, c_yaw);
}

// ---- pipelined batches: submit returns as soon as the batch is uploaded and its kernels are queued; several batches (one per
// lane, round robin) run concurrently, so the slow tail of one batch overlaps the bulk of the next ----
extern "C" int ualm_submit_batch(ualm_ctx_t *c, int B, const int32_t *N, const int32_t *M, const double *bnd, const double *total_time,
                                 const double *inner_xy, const double *inner_yaw, int depth, int *ticket)
{
    if (!c || !ticket) return fail(UALM_EINVAL, "null argument");
    if (depth < 1 || depth > UALM_MAX_LANES) return fail(UALM_EINVAL, "depth out of range [1, UALM_MAX_LANES]");
    const int lane = c->next_submit % depth;
    if (c->tp) {
        if (ualm_tp::tp_lane_in_flight(c->tp, lane)) return fail(UALM_ESTATE, "all lanes of this depth are in flight: ualm_wait_batch the oldest ticket first");
        std::string em;
        int rc = ualm_tp::tp_upload(c->tp, lane, B, N, M, bnd, total_time, inner_xy, inner_yaw, &em);
        if (!rc) rc = ualm_tp::tp_admit(c->tp, lane, &em);
        if (rc) return fail(rc, em);
        *ticket = lane; c->next_submit = (lane + 1) % depth;
        return UALM_OK;
    }
    if (c->lanes[lane].in_flight) return fail(UALM_ESTATE, "all lanes of this depth are in flight: ualm_wait_batch the oldest ticket first");
    const int keep = c->cur;
    int rc = ualm_select_lane(c, lane);
    if (!rc) rc = ualm_upload(c, B, N, M, bnd, total_time, inner_xy, inner_yaw);
    if (!rc) rc = ualm_solve_resident(c);
    if (!rc) { c->lanes[lane].in_flight = true; *ticket = lane; c->next_submit = (lane + 1) % depth; }
    c->cur = keep; c->b = &c->lanes[keep];
    return rc;
}
extern "C" int ualm_wait_batch(ualm_ctx_t *c, int ticket, ualm_result_t *results, double *c_xy, double *c_yaw)
{
    if (!c || ticket < 0 || ticket >= UALM_MAX_LANES) return fail(UALM_EINVAL, "bad ticket");
    if (c->tp) {
        if (!ualm_tp::tp_lane_in_flight(c->tp, ticket)) return fail(UALM_ESTATE, "ticket is not in flight");
        TP_CALL(ualm_tp::tp_download(c->tp, ticket, results, c_xy, c_yaw, err));
    }
    if (!c->lanes[ticket].in_flight) return fail(UALM_ESTATE, "ticket is not in flight");
    const int keep = c->cur;
    c->cur = ticket; c->b = &c->lanes[ticket];
    const int rc = ualm_download(c, results, c_xy, c_yaw);
    c->lanes[ticket].in_flight = false;
    c->cur = keep; c->b = &c->lanes[keep];
    return rc;
}

// ---- one host process, several GPUs: contexts on different devices (same params and map set on each), the batch dealt over
// them (cost-sorted snake, like uneven_planner_b200/distributed.py), solved concurrently, results scattered back in problem order.
// No collective: a single host gathers by D2H copies.  (The one-process-per-GPU variant with an NCCL all-gather of result
// records is ualm_pack_records_device + the caller's communicator.) ----
extern "C" int ualm_solve_batch_multi(ualm_ctx_t **ctxs, int nctx, int B, const int32_t *N, const int32_t *M, const double *bnd,
                                      const double *total_time, const double *inner_xy, const double *inner_yaw, ualm_result_t *results,
                                      double *c_xy, double *c_yaw)
{
    if (!ctxs || nctx < 1 || B < 0) return fail(UALM_EINVAL, "bad argument");
    for (int r = 0; r < nctx; r++) if (!ctxs[r]) return fail(UALM_EINVAL, "null ctx in list");
    if (B == 0) return UALM_OK;
    if (!N || !M || !bnd || !total_time) return fail(UALM_EINVAL, "null argument");
    std::vector<long long> oxy(B + 1, 0), oyw(B + 1, 0), ocx(B + 1, 0), ocy(B + 1, 0);
    for (int b = 0; b < B; b++) {
        if (N[b] < 1 || M[b] < 1) return fail(UALM_EINVAL, "piece counts must be >= 1");
        oxy[b + 1] = oxy[b] + 2LL * (N[b] - 1); oyw[b + 1] = oyw[b] + (M[b] - 1);
        ocx[b + 1] = ocx[b] + 12LL * N[b]; ocy[b + 1] = ocy[b] + 6LL * M[b];
    }
    std::vector<int> ord(B);
    std::iota(ord.begin(), ord.end(), 0);
    std::stable_sort(ord.begin(), ord.end(), [&](int a, int b2) { return N[a] > N[b2]; });
    std::vector<std::vector<int>> shard(nctx);
    for (int pos = 0; pos < B; pos++) {
        const int rnd = pos / nctx, k = pos % nctx;
        shard[(rnd % 2 == 0) ? k : nctx - 1 - k].push_back(ord[pos]);
    }
    for (auto &s : shard) std::sort(s.begin(), s.end());
    struct Sub { std::vector<int32_t> N, M; std::vector<double> bnd, T, ixy, iyw, cxy, cyw; std::vector<ualm_result_t> res; };
    std::vector<Sub> sub(nctx);
    for (int r = 0; r < nctx; r++) {
        Sub &s = sub[r];
        for (int b : shard[r]) {
            s.N.push_back(N[b]); s.M.push_back(M[b]); s.T.push_back(total_time[b]);
            s.bnd.insert(s.bnd.end(), bnd + 18 * (size_t)b, bnd + 18 * (size_t)b + 18);
            if (oxy[b + 1] > oxy[b]) s.ixy.insert(s.ixy.end(), inner_xy + oxy[b], inner_xy + oxy[b + 1]);
            if (oyw[b + 1] > oyw[b]) s.iyw.insert(s.iyw.end(), inner_yaw + oyw[b], inner_yaw + oyw[b + 1]);
        }
        long long ncx = 0, ncy = 0;
        for (int b : shard[r]) { ncx += 12LL * N[b]; ncy += 6LL * M[b]; }
        s.cxy.assign(ncx, 0.0); s.cyw.assign(ncy, 0.0); s.res.resize(shard[r].size());
        if (s.ixy.empty()) s.ixy.push_back(0.0);
        if (s.iyw.empty()) s.iyw.push_back(0.0);
    }
    // upload + launch everywhere first (asynchronous per device), then collect
    for (int r = 0; r < nctx; r++) {
        if (shard[r].empty()) continue;
        int rc = ualm_upload(ctxs[r], (int)shard[r].size(), sub[r].N.data(), sub[r].M.data(), sub[r].bnd.data(), sub[r].T.data(), sub[r].ixy.data(), sub[r].iyw.data());
        if (!rc) rc = ualm_solve_resident(ctxs[r]);
        if (rc) return rc;
    }
    for (int r = 0; r < nctx; r++) {
        if (shard[r].empty()) continue;
        int rc = ualm_download(ctxs[r], sub[r].res.data(), sub[r].cxy.data(), sub[r].cyw.data());
        if (rc) return rc;
        long long px = 0, py = 0;
        for (size_t q = 0; q < shard[r].size(); q++) {
            const int b = shard[r][q];
            if (results) results[b] = sub[r].res[q];
            if (c_xy) memcpy(c_xy + ocx[b], sub[r].cxy.data() + px, sizeof(double) * 12 * N[b]);
            if (c_yaw) memcpy(c_yaw + ocy[b], sub[r].cyw.data() + py, sizeof(double) * 6 * M[b]);
            px += 12LL * N[b]; py += 6LL * M[b];
        }
    }
    return UALM_OK;
}

extern "C" int ualm_pack_records_device(ualm_ctx_t *c, double *d_records, int stride)
{
    if (c && c->tp) {
        if (!d_records) return fail(UALM_EINVAL, "null buffer");
        TP_CALL(ualm_tp::tp_pack_records(c->tp, c->cur, d_records, stride, err));
    }
    if (!c || !c->b->solved || !d_records) return fail(UALM_ESTATE, "nothing solved / null buffer");
    Lane *l = c->b;
    if (stride < 12 + 12 * l->Nmax + 6 * l->Mmax) return fail(UALM_EINVAL, "record stride too small");
    CK(cudaSetDevice(c->device));
    if (l->B > 0) {
        pack_records_kernel<<<l->B, 128, 0, l->stream>>>(batch_ptrs(c), l->B, d_records, stride);
        CK(cudaGetLastError());
    }
    CK(cudaStreamSynchronize(l->stream));
    return UALM_OK;
}
// the same without the host-side wait (pipelined callers synchronise the lane themselves before reading the records)
extern "C" int ualm_pack_records_device_async(ualm_ctx_t *c, double *d_records, int stride)
{
    if (c && c->tp) return ualm_pack_records_device(c, d_records, stride);     // the engine gathers a batch only once it is complete
    if (!c || !c->b->solved || !d_records) return fail(UALM_ESTATE, "nothing solved / null buffer");
    Lane *l = c->b;
    if (stride < 12 + 12 * l->Nmax + 6 * l->Mmax) return fail(UALM_EINVAL, "record stride too small");
    CK(cudaSetDevice(c->device));
    if (l->B > 0) {
        pack_records_kernel<<<l->B, 128, 0, l->stream>>>(batch_ptrs(c), l->B, d_records, stride);
        CK(cudaGetLastError());
    }
    return UALM_OK;
}

// upload an optional host array (or a constant fill) into a device buffer
static int put(ualm_ctx *c, double *dst, const double *src, size_t n, double fill)
{
    if (n == 0) return UALM_OK;
    if (src) { CK(cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyHostToDevice, c->b->stream)); }
    else {
        std::vector<double> tmp(n, fill);
        CK(cudaMemcpyAsync(dst, tmp.data(), n * sizeof(double), cudaMemcpyHostToDevice, c->b->stream));
        CK(cudaStreamSynchronize(c->b->stream));
    }
    return UALM_OK;
}

extern "C" int ualm_eval_batch(ualm_ctx_t *c, const double *x, const double *lambda, const double *mu, const double *scale_cx,
                               const double *scale_fx, double rho, double *f, double *grad, double *hx, double *gx, double *c_xy,
                               double *c_yaw)
{
    if (c && c->tp) TP_CALL(ualm_tp::tp_eval(c->tp, c->cur, x, lambda, mu, scale_cx, scale_fx, rho, f, grad, hx, gx, c_xy, c_yaw, err));
    if (!c || !c->b->have_batch || !c->have_map) return fail(UALM_ESTATE, "upload and set_map first");
    Lane *l = c->b;
    if (l->n_active != l->B) return fail(UALM_ELIMIT, "ualm_eval_batch: the uploaded batch holds problems over the compiled limits");
    CK(cudaSetDevice(c->device));
    int rc;
    if (x) { if ((rc = put(c, l->d_x0.p, x, l->tot_x, 0.0))) return rc; }
    if ((rc = put(c, l->d_lambda.p, lambda, l->tot_s, 0.0))) return rc;
    if ((rc = put(c, l->d_mu.p, mu, 6 * l->tot_s, 0.0))) return rc;
    if ((rc = put(c, l->d_scale_cx.p, scale_cx, 7 * l->tot_s, 1.0))) return rc;
    if ((rc = put(c, l->d_sfx.p, scale_fx, l->B, 1.0))) return rc;
    if (l->B > 0) {
        eval_kernel<<<(l->B + UALM_WPB - 1) / UALM_WPB, UALM_THREADS * UALM_WPB, l->smem_bytes, l->stream>>>(batch_ptrs(c), c->dp, c->dm, l->L, rho);
        CK(cudaGetLastError());
        if (f) CK(cudaMemcpyAsync(f, l->d_f.p, sizeof(double) * l->B, cudaMemcpyDeviceToHost, l->stream));
        if (grad) CK(cudaMemcpyAsync(grad, l->d_grad.p, sizeof(double) * l->tot_x, cudaMemcpyDeviceToHost, l->stream));
        if (hx) CK(cudaMemcpyAsync(hx, l->d_hx.p, sizeof(double) * l->tot_s, cudaMemcpyDeviceToHost, l->stream));
        if (gx) CK(cudaMemcpyAsync(gx, l->d_gx.p, sizeof(double) * 6 * l->tot_s, cudaMemcpyDeviceToHost, l->stream));
        if (c_xy) CK(cudaMemcpyAsync(c_xy, l->d_cxy.p, sizeof(double) * l->tot_cxy, cudaMemcpyDeviceToHost, l->stream));
        if (c_yaw) CK(cudaMemcpyAsync(c_yaw, l->d_cyaw.p, sizeof(double) * l->tot_cyaw, cudaMemcpyDeviceToHost, l->stream));
    }
    CK(cudaStreamSynchronize(l->stream));
    return UALM_OK;
}

extern "C" int ualm_init_scaling_batch(ualm_ctx_t *c, double *scale_fx, double *scale_cx)
{
    if (c && c->tp) TP_CALL(ualm_tp::tp_init_scaling(c->tp, c->cur, scale_fx, scale_cx, err));
    if (!c || !c->b->have_batch || !c->have_map) return fail(UALM_ESTATE, "upload and set_map first");
    Lane *l = c->b;
    if (l->n_active != l->B) return fail(UALM_ELIMIT, "ualm_init_scaling_batch: the uploaded batch holds problems over the compiled limits");
    CK(cudaSetDevice(c->device));
    if (l->B > 0) {
        scaling_kernel<<<(l->B + UALM_WPB - 1) / UALM_WPB, UALM_THREADS * UALM_WPB, l->smem_bytes, l->stream>>>(batch_ptrs(c), c->dp, c->dm, l->L);
        CK(cudaGetLastError());
        if (scale_fx) CK(cudaMemcpyAsync(scale_fx, l->d_sfx.p, sizeof(double) * l->B, cudaMemcpyDeviceToHost, l->stream));
        if (scale_cx) CK(cudaMemcpyAsync(scale_cx, l->d_scale_cx.p, sizeof(double) * 7 * l->tot_s, cudaMemcpyDeviceToHost, l->stream));
    }
    CK(cudaStreamSynchronize(l->stream));
    return UALM_OK;
}

extern "C" int ualm_time_penalty_kernel(ualm_ctx_t *c, int reps, float *ms_per_launch, double *algorithmic_bytes)
{
    if (reps < 1) return fail(UALM_EINVAL, "reps < 1");
    if (c && c->tp) TP_CALL(ualm_tp::tp_time_penalty(c->tp, c->cur, reps, (getenv("UALM_TP_TMA") && atoi(getenv("UALM_TP_TMA"))) ? 1 : 0, ms_per_launch, algorithmic_bytes, err));
    if (!c || !c->b->have_batch || !c->have_map) return fail(UALM_ESTATE, "upload and set_map first");
    Lane *l = c->b;
    if (l->n_active != l->B) return fail(UALM_ELIMIT, "ualm_time_penalty_kernel: the uploaded batch holds problems over the compiled limits");
    if (ms_per_launch) *ms_per_launch = 0.f;
    if (algorithmic_bytes) *algorithmic_bytes = 0.0;
    if (l->B == 0) return UALM_OK;
    CK(cudaSetDevice(c->device));
    int rc;
    if ((rc = put(c, l->d_lambda.p, nullptr, l->tot_s, 0.0))) return rc;
    if ((rc = put(c, l->d_mu.p, nullptr, 6 * l->tot_s, 0.0))) return rc;
    if ((rc = put(c, l->d_scale_cx.p, nullptr, 7 * l->tot_s, 1.0))) return rc;
    penalty_only_kernel<<<(l->B + UALM_WPB - 1) / UALM_WPB, UALM_THREADS * UALM_WPB, l->smem_bytes, l->stream>>>(batch_ptrs(c), c->dp, c->dm, l->L, 1); // warm-up
    CK(cudaEventRecord(l->ev0, l->stream));
    penalty_only_kernel<<<(l->B + UALM_WPB - 1) / UALM_WPB, UALM_THREADS * UALM_WPB, l->smem_bytes, l->stream>>>(batch_ptrs(c), c->dp, c->dm, l->L, reps);
    CK(cudaEventRecord(l->ev1, l->stream));
    CK(cudaGetLastError());
    CK(cudaEventSynchronize(l->ev1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, l->ev0, l->ev1));
    if (ms_per_launch) *ms_per_launch = ms / reps;
    if (algorithmic_bytes) {
        // SURVEY 8d: per trajectory per evaluation S*45e + (25N + 13M)e
        double bytes = 0;
        for (auto &d : l->desc) bytes += (double)d.S * 45 * 8 + (25.0 * d.N + 13.0 * d.M) * 8;
        *algorithmic_bytes = bytes;
    }
    return UALM_OK;
}

// developer aid: per-phase SM cycle counters of the last solve (thread 0 of every CTA), summed over the batch.
// enable != 0 turns collection on for subsequent solves; out16 (may be NULL) receives the sums of the last solve.
extern "C" int ualm_profile(ualm_ctx_t *c, int enable, long long *out16)
{
    if (!c) return fail(UALM_EINVAL, "null ctx");
    if (c->tp) TP_UNSUPPORTED("ualm_profile");
    Lane *l = c->b;
    CK(cudaSetDevice(c->device));
    if (out16 && c->profile && l->solved && l->B > 0) {
        std::vector<long long> h((size_t)l->B * UALM_NPROF);
        CK(cudaMemcpyAsync(h.data(), l->d_prof.p, h.size() * sizeof(long long), cudaMemcpyDeviceToHost, l->stream));
        CK(cudaStreamSynchronize(l->stream));
        if (enable == 2) { // raw: out16 has room for B x 16 values, rows in problem order
            for (size_t q = 0; q < h.size(); q++) out16[q] = h[q];
        } else {
            for (int q = 0; q < UALM_NPROF; q++) out16[q] = 0;
            for (int b = 0; b < l->B; b++) if (!l->skip[b]) for (int q = 0; q < UALM_NPROF; q++) out16[q] += h[(size_t)b * UALM_NPROF + q];
        }
    }
    c->profile = enable != 0;
    return UALM_OK;
}

namespace ualm {
__global__ void piece_T_from_results(const ualm_result_t *res, int B, double *piece_T)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) { piece_T[2 * b] = res[b].piece_T_xy; piece_T[2 * b + 1] = res[b].piece_T_yaw; }
}
} // namespace ualm

// the scan over coefficients that already sit on the device (B problems, ragged offsets from N / M, piece durations from the records)
static int feasibility_from_device(ualm_ctx *c, int B, const int32_t *N, const int32_t *M, const ualm_result_t *d_res, const double *d_cxy, const double *d_cyaw,
                                   double dt, double *out10)
{
    struct Tmp { DevBuf<ProbDesc> desc; DevBuf<double> pt, feas; ~Tmp() { desc.release(); pt.release(); feas.release(); } } t;
    std::vector<ProbDesc> desc(B);
    long long ocx = 0, ocy = 0;
    for (int b = 0; b < B; b++) {
        memset(&desc[b], 0, sizeof(ProbDesc));
        desc[b].N = N[b]; desc[b].M = M[b]; desc[b].off_cxy = ocx; desc[b].off_cyaw = ocy;
        desc[b].S = (N[b] > UALM_NMAX || M[b] > UALM_MMAX) ? 0 : 1;      // S == 0 marks a problem that was not solved
        ocx += 12LL * N[b]; ocy += 6LL * M[b];
    }
    CK(t.desc.ensure(B)); CK(t.pt.ensure(2 * (size_t)B)); CK(t.feas.ensure(10 * (size_t)B));
    CK(cudaMemcpy(t.desc.p, desc.data(), sizeof(ProbDesc) * B, cudaMemcpyHostToDevice));
    piece_T_from_results<<<(B + 127) / 128, 128>>>(d_res, B, t.pt.p);
    BatchPtrs bp;
    memset(&bp, 0, sizeof(bp));
    bp.B = B; bp.desc = t.desc.p; bp.c_xy = const_cast<double *>(d_cxy); bp.c_yaw = const_cast<double *>(d_cyaw); bp.piece_T = t.pt.p;
    feasibility_kernel<<<(B + UALM_WPB - 1) / UALM_WPB, UALM_THREADS * UALM_WPB>>>(bp, c->dp, c->dm, dt, t.feas.p);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out10, t.feas.p, sizeof(double) * 10 * B, cudaMemcpyDeviceToHost));
    return UALM_OK;
}

extern "C" int ualm_feasibility_batch(ualm_ctx_t *c, double dt, double *out10)
{
    if (!c || !out10 || !(dt > 0.0)) return fail(UALM_EINVAL, "null argument or dt <= 0");
    if (c->tp) {
        const ualm_result_t *d_res; const double *d_cxy, *d_cyaw;
        int B = 0; const int32_t *N = nullptr, *M = nullptr;
        if (ualm_tp::tp_lane_outputs(c->tp, c->cur, &d_res, &d_cxy, &d_cyaw, &B, &N, &M) != UALM_OK)
            return fail(UALM_ESTATE, "ualm_feasibility_batch needs a solved, collected batch (ualm_sync / ualm_download first)");
        CK(cudaSetDevice(c->device));
        if (B == 0) return UALM_OK;
        return feasibility_from_device(c, B, N, M, d_res, d_cxy, d_cyaw, dt, out10);
    }
    Lane *l = c->b;
    if (!c->have_map || !c->have_params || !l->have_batch || !l->solved) return fail(UALM_ESTATE, "ualm_feasibility_batch needs a solved resident batch");
    CK(cudaSetDevice(c->device));
    if (l->B == 0) return UALM_OK;
    const BatchPtrs bp = batch_ptrs(c);
    feasibility_kernel<<<(l->B + UALM_WPB - 1) / UALM_WPB, UALM_THREADS * UALM_WPB, 0, l->stream>>>(bp, c->dp, c->dm, dt, l->d_feas.p);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out10, l->d_feas.p, sizeof(double) * 10 * l->B, cudaMemcpyDeviceToHost, l->stream));
    CK(cudaStreamSynchronize(l->stream));
    return UALM_OK;
}

// ---------------------------------------------------------------------------------------------
// SURVEY 8f-3: SE2Traj message + the MPC side's MINCO re-solve + planned-vs-tracked deviation for a solved batch (mpc_export_kernel)
// ---------------------------------------------------------------------------------------------
static int mpc_export_run(ualm_ctx *c, const BatchPtrs &bp, int B, const int32_t *N, const int32_t *M, double dt, const double *init_v, const double *init_a,
                          double *pos_pts, double *posT_pts, double *angle_pts, double *angleT_pts, double *c_mpc_xy, double *c_mpc_yaw, double *dev4, cudaStream_t st)
{
    long long sN = 0, sM = 0;
    for (int b = 0; b < B; b++) { sN += N[b]; sM += M[b]; }
    struct Tmp { DevBuf<double> buf; ~Tmp() { buf.release(); } } t;
    const size_t n_pp = 2 * (size_t)(sN + B), n_pt = (size_t)sN, n_ap = (size_t)(sM + B), n_at = (size_t)sM, n_cx = 12 * (size_t)sN, n_cy = 6 * (size_t)sM, n_dv = 4 * (size_t)B;
    const size_t n_band = 13 * (6 * (size_t)sN + 6 * (size_t)sM);
    CK(t.buf.ensure(n_pp + n_pt + n_ap + n_at + n_cx + n_cy + n_dv + n_band));
    MpcOut o;
    double *q = t.buf.p;
    o.pos_pts = q; q += n_pp; o.posT_pts = q; q += n_pt; o.angle_pts = q; q += n_ap; o.angleT_pts = q; q += n_at;
    o.c_mpc_xy = q; q += n_cx; o.c_mpc_yaw = q; q += n_cy; o.dev = q; q += n_dv; o.band = q;
    for (int k = 0; k < 3; k++) { o.init_v[k] = init_v ? init_v[k] : 0.0; o.init_a[k] = init_a ? init_a[k] : 0.0; }
    mpc_export_kernel<<<(B + UALM_WPB - 1) / UALM_WPB, UALM_THREADS * UALM_WPB, 0, st>>>(bp, dt, o);
    CK(cudaGetLastError());
    struct { double *h; const double *d; size_t n; } cp[7] = {{pos_pts, o.pos_pts, n_pp}, {posT_pts, o.posT_pts, n_pt}, {angle_pts, o.angle_pts, n_ap},
        {angleT_pts, o.angleT_pts, n_at}, {c_mpc_xy, o.c_mpc_xy, n_cx}, {c_mpc_yaw, o.c_mpc_yaw, n_cy}, {dev4, o.dev, n_dv}};
    for (auto &e : cp) if (e.h && e.n) CK(cudaMemcpyAsync(e.h, e.d, sizeof(double) * e.n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return UALM_OK;
}

extern "C" int ualm_mpc_export_batch(ualm_ctx_t *c, double dt, const double *init_v, const double *init_a, double *pos_pts, double *posT_pts, double *angle_pts,
                                     double *angleT_pts, double *c_mpc_xy, double *c_mpc_yaw, double *dev4)
{
    if (!c || !(dt > 0.0)) return fail(UALM_EINVAL, "null ctx or dt <= 0");
    if (c->tp) {
        const ualm_result_t *d_res; const double *d_cxy, *d_cyaw;
        int B = 0; const int32_t *N = nullptr, *M = nullptr;
        if (ualm_tp::tp_lane_outputs(c->tp, c->cur, &d_res, &d_cxy, &d_cyaw, &B, &N, &M) != UALM_OK)
            return fail(UALM_ESTATE, "ualm_mpc_export_batch needs a solved, collected batch (ualm_sync / ualm_download first)");
        CK(cudaSetDevice(c->device));
        if (B == 0) return UALM_OK;
        struct Tmp { DevBuf<ProbDesc> desc; DevBuf<double> pt; ~Tmp() { desc.release(); pt.release(); } } t;
        std::vector<ProbDesc> desc(B);
        long long ocx = 0, ocy = 0;
        for (int b = 0; b < B; b++) {
            memset(&desc[b], 0, sizeof(ProbDesc));
            desc[b].N = N[b]; desc[b].M = M[b]; desc[b].off_cxy = ocx; desc[b].off_cyaw = ocy;
            desc[b].S = (N[b] > UALM_NMAX || M[b] > UALM_MMAX) ? 0 : 1;
            ocx += 12LL * N[b]; ocy += 6LL * M[b];
        }
        CK(t.desc.ensure(B)); CK(t.pt.ensure(2 * (size_t)B));
        CK(cudaMemcpy(t.desc.p, desc.data(), sizeof(ProbDesc) * B, cudaMemcpyHostToDevice));
        piece_T_from_results<<<(B + 127) / 128, 128>>>(d_res, B, t.pt.p);
        BatchPtrs bp;
        memset(&bp, 0, sizeof(bp));
        bp.B = B; bp.desc = t.desc.p; bp.c_xy = const_cast<double *>(d_cxy); bp.c_yaw = const_cast<double *>(d_cyaw); bp.piece_T = t.pt.p;
        return mpc_export_run(c, bp, B, N, M, dt, init_v, init_a, pos_pts, posT_pts, angle_pts, angleT_pts, c_mpc_xy, c_mpc_yaw, dev4, 0);
    }
    Lane *l = c->b;
    if (!l->have_batch || !l->solved) return fail(UALM_ESTATE, "ualm_mpc_export_batch needs a solved resident batch");
    CK(cudaSetDevice(c->device));
    if (l->B == 0) return UALM_OK;
    std::vector<int32_t> N(l->B), M(l->B);
    for (int b = 0; b < l->B; b++) { N[b] = l->desc[b].N; M[b] = l->desc[b].M; }
    return mpc_export_run(c, batch_ptrs(c), l->B, N.data(), M.data(), dt, init_v, init_a, pos_pts, posT_pts, angle_pts, angleT_pts, c_mpc_xy, c_mpc_yaw, dev4, l->stream);
}

// ---------------------------------------------------------------------------------------------
// UnevenMap construction on the device (SURVEY 8f-1).  HBM-bound gather: one thread per cell, yaw fastest so that the 64
// threads of a CTA share (x, y) and read the same few cloud bins through L1.
// ---------------------------------------------------------------------------------------------
namespace ualm {
__global__ void __launch_bounds__(64) map_build_kernel(UalmMapPrep prep, ualm_map_geom_t geom, float4 *cells)
{
    const int W = geom.voxel_num[2], Y = geom.voxel_num[1];
    const long long cell = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)geom.voxel_num[0] * Y * W;
    if (cell >= total) return;
    const int w = (int)(cell % W), y = (int)((cell / W) % Y), x = (int)(cell / ((long long)W * Y));
    float o[4];
    ualm_map_cell(prep, geom, x, y, w, o);
    cells[cell] = make_float4(o[0], o[1], o[2], o[3]);
}
} // namespace ualm

extern "C" int ualm_map_build_device(ualm_ctx_t *c, const float *pin, int64_t npts, const ualm_map_geom_t *g, double ex, double ey, double ez,
                                     int iter_num, float *cells, float *kernel_ms)
{
    if (!c || !pin || !g || !cells || npts < 0) return fail(UALM_EINVAL, "null argument");
    CK(cudaSetDevice(c->device));
    UalmMapHostPrep prep;
    ualm_map_preprocess(pin, npts, ex, ey, ez, prep);
    UalmMapPrep view = prep.view(ex, ey, ez, iter_num);
    const long long total = (long long)g->voxel_num[0] * g->voxel_num[1] * g->voxel_num[2];
    // scratch buffers and events are released on every exit path (CK returns on the first CUDA error)
    struct Scratch {
        DevBuf<float> pts; DevBuf<int> start; DevBuf<float4> cells;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        ~Scratch() { pts.release(); start.release(); cells.release(); if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); }
    } sc;
    CK(sc.pts.ensure(std::max<size_t>(prep.pts.size(), 3)));
    CK(sc.start.ensure(prep.start.size()));
    CK(sc.cells.ensure((size_t)total));
    CK(cudaEventCreate(&sc.e0)); CK(cudaEventCreate(&sc.e1));
    if (!prep.pts.empty()) CK(cudaMemcpyAsync(sc.pts.p, prep.pts.data(), sizeof(float) * prep.pts.size(), cudaMemcpyHostToDevice, c->b->stream));
    CK(cudaMemcpyAsync(sc.start.p, prep.start.data(), sizeof(int) * prep.start.size(), cudaMemcpyHostToDevice, c->b->stream));
    view.pts = sc.pts.p; view.start = sc.start.p;
    CK(cudaEventRecord(sc.e0, c->b->stream));
    map_build_kernel<<<(unsigned)((total + 63) / 64), 64, 0, c->b->stream>>>(view, *g, sc.cells.p);
    CK(cudaGetLastError());
    CK(cudaEventRecord(sc.e1, c->b->stream));
    CK(cudaMemcpyAsync(cells, sc.cells.p, sizeof(float4) * total, cudaMemcpyDeviceToHost, c->b->stream));
    CK(cudaStreamSynchronize(c->b->stream));
    if (kernel_ms) CK(cudaEventElapsedTime(kernel_ms, sc.e0, sc.e1));
    return UALM_OK;
}

// ---- the front-end on the device (csrc/ualm_front_end.cu) ----
extern "C" int ualm_set_front_end_map(ualm_ctx_t *c, const ualm_astar_map_t *m)
{
    if (!c || !m) return fail(UALM_EINVAL, "null argument");
    CK(cudaSetDevice(c->device));
    std::string err;
    const int rc = ualm_fe::set_map(&c->fe, m, err);
    return rc < 0 ? fail(rc, err) : rc;
}

extern "C" int ualm_front_end_batch_device(ualm_ctx_t *c, const ualm_astar_params_t *ap, const ualm_resample_params_t *rp, int B, const double *starts,
                                           const double *goals, int32_t *N, int32_t *M, double *bnd, double *total_time, double *inner_xy,
                                           long long cap_xy, double *inner_yaw, long long cap_yaw, int32_t *packed, int32_t *n_expanded,
                                           double *path_xyyaw, long long cap_path, int64_t *path_off, float *search_ms)
{
    if (!c) return fail(UALM_EINVAL, "null ctx");
    CK(cudaSetDevice(c->device));
    std::string err;
    const int rc = ualm_fe::batch(c->fe, ap, rp, B, starts, goals, N, M, bnd, total_time, inner_xy, cap_xy, inner_yaw, cap_yaw, packed, n_expanded,
                                  path_xyyaw, cap_path, path_off, search_ms, err);
    return rc < 0 ? fail(rc, err) : rc;
}

extern "C" int ualm_front_end_path_cap(const ualm_astar_params_t *ap, const ualm_resample_params_t *rp)
{
    if (!ap || !rp) return fail(UALM_EINVAL, "null argument");
    return ualm_fe::path_cap(ap, rp);
}
