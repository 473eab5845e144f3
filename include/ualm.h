/*
 * ualm.h -- C ABI of the B200-native batched MINCO / augmented-Lagrangian trajectory optimizer.
 *
 * Drop-in boundary for ONE hot path of ZJU-FAST-Lab/uneven_planner: the back-end
 *   uneven_planner::ALMTrajOpt::optimizeSE2Traj(...)            back_end/include/back_end/alm_traj_opt.h:92-98
 *   uneven_planner::ALMTrajOpt::getTraj()                        alm_traj_opt.h:165-168
 * with its environment binding
 *   ALMTrajOpt::setEnvironment(UnevenMap::Ptr)                   alm_traj_opt.h:127-130
 *   ALMTrajOpt::init(nh)  (the alm_traj_opt/ * rosparams)        back_end/src/alm_traj_opt.cpp:5-45
 * (paths relative to /root/reference/src/uneven_planner/).  Plain pointers and sizes only; no
 * torch / Eigen / ROS types.  Every entry point returns 0 on success or a negative UALM_E* code
 * and never falls back to a CPU implementation: without a CUDA device the compute calls fail.
 *
 * All matrices use the reference's (Eigen column-major) layouts:
 *   init_xy / end_xy : 2x3  [px,py, vx,vy, ax,ay]       (alm_traj_opt.cpp:183-186, pm.cpp:80-94)
 *   inner_xy         : 2x(N-1) [x1,y1, x2,y2, ...]      (alm_traj_opt.cpp:211,215)
 *   c_xy             : 6N x 2  (x column then y column; per piece 6 coefficients low->high power,
 *                      se2traj.hpp:585, 712-715);  c_yaw : 6M
 */
#ifndef UALM_H
#define UALM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UALM_OK 0
#define UALM_ENOCUDA (-1)   /* no usable CUDA device / CUDA runtime error (message via ualm_last_error) */
#define UALM_EINVAL (-2)    /* bad argument */
#define UALM_ESTATE (-3)    /* call order (no map / no params / nothing uploaded) */
#define UALM_ELIMIT (-4)    /* problem exceeds compiled limits (N, M, int_K) */

/* ---- parameters: the 21 alm_traj_opt/ * values (alm_traj_opt.cpp:7-27) + uneven_map/gravity ---- */
typedef struct {
    double rho_T, rho_ter, max_vel, max_acc_lon, max_acc_lat, max_kap, min_cxi, max_sig;
    int    use_scaling;
    double rho, beta, gamma, epsilon_con, max_iter;
    double g_epsilon, min_step, inner_max_iter, delta;
    int    mem_size, past, int_K;
    double gravity;          /* UnevenMap::getGravity(), uneven_map.cpp:85 */
} ualm_params_t;

/* run_hill.yaml defaults (plan_manager/params/run_hill.yaml:30-55) */
void ualm_default_params(ualm_params_t *p);

/* ---- environment: what ALMTrajOpt reads of UnevenMap (uneven_map.h:258-377, 398-454) ---- */
typedef struct {
    int    voxel_num[3];     /* X, Y, Yaw cells (uneven_map.cpp:108-110) */
    double origin[3];        /* map_origin = min_boundary (uneven_map.cpp:99-101) */
    double max_boundary[3];
    double xy_resolution, yaw_resolution;
} ualm_map_geom_t;

/* geometry for map_size_x/y and resolutions exactly as UnevenMap::init computes it (uneven_map.cpp:96-114) */
void ualm_map_geometry(double map_size_x, double map_size_y, double xy_resolution, double yaw_resolution,
                       ualm_map_geom_t *g);

/* ---- per-problem result record (what the reference prints / returns: alm_traj_opt.cpp:176,252,267,272-273;
 *      alm_traj_opt.h:142) ---- */
typedef struct {
    int32_t ret_code;        /* 0 converged / 1 L-BFGS hard error / 2 ALM max_iter (the reference's codes); UALM_ELIMIT (-4): this
                                problem exceeds the compiled limits (N <= 64, M <= 128) and was not solved -- the rest of its
                                batch is unaffected */
    int32_t outer_iters;
    int32_t n_evals;         /* cost+gradient evaluations */
    int32_t n_lbfgs_iters;   /* accepted line searches */
    int32_t last_lbfgs_ret;
    int32_t max_bound;
    int32_t sum_bound;       /* sum over L-BFGS iterations of the history depth used (bytes accounting) */
    int32_t reserved;
    double  inner_cost, jerk_cost, total_T, res_h, res_g, scale_fx, rho_final;
    double  piece_T_xy, piece_T_yaw;   /* the uniform piece durations getTraj() carries: T1(i) of the LAST evaluation
                                          (alm_traj_opt.h:257-261, se2traj.hpp:682-695); total_T is their N-fold sum */
} ualm_result_t;

typedef struct ualm_ctx ualm_ctx_t;

/* precision: 64 = parity path (IEEE double, bit-identical to the CPU oracle / the reference sources); 65 = "fast64", the
 * throughput path in double (re-associated reductions, FMA, prefactored MINCO system: not bit-reproducible); 32 = the
 * throughput path in float.  device = CUDA ordinal. */
int ualm_create(ualm_ctx_t **ctx, int device, int precision);
int ualm_destroy(ualm_ctx_t *ctx);
const char *ualm_last_error(void);
/* Run the work of the selected lane on a caller-owned CUDA stream.  The handle is taken literally: NULL is the legacy
 * default stream (torch.cuda.current_stream().cuda_stream == 0 when torch runs on its default stream).  ualm_reset_stream
 * goes back to the lane's own non-blocking stream.  ualm_solve_resident is asynchronous on that stream: follow it with
 * ualm_sync (or a stream-ordered consumer on the SAME stream) before touching its outputs. */
int ualm_set_stream(ualm_ctx_t *ctx, void *cuda_stream);
int ualm_reset_stream(ualm_ctx_t *ctx);
/* ALMTrajOpt::init.  int_K, mem_size and past are baked into uploaded batches: a parameter change invalidates every resident
 * batch (upload again before the next solve / eval); it is refused while a submitted batch is in flight. */
int ualm_set_params(ualm_ctx_t *ctx, const ualm_params_t *p);
/* cells: host, [X][Y][Yaw][4] float {z, sigma, zbx, zby}, address x*Y*Yaw + y*Yaw + yaw (uneven_map.h:427-435).
 * One-time upload (replaces setEnvironment; the reference's map_buffer is private, uneven_map.h:91). */
int ualm_set_map(ualm_ctx_t *ctx, const ualm_map_geom_t *g, const float *cells);
/* The reference's own grid: UnevenMap::map_buffer is RXS2 {double z, sigma; Vector2d zb} (uneven_map.h:36-64), i.e. 4 doubles
 * per cell in the same address order.  repack_to_float = 0 keeps the doubles on the device (82 MB for 200x200x64: bit parity
 * for maps built in-process by the reference); != 0 rounds them to the float4 grid of ualm_set_map (41 MB, what a map read
 * back from this repo's .umap file or from the reference's 6-digit CSV cache holds anyway). */
int ualm_set_map_f64(ualm_ctx_t *ctx, const ualm_map_geom_t *g, const double *cells, int repack_to_float);

/* ---- batch solve = B independent optimizeSE2Traj calls ----
 * Ragged inputs are packed back to back in problem order: inner_xy has sum 2(N_b-1) doubles,
 * inner_yaw sum (M_b-1); outputs c_xy sum 12 N_b, c_yaw sum 6 M_b.  bnd is B x 18:
 * [init_xy(6) | end_xy(6) | init_yaw(3) | end_yaw(3)].  Host pointers. */
int ualm_solve_batch(ualm_ctx_t *ctx, int B, const int32_t *N, const int32_t *M, const double *bnd,
                     const double *total_time, const double *inner_xy, const double *inner_yaw,
                     ualm_result_t *results, double *c_xy, double *c_yaw);

/* The same in three steps, so a caller can keep inputs resident in HBM (bench `value`):
 *   upload (H2D) -> solve_resident (kernels only, asynchronous on the context stream) -> download (D2H). */
int ualm_upload(ualm_ctx_t *ctx, int B, const int32_t *N, const int32_t *M, const double *bnd,
                const double *total_time, const double *inner_xy, const double *inner_yaw);
int ualm_solve_resident(ualm_ctx_t *ctx);
int ualm_sync(ualm_ctx_t *ctx);
int ualm_download(ualm_ctx_t *ctx, ualm_result_t *results, double *c_xy, double *c_yaw);
/* elapsed GPU time of the last solve_resident in ms (CUDA events on the context stream) and the
 * number of kernel launches it made */
int ualm_last_solve_ms(ualm_ctx_t *ctx, float *ms, int *launches);

/* ---- several batches in flight on one context ("lanes") ----
 * A lane is one resident batch with its own buffers, launch plan and streams; kernels of different lanes run concurrently, so
 * the slow tail of batch k (a few long-running trajectories) overlaps the bulk of batch k+1.
 *   ualm_select_lane(ctx, i): upload / solve_resident / sync / download / pack_records / last_solve_ms / eval / feasibility act
 *                             on lane i (0 <= i < ualm_max_lanes(); lane 0 is selected at creation).
 *   ualm_submit_batch:  upload + launch on the next lane of a `depth`-deep ring, returns a ticket without waiting for the solve
 *                       (host inputs are consumed before it returns).  UALM_ESTATE when that lane is still in flight.
 *   ualm_wait_batch:    blocks until the ticket's batch is complete, D2H of its results (same outputs as ualm_solve_batch).
 *   ualm_mark_begin / ualm_mark_end: CUDA-event time (ms) from the selected lane's stream at mark_begin to the completion of the
 *                       last solve of every lane at mark_end. */
int ualm_max_lanes(void);
int ualm_select_lane(ualm_ctx_t *ctx, int lane);
int ualm_submit_batch(ualm_ctx_t *ctx, int B, const int32_t *N, const int32_t *M, const double *bnd, const double *total_time,
                      const double *inner_xy, const double *inner_yaw, int depth, int *ticket);
int ualm_wait_batch(ualm_ctx_t *ctx, int ticket, ualm_result_t *results, double *c_xy, double *c_yaw);
int ualm_mark_begin(ualm_ctx_t *ctx);
int ualm_mark_end(ualm_ctx_t *ctx, float *ms);

/* ---- several GPUs from one host process (SURVEY 8b item 4) ----
 * ctxs[r] lives on its own device with the same parameters and map bound.  The batch is dealt over the contexts (cost-sorted
 * snake), every device solves its shard concurrently, and the results come back in problem order.  There is no collective: the
 * problems never interact and one host gathers by D2H copies.  (One process per GPU: ualm_pack_records_device + an NCCL
 * all-gather of the records on the caller's communicator, uneven_planner_b200/distributed.py.) */
int ualm_solve_batch_multi(ualm_ctx_t **ctxs, int nctx, int B, const int32_t *N, const int32_t *M, const double *bnd,
                           const double *total_time, const double *inner_xy, const double *inner_yaw, ualm_result_t *results,
                           double *c_xy, double *c_yaw);

/* Fixed-stride result records for the multi-GPU all-gather: writes B records of `stride` doubles into
 * a DEVICE buffer (e.g. a torch tensor): [ret, outer, evals, iters, cost, jerk, T, res_h, res_g, N, M, pad,
 * c_xy(12N) , c_yaw(6M), zero pad].  stride >= 12 + 12 Nmax + 6 Mmax.  The _async form does not wait for the kernel. */
int ualm_pack_records_device(ualm_ctx_t *ctx, double *d_records, int stride);
int ualm_pack_records_device_async(ualm_ctx_t *ctx, double *d_records, int stride);

/* ---- phase entry points (kernel-level parity; SURVEY 8b item 3) ----
 * One innerCallback evaluation (alm_traj_opt.cpp:280-347) per problem of the uploaded batch at the given
 * decision vectors x (packed, n_b = 1+2(N_b-1)+(M_b-1)) with duals lambda[S_b], mu[6 S_b], scale_cx[7 S_b]
 * in the reference's index layout (alm_traj_opt.cpp:705-707, 832-946), S_b = N_b (int_K+1).
 * Outputs (host): f[B], grad (packed n_b), hx (packed S_b), gx (packed 6 S_b). Any input dual may be
 * NULL (zeros / ones).  scale_fx[B], rho scalar. */
int ualm_eval_batch(ualm_ctx_t *ctx, const double *x, const double *lambda, const double *mu,
                    const double *scale_cx, const double *scale_fx, double rho,
                    double *f, double *grad, double *hx, double *gx, double *c_xy, double *c_yaw);
/* initScaling (alm_traj_opt.cpp:349-661) at the uploaded initial guesses: scale_fx[B], scale_cx packed 7 S_b */
int ualm_init_scaling_batch(ualm_ctx_t *ctx, double *scale_fx, double *scale_cx);
/* time `reps` back-to-back launches of the penalty-sampling kernel alone over the uploaded batch
 * (roofline of calConstrainCostGrad, alm_traj_opt.cpp:663-991): average ms per launch */
int ualm_time_penalty_kernel(ualm_ctx_t *ctx, int reps, float *ms_per_launch, double *algorithmic_bytes);

/* developer aid: per-phase SM-cycle counters of the last solve (thread 0 of every CTA) summed over the batch into out16[16]
 * (order: fill, LU, solve, jerk, tables, samples, accumulate, combine, adjoint, tail, two-loop, line-search, initScaling,
 * dual-update, other, total).  enable != 0 switches collection on for the following solves. */
int ualm_profile(ualm_ctx_t *ctx, int enable, long long *out16);

/* Post-solve quality scan of the solved resident batch (SURVEY 8f-4): ALMTrajOpt::getMaxVxAxAyCurAttSig
 * (alm_traj_opt.h:170-229) and SE2Trajectory::getNonHolError (se2traj.hpp:551-561), sampled every dt (0.01 in the
 * reference).  out10[10 * b + ...] = {max_vx, max_ax, max_ay, max_cur, max_att (= -min cos xi), max_sig, nonhol_error,
 * number of samples, T_xy piece duration, T_yaw piece duration}.  A trajectory whose duration would need more than 4e6 samples (a
 * diverged solve) is not scanned: zeros and a sample count of -1. */
int ualm_feasibility_batch(ualm_ctx_t *ctx, double dt, double *out10);

/* Hand-over to the MPC for the solved batch of the selected lane, on the device (SURVEY 8f-3):
 *   (1) the mpc_controller/SE2Traj message PlanManager publishes (plan_manager.cpp:151-185, msg/SE2Traj.msg:1-9): pos_pts = the
 *       start point of every xy piece and the end point, (N + 1) x {x, y} per problem, posT_pts = the N piece durations,
 *       angle_pts (M + 1) / angleT_pts (M) likewise for yaw; problems packed back to back;
 *   (2) the trajectory the MPC tracks: TrajAnalyzer::setTraj (traj_anal.hpp:125-181) re-solves MINCO over those points with the
 *       message's init_v / init_a = {x, y, yaw} (NULL = zero, what the reference publishes) and zero tail derivatives, using
 *       MinJerkOpt::generate (minco_traj.hpp:365-444): c_mpc_xy / c_mpc_yaw in the layout of ualm_solve_batch's c_xy / c_yaw,
 *       bit-identical to that header compiled unmodified (tests/test_ref_pin.py + tests/test_gpu_mpc_export.py);
 *   (3) dev4[4 * b + ..] = {max |planned - tracked| position (m), its time, max |planned - tracked| yaw (rad), its time}, sampled
 *       every dt: the planned spline carries the boundary speed of plan_manager.cpp:93-94, the message does not.
 * Any output pointer may be NULL.  Unsolved problems (ret_code UALM_ELIMIT) produce zeros. */
int ualm_mpc_export_batch(ualm_ctx_t *ctx, double dt, const double *init_v, const double *init_a, double *pos_pts, double *posT_pts,
                          double *angle_pts, double *angleT_pts, double *c_mpc_xy, double *c_mpc_yaw, double *dev4);

/* UnevenMap construction on the GPU (SURVEY 8f-1: UnevenMap::init preprocessing on the host, then constructMap + filter,
 * uneven_map.cpp:317-398, 5-43, one thread per (x, y, yaw) cell).  Same arguments and the same arithmetic as ualm_map_build
 * below (csrc/map_cell.h is compiled for both sides): the cells are bit-identical to the host builder's.  cells: host
 * buffer [X][Y][Yaw][4] float; kernel_ms (optional): CUDA-event time of the cell kernel. */
int ualm_map_build_device(ualm_ctx_t *ctx, const float *pts, int64_t npts, const ualm_map_geom_t *g, double ellipsoid_x,
                          double ellipsoid_y, double ellipsoid_z, int iter_num, float *cells, float *kernel_ms);

/* =====================  host-side input pipeline (no GPU needed)  ===================== */

/* UnevenMap::init cloud preprocessing + constructMap (uneven_map.cpp:127-163, 317-398, 5-43) on host
 * threads.  pts: npts x 3 float (x,y,z) as read from the .pcd.  cells out: [X][Y][Yaw][4] float.
 * ellipsoid = {0.2,0.1,0.1}, iter_num = 2 in every reference yaml. */
int ualm_map_build(const float *pts, int64_t npts, const ualm_map_geom_t *g, double ellipsoid_x,
                   double ellipsoid_y, double ellipsoid_z, int iter_num, int nthreads, float *cells);
/* the cloud ualm_map_build / ualm_map_build_device work on: UnevenMap::init's CropBox + 1 cm VoxelGrid (uneven_map.cpp:133-143), as xyz
 * floats.  Returns the number of points (pts_out may be NULL to query it; UALM_ELIMIT when max_pts is too small). */
int64_t ualm_map_preprocess_cloud(const float *pts, int64_t npts, double ellipsoid_x, double ellipsoid_y, double ellipsoid_z, float *pts_out,
                                  int64_t max_pts);
/* occupancy (uneven_map.cpp:169-179): occ3[X*Y*Yaw], occ2[X*Y] (1 = occupied) */
int ualm_map_occupancy(const float *cells, const ualm_map_geom_t *g, double min_cnormal, double max_rho,
                       uint8_t *occ3, uint8_t *occ2);

/* Initial-guess path (stands in for KinoAstar::plan, front_end/src/kino_astar.cpp:67-236, whose one-shot is
 * the same Dubins curve family, kino_astar.h:242-258): shortest forward Dubins path start->goal with
 * turning radius `radius`, sampled every `ds` metres as (x,y,yaw).  Returns the number of points written
 * (<= max_pts) or a negative error. */
int ualm_dubins_path(const double start[3], const double goal[3], double radius, double ds, double *path_xyyaw,
                     int max_pts);

/* PlanManager::rcvWpsCallBack input contract (plan_manager/src/plan_manager.cpp:62-122): yaw unwrap, boundary
 * states, arc-length resampling into inner xy / yaw waypoints, total_time.  Outputs: bnd[18], inner_xy
 * (2 x (N-1)), inner_yaw (M-1); returns 0 and sets *N, *M, *total_time. */
int ualm_resample_path(const double *path_xyyaw, int npts, double piece_len, double yaw_piece_times,
                       double mean_vel, double init_time_times, double init_sig_vel, double *bnd,
                       double *inner_xy, int max_inner_xy, double *inner_yaw, int max_inner_yaw, int32_t *N,
                       int32_t *M, double *total_time);

/* ---- front-end: KinoAstar (SURVEY 8f-2) ---- */
/* kino_astar/* parameters (front_end/src/kino_astar.cpp:7-20) */
typedef struct {
    double yaw_resolution, lambda_heu, weight_r2, weight_so2, weight_v_change, weight_delta_change, weight_sigma;
    double time_interval, collision_interval, oneshot_range, wheel_base, max_steer, max_vel;
} ualm_astar_params_t;
/* plan_manager/params/run_*.yaml:16-30 (the same values in every terrain file) */
void ualm_astar_default_params(ualm_astar_params_t *p);
/* what KinoAstar reads of UnevenMap (isOccupancy, isOccupancyXY, isInMap, getTerrainSig; uneven_map.h:389-500): the cell grid
 * ([X][Y][Yaw][4] = z, sigma, zb.x, zb.y; float as ualm_set_map takes it, or double as ualm_set_map_f64 does -- one of the two) and
 * the occupancy grids of ualm_map_occupancy (occ3: [X][Y][Yaw], occ2: [X][Y]) */
typedef struct {
    const ualm_map_geom_t *geom;
    const float *cells;
    const double *cells64;
    const uint8_t *occ3, *occ2;
} ualm_astar_map_t;
/* plan_manager/* parameters of the resampler (plan_manager.cpp:24-30; run_hill.yaml:57-62) */
typedef struct { double piece_len, yaw_piece_times, mean_vel, init_time_times, init_sig_vel; } ualm_resample_params_t;

/* KinoAstar::plan(start_state, end_state) (front_end/src/kino_astar.cpp:67-236): hybrid A* over (x, y, yaw) with 3 x 5 motion
 * primitives and a Dubins one-shot near the goal.  Writes the (x, y, yaw) polyline start .. goal and returns its number of points;
 * 0 = no path (start or goal occupied, open set exhausted, node pool exhausted), like the reference's empty vector.
 * n_expanded (optional): nodes closed.  The Dubins curve is OMPL's in the reference (absent here): csrc/dubins.h restates it. */
int ualm_kino_astar_plan(const ualm_astar_map_t *map, const ualm_astar_params_t *p, const double start[3], const double goal[3],
                         double *path_xyyaw, int max_pts, int *n_expanded);

/* The one-shot curve of KinoAstar::asignShotTraj alone (kino_astar.h:246-258, without its occupancy test): the shortest Dubins curve of
 * turning radius `radius` sampled every `interval` metres from its start; *length (optional) receives its length. */
int ualm_dubins_shot(const double start[3], const double goal[3], double radius, double interval, double *path_xyyaw, int max_pts, double *length);

/* The reference's whole front half for B (start, goal) pairs, one search per host thread (nthreads <= 0: all cores):
 * KinoAstar::plan -> PlanManager's resampler (ualm_resample_path).  Outputs are the ragged arrays ualm_solve_batch /
 * ualm_submit_batch take, packed back to back for the problems that have a path and fit the optimizer's limits; packed[b] = index of
 * pair b in them or -1; n_expanded[b] (optional) = nodes closed.  Returns the number of packed problems (or a negative error;
 * UALM_ELIMIT when cap_xy / cap_yaw doubles are not enough). */
int ualm_front_end_batch(const ualm_astar_map_t *map, const ualm_astar_params_t *ap, const ualm_resample_params_t *rp, int B,
                         const double *starts, const double *goals, int nthreads, int32_t *N, int32_t *M, double *bnd, double *total_time,
                         double *inner_xy, long long cap_xy, double *inner_yaw, long long cap_yaw, int32_t *packed, int32_t *n_expanded);

/* The same search on the host with include/ualm_detmath.h's sin / cos / tan / atan2 / acos instead of the C library's: bit for bit
 * what ualm_front_end_batch_device computes for one pair.  For tests; it differs from ualm_kino_astar_plan only in the trigonometry. */
int ualm_kino_astar_plan_det(const ualm_astar_map_t *map, const ualm_astar_params_t *p, const double start[3], const double goal[3],
                             double *path_xyyaw, int max_pts, int *n_expanded);

/* ---- the front-end on the GPU (csrc/ualm_front_end.cu): one warp per KinoAstar search ----
 * ualm_set_front_end_map: uploads the occupancy grids and the cell grid (double when map->cells64 is set, float otherwise, as the host
 * search reads it) to the context's device.
 * ualm_front_end_batch_device: ualm_front_end_batch's outputs for B pairs, searched on the device with ualm_kino_astar_plan_det's
 * arithmetic (bit-identical to it; the trigonometry makes it differ from ualm_front_end_batch in the last bits), resampled on the host by
 * ualm_resample_path.  A polyline longer than ualm_front_end_path_cap points cannot pass the optimizer's limits: it is left out
 * (packed = -1) and returned empty.  Optional: path_xyyaw (room for cap_path points) + path_off[B + 1], the raw polylines back to back;
 * search_ms, the CUDA-event time of the search kernel.  Poses must be finite with |yaw| <= 1e4 and the A* parameters finite. */
int ualm_set_front_end_map(ualm_ctx_t *ctx, const ualm_astar_map_t *map);
int ualm_front_end_batch_device(ualm_ctx_t *ctx, const ualm_astar_params_t *ap, const ualm_resample_params_t *rp, int B, const double *starts,
                                const double *goals, int32_t *N, int32_t *M, double *bnd, double *total_time, double *inner_xy, long long cap_xy,
                                double *inner_yaw, long long cap_yaw, int32_t *packed, int32_t *n_expanded, double *path_xyyaw, long long cap_path,
                                int64_t *path_off, float *search_ms);
/* the most points one device search returns for these parameters: every polyline the resampler can accept within N <= 64, M <= 128 fits */
int ualm_front_end_path_cap(const ualm_astar_params_t *ap, const ualm_resample_params_t *rp);

#ifdef __cplusplus
}
#endif
#endif
