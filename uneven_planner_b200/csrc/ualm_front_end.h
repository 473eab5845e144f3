// ualm_front_end.h -- the front-end's host helpers shared by the host batch (csrc/kino_astar.cpp) and the device batch
// (csrc/ualm_front_end.cu), and the device batch as ualm_api.cu's context calls it
#pragma once
#include <string>
#include <vector>

#include "ualm.h"

namespace ualm_fe {

// one polyline through PlanManager's resampler with the optimizer's limits (N <= 64, M <= 128); ok = 0 without a path or over them
struct Resampled { int ok = 0; int32_t N = 0, M = 0; double T = 0; double bnd[18]; std::vector<double> ixy, iyaw; };
void resample(const double *path, int npts, const ualm_resample_params_t *rp, Resampled &o);
// the resampled problems packed back to back in pair order: packed[b] = index or -1.  Returns their number or UALM_ELIMIT
int pack(const std::vector<Resampled> &res, int32_t *N, int32_t *M, double *bnd, double *total_time, double *inner_xy, long long cap_xy,
         double *inner_yaw, long long cap_yaw, int32_t *packed);

struct FrontEnd;      // the uploaded map, the per-warp workspaces and the batch buffers of one context

int set_map(FrontEnd **fe, const ualm_astar_map_t *m, std::string &err);
void release(FrontEnd *fe);
int batch(FrontEnd *fe, const ualm_astar_params_t *ap, const ualm_resample_params_t *rp, int B, const double *starts, const double *goals,
          int32_t *N, int32_t *M, double *bnd, double *total_time, double *inner_xy, long long cap_xy, double *inner_yaw, long long cap_yaw,
          int32_t *packed, int32_t *n_expanded, double *path_xyyaw, long long cap_path, int64_t *path_off, float *search_ms, std::string &err);
// the longest polyline one search may return for these parameters (ualm_front_end_path_cap)
int path_cap(const ualm_astar_params_t *ap, const ualm_resample_params_t *rp);

}  // namespace ualm_fe
