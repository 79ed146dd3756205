// fe_register.h — the interface between the host code of fe_register_matches* (fe_api.cu) and the registration
// kernel (fe_register.cu).  Internal to libfe_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/fe_b200.h"

namespace fe_register {

struct Params {
  double r2, sep2, twoR;  // inlier_radius^2, min_separation^2, 2 * inlier_radius
  int maxH, minInliers, refine;
};

// Per group: pose[4g..4g+3], rms[g], nInl[g], nHyp[g], status[g]; per query row i (absolute row qo[0] + i): assoc[i].
// *err is set to 1 when an entry of `best` is neither -1 nor a reference row of its group.
struct Out {
  double* pose;
  double* rms;
  long long* assoc;
  int* nInl;
  int* nHyp;
  int* status;
  int* err;
};

// Per query row i, for the kernel's own use: the correspondence list of each group and a second evaluation.
struct Scratch {
  int* corr;
  long long* assocNew;
  double* d2Cur;
  double* d2New;
};

// Query row k is at q[k - qBias], reference row j at r[j - rBias], best of row k at best[k - qo[0]]; d_qo and d_ro are
// the n_groups + 1 offsets in device memory.
cudaError_t launch(const fe_point_t* q, int64_t qBias, const fe_point_t* r, int64_t rBias, const long long* best,
                   const int64_t* d_qo, const int64_t* d_ro, int nGroups, Params p, Out o, Scratch s, cudaStream_t stream);

}  // namespace fe_register
