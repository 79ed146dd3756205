// fe_odometry.h — the interface between the host code of fe_odometry* (fe_api.cu) and the odometry kernels
// (fe_odometry.cu).  Internal to libfe_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "../../include/fe_b200.h"
#include "fe_register.h"

namespace fe_odo {

// Sequence i of a step: absolute scan `scan` of the sequence whose first scan is `first`.
struct Item {
  int scan, first;
};

// Step t: items [item0, item0 + n) of the item table; its 2n + 1 query offsets start at offs0 of the offsets table and
// its 2n + 1 reference offsets follow them.  Group 2i registers item i into its slot of reference rows; group 2i + 1
// has no query rows and covers the slot's unused tail (the placement kernel writes its start, ro[2i + 1]).  Query rows
// and reference slots are numbered from 0 in every step.
struct Step {
  int64_t item0, offs0;
  int n;
};

// Device tables of one call, uploaded once.
struct Tables {
  const int64_t* ko;  // keypoint offsets, B + 1
  const int64_t* so;  // sequence offsets, S + 1
  const Item* items;
  int64_t* offs;      // every step's query then reference offsets
};

// Device buffers that every step reuses: the compact query rows, `best` remapped to slot rows, the placed reference
// rows, the window's first absolute row per item, and registration's outputs and scratch.
struct Work {
  fe_point_t *q, *r;
  long long* best;
  int64_t* winLo;
  fe_register::Out reg;
  fe_register::Scratch scratch;
};

// Results: per scan pose, motion (4 doubles each), rms, source, status, nInl, nHyp; per row of [ko[0], ko[B]) assoc.
// *err is set to 1 when an entry of `best` that a step reads is neither -1 nor a row of the previous scan.
struct Out {
  double *pose, *motion, *rms;
  long long* assoc;
  int *source, *status, *nInl, *nHyp, *err;
};

// Keypoint row k is at kp[k - kpBias]; `best` of row k at best[k - ko[1]].  Launches 1 + 3 * steps.size() kernels.
cudaError_t run(const fe_point_t* kp, int64_t kpBias, const long long* best, int nSeq, int W,
                const std::vector<Step>& steps, Tables T, Work w, Out o, fe_register::Params p, cudaStream_t stream);

}  // namespace fe_odo
