// fe_loop.h — the interface between the host code of fe_loop_closures* (fe_api.cu) and the loop-closure kernels
// (fe_loop.cu).  Internal to libfe_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/fe_b200.h"
#include "fe_match.h"
#include "fe_register.h"

namespace fe_loop {

constexpr int MAX_CANDIDATES = 16;

// Eligible scan e: absolute scan `scan` of the sequence whose first scan is `first`; its K verification slots are
// e * K .. e * K + K - 1.
struct Scan {
  int scan, first;
};

// Verification slot i (scan e = i / K, rank k = i % K): query rows [q0, q0 + n_t) are a copy of scan t's keypoints,
// reference rows [r0, r0 + cap) hold scan j's keypoints and then an unused tail.  Its pass-2 items are
// [item0, item0 + nseg * tiles), segment outer; segment g reads reference rows [ko[j] + g * ITEM_REFS, ...).
struct Slot {
  int64_t q0, r0, cap;
  int64_t item0;
  int32_t tiles, nseg;
};

// Device tables of one call, uploaded once.  Registration groups 2i (slot i) and 2i + 1 (its unused tail): query
// offsets qo[0..2n], reference offsets ro[0..2n]; ro[2i + 1] is written by k_loop_place.
struct Tables {
  const int64_t* ko;      // keypoint offsets, B + 1
  const int* elig;        // B: eligible index e of each scan, or -1
  const Scan* scans;      // E eligible scans
  const Slot* slots;      // E * K
  fe_match::Item* items;  // pass-2 items (r0 and nr written by k_loop_place)
  const int64_t* qo;
  int64_t* ro;
};

// Device work buffers: retrieval's best per row of [ko[0], ko[B]), each row's voted scan and vote key; the slot rows,
// pass-2 best (absolute rows of scan j), its remap to slot rows, and registration's outputs and scratch.
struct Work {
  const long long* best1;
  int* voteScan;
  unsigned long long* voteKey;
  fe_point_t *q, *r;
  long long* best2;
  long long* slotBest;
  fe_register::Out reg;
  fe_register::Scratch scratch;
};

// Results: per scan loop, loopScan, pose (4 doubles), rms, nInl, nHyp; per scan x K candidate scan, votes, status,
// inliers, hypotheses, rms, pose; per row of [ko[0], ko[B]) assoc.
struct Out {
  int *loop, *loopScan, *nInl, *nHyp;
  double *pose, *rms;
  int *cScan, *cVotes, *cStatus, *cInl, *cHyp;
  double *cRms, *cPose;
  long long* assoc;
};

// E eligible scans, whose databases end `gap` scans before them.  Each launcher launches one kernel, or none when
// there is nothing to do.
cudaError_t vote(int E, int K, int gap, Tables T, Work w, Out o, cudaStream_t stream);
// Keypoint row k is at kp[k - kpBias].
cudaError_t place(const fe_point_t* kp, int64_t kpBias, int nSlots, int K, Tables T, Work w, Out o, cudaStream_t stream);
cudaError_t remap(int nSlots, int K, Tables T, Work w, Out o, cudaStream_t stream);
cudaError_t select(int B, int K, Tables T, Work w, Out o, cudaStream_t stream);

}  // namespace fe_loop
