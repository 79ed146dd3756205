// fe_match.h — the interface between the host code of fe_match_descriptors* (fe_api.cu) and the matcher's
// kernels (fe_match.cu).  Internal to libfe_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace fe_match {

constexpr int ITEM_QUERIES = 4;       // query rows per work item (one warp)
constexpr int64_t ITEM_REFS = 1024;   // reference rows per work item: a larger group is split into segments

// One work item: query rows [q0, q0 + nq) of a group against its reference rows [r0, r0 + nr) (absolute row indices
// of the caller's arrays).  Output row of query q0 + i is out + i.  A group of more than ITEM_REFS reference rows is cut
// into nseg segments; item `seg` of them writes the partial of query i at part + i * nseg + seg.
struct Item {
  int64_t q0, r0, out, part;
  int32_t nq, nr, nseg, seg;
};

struct Partial {
  float d, sd;  // best distance, smallest row minimum of the segment's other rows
  long long r;  // best row (-1: none)
  int s;        // its shift (-1: none)
};

struct Result {
  long long* best;
  int* shift;
  float* dist2;
  float* second;
};

size_t smem_bytes();
cudaError_t set_attributes();
// Row i of the query side is at q + (i - qBias) * qStride (likewise for the references).  `split`: some item has nseg > 1.
cudaError_t launch(const float* q, int64_t qStride, int64_t qBias, const float* r, int64_t rStride, int64_t rBias,
                   const Item* d_items, int nItems, bool split, Partial* d_part, Result res, cudaStream_t stream);

}  // namespace fe_match
