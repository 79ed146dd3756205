// fe_match_oracle.cpp — CPU restatement of fe_match_descriptors (include/fe_b200.h, "descriptor matching").
// TEST INFRASTRUCTURE ONLY, like oracle/fe_oracle.cpp.  A literal loop over the contract: the 144 chains P(la, lb) with
// std::fmaf, the 12 shift sums as unfused float adds in ascending l, candidates visited in ascending (r, s) and
// taken only when strictly smaller.  Built with -ffp-contract=off.  Queries are split over n_threads threads; a
// query's result depends on nothing but its group, so the split does not change it.
#include <cmath>
#include <algorithm>
#include <cstdint>
#include <limits>
#include <thread>
#include <vector>

namespace {

constexpr int L = 12, BLK = 165;

float shift_distance(const float* a, const float* b, int s) {
  float d = 0.0f;
  for (int l = 0; l < L; l++) {
    const float* x = a + l * BLK;
    const float* y = b + ((l + s) % L) * BLK;
    float acc = 0.0f;
    for (int m = 0; m < BLK; m++) {
      const float t = x[m] - y[m];
      acc = std::fmaf(t, t, acc);
    }
    d = d + acc;
  }
  return d;
}

}  // namespace

extern "C" {

// Returns 0, or 1 (FE_ERR_INVALID) on the argument errors fe_match_descriptors rejects.
int feo_match_descriptors(const float* query, int64_t query_stride, const int64_t* query_offsets, const float* ref,
                          int64_t ref_stride, const int64_t* ref_offsets, int32_t n_groups, int32_t n_threads,
                          int64_t* best, int32_t* shift, float* dist2, float* second_dist2) {
  if (n_groups < 0 || query_stride < 1980 || ref_stride < 1980 || !query_offsets || !ref_offsets) return 1;
  for (int32_t g = 0; g < n_groups; g++)
    if (query_offsets[g + 1] < query_offsets[g] || ref_offsets[g + 1] < ref_offsets[g]) return 1;
  if (query_offsets[0] < 0 || ref_offsets[0] < 0) return 1;
  const int64_t q0 = query_offsets[0], nQ = query_offsets[n_groups] - q0;
  if ((nQ > 0 && !query) || (ref_offsets[n_groups] > ref_offsets[0] && !ref)) return 1;
  const float INF = std::numeric_limits<float>::infinity();

  // group of every query row
  std::vector<int32_t> grp((size_t)nQ);
  for (int32_t g = 0; g < n_groups; g++)
    for (int64_t i = query_offsets[g]; i < query_offsets[g + 1]; i++) grp[(size_t)(i - q0)] = g;

  auto run = [&](int64_t lo, int64_t hi) {
    std::vector<float> rowMin;
    std::vector<int32_t> rowS;
    for (int64_t i = lo; i < hi; i++) {
      const int32_t g = grp[(size_t)i];
      const float* a = query + (q0 + i) * query_stride;
      const int64_t r0 = ref_offsets[g], r1 = ref_offsets[g + 1];
      rowMin.assign((size_t)(r1 - r0), INF);
      rowS.assign((size_t)(r1 - r0), -1);
      float bd = INF;
      int64_t br = -1;
      int32_t bs = -1;
      for (int64_t r = r0; r < r1; r++) {
        const float* b = ref + r * ref_stride;
        for (int s = 0; s < L; s++) {
          const float d = shift_distance(a, b, s);
          if (d < rowMin[(size_t)(r - r0)]) { rowMin[(size_t)(r - r0)] = d; rowS[(size_t)(r - r0)] = s; }
          if (d < bd) { bd = d; br = r; bs = s; }
        }
      }
      float sd = INF;
      for (int64_t r = r0; r < r1; r++)
        if (r != br && rowMin[(size_t)(r - r0)] < sd) sd = rowMin[(size_t)(r - r0)];
      best[i] = br;
      shift[i] = bs;
      dist2[i] = bd;
      second_dist2[i] = sd;
    }
  };
  const int T = (int)std::max<int64_t>(1, std::min<int64_t>(n_threads, nQ));
  if (T == 1) {
    run(0, nQ);
  } else {
    // queries interleaved over the threads: groups of very different sizes spread evenly
    std::vector<std::thread> th;
    for (int t = 0; t < T; t++)
      th.emplace_back([&, t] {
        for (int64_t i = t; i < nQ; i += T) run(i, i + 1);
      });
    for (auto& x : th) x.join();
  }
  return 0;
}

}  // extern "C"
