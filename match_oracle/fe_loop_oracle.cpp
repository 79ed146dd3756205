// fe_loop_oracle.cpp — CPU restatement of fe_loop_closures (include/fe_b200.h, "loop closures").
// TEST INFRASTRUCTURE ONLY, like fe_odometry_oracle.cpp.  A literal loop over the contract: scan after scan, the
// database materialised as one group for feo_match_descriptors, the votes counted in a map, and every candidate
// matched and registered as one group by feo_match_descriptors and feo_register_matches.  Built with
// -ffp-contract=off, so every double operation is rounded on its own.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <map>
#include <utility>
#include <vector>

extern "C" int feo_match_descriptors(const float* query, int64_t query_stride, const int64_t* query_offsets,
                                     const float* ref, int64_t ref_stride, const int64_t* ref_offsets, int32_t n_groups,
                                     int32_t n_threads, int64_t* best, int32_t* shift, float* dist2, float* second_dist2);
extern "C" int feo_register_matches(const float* query_kp, const float* ref_kp, const int64_t* best, const int64_t* qo,
                                    const int64_t* ro, int32_t G, double inlier_radius, double min_separation,
                                    int32_t max_hypotheses, int32_t min_inliers, int32_t refine_iterations, double* pose,
                                    double* rms, int32_t* n_inliers, int32_t* n_hypotheses, int32_t* status,
                                    int64_t* assoc);

namespace {

// feo_match_descriptors on one group -> best per query row
std::vector<int64_t> match(const float* desc, int64_t stride, int64_t q0, int64_t q1, int64_t r0, int64_t r1, int32_t threads) {
  const size_t n = (size_t)(q1 - q0);
  std::vector<int64_t> best(n);
  std::vector<int32_t> shift(n);
  std::vector<float> d(n), sd(n);
  const int64_t qo[2] = {q0, q1}, ro[2] = {r0, r1};
  feo_match_descriptors(desc, stride, qo, desc, stride, ro, 1, threads, best.data(), shift.data(), d.data(), sd.data());
  return best;
}

}  // namespace

extern "C" {

// Returns 0, or 1 (FE_ERR_INVALID) on the argument errors fe_loop_closures rejects.  Outputs as fe_loop_result_t:
// per scan loop, loop_scan, pose (B x 4), rms, n_inliers, n_hypotheses; per scan x K cand_scan, cand_votes,
// cand_status, cand_inliers, cand_hypotheses, cand_rms, cand_pose (B x K x 4); assoc per row of [ko[0], ko[B]).
int feo_loop_closures(const float* kp, const float* desc, int64_t stride, const int64_t* ko, int32_t B, const int64_t* so,
                      int32_t S, int32_t min_gap, int32_t K, double inlier_radius, double min_separation,
                      int32_t max_hypotheses, int32_t min_inliers, int32_t refine_iterations, int32_t n_threads,
                      int32_t* loop, int32_t* loop_scan, double* pose, double* rms, int32_t* n_inliers,
                      int32_t* n_hypotheses, int32_t* cand_scan, int32_t* cand_votes, int32_t* cand_status,
                      int32_t* cand_inliers, int32_t* cand_hypotheses, double* cand_rms, double* cand_pose,
                      int64_t* assoc) {
  if (!(std::isfinite(inlier_radius) && inlier_radius > 0) || !(std::isfinite(min_separation) && min_separation > 0) ||
      max_hypotheses < 1 || max_hypotheses > 65536 || min_inliers < 1 || refine_iterations < 0 || refine_iterations > 1000)
    return 1;
  if (B < 0 || S < 0 || !ko || !so || K < 1 || K > 16 || min_gap < 1 || stride < 1980) return 1;
  if (ko[0] < 0 || so[0] != 0 || so[S] != B) return 1;
  for (int32_t b = 0; b < B; b++)
    if (ko[b + 1] < ko[b] || ko[b + 1] - ko[b] >= (1LL << 24)) return 1;
  for (int32_t q = 0; q < S; q++)
    if (so[q + 1] < so[q]) return 1;
  if (ko[B] - ko[0] >= (1LL << 31)) return 1;
  if (ko[B] > ko[0] && (!kp || !desc)) return 1;
  const double id[4] = {1.0, 0.0, 0.0, 0.0};

  for (int64_t s = 0; s < B; s++) {
    loop[s] = loop_scan[s] = -1;
    for (int c = 0; c < 4; c++) pose[4 * s + c] = id[c];
    rms[s] = 0.0;
    n_inliers[s] = n_hypotheses[s] = 0;
    for (int64_t k = s * K; k < (s + 1) * K; k++) {
      cand_scan[k] = -1;
      cand_votes[k] = 0;
      cand_status[k] = -1;
      cand_inliers[k] = cand_hypotheses[k] = 0;
      cand_rms[k] = 0.0;
      for (int c = 0; c < 4; c++) cand_pose[4 * k + c] = id[c];
    }
    for (int64_t r = ko[s]; r < ko[s + 1]; r++) assoc[r - ko[0]] = -1;
  }

  for (int32_t q = 0; q < S; q++) {
    const int64_t f = so[q];
    for (int64_t s = f + min_gap; s < so[q + 1]; s++) {
      const int64_t q0 = ko[s], q1 = ko[s + 1];
      if (q1 == q0) continue;
      // retrieval: best over the database, scans f .. s - min_gap; one vote per row for the scan holding its best
      const int64_t last = s - min_gap;
      const std::vector<int64_t> best = match(desc, stride, q0, q1, ko[f], ko[last + 1], n_threads);
      std::map<int64_t, int32_t> votes;
      for (const int64_t b : best) {
        if (b < 0) continue;
        int64_t j = f;
        while (!(ko[j] <= b && b < ko[j + 1])) j++;
        votes[j]++;
      }
      std::vector<std::pair<int32_t, int64_t>> cand;  // (-votes, scan): ascending is the contract's order
      for (const auto& v : votes) cand.push_back({-v.second, v.first});
      std::sort(cand.begin(), cand.end());
      if ((int)cand.size() > K) cand.resize((size_t)K);

      // verification of every candidate, then the choice: status 2, most inliers, lower rank on ties
      int win = -1;
      std::vector<int64_t> winAssoc;
      for (int k = 0; k < (int)cand.size(); k++) {
        const int64_t j = cand[(size_t)k].second, slot = s * K + k;
        cand_scan[slot] = (int32_t)j;
        cand_votes[slot] = -cand[(size_t)k].first;
        const std::vector<int64_t> b2 = match(desc, stride, q0, q1, ko[j], ko[j + 1], 1);
        const int64_t qo[2] = {q0, q1}, ro[2] = {ko[j], ko[j + 1]};
        std::vector<int64_t> a((size_t)(q1 - q0));
        if (feo_register_matches(kp, kp, b2.data(), qo, ro, 1, inlier_radius, min_separation, max_hypotheses,
                                 min_inliers, refine_iterations, cand_pose + 4 * slot, cand_rms + slot,
                                 cand_inliers + slot, cand_hypotheses + slot, cand_status + slot, a.data()) != 0)
          return 1;
        if (cand_status[slot] == 2 && (win < 0 || cand_inliers[slot] > cand_inliers[s * K + win])) {
          win = k;
          winAssoc = a;
        }
      }
      if (win < 0) continue;
      const int64_t slot = s * K + win;
      loop[s] = win;
      loop_scan[s] = cand_scan[slot];
      for (int c = 0; c < 4; c++) pose[4 * s + c] = cand_pose[4 * slot + c];
      rms[s] = cand_rms[slot];
      n_inliers[s] = cand_inliers[slot];
      n_hypotheses[s] = cand_hypotheses[slot];
      for (int64_t r = q0; r < q1; r++) assoc[r - ko[0]] = winAssoc[(size_t)(r - q0)];
    }
  }
  return 0;
}

}  // extern "C"
