// fe_odometry_oracle.cpp — CPU restatement of fe_odometry (include/fe_b200.h, "odometry").
// TEST INFRASTRUCTURE ONLY, like fe_register_oracle.cpp.  A literal loop over the contract: sequence after sequence,
// step after step, each step's window materialised and registered by feo_register_matches as one group.  Built with
// -ffp-contract=off, so every double operation is rounded on its own.
#include <cmath>
#include <cstdint>
#include <vector>

extern "C" int feo_register_matches(const float* query_kp, const float* ref_kp, const int64_t* best, const int64_t* qo,
                                    const int64_t* ro, int32_t G, double inlier_radius, double min_separation,
                                    int32_t max_hypotheses, int32_t min_inliers, int32_t refine_iterations, double* pose,
                                    double* rms, int32_t* n_inliers, int32_t* n_hypotheses, int32_t* status,
                                    int64_t* assoc);

namespace {

struct Pt { float x, y, z, w; };
struct Motion { double c, s, tx, ty; };

Motion inv(const Motion& a) { return {a.c, -a.s, -(a.c * a.tx + a.s * a.ty), a.s * a.tx - a.c * a.ty}; }

Motion compose(const Motion& a, const Motion& b) {
  return {a.c * b.c - a.s * b.s, a.s * b.c + a.c * b.s, (a.c * b.tx - a.s * b.ty) + a.tx, (a.s * b.tx + a.c * b.ty) + a.ty};
}

Motion get(const double* m, int64_t s) { return {m[4 * s], m[4 * s + 1], m[4 * s + 2], m[4 * s + 3]}; }

void put(double* m, int64_t s, const Motion& a) {
  m[4 * s] = a.c; m[4 * s + 1] = a.s; m[4 * s + 2] = a.tx; m[4 * s + 3] = a.ty;
}

}  // namespace

extern "C" {

// Returns 0, or 1 (FE_ERR_INVALID) on the argument errors fe_odometry rejects.  Outputs as fe_odometry_result_t:
// pose, motion B x 4, rms, source, status, n_inliers, n_hypotheses per scan, assoc per row of [ko[0], ko[B]).
int feo_odometry(const float* kp, const int64_t* ko, int32_t B, const int64_t* best, const int64_t* so, int32_t S,
                 int32_t W, double inlier_radius, double min_separation, int32_t max_hypotheses, int32_t min_inliers,
                 int32_t refine_iterations, double* pose, double* motion, double* rms, int32_t* source, int32_t* status,
                 int32_t* n_inliers, int32_t* n_hypotheses, int64_t* assoc) {
  if (!(std::isfinite(inlier_radius) && inlier_radius > 0) || !(std::isfinite(min_separation) && min_separation > 0) ||
      max_hypotheses < 1 || max_hypotheses > 65536 || min_inliers < 1 || refine_iterations < 0 || refine_iterations > 1000)
    return 1;
  if (B < 0 || S < 0 || !ko || !so || W < 1 || W > 64) return 1;
  if (ko[0] < 0 || so[0] != 0 || so[S] != B) return 1;
  for (int32_t b = 0; b < B; b++)
    if (ko[b + 1] < ko[b] || ko[b + 1] - ko[b] >= (1LL << 24)) return 1;
  for (int32_t q = 0; q < S; q++)
    if (so[q + 1] < so[q]) return 1;
  if (ko[B] - ko[0] >= (1LL << 31)) return 1;
  bool steps = false, rows = false;
  for (int32_t q = 0; q < S; q++)
    for (int64_t s = so[q] + 1; s < so[q + 1]; s++) {
      steps = true;
      rows |= ko[s + 1] > ko[s];
      for (int64_t k = ko[s]; best && k < ko[s + 1]; k++) {
        const int64_t b = best[k - ko[1]];
        if (b != -1 && (b < ko[s - 1] || b >= ko[s])) return 1;
      }
    }
  if ((rows && !best) || (steps && ko[B] > ko[0] && !kp)) return 1;
  const Pt* P = (const Pt*)kp;
  const Motion id = {1.0, 0.0, 0.0, 0.0};

  for (int32_t q = 0; q < S; q++) {
    const int64_t f = so[q], L = so[q + 1] - so[q];
    if (L == 0) continue;
    put(pose, f, id);
    put(motion, f, id);
    rms[f] = 0.0;
    source[f] = 0;
    status[f] = -1;
    n_inliers[f] = 0;
    n_hypotheses[f] = 0;
    for (int64_t k = ko[f]; k < ko[f + 1]; k++) assoc[k - ko[0]] = -1;
    for (int64_t t = 1; t < L; t++) {
      const int64_t s = f + t;
      // window: scan t-1, then t-2, ... down to t-W, stopping before the first scan whose link was predicted
      int64_t first = s - 1;
      for (int64_t j = s - 2; j >= f && j >= s - W; j--) {
        if (source[j + 1] != 1) break;
        first = j;
      }
      const int64_t winLo = ko[first];
      std::vector<Pt> ref((size_t)(ko[s] - winLo));
      for (int64_t k = ko[s - 1]; k < ko[s]; k++) ref[(size_t)(k - winLo)] = P[k];
      Motion Pj = inv(get(motion, s - 1));  // P_{t-2}
      for (int64_t j = s - 2; j >= first; j--) {
        if (j < s - 2) Pj = compose(Pj, inv(get(motion, j + 1)));
        for (int64_t k = ko[j]; k < ko[j + 1]; k++) {
          Pt p = P[k];
          const double px = (double)p.x, py = (double)p.y;
          p.x = (float)((Pj.c * px - Pj.s * py) + Pj.tx);
          p.y = (float)((Pj.s * px + Pj.c * py) + Pj.ty);
          ref[(size_t)(k - winLo)] = p;
        }
      }
      const int64_t nq = ko[s + 1] - ko[s];
      std::vector<int64_t> b((size_t)nq), a((size_t)nq + 1);
      for (int64_t k = ko[s]; k < ko[s + 1]; k++) {
        const int64_t e = best[k - ko[1]];
        b[(size_t)(k - ko[s])] = e < 0 ? -1 : e - winLo;
      }
      const int64_t qo[2] = {ko[s], ko[s + 1]}, ro[2] = {0, (int64_t)ref.size()};
      double gp[4], grms;
      int32_t gin, ghyp, gst;
      if (feo_register_matches(kp, ref.empty() ? nullptr : (const float*)ref.data(), nq ? b.data() : nullptr, qo, ro, 1,
                               inlier_radius, min_separation, max_hypotheses, min_inliers, refine_iterations, gp, &grms,
                               &gin, &ghyp, &gst, a.data()) != 0)
        return 1;
      const Motion M = gst == 2 ? Motion{gp[0], gp[1], gp[2], gp[3]} : t == 1 ? id : get(motion, s - 1);
      put(motion, s, M);
      put(pose, s, compose(get(pose, s - 1), M));
      source[s] = gst == 2 ? 1 : 2;
      status[s] = gst;
      rms[s] = grms;
      n_inliers[s] = gin;
      n_hypotheses[s] = ghyp;
      for (int64_t k = ko[s]; k < ko[s + 1]; k++) {
        const int64_t j = a[(size_t)(k - ko[s])];
        assoc[k - ko[0]] = j < 0 ? -1 : winLo + j;
      }
    }
  }
  return 0;
}

}  // extern "C"
