// fe_register_oracle.cpp — CPU restatement of fe_register_matches (include/fe_b200.h, "registration").
// TEST INFRASTRUCTURE ONLY, like fe_match_oracle.cpp.  A literal loop over the contract, one group after the other:
// hypotheses in ascending h, query rows and reference rows in ascending order, every sum sequential.  Built with
// -ffp-contract=off, so every double operation is rounded on its own.
#include <cmath>
#include <cstdint>
#include <vector>

namespace {

struct Pt { float x, y, z, w; };
struct Motion { double c, s, tx, ty; };

struct Eval {
  int score = 0;
  std::vector<int64_t> assoc;  // per query row of the group
  std::vector<double> d2;
};

Eval evaluate(const Motion& M, const Pt* q, int64_t q0, int64_t q1, const Pt* r, int64_t r0, int64_t r1, double r2) {
  Eval e;
  for (int64_t k = q0; k < q1; k++) {
    const double px = (double)q[k].x, py = (double)q[k].y;
    const double wx = (M.c * px - M.s * py) + M.tx, wy = (M.s * px + M.c * py) + M.ty;
    double cur = r2;
    int64_t jj = -1;
    for (int64_t j = r0; j < r1; j++) {
      const double dx = wx - (double)r[j].x, dy = wy - (double)r[j].y;
      const double d2 = dx * dx + dy * dy;
      if (d2 < cur) { cur = d2; jj = j; }
    }
    e.assoc.push_back(jj);
    e.d2.push_back(cur);
    if (jj >= 0) e.score++;
  }
  return e;
}

}  // namespace

extern "C" {

// Returns 0, or 1 (FE_ERR_INVALID) on the argument errors fe_register_matches rejects.  Outputs as fe_register_result_t:
// pose n_groups x 4, rms, n_inliers, n_hypotheses, status per group, assoc per query row.
int feo_register_matches(const float* query_kp, const float* ref_kp, const int64_t* best, const int64_t* qo,
                         const int64_t* ro, int32_t G, double inlier_radius, double min_separation,
                         int32_t max_hypotheses, int32_t min_inliers, int32_t refine_iterations, double* pose,
                         double* rms, int32_t* n_inliers, int32_t* n_hypotheses, int32_t* status, int64_t* assoc) {
  if (G < 0 || !qo || !ro) return 1;
  if (!(std::isfinite(inlier_radius) && inlier_radius > 0) || !(std::isfinite(min_separation) && min_separation > 0) ||
      max_hypotheses < 1 || max_hypotheses > 65536 || min_inliers < 1 || refine_iterations < 0 || refine_iterations > 1000)
    return 1;
  if (qo[0] < 0 || ro[0] < 0) return 1;
  for (int32_t g = 0; g < G; g++)
    if (qo[g + 1] < qo[g] || ro[g + 1] < ro[g] || qo[g + 1] - qo[g] >= (1LL << 24)) return 1;
  const int64_t base = qo[0];
  if ((qo[G] > base && (!query_kp || !best)) || (ro[G] > ro[0] && !ref_kp)) return 1;
  for (int32_t g = 0; g < G; g++)
    for (int64_t k = qo[g]; k < qo[g + 1]; k++) {
      const int64_t b = best[k - base];
      if (b != -1 && (b < ro[g] || b >= ro[g + 1])) return 1;
    }
  const Pt* q = (const Pt*)query_kp;
  const Pt* r = (const Pt*)ref_kp;
  const double r2 = inlier_radius * inlier_radius, sep2 = min_separation * min_separation, twoR = 2.0 * inlier_radius;

  for (int32_t g = 0; g < G; g++) {
    const int64_t q0 = qo[g], q1 = qo[g + 1], r0 = ro[g], r1 = ro[g + 1];
    std::vector<int64_t> corr;
    for (int64_t k = q0; k < q1; k++)
      if (best[k - base] >= 0) corr.push_back(k);
    const int64_t nc = (int64_t)corr.size(), P = nc * (nc - 1) / 2;
    const int64_t H = P < max_hypotheses ? P : max_hypotheses;

    auto hypothesis = [&](int64_t h, Motion& M) {
      int64_t idx = h * P / H, a = 0;
      while (idx >= nc - 1 - a) { idx -= nc - 1 - a; a++; }
      const int64_t b = a + 1 + idx;
      const int64_t ka = corr[(size_t)a], kb = corr[(size_t)b];
      const int64_t ja = best[ka - base], jb = best[kb - base];
      const double pax = q[ka].x, pay = q[ka].y, pbx = q[kb].x, pby = q[kb].y;
      const double qax = r[ja].x, qay = r[ja].y, qbx = r[jb].x, qby = r[jb].y;
      const double ux = pbx - pax, uy = pby - pay, vx = qbx - qax, vy = qby - qay;
      const double lu = ux * ux + uy * uy, lv = vx * vx + vy * vy;
      if (lu < sep2 || lv < sep2) return false;
      if (std::fabs(std::sqrt(lu) - std::sqrt(lv)) >= twoR) return false;
      const double nn = std::sqrt(lu * lv);
      M.c = (ux * vx + uy * vy) / nn;
      M.s = (ux * vy - uy * vx) / nn;
      const double mpx = (pax + pbx) * 0.5, mpy = (pay + pby) * 0.5;
      const double mqx = (qax + qbx) * 0.5, mqy = (qay + qby) * 0.5;
      M.tx = mqx - (M.c * mpx - M.s * mpy);
      M.ty = mqy - (M.s * mpx + M.c * mpy);
      return true;
    };

    int32_t nHyp = 0;
    int bestScore = -1;
    int64_t bestH = -1;
    for (int64_t h = 0; h < H; h++) {
      Motion M;
      if (!hypothesis(h, M)) continue;
      nHyp++;
      const int sc = evaluate(M, q, q0, q1, r, r0, r1, r2).score;
      if (sc > bestScore) { bestScore = sc; bestH = h; }
    }
    double* po = pose + 4 * (int64_t)g;
    if (nHyp == 0) {
      po[0] = 1.0; po[1] = 0.0; po[2] = 0.0; po[3] = 0.0;
      rms[g] = 0.0;
      n_inliers[g] = 0;
      n_hypotheses[g] = 0;
      status[g] = 0;
      for (int64_t k = q0; k < q1; k++) assoc[k - base] = -1;
      continue;
    }
    Motion M;
    hypothesis(bestH, M);
    Eval cur = evaluate(M, q, q0, q1, r, r0, r1, r2);
    for (int32_t it = 0; it < refine_iterations; it++) {
      if (cur.score < 2) break;
      const double m = (double)cur.score;
      double spx = 0.0, spy = 0.0, sqx = 0.0, sqy = 0.0;
      for (int64_t k = q0; k < q1; k++) {
        const int64_t j = cur.assoc[(size_t)(k - q0)];
        if (j < 0) continue;
        spx = spx + (double)q[k].x; spy = spy + (double)q[k].y;
        sqx = sqx + (double)r[j].x; sqy = sqy + (double)r[j].y;
      }
      const double mpx = spx / m, mpy = spy / m, mqx = sqx / m, mqy = sqy / m;
      double A = 0.0, B = 0.0;
      for (int64_t k = q0; k < q1; k++) {
        const int64_t j = cur.assoc[(size_t)(k - q0)];
        if (j < 0) continue;
        const double ax = (double)q[k].x - mpx, ay = (double)q[k].y - mpy;
        const double bx = (double)r[j].x - mqx, by = (double)r[j].y - mqy;
        A = A + (ax * bx + ay * by);
        B = B + (ax * by - ay * bx);
      }
      const double n = std::sqrt(A * A + B * B);
      if (n == 0.0) break;
      Motion N;
      N.c = A / n;
      N.s = B / n;
      N.tx = mqx - (N.c * mpx - N.s * mpy);
      N.ty = mqy - (N.s * mpx + N.c * mpy);
      Eval nxt = evaluate(N, q, q0, q1, r, r0, r1, r2);
      if (nxt.score < cur.score) break;
      const bool changed = nxt.assoc != cur.assoc;
      M = N;
      cur = nxt;
      if (!changed) break;
    }
    double sd = 0.0;
    for (int64_t k = q0; k < q1; k++)
      if (cur.assoc[(size_t)(k - q0)] >= 0) sd = sd + cur.d2[(size_t)(k - q0)];
    po[0] = M.c; po[1] = M.s; po[2] = M.tx; po[3] = M.ty;
    rms[g] = cur.score > 0 ? std::sqrt(sd / (double)cur.score) : 0.0;
    n_inliers[g] = cur.score;
    n_hypotheses[g] = nHyp;
    status[g] = cur.score >= min_inliers ? 2 : 1;
    for (int64_t k = q0; k < q1; k++) assoc[k - base] = cur.assoc[(size_t)(k - q0)];
  }
  return 0;
}

}  // extern "C"
