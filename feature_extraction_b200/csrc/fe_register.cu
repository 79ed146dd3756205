// fe_register.cu — planar registration of matched keypoints (fe_register_matches*).  A translation unit of its own, so
// that the pipeline's kernels in fe_api.cu and the matcher's in fe_match.cu compile exactly as they did.
//
// The arithmetic is the contract of include/fe_b200.h ("registration"): doubles, each operation rounded on its own
// (the library builds with -fmad=false), in the order the contract writes them.
//
// Decomposition.  One warp owns one group.  It checks the group's `best` entries and compacts its correspondences with
// ballots, then each lane takes hypotheses h = lane, lane + 32, ... and scores each against every (query, reference)
// pair of the group; the warp keeps the maximum of the key (score + 1) << 32 | (2^32 - 1 - h), i.e. the highest
// score, then the lowest h (0: nothing survived).  The winner's motion is recomputed by every lane and evaluated with
// lanes over query rows.  Refinement needs its sums in ascending query row, so lane 0 forms them alone: O(inliers) per
// round, against O(n_q * n_r) for the evaluation the lanes share.  Positions are read from global memory (L1): all
// lanes of the warp read the same reference row at the same time.
#include <cuda_runtime.h>
#include <stdint.h>

#include "fe_register.h"

namespace fe_register {

constexpr int WARPS = 4;  // warps per block (independent: each runs its own group)
constexpr unsigned FULL = 0xffffffffu;

struct Motion {
  double c, s, tx, ty;
};

// row i of an array whose first element is row `bias`
__device__ __forceinline__ void xy(const fe_point_t* p, int64_t bias, int64_t i, double& x, double& y) {
  x = (double)__ldg(&p[i - bias].x);
  y = (double)__ldg(&p[i - bias].y);
}

// Nearest reference row of [r0, r1) within the radius to the query position (px, py) mapped by M: -1 if none.
__device__ __forceinline__ long long associate(const Motion& M, double px, double py, const fe_point_t* r, int64_t rBias,
                                               int64_t r0, int64_t r1, double r2, double& d2out) {
  const double wx = (M.c * px - M.s * py) + M.tx, wy = (M.s * px + M.c * py) + M.ty;
  double cur = r2;
  long long jj = -1;
  for (int64_t j = r0; j < r1; j++) {
    double rx, ry;
    xy(r, rBias, j, rx, ry);
    const double dx = wx - rx, dy = wy - ry;
    const double d2 = dx * dx + dy * dy;
    if (d2 < cur) { cur = d2; jj = j; }
  }
  d2out = cur;
  return jj;
}

__global__ void __launch_bounds__(WARPS * 32)
k_register(const fe_point_t* __restrict__ q, int64_t qBias, const fe_point_t* __restrict__ r, int64_t rBias,
           const long long* __restrict__ best, const int64_t* __restrict__ qo, const int64_t* __restrict__ ro, int G,
           Params P, Out o, Scratch S) {
  const int lane = threadIdx.x & 31;
  const int g = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (g >= G) return;
  const int64_t base = qo[0];
  const int64_t q0 = qo[g], q1 = qo[g + 1], r0 = ro[g], r1 = ro[g + 1];
  const int64_t gi = q0 - base;  // the group's first query row in the per-row arrays

  // check `best`, and list the correspondences in ascending row order
  bool bad = false;
  int nc = 0;
  for (int64_t k0 = q0; k0 < q1; k0 += 32) {
    const int64_t k = k0 + lane;
    long long b = -1;
    if (k < q1) {
      b = best[k - base];
      bad |= b != -1 && (b < r0 || b >= r1);
    }
    const unsigned m = __ballot_sync(FULL, k < q1 && b >= 0);
    if (k < q1 && b >= 0) S.corr[gi + nc + __popc(m & ((1u << lane) - 1u))] = (int)(k - base);
    nc += __popc(m);
  }
  if (__any_sync(FULL, bad)) {
    if (lane == 0) atomicOr(o.err, 1);
    return;
  }
  __syncwarp();

  const int64_t nP = (int64_t)nc * (nc - 1) / 2;
  const int64_t H = nP < P.maxH ? nP : P.maxH;
  auto hypothesis = [&](int64_t h, Motion& M) {
    int64_t idx = h * nP / H, a = 0;
    while (idx >= nc - 1 - a) { idx -= nc - 1 - a; a++; }
    const int64_t ka = (int64_t)S.corr[gi + a] + base, kb = (int64_t)S.corr[gi + a + 1 + idx] + base;
    const long long ja = best[ka - base], jb = best[kb - base];
    double pax, pay, pbx, pby, qax, qay, qbx, qby;
    xy(q, qBias, ka, pax, pay);
    xy(q, qBias, kb, pbx, pby);
    xy(r, rBias, ja, qax, qay);
    xy(r, rBias, jb, qbx, qby);
    const double ux = pbx - pax, uy = pby - pay, vx = qbx - qax, vy = qby - qay;
    const double lu = ux * ux + uy * uy, lv = vx * vx + vy * vy;
    if (lu < P.sep2 || lv < P.sep2) return false;
    if (fabs(sqrt(lu) - sqrt(lv)) >= P.twoR) return false;
    const double nn = sqrt(lu * lv);
    M.c = (ux * vx + uy * vy) / nn;
    M.s = (ux * vy - uy * vx) / nn;
    const double mpx = (pax + pbx) * 0.5, mpy = (pay + pby) * 0.5;
    const double mqx = (qax + qbx) * 0.5, mqy = (qay + qby) * 0.5;
    M.tx = mqx - (M.c * mpx - M.s * mpy);
    M.ty = mqy - (M.s * mpx + M.c * mpy);
    return true;
  };

  unsigned long long key = 0;
  int nHyp = 0;
  for (int64_t h = lane; h < H; h += 32) {
    Motion M;
    if (!hypothesis(h, M)) continue;
    nHyp++;
    unsigned long long score = 0;
    for (int64_t k = q0; k < q1; k++) {
      double px, py, d2;
      xy(q, qBias, k, px, py);
      score += associate(M, px, py, r, rBias, r0, r1, P.r2, d2) >= 0;
    }
    const unsigned long long kk = ((score + 1) << 32) | (0xffffffffull - (unsigned long long)h);
    key = kk > key ? kk : key;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const unsigned long long ok = __shfl_xor_sync(FULL, key, off);
    key = ok > key ? ok : key;
    nHyp += __shfl_xor_sync(FULL, nHyp, off);
  }

  if (key == 0) {  // no hypothesis survived
    for (int64_t k = q0 + lane; k < q1; k += 32) o.assoc[k - base] = -1;
    if (lane == 0) {
      o.pose[4 * g] = 1.0; o.pose[4 * g + 1] = 0.0; o.pose[4 * g + 2] = 0.0; o.pose[4 * g + 3] = 0.0;
      o.rms[g] = 0.0;
      o.nInl[g] = 0;
      o.nHyp[g] = 0;
      o.status[g] = 0;
    }
    return;
  }

  // evaluate M into (assoc, d2) with lanes over query rows; -> score; *changed: some assoc differs from `cmp`
  auto evaluate = [&](const Motion& M, long long* assoc, double* d2s, const long long* cmp, bool* changed) {
    int cnt = 0;
    bool ch = false;
    for (int64_t k = q0 + lane; k < q1; k += 32) {
      double px, py, d2;
      xy(q, qBias, k, px, py);
      const long long j = associate(M, px, py, r, rBias, r0, r1, P.r2, d2);
      assoc[k - base] = j;
      d2s[k - base] = d2;
      cnt += j >= 0;
      if (cmp) ch |= cmp[k - base] != j;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) cnt += __shfl_xor_sync(FULL, cnt, off);
    if (changed) *changed = __any_sync(FULL, ch);
    __syncwarp();  // the per-row arrays are read by other lanes next
    return cnt;
  };

  Motion M;
  hypothesis((int64_t)(0xffffffffull - (key & 0xffffffffull)), M);
  int score = evaluate(M, o.assoc, S.d2Cur, nullptr, nullptr);
  for (int it = 0; it < P.refine; it++) {
    if (score < 2) break;
    Motion N = {0.0, 0.0, 0.0, 0.0};
    double n = 0.0;
    if (lane == 0) {  // the contract's sums run in ascending row order
      const double m = (double)score;
      double spx = 0.0, spy = 0.0, sqx = 0.0, sqy = 0.0;
      for (int64_t k = q0; k < q1; k++) {
        const long long j = o.assoc[k - base];
        if (j < 0) continue;
        double px, py, rx, ry;
        xy(q, qBias, k, px, py);
        xy(r, rBias, j, rx, ry);
        spx = spx + px; spy = spy + py;
        sqx = sqx + rx; sqy = sqy + ry;
      }
      const double mpx = spx / m, mpy = spy / m, mqx = sqx / m, mqy = sqy / m;
      double A = 0.0, B = 0.0;
      for (int64_t k = q0; k < q1; k++) {
        const long long j = o.assoc[k - base];
        if (j < 0) continue;
        double px, py, rx, ry;
        xy(q, qBias, k, px, py);
        xy(r, rBias, j, rx, ry);
        const double ax = px - mpx, ay = py - mpy, bx = rx - mqx, by = ry - mqy;
        A = A + (ax * bx + ay * by);
        B = B + (ax * by - ay * bx);
      }
      n = sqrt(A * A + B * B);
      if (n != 0.0) {
        N.c = A / n;
        N.s = B / n;
        N.tx = mqx - (N.c * mpx - N.s * mpy);
        N.ty = mqy - (N.s * mpx + N.c * mpy);
      }
    }
    n = __shfl_sync(FULL, n, 0);
    if (n == 0.0) break;
    N.c = __shfl_sync(FULL, N.c, 0);
    N.s = __shfl_sync(FULL, N.s, 0);
    N.tx = __shfl_sync(FULL, N.tx, 0);
    N.ty = __shfl_sync(FULL, N.ty, 0);
    bool changed;
    const int sc = evaluate(N, S.assocNew, S.d2New, o.assoc, &changed);
    if (sc < score) break;
    M = N;
    score = sc;
    for (int64_t k = q0 + lane; k < q1; k += 32) {
      o.assoc[k - base] = S.assocNew[k - base];
      S.d2Cur[k - base] = S.d2New[k - base];
    }
    __syncwarp();
    if (!changed) break;
  }
  if (lane == 0) {
    double sd = 0.0;
    for (int64_t k = q0; k < q1; k++)
      if (o.assoc[k - base] >= 0) sd = sd + S.d2Cur[k - base];
    o.pose[4 * g] = M.c; o.pose[4 * g + 1] = M.s; o.pose[4 * g + 2] = M.tx; o.pose[4 * g + 3] = M.ty;
    o.rms[g] = score > 0 ? sqrt(sd / (double)score) : 0.0;
    o.nInl[g] = score;
    o.nHyp[g] = nHyp;
    o.status[g] = score >= P.minInliers ? 2 : 1;
  }
}

cudaError_t launch(const fe_point_t* q, int64_t qBias, const fe_point_t* r, int64_t rBias, const long long* best,
                   const int64_t* d_qo, const int64_t* d_ro, int nGroups, Params p, Out o, Scratch s, cudaStream_t stream) {
  if (nGroups <= 0) return cudaSuccess;
  k_register<<<(nGroups + WARPS - 1) / WARPS, WARPS * 32, 0, stream>>>(q, qBias, r, rBias, best, d_qo, d_ro, nGroups, p, o, s);
  return cudaGetLastError();
}

}  // namespace fe_register
