// fe_odometry.cu — odometry over scan sequences (fe_odometry*).  A translation unit of its own, so that the kernels of
// fe_api.cu, fe_match.cu and fe_register.cu compile exactly as they did.
//
// The arithmetic is the contract of include/fe_b200.h ("odometry"): doubles, each operation rounded on its own (the
// library builds with -fmad=false), in the order the contract writes them.
//
// Decomposition.  Steps t = 1, 2, ... run one after the other on the stream, three launches each, with no host round
// trip in between:
//   k_odo_place   a warp per sequence: gathers scan t's rows and remaps their `best` to slot rows, finds the window
//                 from the `source` of the links the earlier steps decided, and writes the placed reference rows;
//   k_register    fe_register.cu's kernel, unchanged, on the step's 2n groups (each slot, then its unused tail);
//   k_odo_update  a warp per sequence: motion, source and pose of scan t, and assoc back to absolute rows (the window is
//                 one contiguous range of absolute rows copied in order, so this is a subtraction).
// One k_odo_init before the first step writes the first scans' results.
#include <cuda_runtime.h>
#include <stdint.h>

#include "fe_odometry.h"

namespace fe_odo {

constexpr int WARPS = 4;  // warps per block, each on its own sequence

using fe_register::Motion;

__device__ __forceinline__ Motion load(const double* m) { return Motion{m[0], m[1], m[2], m[3]}; }

__device__ __forceinline__ void store(double* m, const Motion& a) {
  m[0] = a.c; m[1] = a.s; m[2] = a.tx; m[3] = a.ty;
}

__device__ __forceinline__ Motion inv(const Motion& a) {
  return Motion{a.c, -a.s, -(a.c * a.tx + a.s * a.ty), a.s * a.tx - a.c * a.ty};
}

__device__ __forceinline__ Motion compose(const Motion& a, const Motion& b) {
  return Motion{a.c * b.c - a.s * b.s, a.s * b.c + a.c * b.s, (a.c * b.tx - a.s * b.ty) + a.tx,
                (a.s * b.tx + a.c * b.ty) + a.ty};
}

__global__ void __launch_bounds__(WARPS * 32) k_odo_init(int nSeq, Tables T, Out o) {
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (q >= nSeq) return;
  const int64_t s = T.so[q];
  if (s == T.so[q + 1]) return;  // empty sequence
  const int64_t base = T.ko[0];
  for (int64_t k = T.ko[s] + lane; k < T.ko[s + 1]; k += 32) o.assoc[k - base] = -1;
  if (lane == 0) {
    const Motion id = {1.0, 0.0, 0.0, 0.0};
    store(o.pose + 4 * s, id);
    store(o.motion + 4 * s, id);
    o.rms[s] = 0.0;
    o.source[s] = 0;
    o.status[s] = -1;
    o.nInl[s] = 0;
    o.nHyp[s] = 0;
  }
}

__global__ void __launch_bounds__(WARPS * 32)
k_odo_place(const fe_point_t* __restrict__ kp, int64_t kpBias, const long long* __restrict__ best, Step st, int W,
            Tables T, Work w, Out o) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (i >= st.n) return;
  const Item it = T.items[st.item0 + i];
  const int s = it.scan;
  const int64_t* qo = T.offs + st.offs0;
  int64_t* ro = T.offs + st.offs0 + 2 * st.n + 1;
  const int64_t qDst = qo[2 * i], rDst = ro[2 * i];
  const int64_t* ko = T.ko;

  // window: scan s-1, then earlier scans down to max(first, s-W) while their link was registered
  int m = 1;
  const int lo = s - W > it.first ? s - W : it.first;
  for (int j = s - 2; j >= lo && o.source[j + 1] == 1; j--) m++;
  const int64_t winLo = ko[s - m], prev0 = ko[s - 1], winHi = ko[s];
  if (lane == 0) {
    ro[2 * i + 1] = rDst + (winHi - winLo);
    w.winLo[i] = winLo;
  }

  // query rows and their `best`, as slot rows of scan s-1 (-2 for a bad entry: k_register rejects it as well)
  bool bad = false;
  for (int64_t k = ko[s] + lane; k < ko[s + 1]; k += 32) {
    const int64_t d = qDst + (k - ko[s]);
    w.q[d] = kp[k - kpBias];
    const long long b = best[k - ko[1]];
    const bool ok = b == -1 || (b >= prev0 && b < winHi);
    bad |= !ok;
    w.best[d] = b == -1 ? -1 : ok ? rDst + (b - winLo) : -2;
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(o.err, 1);

  // scan s-1 unchanged; scan j < s-1 by P_j = P_{j+1} o inv(motion_{j+1}), P_{s-2} = inv(motion_{s-1})
  for (int64_t k = prev0 + lane; k < winHi; k += 32) w.r[rDst + (k - winLo)] = kp[k - kpBias];
  Motion P = inv(load(o.motion + 4 * (s - 1)));
  for (int j = s - 2; j >= s - m; j--) {
    if (j < s - 2) P = compose(P, inv(load(o.motion + 4 * (j + 1))));
    for (int64_t k = ko[j] + lane; k < ko[j + 1]; k += 32) {
      fe_point_t p = kp[k - kpBias];
      const double px = (double)p.x, py = (double)p.y;
      p.x = (float)((P.c * px - P.s * py) + P.tx);
      p.y = (float)((P.s * px + P.c * py) + P.ty);
      w.r[rDst + (k - winLo)] = p;
    }
  }
}

__global__ void __launch_bounds__(WARPS * 32) k_odo_update(Step st, Tables T, Work w, Out o) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (i >= st.n) return;
  const Item it = T.items[st.item0 + i];
  const int s = it.scan;
  const int64_t* qo = T.offs + st.offs0;
  const int64_t* ro = qo + 2 * st.n + 1;
  const int64_t qSrc = qo[2 * i], rSrc = ro[2 * i], winLo = w.winLo[i];
  const int64_t k0 = T.ko[s], k1 = T.ko[s + 1], base = T.ko[0];
  for (int64_t k = k0 + lane; k < k1; k += 32) {
    const long long a = w.reg.assoc[qSrc + (k - k0)];
    o.assoc[k - base] = a < 0 ? -1 : winLo + (a - rSrc);
  }
  if (lane == 0) {
    const int g = 2 * i, status = w.reg.status[g];
    Motion M;
    if (status == 2) M = load(w.reg.pose + 4 * g);
    else if (s - it.first == 1) M = Motion{1.0, 0.0, 0.0, 0.0};
    else M = load(o.motion + 4 * (s - 1));
    store(o.motion + 4 * s, M);
    store(o.pose + 4 * s, compose(load(o.pose + 4 * (s - 1)), M));
    o.source[s] = status == 2 ? 1 : 2;
    o.status[s] = status;
    o.rms[s] = w.reg.rms[g];
    o.nInl[s] = w.reg.nInl[g];
    o.nHyp[s] = w.reg.nHyp[g];
  }
}

cudaError_t run(const fe_point_t* kp, int64_t kpBias, const long long* best, int nSeq, int W,
                const std::vector<Step>& steps, Tables T, Work w, Out o, fe_register::Params p, cudaStream_t stream) {
  if (nSeq <= 0) return cudaSuccess;
  k_odo_init<<<(nSeq + WARPS - 1) / WARPS, WARPS * 32, 0, stream>>>(nSeq, T, o);
  cudaError_t e = cudaGetLastError();
  for (const Step& st : steps) {
    if (e != cudaSuccess) return e;
    const int blocks = (st.n + WARPS - 1) / WARPS;
    k_odo_place<<<blocks, WARPS * 32, 0, stream>>>(kp, kpBias, best, st, W, T, w, o);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    const int64_t* qo = T.offs + st.offs0;
    e = fe_register::launch(w.q, 0, w.r, 0, w.best, qo, qo + 2 * st.n + 1, 2 * st.n, p, w.reg, w.scratch, stream);
    if (e != cudaSuccess) return e;
    k_odo_update<<<blocks, WARPS * 32, 0, stream>>>(st, T, w, o);
    e = cudaGetLastError();
  }
  return e;
}

}  // namespace fe_odo
