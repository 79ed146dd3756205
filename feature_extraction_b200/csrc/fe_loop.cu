// fe_loop.cu — loop closures within scan sequences (fe_loop_closures*).  A translation unit of its own, so that the
// kernels of fe_api.cu, fe_match.cu, fe_register.cu and fe_odometry.cu compile exactly as they did.
//
// The contract is include/fe_b200.h ("loop closures").  The call is a fixed chain of launches on the context's stream,
// whatever the sequence length, with no host round trip between retrieval and verification:
//   k_match_tiles (+ k_match_merge)  retrieval: every eligible scan's rows against its database (host-built items)
//   k_loop_vote    a warp per eligible scan: each row's vote, the votes per scan, the top K in contract order
//   k_loop_place   a warp per (scan, candidate) slot: copies scan t's and scan j's keypoints into the slot, writes the
//                  pass-2 items' r0 / nr and the start of the slot's unused tail (registration group 2i + 1)
//   k_match_tiles (+ k_match_merge)  verification matching: scan t against scan j, in place in the descriptor rows
//   k_loop_remap   pass-2 `best` (rows of scan j) -> rows of the slot
//   k_register     fe_register.cu's kernel, unchanged, on the slots
//   k_loop_select  a warp per scan: the candidates' outputs, the choice, and assoc as absolute rows of scan j
#include <cuda_runtime.h>
#include <stdint.h>

#include "fe_loop.h"

namespace fe_loop {

constexpr int WARPS = 4;  // warps per block, each on its own scan or slot
constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ unsigned long long warp_max(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long x = __shfl_xor_sync(FULL, v, o);
    v = x > v ? x : v;
  }
  return v;
}

// One warp per eligible scan.  Row k's vote is the scan j of [first, s - gap] with ko[j] <= best < ko[j + 1] (the
// largest j with ko[j] <= best: empty scans hold no row).  A row's key is (votes of its scan) << 32 | (2^32 - 1 - j),
// unique per scan and ordered as the contract orders candidates; rank c is the largest key below rank c - 1's.
__global__ void __launch_bounds__(WARPS * 32)
k_loop_vote(int E, int K, int gap, Tables T, Work w, Out o) {
  const int lane = threadIdx.x & 31;
  const int e = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (e >= E) return;
  const Scan sc = T.scans[e];
  const int64_t* ko = T.ko;
  const int64_t base = ko[0], k0 = ko[sc.scan], k1 = ko[sc.scan + 1];
  const int hi = sc.scan - gap;
  for (int64_t k = k0 + lane; k < k1; k += 32) {
    const long long b = w.best1[k - base];
    int j = -1;
    if (b >= 0) {
      int lo = sc.first, up = hi;
      while (lo < up) {
        const int m = (lo + up + 1) >> 1;
        if (ko[m] <= b) lo = m;
        else up = m - 1;
      }
      j = lo;
    }
    w.voteScan[k - base] = j;
  }
  __syncwarp();
  for (int64_t k = k0 + lane; k < k1; k += 32) {
    const int j = w.voteScan[k - base];
    unsigned long long kk = 0;
    if (j >= 0) {
      unsigned n = 0;
      for (int64_t x = k0; x < k1; x++) n += w.voteScan[x - base] == j;
      kk = ((unsigned long long)n << 32) | (0xffffffffu - (unsigned)j);
    }
    w.voteKey[k - base] = kk;
  }
  __syncwarp();
  unsigned long long prev = ~0ull;
  for (int c = 0; c < K; c++) {
    unsigned long long m = 0;
    for (int64_t k = k0 + lane; k < k1; k += 32) {
      const unsigned long long kk = w.voteKey[k - base];
      if (kk < prev && kk > m) m = kk;
    }
    m = warp_max(m);
    if (lane == 0) {
      o.cScan[(int64_t)sc.scan * K + c] = m ? (int)(0xffffffffu - (unsigned)m) : -1;
      o.cVotes[(int64_t)sc.scan * K + c] = (int)(m >> 32);
    }
    prev = m;
  }
}

// One warp per slot: the slot's rows, its pass-2 items' reference segments and the start of its unused tail.
__global__ void __launch_bounds__(WARPS * 32)
k_loop_place(const fe_point_t* __restrict__ kp, int64_t kpBias, int nSlots, int K, Tables T, Work w, Out o) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (i >= nSlots) return;
  const Slot sl = T.slots[i];
  const int s = T.scans[i / K].scan;
  const int j = o.cScan[(int64_t)s * K + i % K];
  const int64_t* ko = T.ko;
  const int64_t nq = ko[s + 1] - ko[s], r0 = j >= 0 ? ko[j] : 0, nr = j >= 0 ? ko[j + 1] - ko[j] : 0;
  for (int64_t k = lane; k < nq; k += 32) w.q[sl.q0 + k] = kp[ko[s] + k - kpBias];
  for (int64_t k = lane; k < nr; k += 32) w.r[sl.r0 + k] = kp[r0 + k - kpBias];
  const int64_t n = (int64_t)sl.nseg * sl.tiles;
  for (int64_t x = lane; x < n; x += 32) {
    const int64_t g = x / sl.tiles, left = nr - g * fe_match::ITEM_REFS;
    fe_match::Item& it = T.items[sl.item0 + x];
    it.r0 = r0 + g * fe_match::ITEM_REFS;
    it.nr = (int32_t)(left < 0 ? 0 : left < fe_match::ITEM_REFS ? left : fe_match::ITEM_REFS);
  }
  if (lane == 0) T.ro[2 * i + 1] = sl.r0 + nr;
}

// One warp per slot: pass-2 best, an absolute row of scan j, as a row of the slot.
__global__ void __launch_bounds__(WARPS * 32) k_loop_remap(int nSlots, int K, Tables T, Work w, Out o) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (i >= nSlots) return;
  const Slot sl = T.slots[i];
  const int s = T.scans[i / K].scan;
  const int j = o.cScan[(int64_t)s * K + i % K];
  const int64_t nq = T.ko[s + 1] - T.ko[s], r0 = j >= 0 ? T.ko[j] : 0;
  for (int64_t k = lane; k < nq; k += 32) {
    const long long b = w.best2[sl.q0 + k];
    w.slotBest[sl.q0 + k] = b < 0 ? -1 : sl.r0 + (b - r0);
  }
}

// One warp per scan: lane k < K reads candidate k's registration, the warp picks the loop (status 2, most inliers,
// lowest rank: the largest n_inliers << 5 | (31 - k)), and the lanes write assoc under it.
__global__ void __launch_bounds__(WARPS * 32) k_loop_select(int B, int K, Tables T, Work w, Out o) {
  const int lane = threadIdx.x & 31;
  const int s = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (s >= B) return;
  const int e = T.elig[s];
  const int64_t c = (int64_t)s * K + lane;
  unsigned long long key = 0;
  if (lane < K) {
    const int j = e >= 0 ? o.cScan[c] : -1;
    double p[4] = {1.0, 0.0, 0.0, 0.0}, rms = 0.0;
    int st = -1, inl = 0, hyp = 0;
    if (j >= 0) {
      const int g = 2 * (e * K + lane);
      for (int x = 0; x < 4; x++) p[x] = w.reg.pose[4 * g + x];
      rms = w.reg.rms[g];
      st = w.reg.status[g];
      inl = w.reg.nInl[g];
      hyp = w.reg.nHyp[g];
    } else {
      o.cScan[c] = -1;
      o.cVotes[c] = 0;
    }
    for (int x = 0; x < 4; x++) o.cPose[4 * c + x] = p[x];
    o.cRms[c] = rms;
    o.cStatus[c] = st;
    o.cInl[c] = inl;
    o.cHyp[c] = hyp;
    if (st == 2) key = ((unsigned long long)(unsigned)inl << 5 | (unsigned)(31 - lane)) + 1;
  }
  key = warp_max(key);
  const int win = key ? 31 - (int)((key - 1) & 31) : -1;
  const int64_t base = T.ko[0], k0 = T.ko[s], k1 = T.ko[s + 1];
  if (win < 0) {
    for (int64_t k = k0 + lane; k < k1; k += 32) o.assoc[k - base] = -1;
    if (lane == 0) {
      o.loop[s] = -1;
      o.loopScan[s] = -1;
      o.pose[4 * s] = 1.0; o.pose[4 * s + 1] = 0.0; o.pose[4 * s + 2] = 0.0; o.pose[4 * s + 3] = 0.0;
      o.rms[s] = 0.0;
      o.nInl[s] = 0;
      o.nHyp[s] = 0;
    }
    return;
  }
  const int i = e * K + win, g = 2 * i;
  const int j = o.cScan[(int64_t)s * K + win];
  const Slot sl = T.slots[i];
  const int64_t r0 = T.ko[j];
  for (int64_t k = k0 + lane; k < k1; k += 32) {
    const long long a = w.reg.assoc[sl.q0 + (k - k0)];
    o.assoc[k - base] = a < 0 ? -1 : r0 + (a - sl.r0);
  }
  if (lane == 0) {
    o.loop[s] = win;
    o.loopScan[s] = j;
    for (int x = 0; x < 4; x++) o.pose[4 * s + x] = w.reg.pose[4 * g + x];
    o.rms[s] = w.reg.rms[g];
    o.nInl[s] = w.reg.nInl[g];
    o.nHyp[s] = w.reg.nHyp[g];
  }
}

cudaError_t vote(int E, int K, int gap, Tables T, Work w, Out o, cudaStream_t stream) {
  if (E <= 0) return cudaSuccess;
  k_loop_vote<<<(E + WARPS - 1) / WARPS, WARPS * 32, 0, stream>>>(E, K, gap, T, w, o);
  return cudaGetLastError();
}

cudaError_t place(const fe_point_t* kp, int64_t kpBias, int nSlots, int K, Tables T, Work w, Out o, cudaStream_t stream) {
  if (nSlots <= 0) return cudaSuccess;
  k_loop_place<<<(nSlots + WARPS - 1) / WARPS, WARPS * 32, 0, stream>>>(kp, kpBias, nSlots, K, T, w, o);
  return cudaGetLastError();
}

cudaError_t remap(int nSlots, int K, Tables T, Work w, Out o, cudaStream_t stream) {
  if (nSlots <= 0) return cudaSuccess;
  k_loop_remap<<<(nSlots + WARPS - 1) / WARPS, WARPS * 32, 0, stream>>>(nSlots, K, T, w, o);
  return cudaGetLastError();
}

cudaError_t select(int B, int K, Tables T, Work w, Out o, cudaStream_t stream) {
  if (B <= 0) return cudaSuccess;
  k_loop_select<<<(B + WARPS - 1) / WARPS, WARPS * 32, 0, stream>>>(B, K, T, w, o);
  return cudaGetLastError();
}

}  // namespace fe_loop
