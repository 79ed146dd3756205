// fe_ring_runs.cuh — K2, the per-ring EuclideanClusterExtraction + getCylinderSegments gate of
// reference src:261-327, built around the structure of a lidar ring instead of a general grid.
//
// A ring's returns arrive in firing (azimuth) order, so consecutive returns on one surface are
// closer than the cluster tolerance: one linear sweep d2(e-1, e) < r2f cuts the ring into RUNS, each
// of which lies inside one connected component of the radius graph {d2 < r2f}.  What is left is to find
// the links BETWEEN runs: run pairs whose xy bounding boxes come within the tolerance are tested point
// against point (the larger run first pruned against the smaller run's box), stopping at the first
// link, and joined in a union-find over runs.  Components of runs = PCL's clusters, exactly: every
// accept/reject is the same float predicate (FLANN L2_Simple, unfused), boxes only pre-select with slack.
// A run's first entry is its smallest entry, so a component's root (smallest run) gives PCL's discovery
// order and indices[0]; sizes are sums of run lengths; members ascend run by run.
//
// Work layout: one block of NT_RR threads per scan.  Phase A buckets the scan's crop survivors by ring
// (stable) into a global scratch slot of the scan — L2-resident, any size, no shared-memory capacity
// chain.  Phase B: every warp takes rings off a block-wide counter and does sweep, run links, size gate,
// PCL's cluster order (sort_replay.h), the xy-diagonal gate and the double centroid sums all by itself:
// no block barrier after phase A.  Input in arbitrary order still gives the exact result (runs of one
// entry); when a ring has more than RW runs the scan is handed to the grid-based kernels of
// fe_kernels.cuh (k_cluster_rings), which remain the general fallback and the cross-check.
#pragma once

namespace fe {

constexpr int NT_RR = 128;       // threads per scan block (4 warps)
constexpr int NW_RR = NT_RR / 32;
constexpr int RW = 128;          // runs of one ring a warp of the first kernel keeps in shared memory (7 KB per warp: 12+ blocks / SM)
constexpr int RW2 = 256;         // ... of the second kernel, which takes the scans with a ring beyond RW (hundreds of poles in one ring)

template <int RWT>
struct RunBufT {                 // one per warp, shared memory
  float minx[RWT], maxx[RWT], miny[RWT], maxy[RWT];  // xy box of every run
  int start[RWT + 1];            // first entry of every run (start[R] = n)
  int csize[RWT];                // at a root: entries of the component
  unsigned short parent[RWT];    // union-find over runs, root = smallest run
  unsigned short list[RWT];      // kept clusters (root runs) in output order
  static constexpr int cap = RWT;
};

constexpr int NW_RR_SMALL = 16;  // warps per scan block when a call holds only a handful of scans: a warp per ring at once

template <int RWT, int NW = NW_RR>
struct RingRunsSmT {
  int pre[MAXCHUNK + 1];
  int sc[40];
  int cnt[NW][17];               // phase A: entries per (warp, ring); [16] = entries in no ring
  int ringBase[18];
  int nextRing;
  int defer;
  RunBufT<RWT> rb[NW];
};

__device__ __forceinline__ int f2ord(float f) {  // monotone float -> int
  const int i = __float_as_int(f);
  return i ^ ((i >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }

// ring membership of a crop survivor: K1's code = first ring | 16 (also the next ring) | 32 (no ring)
__device__ __forceinline__ unsigned ring_mask_of(unsigned cd, int single_ring) {
  if (cd & 32u) return 0u;
  if (single_ring) return 1u;
  const unsigned r = cd & 15u;
  return (1u << r) | ((cd & 16u) ? (1u << (r + 1)) : 0u);
}

// Every lane of the warp walks the same chain (read-only: links are only ever written by lane 0 between
// __syncwarp()s, and a root is the smallest run of its set, so chains are short).
__device__ __forceinline__ unsigned rr_find(const unsigned short* parent, unsigned x) {
  unsigned p = parent[x];
  while (p != x) { x = p; p = parent[x]; }
  return x;
}

// Is any entry of run a within the tolerance of any entry of run b?  Warp-uniform.
template <class RB>
__device__ bool rr_runs_linked(const RB& B, const float4* P, int a, int b, float r2f, float r2box) {
  const int lane = threadIdx.x & 31;
  int big = a, small = b;
  if (B.start[b + 1] - B.start[b] > B.start[a + 1] - B.start[a]) { big = b; small = a; }
  const float bx0 = B.minx[small], bx1 = B.maxx[small], by0 = B.miny[small], by1 = B.maxy[small];
  const int s0 = B.start[small], s1 = B.start[small + 1];
  const int e1 = B.start[big + 1];
  for (int i0 = B.start[big]; i0 < e1; i0 += 32) {
    const int i = i0 + lane;
    bool near = false;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < e1) {
      p = P[i];
      const float dx = fmaxf(0.0f, fmaxf(bx0 - p.x, p.x - bx1)), dy = fmaxf(0.0f, fmaxf(by0 - p.y, p.y - by1));
      near = dx * dx + dy * dy <= r2box;
    }
    unsigned nm = __ballot_sync(FE_FULL, near);
    while (nm) {
      const int src = __ffs(nm) - 1;
      nm &= nm - 1;
      const float px = __shfl_sync(FE_FULL, p.x, src), py = __shfl_sync(FE_FULL, p.y, src), pz = __shfl_sync(FE_FULL, p.z, src);
      for (int j0 = s0; j0 < s1; j0 += 32) {
        const int j = j0 + lane;
        bool hit = false;
        if (j < s1) {
          const float4 q = P[j];
          hit = l2_simple(px, py, pz, q.x, q.y, q.z) < r2f;
        }
        if (__ballot_sync(FE_FULL, hit)) return true;
      }
    }
  }
  return false;
}

// (P is the block's own scratch, written in phase A of the same kernel: plain pointers, no read-only path.)
// One ring: entries P[0, n) in original order.  Returns false when the ring has more runs than the buffer
// holds (nothing has been written then).  Warp-uniform; all 32 lanes call.
// gate...: nothing, or a GateCount whose cnt is the ring's slot of the kind-6 count.
template <class RB, class... G>
__device__ bool rr_cluster_ring(RB& B, const float4* P, const int n, const DevParams& Pm,
                                float4* __restrict__ kfPool, int kfCap, int* __restrict__ kfBaseOut, int* __restrict__ kfCntOut,
                                float4* __restrict__ kcPool, int kcCap, int* __restrict__ kcBaseOut, int* __restrict__ kcCntOut,
                                DevCounters* __restrict__ ctr, G... gate) {
  const int lane = threadIdx.x & 31;
  const unsigned le = lanemask_lt() | (1u << lane);
  const float r2f = Pm.r2f_cluster;
  const float r2box = r2f * 1.0001f + 1e-12f;  // boxes pre-select with slack; links are decided by r2f alone
  const int minSz = Pm.min_count, maxSz = Pm.max_count;
  // ---- sweep: runs and their boxes ----
  int R = 0;
  float cx = 0.f, cy = 0.f, cz = 0.f;  // last entry of the previous 32
  for (int e0 = 0; e0 < n; e0 += 32) {
    const int e = e0 + lane;
    const bool valid = e < n;
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) q = P[e];
    float ux = __shfl_up_sync(FE_FULL, q.x, 1), uy = __shfl_up_sync(FE_FULL, q.y, 1), uz = __shfl_up_sync(FE_FULL, q.z, 1);
    if (lane == 0) { ux = cx; uy = cy; uz = cz; }
    const bool head = valid && (e == 0 || !(l2_simple(ux, uy, uz, q.x, q.y, q.z) < r2f));
    const unsigned hm = __ballot_sync(FE_FULL, head);
    const int nv = min(32, n - e0);
    if (R + __popc(hm) > B.cap) return false;
    if (valid) {
      const unsigned below = hm & le;                      // heads at or below this lane
      const int segStart = below ? 31 - __clz(below) : 0;  // none: the run continues from the previous 32
      const unsigned above = hm & ~le;
      const int segEnd = above ? __ffs(above) - 1 : nv;    // exclusive
      const unsigned segMask = ((segEnd >= 32) ? 0xffffffffu : ((1u << segEnd) - 1u)) & ~((1u << segStart) - 1u);
      const int mnx = __reduce_min_sync(segMask, f2ord(q.x)), mxx = __reduce_max_sync(segMask, f2ord(q.x));
      const int mny = __reduce_min_sync(segMask, f2ord(q.y)), mxy = __reduce_max_sync(segMask, f2ord(q.y));
      if (lane == segStart) {
        const int r = R + __popc(below) - 1;
        if (below) {  // a run starts here
          B.minx[r] = ord2f(mnx); B.maxx[r] = ord2f(mxx); B.miny[r] = ord2f(mny); B.maxy[r] = ord2f(mxy);
          B.start[r] = e;
        } else {
          B.minx[r] = fminf(B.minx[r], ord2f(mnx)); B.maxx[r] = fmaxf(B.maxx[r], ord2f(mxx));
          B.miny[r] = fminf(B.miny[r], ord2f(mny)); B.maxy[r] = fmaxf(B.maxy[r], ord2f(mxy));
        }
      }
    }
    R += __popc(hm);
    cx = __shfl_sync(FE_FULL, q.x, 31); cy = __shfl_sync(FE_FULL, q.y, 31); cz = __shfl_sync(FE_FULL, q.z, 31);
    __syncwarp();  // the run records written here are read (lane 0 extends a run) in the next round
  }
  if (lane == 0) B.start[R] = n;
  __syncwarp();
  for (int r = lane; r < R; r += 32) { B.parent[r] = (unsigned short)r; B.csize[r] = B.start[r + 1] - B.start[r]; }
  __syncwarp();
  // ---- links between runs ----
  for (int a = 0; a + 1 < R; a++) {
    const float ax0 = B.minx[a], ax1 = B.maxx[a], ay0 = B.miny[a], ay1 = B.maxy[a];
    for (int b0 = a + 1; b0 < R; b0 += 32) {
      const int b = b0 + lane;
      bool cand = false;
      if (b < R) {
        const float dx = fmaxf(0.0f, fmaxf(ax0 - B.maxx[b], B.minx[b] - ax1)), dy = fmaxf(0.0f, fmaxf(ay0 - B.maxy[b], B.miny[b] - ay1));
        cand = dx * dx + dy * dy <= r2box;
      }
      unsigned cm = __ballot_sync(FE_FULL, cand);
      while (cm) {
        const int bb = b0 + __ffs(cm) - 1;
        cm &= cm - 1;
        const unsigned ra = rr_find(B.parent, (unsigned)a), rb = rr_find(B.parent, (unsigned)bb);
        if (ra == rb) continue;
        if (B.csize[ra] > maxSz && B.csize[rb] > maxSz) continue;  // both components are already dropped whole
        if (rr_runs_linked(B, P, a, bb, r2f, r2box)) {
          __syncwarp();
          if (lane == 0) {
            const unsigned lo = min(ra, rb), hi = max(ra, rb);
            B.parent[hi] = (unsigned short)lo;
            B.csize[lo] += B.csize[hi];
          }
          __syncwarp();
        }
      }
    }
  }
  __syncwarp();
  // ---- flatten (through `list`, free until the clusters are listed); clusters that pass the size gate in
  //      discovery order (ascending root) ----
  for (int r = lane; r < R; r += 32) {
    unsigned x = (unsigned)r, p = B.parent[x];
    while (p != x) { x = p; p = B.parent[x]; }
    B.list[r] = (unsigned short)x;
  }
  __syncwarp();
  for (int r = lane; r < R; r += 32) B.parent[r] = B.list[r];
  __syncwarp();
  int nC = 0;
  for (int r0 = 0; r0 < R; r0 += 32) {
    const int r = r0 + lane;
    const bool keep = r < R && B.parent[r] == r && B.csize[r] >= minSz && B.csize[r] <= maxSz;
    const unsigned km = __ballot_sync(FE_FULL, keep);
    if (keep) B.list[nC + __popc(km & lanemask_lt())] = (unsigned short)r;
    nC += __popc(km);
  }
  __syncwarp();
  if (nC == 0) return true;  // (all lanes are past their last read of the run buffer: the __syncwarp above)
  // ---- PCL's final std::sort(rbegin, rend, size<) ----
  if (nC > 1 && lane == 0) {
    const int* cs = B.csize;
    unsigned short* lst = B.list;
    pcl_cluster_order(lst, nC, [=](unsigned short id) { return cs[id]; });
  }
  __syncwarp();
  // ---- getCylinderSegments gate (src:282-325): xy box diagonal of the cluster, strict < 2*threshold ----
  // pass 0 gates every cluster on the union of its runs' boxes (min / max do not depend on the order; the
  // +-1000 initial values of src:289-290 are kept) and counts; pass 1 sums the survivors' members in
  // ascending order, in double, like the reference loop.
  int nOk = 0, nMem = 0;
  for (int i0 = 0; i0 < nC; i0 += 32) {
    const int i = i0 + lane;
    bool ok = false;
    int size = 0;
    if (i < nC) {
      const int root = B.list[i];
      size = B.csize[root];
      double minx = 1000.0, maxx = -1000.0, miny = 1000.0, maxy = -1000.0;
      int left = size;
      for (int r = root; r < R && left > 0; r++) {
        if (B.parent[r] != root) continue;
        left -= B.start[r + 1] - B.start[r];
        const double x0 = B.minx[r], x1 = B.maxx[r], y0 = B.miny[r], y1 = B.maxy[r];
        if (x0 < minx) minx = x0;
        if (y0 < miny) miny = y0;
        if (x1 > maxx) maxx = x1;
        if (y1 > maxy) maxy = y1;
      }
      const double ddx = maxx - minx, ddy = maxy - miny;
      const double diameter = sqrt(__dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy)));  // src:314
      ok = diameter < Pm.two_radius_threshold;
      if constexpr (sizeof...(G) > 0) if (fabs(diameter - Pm.two_radius_threshold) < (gate.eps, ...)) atomicAdd((gate.cnt, ...), 1u);
    }
    const unsigned om = __ballot_sync(FE_FULL, ok);
    // the flag travels in the sign of csize (sizes are > 0)
    if (ok) B.csize[B.list[i]] = -size;
    nOk += __popc(om);
    if (kcPool) {
      int v = ok ? size : 0;
#pragma unroll
      for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(FE_FULL, v, d);
      nMem += v;
    }
  }
  __syncwarp();
  if (nOk == 0) return true;
  int base = 0, kbase = 0;
  if (lane == 0) {
    base = atomicAdd(&ctr->kf_cursor, nOk);
    if (base + nOk > kfCap) { atomicOr(&ctr->err, ERR_KF_POOL); base = -1; }
    if (kcPool) {
      kbase = atomicAdd(&ctr->kc_cursor, nMem);
      if (kbase + nMem > kcCap) { atomicOr(&ctr->err, ERR_KC_POOL); kbase = -1; }
    }
    *kfBaseOut = max(base, 0);
    *kfCntOut = base >= 0 ? nOk : 0;
    if (kcBaseOut) { *kcBaseOut = max(kbase, 0); *kcCntOut = kbase >= 0 ? nMem : 0; }
  }
  base = __shfl_sync(FE_FULL, base, 0);
  kbase = __shfl_sync(FE_FULL, kbase, 0);
  int doneOk = 0, doneMem = 0;
  for (int i0 = 0; i0 < nC; i0 += 32) {
    const int i = i0 + lane;
    bool ok = false;
    int size = 0, root = 0;
    if (i < nC) { root = B.list[i]; size = B.csize[root]; ok = size < 0; size = abs(size); }
    const unsigned om = __ballot_sync(FE_FULL, ok);
    int memBefore = 0;  // members of the ok clusters of lower lanes
    if (kcPool) {
      int inc = ok ? size : 0;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(FE_FULL, inc, d); if (lane >= d) inc += t; }
      memBefore = inc - (ok ? size : 0);
      const int tot = __shfl_sync(FE_FULL, inc, 31);
      if (ok && kbase >= 0) {
        int o = kbase + doneMem + memBefore, left = size;
        for (int r = root; r < R && left > 0; r++) {
          if (B.parent[r] != root) continue;
          for (int e = B.start[r]; e < B.start[r + 1]; e++) kcPool[o++] = P[e];
          left -= B.start[r + 1] - B.start[r];
        }
      }
      doneMem += tot;
    }
    if (ok && base >= 0) {
      double sumx = 0.0, sumy = 0.0, sumz = 0.0;
      int left = size;
      for (int r = root; r < R && left > 0; r++) {
        if (B.parent[r] != root) continue;
        for (int e = B.start[r]; e < B.start[r + 1]; e++) {
          const float4 q = P[e];
          sumx += (double)q.x; sumy += (double)q.y; sumz += (double)q.z;
        }
        left -= B.start[r + 1] - B.start[r];
      }
      float4 cen;
      cen.x = (float)(sumx / (double)size);
      cen.y = (float)(sumy / (double)size);
      cen.z = (float)(sumz / (double)size);
      cen.w = P[B.start[root]].w;  // intensity of indices[0] (src:320)
      kfPool[base + doneOk + __popc(om & lanemask_lt())] = cen;
    }
    doneOk += __popc(om);
  }
  __syncwarp();  // the next ring reuses the run buffer
  return true;
}

// Phase B for one scan whose ring segments [ringBase[r], ringBase[r+1]) are in place at RP: the warps take rings
// off the block's counter.  A ring with more runs than a warp's buffer holds is listed for the wide kernel (its
// outputs are untouched); the other rings of the scan are finished here.
template <int RWT, int NW, class... G>
__device__ void rr_scan_rings(RingRunsSmT<RWT, NW>& S, const int s, const float4* RP, const int nRings, const DevParams& P,
                              float4* __restrict__ kfPool, int kfCap, int* __restrict__ kfBase, int* __restrict__ kfCnt,
                              float4* __restrict__ kcPool, int kcCap, int* __restrict__ kcBase, int* __restrict__ kcCnt,
                              DevCounters* __restrict__ ctr, int* __restrict__ ovfRuns, int* __restrict__ ovfRunsCount,
                              G... gate) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  RunBufT<RWT>& B = S.rb[w];
  for (;;) {
    int ring = 0;
    if (lane == 0) ring = atomicAdd(&S.nextRing, 1);
    ring = __shfl_sync(FE_FULL, ring, 0);
    if (ring >= nRings) break;
    const int r0 = S.ringBase[ring], n = S.ringBase[ring + 1] - r0;
    if (n == 0) continue;
    const bool done = rr_cluster_ring(B, RP + r0, n, P, kfPool, kfCap, &kfBase[s * 16 + ring], &kfCnt[s * 16 + ring], kcPool, kcCap,
                                      kcBase ? &kcBase[s * 16 + ring] : nullptr, kcBase ? &kcCnt[s * 16 + ring] : nullptr, ctr,
                                      gate.at(s * 16 + ring)...);
    if (!done && lane == 0) ovfRuns[atomicAdd(ovfRunsCount, 1)] = s * 16 + ring;
  }
}

// First kernel: one block per scan, every scan.  A ring of more than RW runs is handed to the second kernel (the
// ring segments and their offsets stay in global memory, so nothing is bucketed twice); a scan with more ring
// entries than its scratch slot goes straight to the grid-based kernels.
// gate...: nothing, or the GateCount of the boundary report's kind 6 (zeroed here for the scan's 16 rings).
template <int NW, class... G>
__global__ void __launch_bounds__(NW * 32, NW == NW_RR ? 12 : 1) k_ring_runs(
    const float4* __restrict__ crop, const unsigned* __restrict__ cropMeta, const int* __restrict__ cropCnt,
    const long long* __restrict__ scan_off, const int* __restrict__ chunk_off, DevParams P, int single_ring,
    float4* ringPts, int* __restrict__ ringBaseOut, float4* __restrict__ kfPool, int kfCap, int* __restrict__ kfBase, int* __restrict__ kfCnt,
    float4* __restrict__ kcPool, int kcCap, int* __restrict__ kcBase, int* __restrict__ kcCnt,
    DevCounters* __restrict__ ctr, int* __restrict__ ovfRuns, int* __restrict__ ovfRunsCount, int* __restrict__ scanFlag,
    int* __restrict__ ovfList, int* __restrict__ ovfCount, G... gate) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  RingRunsSmT<RW, NW>& S = *reinterpret_cast<RingRunsSmT<RW, NW>*>(smem_raw);
  const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const long long base = scan_off[s];
  const int nScan = (int)(scan_off[s + 1] - base);
  const int nch = chunk_off[s + 1] - chunk_off[s];
  if (tid < 16) { kfBase[s * 16 + tid] = 0; kfCnt[s * 16 + tid] = 0; if (kcBase) { kcBase[s * 16 + tid] = 0; kcCnt[s * 16 + tid] = 0; } }
  if (tid == 0) scanFlag[s] = 0;  // the wide kernel sets it when it sends the scan on to the grid-based kernels
  if constexpr (sizeof...(G) > 0) if (tid < 16) (gate.cnt, ...)[s * 16 + tid] = 0;
  if (nch > MAXCHUNK) { if (tid == 0) atomicOr(&ctr->err, ERR_CHUNKS); return; }
  if (tid < NW * 17) (&S.cnt[0][0])[tid] = 0;
  if (tid == 0) { S.nextRing = 0; S.defer = 0; }
  const int Nc = chunk_prefix<NW * 32>(cropCnt + chunk_off[s], nch, S.pre, S.sc);  // ends with a barrier
  if (Nc == 0) return;
  const int nRings = single_ring ? 1 : 16;
  // ---- phase A: stable bucketing of the crop survivors by ring ----
  // every warp owns a contiguous range of the survivors; (1) per-warp counts, (2) offsets, (3) scatter
  const int lo = (int)((long long)Nc * w / NW), hi = (int)((long long)Nc * (w + 1) / NW);
  int* mycnt = S.cnt[w];
  for (int i0 = lo; i0 < hi; i0 += 32) {
    const int i = i0 + lane;
    unsigned m = 0;
    if (i < hi) m = ring_mask_of(cropMeta[piece_pos(S.pre, nch, i, base)] & 63u, single_ring);
    const int first = m ? __ffs(m) - 1 : 16;
    const unsigned peers = __match_any_sync(FE_FULL, first);
    if (i < hi && lane == __ffs(peers) - 1) mycnt[first] += __popc(peers);
    __syncwarp();
    unsigned dual = __ballot_sync(FE_FULL, __popc(m) > 1);  // on a window's end value: also in the next ring (rare)
    while (dual) {
      const int src = __ffs(dual) - 1;
      dual &= dual - 1;
      const int f2 = __shfl_sync(FE_FULL, first, src) + 1;
      if (lane == 0) mycnt[f2] += 1;
      __syncwarp();
    }
  }
  __syncthreads();
  if (tid < 16) {
    // S.cnt[w][h] becomes the first slot of warp w's entries of ring h inside the ring's segment
    int run = 0;
    for (int ww = 0; ww < NW; ww++) { const int c = S.cnt[ww][tid]; S.cnt[ww][tid] = run; run += c; }
    S.ringBase[tid + 1] = run;  // totals for now
  }
  __syncthreads();
  if (tid == 0) {
    int run = 0;
    S.ringBase[0] = 0;
    for (int h = 0; h < 16; h++) { const int c = S.ringBase[h + 1]; S.ringBase[h + 1] = run + c; run += c; }
    if (run > nScan) {  // more ring entries than the scan's slot holds (end-value points count twice): grid path
      S.defer = 1;
      ovfList[atomicAdd(ovfCount, 1)] = s;
    }
  }
  __syncthreads();
  if (S.defer) return;
  float4* RP = ringPts + base;
  for (int i0 = lo; i0 < hi; i0 += 32) {
    const int i = i0 + lane;
    unsigned m = 0;
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < hi) {
      const long long pp = piece_pos(S.pre, nch, i, base);
      m = ring_mask_of(cropMeta[pp] & 63u, single_ring);
      if (m) q = crop[pp];
    }
    const int first = m ? __ffs(m) - 1 : 16;
    const unsigned anyDual = __ballot_sync(FE_FULL, __popc(m) > 1);
    if (!anyDual) {
      const unsigned peers = __match_any_sync(FE_FULL, first);
      const int leader = __ffs(peers) - 1;
      int old = 0;
      if (lane == leader) { old = mycnt[first]; mycnt[first] = old + __popc(peers); }
      old = __shfl_sync(FE_FULL, old, leader);
      if (m) RP[S.ringBase[first] + old + __popc(peers & lanemask_lt())] = q;
      __syncwarp();
    } else {  // a point of this window belongs to two rings: ring by ring, so that every ring keeps the original order
      for (int h = 0; h < nRings; h++) {
        const bool in = (m >> h) & 1u;
        const unsigned bm = __ballot_sync(FE_FULL, in);
        if (!bm) continue;
        const int old = mycnt[h];
        if (in) RP[S.ringBase[h] + old + __popc(bm & lanemask_lt())] = q;
        __syncwarp();
        if (lane == 0) mycnt[h] = old + __popc(bm);
        __syncwarp();
      }
    }
  }
  __syncthreads();  // the block's global writes are visible to all its threads from here on
  // ---- phase B: a warp per ring, rings handed out dynamically ----
  if (tid < 17) ringBaseOut[s * 17 + tid] = S.ringBase[tid];  // for the wide kernel, should a ring of this scan need it
  rr_scan_rings<RW, NW>(S, s, RP, nRings, P, kfPool, kfCap, kfBase, kfCnt, kcPool, kcCap, kcBase, kcCnt, ctr, ovfRuns, ovfRunsCount, gate...);
}

// Second kernel: the rings the first one listed (hundreds of poles in one ring), a warp per ring with RW2 runs;
// what exceeds that — entries in arbitrary order, mostly — sends the ring's whole scan to the grid-based kernels.
template <class... G>
__device__ __forceinline__ void ring_runs_wide_blocks(
    const long long* __restrict__ scan_off, const DevParams& P, const float4* ringPts, const int* __restrict__ ringBaseIn,
    float4* __restrict__ kfPool, int kfCap, int* __restrict__ kfBase, int* __restrict__ kfCnt,
    float4* __restrict__ kcPool, int kcCap, int* __restrict__ kcBase, int* __restrict__ kcCnt,
    DevCounters* __restrict__ ctr, const int* __restrict__ ringList, const int* __restrict__ nList, int* __restrict__ scanFlag,
    int* __restrict__ ovfList, int* __restrict__ ovfCount, G... gate) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  RunBufT<RW2>* bufs = reinterpret_cast<RunBufT<RW2>*>(smem_raw);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  RunBufT<RW2>& B = bufs[w];
  const int nl = *nList;
  for (int li = blockIdx.x * NW_RR + w; li < nl; li += gridDim.x * NW_RR) {
    const int id = ringList[li], s = id >> 4, ring = id & 15;
    const int r0 = ringBaseIn[s * 17 + ring], n = ringBaseIn[s * 17 + ring + 1] - r0;
    const bool done = rr_cluster_ring(B, ringPts + scan_off[s] + r0, n, P, kfPool, kfCap, &kfBase[s * 16 + ring], &kfCnt[s * 16 + ring],
                                      kcPool, kcCap, kcBase ? &kcBase[s * 16 + ring] : nullptr, kcBase ? &kcCnt[s * 16 + ring] : nullptr, ctr,
                                      gate.at(s * 16 + ring)...);
    if (!done && lane == 0 && atomicExch(&scanFlag[s], 1) == 0) ovfList[atomicAdd(ovfCount, 1)] = s;
  }
}

template <class... G>
__global__ void __launch_bounds__(NT_RR) k_ring_runs_wide(
    const long long* __restrict__ scan_off, DevParams P, const float4* ringPts, const int* __restrict__ ringBaseIn,
    float4* __restrict__ kfPool, int kfCap, int* __restrict__ kfBase, int* __restrict__ kfCnt,
    float4* __restrict__ kcPool, int kcCap, int* __restrict__ kcBase, int* __restrict__ kcCnt,
    DevCounters* __restrict__ ctr, const int* __restrict__ ringList, const int* __restrict__ nList, int* __restrict__ scanFlag,
    int* __restrict__ ovfList, int* __restrict__ ovfCount, G... gate) {
  ring_runs_wide_blocks(scan_off, P, ringPts, ringBaseIn, kfPool, kfCap, kfBase, kfCnt, kcPool, kcCap, kcBase, kcCnt, ctr, ringList, nList,
                        scanFlag, ovfList, ovfCount, gate...);
}

}  // namespace fe
