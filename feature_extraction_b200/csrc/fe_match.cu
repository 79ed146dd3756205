// fe_match.cu — 3DSC descriptor matching minimised over the 12 azimuth shifts (fe_match_descriptors*).
// A translation unit of its own, so that the pipeline's kernels in fe_api.cu compile exactly as they did.
//
// The distance is the contract of include/fe_b200.h: for a query row a and a reference row b,
//   P(la, lb) = fmaf chain over m = 0..164 of (a[la*165+m] - b[lb*165+m])^2,
//   d_s       = P(0, s) + P(1, (1+s)%12) + ... + P(11, (11+s)%12), float adds in that order.
//
// Decomposition.  One warp owns one work item: a tile of up to MQ = 4 query rows of one group against one
// segment of up to ITEM_REFS (fe_match.h) reference rows of that group.  Lane = qi * 8 + ri holds the pair (query qi, reference
// ri) of the current 4 x 8 tile and all 144 chains P(la, lb) of it in registers, so every loaded element
// feeds 12 chains: per m step a lane reads 12 query and 12 reference floats (6 LDS.128) for 144 FADD + 144
// FFMA.  The 12 rows of a tile are staged m-chunk by m-chunk (MC = 16) into the warp's own double buffer with
// cp.async, so the copy of the next chunk runs under the arithmetic of this one; no block-wide barrier.
// After the last chunk each lane forms its 12 d_s, keeps the row minimum and folds it into a running top-2;
// at the end of the item the 8 lanes of a query are reduced with shuffles.  An item that covers its whole
// group writes the result; otherwise it writes a partial, and k_match_merge folds the partials of a query.
// The key (d, r, s) is exact and totally ordered, so neither merge depends on the order of the work.
#include <cuda_runtime.h>
#include <stdint.h>

#include "fe_match.h"

namespace fe_match {

constexpr int NBLK = 12;                  // azimuth blocks
constexpr int BLK = 165;                  // 11 elevation x 15 radial bins per block
constexpr int MQ = 4, MR = 8;             // warp tile: 4 queries x 8 reference rows
constexpr int ROWS = MQ + MR;
constexpr int MC = 16;                    // m values staged per chunk
constexpr int NCHUNK = (BLK + MC - 1) / MC;
constexpr int MSTRIDE = ROWS * NBLK + 4;  // floats per staged m: 12 rows x 12 blocks, padded against bank conflicts
constexpr int BUF = MC * MSTRIDE;         // floats per buffer
constexpr int WARPS = 4;                  // warps per block (independent: each runs its own items)
static_assert(MQ * MR == 32, "one pair per lane");
static_assert(MQ == ITEM_QUERIES, "an item is one warp tile of queries");
static_assert(MSTRIDE % 4 == 0, "rows are read with 16-byte loads");

size_t smem_bytes() { return (size_t)WARPS * 2 * BUF * sizeof(float); }

__device__ __forceinline__ void cp_async4(float* dst, const float* src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_1() { asm volatile("cp.async.wait_group 1;\n" ::: "memory"); }

// (d, r) of candidate A orders before that of B.  An empty entry is (+inf, -1); no real candidate has d = +inf
// (a candidate is only taken when d < the current value, which starts at +inf).
__device__ __forceinline__ bool before(float da, long long ra, float db, long long rb) {
  return da < db || (da == db && ra < rb);
}

// top-2 of two disjoint sets of reference rows: best (d, r, s) and the smallest row minimum of the other rows
__device__ __forceinline__ void fold(float& bd, long long& br, int& bs, float& sd, float od, long long orr, int os, float osd) {
  if (before(od, orr, bd, br)) {
    sd = fminf(osd, bd);
    bd = od; br = orr; bs = os;
  } else {
    sd = fminf(sd, od);
  }
}

__global__ void __launch_bounds__(WARPS * 32, 2)
k_match_tiles(const float* __restrict__ q, int64_t qStride, int64_t qBias, const float* __restrict__ r, int64_t rStride,
              int64_t rBias, const Item* __restrict__ items, int nItems, Partial* __restrict__ part, Result res) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int it = blockIdx.x * WARPS + warp;
  if (it >= nItems) return;
  const Item I = items[it];
  float* buf = smem + (size_t)warp * 2 * BUF;
  const int qi = lane >> 3, ri = lane & 7;
  // staging role: lane stages m = mm of rows half*6 .. half*6+5 (rows 0-3 are the queries, 4-11 the references)
  const int mm = lane & 15, half = lane >> 4;
  const int nTiles = (I.nr + MR - 1) / MR;
  const int nSteps = nTiles * NCHUNK;

  const float* src[6];
  bool ok[6];
  auto rows_of_tile = [&](int t) {
#pragma unroll
    for (int k = 0; k < 6; k++) {
      const int row = half * 6 + k;
      if (row < MQ) {
        ok[k] = row < I.nq;
        src[k] = q + (I.q0 + row - qBias) * qStride;
      } else {
        const int rr = t * MR + row - MQ;
        ok[k] = rr < I.nr;
        src[k] = r + (I.r0 + rr - rBias) * rStride;
      }
    }
  };
  auto stage = [&](int step) {  // issue the copies of step `step` (tile step / NCHUNK, chunk step % NCHUNK)
    if (step < nSteps) {
      const int c = step % NCHUNK;
      if (c == 0) rows_of_tile(step / NCHUNK);
      const int m = c * MC + mm;
      float* dst = buf + (step & 1) * BUF + mm * MSTRIDE + half * 6 * NBLK;
      if (m < BLK) {
#pragma unroll
        for (int k = 0; k < 6; k++)
          if (ok[k]) {
#pragma unroll
            for (int lb = 0; lb < NBLK; lb++) cp_async4(dst + k * NBLK + lb, src[k] + lb * BLK + m);
          }
      }
    }
    cp_async_commit();  // an empty group at the end keeps wait_group 1 meaning "the step before the last is in"
  };

  // running top-2 of this lane's pairs: best (d, absolute r, s) and the smallest row minimum of the other rows
  float bd = __int_as_float(0x7f800000), sd = __int_as_float(0x7f800000);
  long long br = -1;
  int bs = -1;
  const bool qValid = qi < I.nq;

  float P[NBLK][NBLK];
#pragma unroll
  for (int i = 0; i < NBLK; i++)
#pragma unroll
    for (int j = 0; j < NBLK; j++) P[i][j] = 0.0f;

  stage(0);
  for (int step = 0; step < nSteps; step++) {
    stage(step + 1);
    cp_async_wait_1();
    __syncwarp();
    const int c = step % NCHUNK;
    const int mlen = min(MC, BLK - c * MC);
    const float* sa = buf + (step & 1) * BUF + qi * NBLK;
    const float* sb = buf + (step & 1) * BUF + (MQ + ri) * NBLK;
#pragma unroll 1
    for (int k = 0; k < mlen; k++) {
      float a[NBLK], b[NBLK];
#pragma unroll
      for (int v = 0; v < NBLK / 4; v++) {
        const float4 x = *reinterpret_cast<const float4*>(sa + k * MSTRIDE + 4 * v);
        const float4 y = *reinterpret_cast<const float4*>(sb + k * MSTRIDE + 4 * v);
        a[4 * v] = x.x; a[4 * v + 1] = x.y; a[4 * v + 2] = x.z; a[4 * v + 3] = x.w;
        b[4 * v] = y.x; b[4 * v + 1] = y.y; b[4 * v + 2] = y.z; b[4 * v + 3] = y.w;
      }
#pragma unroll
      for (int la = 0; la < NBLK; la++)
#pragma unroll
        for (int lb = 0; lb < NBLK; lb++) {
          const float t = __fsub_rn(a[la], b[lb]);
          P[la][lb] = __fmaf_rn(t, t, P[la][lb]);
        }
    }
    __syncwarp();  // the next stage() overwrites this buffer
    if (c == NCHUNK - 1) {
      const int rr = (step / NCHUNK) * MR + ri;
      float rowMin = __int_as_float(0x7f800000);
      int rowS = -1;
#pragma unroll
      for (int s = 0; s < NBLK; s++) {
        float d = 0.0f;
#pragma unroll
        for (int l = 0; l < NBLK; l++) d = __fadd_rn(d, P[l][(l + s) % NBLK]);
        if (d < rowMin) { rowMin = d; rowS = s; }  // NaN never wins; ties keep the lower s
      }
      if (qValid && rr < I.nr && rowS >= 0) {
        // this lane's rows come in ascending order: a tie keeps the earlier (lower) row
        if (rowMin < bd) {
          sd = bd;
          bd = rowMin; br = I.r0 + rr; bs = rowS;
        } else {
          sd = fminf(sd, rowMin);
        }
      }
#pragma unroll
      for (int i = 0; i < NBLK; i++)
#pragma unroll
        for (int j = 0; j < NBLK; j++) P[i][j] = 0.0f;
    }
  }
  // the 8 lanes of one query: disjoint rows
#pragma unroll
  for (int o = 1; o < MR; o <<= 1) {
    const float od = __shfl_xor_sync(0xffffffffu, bd, o), osd = __shfl_xor_sync(0xffffffffu, sd, o);
    const long long orr = __shfl_xor_sync(0xffffffffu, br, o);
    const int os = __shfl_xor_sync(0xffffffffu, bs, o);
    fold(bd, br, bs, sd, od, orr, os, osd);
  }
  if (ri == 0 && qValid) {
    const int64_t out = I.out + qi;
    if (I.nseg == 1) {
      res.best[out] = br;
      res.shift[out] = bs;
      res.dist2[out] = bd;
      res.second[out] = sd;
    } else {
      Partial p;
      p.d = bd; p.sd = sd; p.r = br; p.s = bs;
      part[I.part + (int64_t)qi * I.nseg + I.seg] = p;
    }
  }
}

// one thread per query of an item with seg == 0 of a group split into several segments
__global__ void k_match_merge(const Item* __restrict__ items, int nItems, const Partial* __restrict__ part, Result res) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int it = (int)(t / MQ), qi = (int)(t % MQ);
  if (it >= nItems) return;
  const Item I = items[it];
  if (I.nseg == 1 || I.seg != 0 || qi >= I.nq) return;
  const Partial* p = part + I.part + (int64_t)qi * I.nseg;
  float bd = p[0].d, sd = p[0].sd;
  long long br = p[0].r;
  int bs = p[0].s;
  for (int g = 1; g < I.nseg; g++) fold(bd, br, bs, sd, p[g].d, p[g].r, p[g].s, p[g].sd);
  const int64_t out = I.out + qi;
  res.best[out] = br;
  res.shift[out] = bs;
  res.dist2[out] = bd;
  res.second[out] = sd;
}

cudaError_t set_attributes() {
  return cudaFuncSetAttribute(k_match_tiles, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes());
}

cudaError_t launch(const float* q, int64_t qStride, int64_t qBias, const float* r, int64_t rStride, int64_t rBias,
                   const Item* d_items, int nItems, bool split, Partial* d_part, Result res, cudaStream_t stream) {
  if (nItems <= 0) return cudaSuccess;
  k_match_tiles<<<(nItems + WARPS - 1) / WARPS, WARPS * 32, smem_bytes(), stream>>>(q, qStride, qBias, r, rStride, rBias,
                                                                                     d_items, nItems, d_part, res);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || !split) return e;
  const int64_t threads = (int64_t)nItems * MQ;
  k_match_merge<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(d_items, nItems, d_part, res);
  return cudaGetLastError();
}

}  // namespace fe_match
