// fe_kernels.cuh — the sm_100a kernels of the per-scan keypoint pipeline.
//
//   K1  k_level_crop_ring     getElevationAngles + rotateCloud + filterCloud + ring bucketing
//                             (reference src:147-183, 200-202), fused, one pass over the points;
//                             decodes PointCloud2-style records in place when asked to
//   K2  k_cluster_rings       per-ring EuclideanClusterExtraction + getCylinderSegments gating
//                             (src:261-327): uniform grid (cell = 0.55 x tolerance) built by a block
//                             radix sort of cell keys in shared memory, atomic union-find over the
//                             neighbour cells, segmented per-cluster reductions
//   K3  k_merge_keypoints     cross-ring merge of ring centroids (src:205-257), same machinery
//   K4a k_surface_grid[_smem] 2-D cell sort of the descriptor search surface (cell >= R/5)
//   K4b k_desc_mark           which surface points are inside some keypoint's sphere
//   K4c k_density             3DSC local point density, once per marked point
//   K4d k_desc_hist           1980-bin shape context per keypoint, contributions summed in PCL's order
//
// Batched over scans: every kernel addresses scan s through CSR offsets; blocks never cross scans.
// Per-scan kernels come as chains of instantiations (fast -> large shared memory -> global-memory
// slab): a block that finds its scan too big defers it to a device list for the next one.
#pragma once
#include <math.h>
#include "fe_device.cuh"
#include "glibc_f32.h"
#include "sort_replay.h"
#include "../../include/fe_b200.h"

namespace fe {

constexpr int CH = 2048;        // points per K1 chunk (one block)
constexpr int MAXCHUNK = 512;   // chunks per scan the per-scan kernels can index (1M points)
constexpr int NT2 = 512;        // threads of the per-scan clustering / grid kernels
constexpr int ECAP = 1408;      // cluster entries of the fast instantiation (256 threads, 4 blocks / SM)
constexpr int NTF = 256;
constexpr int ECAP_M = 512;     // K3 fast instantiation: ring centroids per scan (64 threads, many blocks / SM)
constexpr int NTM = 64;
constexpr int NTL = 1024;      // threads of the large K2 instantiation
constexpr int ECAP_G = 65535;   // last resort: per-entry arrays in a global-memory slab (16-bit entry indices)
constexpr int NGLOBAL = 32;     // blocks (and slabs) of the global-memory instantiations
// cluster_extract tests all pairs of a ring while sum(n_r^2)/2 <= this * entries (0: never).  Ring
// points are dense chains (a wall seen by one laser links every point to dozens of others, and
// every link is a union): measured, the pair loop loses there at any threshold (K2 1.90 -> 1.97 ms
// at 4 and 16, 3.95 ms at 256); ring centroids (K3) have few links and win at any size (0.26 -> 0.125 ms).
constexpr int BRUTE_PAIRS_RINGS = 0;
constexpr int BRUTE_PAIRS_MERGE = 256;
constexpr int ECAP_L = 6144;    // the large instantiations (1 block / SM) for scans the fast ones defer

// error bits reported through DevCounters::err
enum {
  ERR_RING_CAP = 1,   // one ring of one scan has more entries than ECAP
  ERR_KF_POOL = 2,    // ring-centroid pool exhausted
  ERR_KP_POOL = 4,    // keypoint pool exhausted
  ERR_MERGE_CAP = 8,  // a scan has more ring centroids than ECAP
  ERR_AXIS_CAP = 16,  // more keypoints in one scan than precomputed 3DSC axes
  ERR_CHUNKS = 32,    // scan has more than MAXCHUNK chunks
  ERR_KC_POOL = 64    // keypoint_cloud pool exhausted
};

// K1 flags
enum { F_ELEV = 1, F_ROT = 2, F_CROP = 4, F_RING = 8, F_SURF = 16 };

struct DevParams {
  // filterCloud limits as pcl::PassThrough stores them (float)
  float xmin, xmax, ymin, ymax, zmin, zmax;
  // descriptor search surface: keep box and 2-D grid (origin sx0,sy0; cell 1/sg_inv)
  float sx0, sx1, sy0, sy1, sz0, sz1;
  float sg_inv;
  int sg_nx, sg_ny, sg_bx;  // key = (cy << sg_bx) | cx
  // ring clustering
  float tol_f, r2f_cluster;
  int min_count, max_count;
  double two_radius_threshold;  // 2*clusterRadiusThreshold (src:316)
  double radius_threshold;      // clusterRadiusThreshold (src:217)
  // merge
  float merge_tol_f, r2f_merge;
  int min_channels;
  // 3DSC
  float R2f, rho2f, Rpad, rhopad;
  float halopad;  // R + R/5 padded: only surface points this close (in x and in y) to a keypoint can matter
  float zs0, zs_inv_range;  // z slabs of the cell grid: slab = clamp(floor((z - zs0) * NS * zs_inv_range), 0, NS-1)
  float radii[16], theta[12], phi[13];
  int estimate_descriptors;
  int angle_libm;  // 0: fdlibm atan2f/acosf (glibc <= 2.40), 1: correctly rounded (glibc >= 2.41)
};

struct DevCounters {
  int kf_cursor;   // ring-centroid pool
  int kp_cursor;   // keypoint pool
  int kc_cursor;   // keypoint_cloud pool
  int err;
  int kp_total;
  int ovf_rings;   // scans deferred from the fast K2 to the medium instantiation
  int ovf_rings2;  // scans deferred from the large K2 to the global-memory instantiation
  int ovf_merge;   // scans deferred from K3 to its large instantiation
  int ovf_surf;    // scans deferred from the shared-memory K4a to the global-memory one
  int desc_unordered;  // keypoints with more than DCAP_L contributions (summed with atomics, not in PCL's order)
  int ovf_merge2;      // scans deferred from the large K3 to the global-memory instantiation
  int ovf_runs;        // scans the first run-based K2 kernel hands to the wide one (a ring with more than RW runs)
  unsigned long long nbr_cursor;  // neighbour-list pool (K4b -> K4d)
  int kd_cursor;                  // next keypoint batch of the fast K4d instantiation
  int kw_cursor;                  // next keypoint of the warp-per-keypoint K4d
  int n_list_m, n_list_l;         // keypoints listed for the medium / large K4d instantiation
  unsigned long long dens_work[2];  // K4c: distance tests, marked points
};

// Kind 6 of the tolerance-boundary report (fe_enable_boundary_report_all): ring clusters whose xy diameter lies within
// eps of the gate 2 * clusterRadiusThreshold (src:316), counted by the K2 kernels where they decide the gate.  The
// K2 kernels and their device functions take it as a trailing parameter pack `gate...`: empty in the instantiations
// that run without that report (their code is what it was without it), one GateCount in the report-on ones
// (k_ring_runs<NW, GateCount>, k_ring_runs_wide<GateCount>, k_cluster_rings<..., GateCount>).
struct GateCount {
  double eps;
  unsigned* cnt;  // [scan][16], zeroed by the first K2 kernel of a scan: the run kernels count ring r in slot r,
                  // the grid kernels (which redo a whole scan) count every cluster of the scan in slot 0
  __device__ GateCount at(int slot) const { return GateCount{eps, cnt + slot}; }
};

// getElevationAngles, src:147-156, literally: double atan2 / cos / sin / atan2.
__device__ __noinline__ float elevation_deg_literal(float xf, float yf, float zf) {
  const double x = xf, y = yf, z = zf;
  const double az = atan2(y, x);
  double sn, cs;
  sincos(az, &sn, &cs);
  const double xp = __dadd_rn(__dmul_rn(cs, x), __dmul_rn(sn, y));
  const double eld = __ddiv_rn(__dmul_rn(atan2(z, xp), 180.0), 3.14159265358979323846);
  return (float)eld;
}

// The same value for the common case without the four double transcendentals.
// cos(atan2(y,x))*x + sin(atan2(y,x))*y is hypot(x,y) up to a few double ulps (the expression is
// stationary in the azimuth), so el = atan(z / hypot(x,y)) in degrees.  For |tan el| < 0.3 (|el| <
// 16.7 deg: every VLP-16 beam) atan is a degree-8 polynomial in q^2 (|error| < 2^-53, fitted at
// Chebyshev nodes).  The result is accepted only if every double within 2^-44 relative of it rounds
// to the same float, i.e. the float the reference's double evaluation produces is not in doubt;
// otherwise (about 1 point in 10^5) the literal evaluation above is used.
__device__ __forceinline__ float elevation_deg(float xf, float yf, float zf) {
  const double x = xf, y = yf, z = zf;
  const double r2 = fma(x, x, y * y);
  if (r2 > 1e-280 && r2 < 1e280) {
    const double q = z * rsqrt(r2);
    if (fabs(q) < 0.2999) {
      const double u = q * q;
      double p = 0.0414062517093382;
      p = fma(p, u, -0.06392744183152536);
      p = fma(p, u, 0.07668228432867163);
      p = fma(p, u, -0.09089657177886407);
      p = fma(p, u, 0.11111072588438455);
      p = fma(p, u, -0.1428571361686184);
      p = fma(p, u, 0.199999999941651);
      p = fma(p, u, -0.3333333333331369);
      p = fma(p, u, 0.9999999999999999);
      const double deg = (q * p) * 57.295779513082320877;
      const double eb = fabs(deg) * 5.6843418860808015e-14;  // 2^-44
      const float lo = (float)(deg - eb), hi = (float)(deg + eb);
      if (lo == hi) return lo;
    }
  }
  return elevation_deg_literal(xf, yf, zf);
}

// 32-bit float at any byte address (PointCloud2 records with point_step 22 are only 2-byte aligned)
__device__ __forceinline__ float load_f32_any(const unsigned char* p) {
  const unsigned long long a = (unsigned long long)p;
  unsigned v;
  if ((a & 3ull) == 0ull) v = __ldg((const unsigned*)p);
  else if ((a & 1ull) == 0ull) v = (unsigned)__ldg((const unsigned short*)p) | ((unsigned)__ldg((const unsigned short*)(p + 2)) << 16);
  else v = (unsigned)__ldg(p) | ((unsigned)__ldg(p + 1) << 8) | ((unsigned)__ldg(p + 2) << 16) | ((unsigned)__ldg(p + 3) << 24);
  return __uint_as_float(v);
}

struct RawLayout {  // records of fe_point_layout_t; raw == nullptr: the input is float4
  const unsigned char* raw;
  int stride, xo, yo, zo;
};

// pcl::transformPointCloud, PCL 1.8.0 scalar form: left to right, unfused, + translation 0
__device__ __forceinline__ float3 level_xyz(const float m[9], const float4 p) {
  float3 q;
  q.x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], p.x), __fmul_rn(m[1], p.y)), __fmul_rn(m[2], p.z)), 0.0f);
  q.y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[3], p.x), __fmul_rn(m[4], p.y)), __fmul_rn(m[5], p.z)), 0.0f);
  q.z = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[6], p.x), __fmul_rn(m[7], p.y)), __fmul_rn(m[8], p.z)), 0.0f);
  return q;
}

// pcl::PassThrough x3 (src:169-183) on a finite point: inclusive float limits
__device__ __forceinline__ bool crop_keeps(const DevParams& P, const float4 q) {
  return !(q.z < P.zmin || q.z > P.zmax) && !(q.y < P.ymin || q.y > P.ymax) && !(q.x < P.xmin || q.x > P.xmax);
}

// K1's chunk table: per chunk {scan, (chunk of the scan << 12) | points, first point lo, hi}.  One warp per scan.
__global__ void __launch_bounds__(256) k_chunk_table(const long long* __restrict__ scan_off, const int* __restrict__ chunk_off,
                                                      int n_scans, int4* __restrict__ tab) {
  const int s = (int)((blockIdx.x * 256u + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (s >= n_scans) return;
  const long long b0 = scan_off[s], n = scan_off[s + 1] - b0;
  const int c0 = chunk_off[s], nc = chunk_off[s + 1] - c0;
  for (int c = lane; c < nc; c += 32) {
    const long long b = b0 + (long long)c * CH;
    tab[c0 + c] = make_int4(s, (int)(((unsigned)c << 12) | (unsigned)min((long long)CH, n - (long long)c * CH)),
                            (int)(unsigned)(b & 0xFFFFFFFFll), (int)(b >> 32));
  }
}

// ============================================================================================
// K1 — fused elevation / level / crop / ring-bucket, order-preserving compaction per chunk.
// Block = one chunk of CH consecutive points of one scan; 256 threads; warp w owns points
// [256w, 256w+256) of the chunk in 8 coalesced rounds (float4 loads).  Survivors are written to
// the chunk's own slot of the output arrays (same CSR as the input) with their counts, so the
// per-scan consumers concatenate pieces in order and no global prefix sum is needed.
// ============================================================================================
template <bool RAW, bool FUSED>
__global__ void __launch_bounds__(256, 6) k_level_crop_ring(
    const float4* __restrict__ pts, const int4* __restrict__ chunkTab, const float* __restrict__ rot, DevParams P,
    int flags_rt, float4* __restrict__ surf, int* __restrict__ surfCnt, float4* __restrict__ crop,
    unsigned* __restrict__ cropMeta, int* __restrict__ cropCnt, float4* __restrict__ full_out,
    RawLayout L, int chunk_base) {
  // FUSED: the cloudCallback path, every stage on (surface stream optional); otherwise run-time flags
  const int flags = FUSED ? (F_ELEV | F_ROT | F_CROP | F_RING | (flags_rt & F_SURF)) : flags_rt;
  __shared__ int s_ws[8], s_wc[8];
  // One tile of shared memory holds the chunk twice over: first its input points, brought in by a single
  // TMA bulk copy (float4 input), then — slot by slot, each written by the thread that read it — the
  // transformed points waiting for their output offsets.
  __shared__ __align__(128) float4 s_o[CH];
  __shared__ __align__(8) unsigned long long s_bar;
  const int chunk = chunk_base + blockIdx.x;  // a batch may be launched in several chunk ranges
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  // chunk -> (scan, chunk of the scan, points, first point), tabulated by the host while it stages the
  // offsets: ONE load stands between the start of the block and its bulk copy (a bisection of chunk_off
  // followed by the scan_off reads was ~15 dependent loads, a sixth of the block's life)
  const int4 ct = __ldg(chunkTab + chunk);
  const int s = ct.x;
  const int c = (int)((unsigned)ct.y >> 12);
  const int nIn = ct.y & 4095;
  const long long base = (long long)(((unsigned long long)(unsigned)ct.w << 32) | (unsigned)ct.z);
  if (!RAW && tid == 0) {
    mbar_init(&s_bar, 1);
    mbar_expect_tx(&s_bar, (unsigned)nIn * 16u);
    tma_load_1d(s_o, pts + base, (unsigned)nIn * 16u, &s_bar);
  }
  float m[9];
#pragma unroll
  for (int i = 0; i < 9; i++) m[i] = (flags & F_ROT) ? rot[s * 9 + i] : 0.0f;
  __syncthreads();
  if (!RAW) mbar_wait(&s_bar, 0);

  unsigned code = 0;             // 8 x 4 bits: ring id of round r (first ring containing el)
  unsigned fl = 0;               // bit r: surf, bit 8+r: crop, bit 16+r: dual ring, bit 24+r: no ring
  unsigned ms[8], mc[8];
#pragma unroll
  for (int r = 0; r < 8; r++) {
    const int j = w * 256 + r * 32 + lane;
    bool fs = false, fc = false;
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j < nIn) {
      float4 p;
      if (RAW) {  // PointCloud2-style records decoded in place (SURVEY.md §8f-1)
        const unsigned char* rec = L.raw + (base + j) * (long long)L.stride;
        p = make_float4(load_f32_any(rec + L.xo), load_f32_any(rec + L.yo), load_f32_any(rec + L.zo), 0.0f);
      } else {
        p = s_o[j];
      }
      float el = p.w;
      if (flags & F_ROT) {
        const float3 l = level_xyz(m, p);
        q.x = l.x; q.y = l.y; q.z = l.z;
      } else {
        q.x = p.x; q.y = p.y; q.z = p.z;
      }
      const bool fin = finite3(q.x, q.y, q.z);
      // pcl::PassThrough: non-finite dropped, inclusive float limits (src:169-183)
      fc = fin;
      if (flags & F_CROP) fc = fin && crop_keeps(P, q);
      // getElevationAngles, src:147-156.  The angle only travels with the cropped cloud (the
      // descriptor surface never reads it), so it is evaluated for the crop survivors alone.
      if ((flags & F_ELEV) && (fc || (!FUSED && full_out))) el = elevation_deg(p.x, p.y, p.z);
      q.w = el;
      if (!FUSED && full_out) full_out[base + j] = q;
      if (fc) {
        unsigned rm = 1u;
        if (flags & F_RING) {
          // ring i keeps (i-7)*2-1 +- 1 inclusive (src:200-202); windows share their end points
          rm = 0u;
          if (isfinite(el)) {
            // i = the ring with lo <= el < lo + 2 (lo = 2i - 16).  The float (el + 16) / 2 can round across
            // an integer, so its floor is off by at most one: one correction step.  An angle exactly on a
            // window's lower end is also the upper end of ring i - 1.  (Far outside angles end at i <= -3
            // or i >= 19 through the clamp: no ring.)
            int i = (int)floorf(fminf(fmaxf((el + 16.0f) * 0.5f, -2.0f), 18.0f));
            float lo = (float)(2 * i - 16);
            if (el < lo) { i--; lo -= 2.0f; }
            else if (el >= lo + 2.0f) { i++; lo += 2.0f; }
            if (i >= 0 && i < 16) rm = 1u << i;
            if (el == lo && i >= 1 && i <= 16) rm |= 1u << (i - 1);
          }
        }
        if (rm == 0u) fl |= 1u << (24 + r);
        else {
          code |= (unsigned)(__ffs(rm) - 1) << (4 * r);
          if (__popc(rm) > 1) fl |= 1u << (16 + r);
        }
      }
      if (flags & F_SURF)
        fs = fin && q.x >= P.sx0 && q.x <= P.sx1 && q.y >= P.sy0 && q.y <= P.sy1 && q.z >= P.sz0 && q.z <= P.sz1;
    }
    s_o[j] = q;
    if (fs) fl |= 1u << r;
    if (fc) fl |= 1u << (8 + r);
    ms[r] = __ballot_sync(FE_FULL, fs);
    mc[r] = __ballot_sync(FE_FULL, fc);
  }
  int ts = 0, tc = 0;
#pragma unroll
  for (int r = 0; r < 8; r++) { ts += __popc(ms[r]); tc += __popc(mc[r]); }
  if (lane == 0) { s_ws[w] = ts; s_wc[w] = tc; }
  __syncthreads();
  int os = 0, oc = 0, tots = 0, totc = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    if (i < w) { os += s_ws[i]; oc += s_wc[i]; }
    tots += s_ws[i]; totc += s_wc[i];
  }
  if (tid == 0) {
    if (surfCnt) surfCnt[chunk] = tots;
    if (cropCnt) cropCnt[chunk] = totc;
  }
  const unsigned lt = lanemask_lt();
#pragma unroll
  for (int r = 0; r < 8; r++) {
    const float4 orr = s_o[w * 256 + r * 32 + lane];
    if (fl & (1u << r)) {
      float4 sq = orr;  // 3DSC reads only x,y,z of the surface: .w carries the point's index in the scan
      sq.w = __int_as_float(c * CH + w * 256 + r * 32 + lane);
      surf[base + os + __popc(ms[r] & lt)] = sq;
    }
    if (fl & (1u << (8 + r))) {
      const long long d = base + oc + __popc(mc[r] & lt);
      crop[d] = orr;
      unsigned cd = (code >> (4 * r)) & 15u;
      if (fl & (1u << (16 + r))) cd |= 16u;
      if (fl & (1u << (24 + r))) cd = 32u;
      const unsigned idx = (unsigned)(c * CH + w * 256 + r * 32 + lane);
      cropMeta[d] = (idx << 6) | cd;
    }
    os += __popc(ms[r]);
    oc += __popc(mc[r]);
  }
}

// ============================================================================================
// Shared-memory workspace of the per-scan clustering kernels.
// ============================================================================================
struct ClusterSm {
  float *x, *y, *z;
  unsigned* gref;          // where the entry lives in the global array it came from
  unsigned char* ring;
  unsigned *keyA, *keyB;
  unsigned short *valA, *valB, *aux, *lst;
  unsigned short* wc;      // NT/32 * 257
  unsigned* base;          // 256 + 32
  int* misc;               // MISC_INTS
};
constexpr int MISC_INTS = MAXCHUNK + 1 + 128;
constexpr size_t cluster_smem_bytes(int cap, int nt) {
  return (size_t)cap * (12 + 4 + 1 + 8 + 8) + (nt / 32) * 257 * 2 + (256 + 32) * 4 + MISC_INTS * 4 + 64;
}

template <int CAP, int NT>
__device__ __forceinline__ void cluster_sm_carve(unsigned char* p, ClusterSm& S) {
  S.x = (float*)p; p += CAP * 4;
  S.y = (float*)p; p += CAP * 4;
  S.z = (float*)p; p += CAP * 4;
  S.gref = (unsigned*)p; p += CAP * 4;
  S.keyA = (unsigned*)p; p += CAP * 4;
  S.keyB = (unsigned*)p; p += CAP * 4;
  S.base = (unsigned*)p; p += (256 + 32) * 4;
  S.misc = (int*)p; p += MISC_INTS * 4;
  S.valA = (unsigned short*)p; p += CAP * 2;
  S.valB = (unsigned short*)p; p += CAP * 2;
  S.aux = (unsigned short*)p; p += CAP * 2;
  S.lst = (unsigned short*)p; p += CAP * 2;
  S.wc = (unsigned short*)p; p += (NT / 32) * 257 * 2;
  S.ring = (unsigned char*)p;
}

// Same workspace with the per-entry arrays in a global-memory slab (entries up to ECAP_G); only the
// radix counters and the small scratch stay in shared memory.
__host__ __device__ constexpr size_t cluster_slab_bytes(int cap) { return ((size_t)cap * 33 + 255) / 256 * 256; }
constexpr size_t cluster_smem_bytes_global(int nt) { return (size_t)(nt / 32) * 257 * 2 + (256 + 32) * 4 + MISC_INTS * 4 + 64; }

template <int CAP, int NT>
__device__ __forceinline__ void cluster_carve_global(unsigned char* g, unsigned char* p, ClusterSm& S) {
  S.x = (float*)g; g += (size_t)CAP * 4;
  S.y = (float*)g; g += (size_t)CAP * 4;
  S.z = (float*)g; g += (size_t)CAP * 4;
  S.gref = (unsigned*)g; g += (size_t)CAP * 4;
  S.keyA = (unsigned*)g; g += (size_t)CAP * 4;
  S.keyB = (unsigned*)g; g += (size_t)CAP * 4;
  S.valA = (unsigned short*)g; g += (size_t)CAP * 2;
  S.valB = (unsigned short*)g; g += (size_t)CAP * 2;
  S.aux = (unsigned short*)g; g += (size_t)CAP * 2;
  S.lst = (unsigned short*)g; g += (size_t)CAP * 2;
  S.ring = (unsigned char*)g;
  S.base = (unsigned*)p; p += (256 + 32) * 4;
  S.misc = (int*)p; p += MISC_INTS * 4;
  S.wc = (unsigned short*)p;
}

struct ClusterOut {
  int nC;                  // clusters that passed the size gate, in PCL's output order
  unsigned short* slotRoot;   // [nC] entry index of the cluster's first (smallest) member
  unsigned* cnt;              // [E] cnt[root] = cluster size
  unsigned short* mem;        // [sum of sizes] members, cluster after cluster, ascending
  unsigned short* slotStart;  // [nC] offset of each cluster in mem
  unsigned* parent;           // [E] root of every entry
};

// pcl::EuclideanClusterExtraction::extract (PCL 1.8.0 extract_clusters.hpp) over the E entries
// held in S (x,y,z,ring), ring by ring: connected components of {d2 < r2f}, size gate applied
// to whole components, members ascending, clusters in discovery order then reordered by the
// std::sort(rbegin, rend, size<) replay.  Entries must be in the original point order.
// misc[96..127] is scratch.
template <int NT>
__device__ void cluster_extract(ClusterSm& S, int E, float tol_f, float r2f, int minSz, int maxSz,
                                int nRings, int brutePairs, ClusterOut& out) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  int* sc = S.misc + MAXCHUNK + 1;        // 128 ints of scratch
  float* bb = (float*)(sc + 40);          // 6 floats
  // ---- small rings: all pairs inside every ring ----
  // A ring of n entries costs n^2/2 distance tests (and a union per linked pair) here, against ~130 warp
  // instructions per entry for the grid machinery below (keys, three radix passes, cells, row
  // searches) that never tests points sharing a cell: the caller says up to which density this wins.
  unsigned *kS = S.keyA, *kT = S.keyB;
  unsigned short *vS = S.valA, *vT = S.valB;
  bool brute = false;
  if (brutePairs > 0) {
    unsigned short* ord = S.valA;  // entries in ring order (stable: ascending entry inside a ring)
    unsigned* ringEnd = S.base;    // block_radix_pass leaves the end offset of every digit (= ring)
    if (nRings > 1) {
      unsigned char* rng = S.ring;
      block_radix_pass<NT, unsigned short>(
          E, [=](int i) { return (unsigned)rng[i]; }, [=](int i, int pos) { ord[pos] = (unsigned short)i; }, S.wc, S.base);
    } else {
      for (int e = tid; e < E; e += NT) ord[e] = (unsigned short)e;
      if (tid == 0) ringEnd[0] = (unsigned)E;
    }
    __syncthreads();
    unsigned long long sumsq = 0;
    for (int r = 0; r < nRings; r++) {
      const unsigned long long nr = ringEnd[r] - (r ? ringEnd[r - 1] : 0u);
      sumsq += nr * nr;
    }
    brute = sumsq <= (unsigned long long)brutePairs * 2ull * (unsigned long long)E;
    if (brute) {
      unsigned* par = S.keyB;
      for (int e = tid; e < E; e += NT) par[e] = (unsigned)e;
      __syncthreads();
      for (int k = tid; k < E; k += NT) {
        const unsigned ei = ord[k];
        const int end = (int)ringEnd[S.ring[ei]];
        const float xi = S.x[ei], yi = S.y[ei], zi = S.z[ei];
        for (int m = k + 1; m < end; m++) {
          const unsigned ej = ord[m];
          if (l2_simple(xi, yi, zi, S.x[ej], S.y[ej], S.z[ej]) < r2f) {
            const volatile unsigned* vp = par;
            if (vp[ei] != vp[ej]) uf_union(par, ei, ej);
          }
        }
      }
      __syncthreads();
      // flatten: the root of a component is its smallest entry (= its first point in the cloud)
      for (int e = tid; e < E; e += NT) { const unsigned r = uf_find_readonly(par, (unsigned)e); S.aux[e] = (unsigned short)r; }
      __syncthreads();
      for (int e = tid; e < E; e += NT) { par[e] = S.aux[e]; S.keyA[e] = 0; }
      __syncthreads();
    }
  }
  if (!brute) {
    // ---- bounding box of the entries (grid origin) ----
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int e = tid; e < E; e += NT) {
      mn[0] = fminf(mn[0], S.x[e]); mx[0] = fmaxf(mx[0], S.x[e]);
      mn[1] = fminf(mn[1], S.y[e]); mx[1] = fmaxf(mx[1], S.y[e]);
      mn[2] = fminf(mn[2], S.z[e]); mx[2] = fmaxf(mx[2], S.z[e]);
    }
  #pragma unroll
    for (int k = 0; k < 3; k++)
  #pragma unroll
      for (int d = 16; d; d >>= 1) {
        mn[k] = fminf(mn[k], __shfl_xor_sync(FE_FULL, mn[k], d));
        mx[k] = fmaxf(mx[k], __shfl_xor_sync(FE_FULL, mx[k], d));
      }
    float* red = (float*)(sc + 48);  // NT/32 * 6 floats <= 96 -> use S.wc area instead (free here)
    red = (float*)S.wc;
    __syncthreads();
    if (lane == 0) {
  #pragma unroll
      for (int k = 0; k < 3; k++) { red[w * 6 + k] = mn[k]; red[w * 6 + 3 + k] = mx[k]; }
    }
    __syncthreads();
    if (tid < 6) {
      float v = red[tid];
      for (int i = 1; i < NT / 32; i++) v = (tid < 3) ? fminf(v, red[i * 6 + tid]) : fmaxf(v, red[i * 6 + tid]);
      bb[tid] = v;
    }
    __syncthreads();
    // Grid cell = 0.55 * tolerance.  Two properties follow, both with several percent of slack
    // against the float rounding of the cell computation and of the d2 predicate:
    //   (i)  two points in the same cell are closer than sqrt(3)*0.55*tol = 0.953*tol: they are
    //        linked by construction and need no distance test;
    //   (ii) two linked points (d < tol) are at most 2 cells apart on every axis.
    // Cell indices clamp to the key's bit budget (x,y: 10 bits, z: 8 bits); the monotone clamp keeps
    // (ii), but merges far cells, so (i) is only trusted when nothing had to be clamped.
    const float inv = 1.0f / (tol_f * 0.55f);
    const float ox = bb[0], oy = bb[1], oz = bb[2];
    const float fx = floorf((bb[3] - ox) * inv), fy = floorf((bb[4] - oy) * inv), fz = floorf((bb[5] - oz) * inv);
    const bool trusted = (fx < 1023.0f) && (fy < 1023.0f) && (fz < 255.0f);
    const int nx = (int)fminf(1023.0f, fmaxf(fx, 0.0f)) + 1;
    const int ny = (int)fminf(1023.0f, fmaxf(fy, 0.0f)) + 1;
    const int nz = (int)fminf(255.0f, fmaxf(fz, 0.0f)) + 1;
    // key = ((ring*nz + cz)*ny + cy)*nx + cx  (< 2^32: 16 * 256 * 1024 * 1024)
    const unsigned unx = (unsigned)nx, uny = (unsigned)ny, unz = (unsigned)nz;
    const unsigned long long nkeys = (unsigned long long)nRings * unz * uny * unx;
    const int keybits = (nkeys <= 1ull) ? 0 : 64 - __clzll((long long)(nkeys - 1ull));
    // ---- keys ----
    for (int e = tid; e < E; e += NT) {
      int cx = (int)floorf((S.x[e] - ox) * inv), cy = (int)floorf((S.y[e] - oy) * inv), cz = (int)floorf((S.z[e] - oz) * inv);
      cx = max(0, min(cx, nx - 1)); cy = max(0, min(cy, ny - 1)); cz = max(0, min(cz, nz - 1));
      S.keyA[e] = (((unsigned)S.ring[e] * unz + (unsigned)cz) * uny + (unsigned)cy) * unx + (unsigned)cx;
      S.valA[e] = (unsigned short)e;
    }
    // ---- radix sort of (key, entry) ----
    kS = S.keyA; kT = S.keyB; vS = S.valA; vT = S.valB;
    for (int shift = 0; shift < keybits; shift += 8) {
      unsigned* ki = kS; unsigned* ko = kT; unsigned short* vi = vS; unsigned short* vo = vT;
      block_radix_pass<NT, unsigned short>(
          E, [=](int i) { return (ki[i] >> shift) & 255u; },
          [=](int i, int pos) { ko[pos] = ki[i]; vo[pos] = vi[i]; }, S.wc, S.base);
      kS = ko; kT = ki; vS = vo; vT = vi;
    }
    __syncthreads();
    // The last pass leaves in S.base[d] the end offset of top digit d: a 256-bucket index into the
    // sorted keys that shortens every lower_bound below (keybits == 0: one bucket, no pass ran).
    const int topShift = (keybits > 0) ? 8 * ((keybits - 1) >> 3) : 32;
    const unsigned* bucketEnd = S.base;
    // ---- units: the runs of equal key (cells); every entry on its own when cells are not trusted ----
    unsigned short* unitStart = S.lst;
    int nU = 0;
    {
      int run = 0;
      for (int p0 = 0; p0 < E; p0 += NT) {
        const int p = p0 + tid;
        const int head = (p < E && (!trusted || p == 0 || kS[p] != kS[p - 1])) ? 1 : 0;
        int tot;
        const int pos = block_excl_scan<NT>(head, &tot, sc);
        if (head) unitStart[run + pos] = (unsigned short)p;
        if (p < E) S.aux[p] = (unsigned short)(run + pos + head - 1);  // unit index of every sorted position
        run += tot;
      }
      nU = run;
    }
    __syncthreads();
    // ---- union-find over sorted positions; a cell's members start out linked to its first ----
    unsigned* parentS = kT;
    constexpr int G = 8;
    const int gl = lane & (G - 1);
    const unsigned gmask = 0xFFu << (lane & 24);
    unsigned short* unitOf = S.aux;
    for (int p = tid; p < E; p += NT) parentS[p] = (unsigned)unitStart[unitOf[p]];
    __syncthreads();
    // One 8-lane group per unit.  The 13 rows (dz,dy) that precede the unit's own cell in key order
    // and can hold linked points are located by 13 binary searches spread over the lanes; the
    // candidates of a row are then visited 8 at a time.  A candidate already in the unit's component
    // is skipped; otherwise it is tested against the unit's members until the first link.
    int* unitCursor = sc + 60;
    if (tid == 0) *unitCursor = 0;
    __syncthreads();
    for (;;) {
      int u = 0;
      if (gl == 0) u = atomicAdd(unitCursor, 1);  // units are handed out dynamically: their cost varies a lot
      u = __shfl_sync(gmask, u, 0, G);
      if (u >= nU) break;
      const int a0 = unitStart[u];
      const int a1 = (u + 1 < nU) ? (int)unitStart[u + 1] : E;
      const unsigned key = kS[a0];
      const int cx = (int)(key % unx);
      const unsigned t1 = key / unx;
      const int cy = (int)(t1 % uny);
      const unsigned t2 = t1 / uny;
      const int cz = (int)(t2 % unz);
      const unsigned rg = t2 / unz;
      int lo[2] = {0, 0}, end[2] = {0, 0};
      unsigned khi[2] = {0u, 0u};
      unsigned mine = 0;  // bit rnd: my row of that round has candidates
  #pragma unroll
      for (int rnd = 0; rnd < 2; rnd++) {
        const int r = gl + 8 * rnd;  // 0..9: dz=-2,-1 x dy=-2..2; 10,11: dz=0, dy=-2,-1; 12: own row
        if (r < 13) {
          const int dz = (r < 5) ? -2 : (r < 10) ? -1 : 0;
          const int dy = (r < 10) ? (r % 5) - 2 : (r == 12) ? 0 : r - 12;
          const int zz = cz + dz, yy = cy + dy;
          if (zz >= 0 && yy >= 0 && yy < ny) {
            const unsigned rowk = ((rg * unz + (unsigned)zz) * uny + (unsigned)yy) * unx;
            const unsigned klo = rowk + (unsigned)max(cx - 2, 0);
            khi[rnd] = rowk + (unsigned)min(cx + 2, nx - 1);
            end[rnd] = (r == 12) ? a0 : E;
            int l = 0, h = end[rnd];  // lower_bound(klo) in kS[0, end), inside klo's top-digit bucket
            if (topShift < 32) {
              const unsigned d = klo >> topShift;
              l = min(d ? (int)bucketEnd[d - 1] : 0, h);
              h = min((int)bucketEnd[d], h);
            }
            while (l < h) {
              const int mid = (l + h) >> 1;
              if (kS[mid] < klo) l = mid + 1; else h = mid;
            }
            lo[rnd] = l;
            if (l < end[rnd] && kS[l] <= khi[rnd]) mine |= 1u << rnd;
          }
        }
      }
      // rows that actually hold candidates: bit (8*rnd + lane)
      unsigned rows = (__ballot_sync(gmask, mine & 1u) >> (lane & 24)) & 0xFFu;
      rows |= ((__ballot_sync(gmask, mine & 2u) >> (lane & 24)) & 0xFFu) << 8;
      while (rows) {
        const int r = __ffs(rows) - 1;
        rows &= rows - 1;
        const int src = r & 7;
        const int rlo = __shfl_sync(gmask, (r < 8) ? lo[0] : lo[1], src, G);
        const int rend = __shfl_sync(gmask, (r < 8) ? end[0] : end[1], src, G);
        const unsigned rkhi = __shfl_sync(gmask, (r < 8) ? khi[0] : khi[1], src, G);
        // Candidate units (cells) of this row — at most five, one lane each.  All points of a unit are
        // in one component, so one root comparison decides whether the unit matters.  Small unit pairs
        // are tested by the lane that owns them; large ones (dense cells) are flagged and then tested
        // by the whole group, the pair tests spread over the 8 lanes, stopping at the first link.
        for (int uu0 = unitOf[rlo];; uu0 += G) {
          const int uu = uu0 + gl;
          bool in = false, heavy = false;
          if (uu < nU) {
            const int b0 = unitStart[uu];
            in = (b0 < rend) && (kS[b0] <= rkhi);
            if (in && uf_find(parentS, (unsigned)b0) != uf_find(parentS, (unsigned)a0)) {
              const int b1 = (uu + 1 < nU) ? (int)unitStart[uu + 1] : E;
              if ((a1 - a0) * (b1 - b0) <= 96) {
                bool linked = false;
                for (int a = a0; a < a1 && !linked; a++) {
                  const unsigned ea = vS[a];
                  const float ax = S.x[ea], ay = S.y[ea], az = S.z[ea];
                  for (int b = b0; b < b1; b++) {
                    const unsigned eb = vS[b];
                    if (l2_simple(ax, ay, az, S.x[eb], S.y[eb], S.z[eb]) < r2f) { linked = true; break; }
                  }
                }
                if (linked) uf_union(parentS, (unsigned)a0, (unsigned)b0);
              } else {
                heavy = true;
              }
            }
          }
          unsigned hv = (__ballot_sync(gmask, heavy) >> (lane & 24)) & 0xFFu;
          while (hv) {
            const int ub = uu0 + __ffs(hv) - 1;
            hv &= hv - 1;
            const int b0 = unitStart[ub];
            const int b1 = (ub + 1 < nU) ? (int)unitStart[ub + 1] : E;
            int differs = 0;  // re-checked (unions happened meanwhile); by lane 0 so that it is uniform
            if (gl == 0) differs = (uf_find(parentS, (unsigned)b0) != uf_find(parentS, (unsigned)a0)) ? 1 : 0;
            differs = __shfl_sync(gmask, differs, 0, G);
            if (!differs) continue;
            bool linked = false;
            for (int a = a0; a < a1; a++) {
              const unsigned ea = vS[a];
              const float ax = S.x[ea], ay = S.y[ea], az = S.z[ea];
              for (int b = b0 + gl; b < b1; b += G) {
                const unsigned eb = vS[b];
                if (l2_simple(ax, ay, az, S.x[eb], S.y[eb], S.z[eb]) < r2f) { linked = true; break; }
              }
              if (__ballot_sync(gmask, linked) != 0u) { linked = true; break; }
            }
            if (linked && gl == 0) uf_union(parentS, (unsigned)a0, (unsigned)b0);
          }
          if (!__shfl_sync(gmask, (int)in, G - 1, G)) break;  // units are in key order: nothing further in range
        }
      }
    }
    __syncthreads();
    // ---- flatten; label every component with its smallest entry (= its first point in the cloud) ----
    // (two steps through S.aux — the unit indices are no longer needed — so that no thread rewrites a link
    // while another one is still walking it)
    for (int p = tid; p < E; p += NT) S.aux[p] = (unsigned short)uf_find_readonly(parentS, (unsigned)p);
    __syncthreads();
    for (int p = tid; p < E; p += NT) parentS[p] = (unsigned)S.aux[p];
    __syncthreads();
    unsigned* minE = kS;
    for (int p = tid; p < E; p += NT) minE[p] = 0xFFFFFFFFu;
    __syncthreads();
    for (int p = tid; p < E; p += NT) atomicMin(&minE[parentS[p]], (unsigned)vS[p]);
    __syncthreads();
    for (int p = tid; p < E; p += NT) {
      vT[p] = (unsigned short)minE[parentS[p]];
      S.aux[vS[p]] = (unsigned short)p;
    }
    __syncthreads();
  }
  unsigned* parent = kT;  // from here on indexed by entry: parent[e] = first entry of e's component
  unsigned* cnt = kS;
  if (!brute) {
    for (int e = tid; e < E; e += NT) { parent[e] = vT[S.aux[e]]; cnt[e] = 0; }
    __syncthreads();
  }
  for (int e = tid; e < E; e += NT) atomicAdd(&cnt[parent[e]], 1u);
  __syncthreads();
  // ---- size-gated roots in discovery order (ascending first member) ----
  int nC = 0;
  {
    int run = 0;
    for (int e0 = 0; e0 < E; e0 += NT) {
      const int e = e0 + tid;
      const int keep = (e < E && parent[e] == (unsigned)e && (int)cnt[e] >= minSz && (int)cnt[e] <= maxSz) ? 1 : 0;
      int tot;
      const int pos = block_excl_scan<NT>(keep, &tot, sc);
      if (keep) vT[run + pos] = (unsigned short)e;
      run += tot;
    }
    nC = run;
  }
  __syncthreads();
  out.nC = nC;
  out.cnt = cnt;
  out.parent = parent;
  out.slotRoot = S.lst;
  if (nC == 0) { out.mem = vS; out.slotStart = S.aux; return; }
  // ---- split by ring (stable), then PCL's final cluster order inside every ring ----
  int* ringEnd = sc + 64;  // 16 ints
  if (nRings > 1) {
    unsigned short* src = vT; unsigned short* dst = S.lst; unsigned char* rng = S.ring;
    block_radix_pass<NT, unsigned short>(
        nC, [=](int i) { return (unsigned)rng[src[i]]; }, [=](int i, int pos) { dst[pos] = src[i]; }, S.wc, S.base);
    if (tid < 16) ringEnd[tid] = (int)S.base[tid];
  } else {
    for (int i = tid; i < nC; i += NT) S.lst[i] = vT[i];
    if (tid < 16) ringEnd[tid] = nC;
  }
  __syncthreads();
  {
    constexpr int STRIDE = NT / 16;  // one thread per ring, spread over the warps
    if ((tid % STRIDE) == 0 && (tid / STRIDE) < nRings) {
      const int r = tid / STRIDE;
      const int b = (r == 0) ? 0 : ringEnd[r - 1];
      const int n = ringEnd[r] - b;
      if (n > 1) {
        const unsigned* c2 = cnt;
        pcl_cluster_order(S.lst + b, n, [=](unsigned short id) { return c2[id]; });
      }
    }
  }
  for (int e = tid; e < E; e += NT) S.aux[e] = 0xFFFFu;
  __syncthreads();
  for (int i = tid; i < nC; i += NT) S.aux[S.lst[i]] = (unsigned short)i;
  __syncthreads();
  // ---- member lists: stable sort of the entries by cluster slot (ascending entry inside) ----
  {
    const int kb = bits_for(nC);  // values 0..nC (nC = not in a kept cluster)
    unsigned short* aux = S.aux;
    const unsigned* par = parent;
    const unsigned nCu = (unsigned)nC;
    unsigned short* o1 = vS;
    block_radix_pass<NT, unsigned short>(
        E, [=](int i) { unsigned s = aux[par[i]]; if (s == 0xFFFFu) s = nCu; return s & 255u; },
        [=](int i, int pos) { o1[pos] = (unsigned short)i; }, S.wc, S.base);
    out.mem = vS;
    if (kb > 8) {
      unsigned short* o2 = vT;
      block_radix_pass<NT, unsigned short>(
          E, [=](int i) { unsigned s = aux[par[o1[i]]]; if (s == 0xFFFFu) s = nCu; return (s >> 8) & 255u; },
          [=](int i, int pos) { o2[pos] = o1[i]; }, S.wc, S.base);
      out.mem = vT;
    }
  }
  __syncthreads();
  // ---- slot offsets ----
  {
    int run = 0;
    for (int i0 = 0; i0 < nC; i0 += NT) {
      const int i = i0 + tid;
      const int v = (i < nC) ? (int)cnt[S.lst[i]] : 0;
      int tot;
      const int pos = block_excl_scan<NT>(v, &tot, sc);
      if (i < nC) S.aux[i] = (unsigned short)(run + pos);
      run += tot;
    }
  }
  out.slotStart = S.aux;
  __syncthreads();
}

// Prefix of a scan's chunk counts into misc[0..nch]; returns the total.  All threads call.
template <int NT>
__device__ int chunk_prefix(const int* __restrict__ cnt, int nch, int* pre, int* sc) {
  int run = 0;
  for (int c0 = 0; c0 < nch; c0 += NT) {
    const int c = c0 + threadIdx.x;
    const int v = (c < nch) ? cnt[c] : 0;
    int tot;
    const int pos = block_excl_scan<NT>(v, &tot, sc);
    if (c < nch) pre[c] = run + pos;
    run += tot;
  }
  if (threadIdx.x == 0) pre[nch] = run;
  __syncthreads();
  return run;
}

// position in the piece-wise array of the i-th survivor of a scan
__device__ __forceinline__ long long piece_pos(const int* pre, int nch, int i, long long base) {
  int lo = 0, hi = nch - 1;  // largest c with pre[c] <= i
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (pre[mid] <= i) lo = mid; else hi = mid - 1;
  }
  return base + (long long)lo * CH + (i - pre[lo]);
}

// ============================================================================================
// K2 — per-ring clustering and getCylinderSegments gating for one scan per block.
// ============================================================================================
template <int CAP, int NT, class... G>
__device__ void cluster_rings_scan(
    ClusterSm& S, const int s, const float4* __restrict__ crop, const unsigned* __restrict__ cropMeta,
    const int* __restrict__ cropCnt, const long long* __restrict__ scan_off,
    const int* __restrict__ chunk_off, const DevParams& P, int single_ring,
    float4* __restrict__ kfPool, int kfCap, int* __restrict__ kfBase, int* __restrict__ kfCnt,
    float4* __restrict__ kcPool, int kcCap, int* __restrict__ kcBase, int* __restrict__ kcCnt,
    DevCounters* __restrict__ ctr, int* __restrict__ ovfList, int* __restrict__ ovfCount, G... gate) {
  const int tid = threadIdx.x;
  int* pre = S.misc;
  int* sc = S.misc + MAXCHUNK + 1;
  int* ringCnt = sc + 80;  // 16
  const long long base = scan_off[s];
  const int nch = chunk_off[s + 1] - chunk_off[s];
  if (tid < 16) { kfBase[s * 16 + tid] = 0; kfCnt[s * 16 + tid] = 0; if (kcBase) { kcBase[s * 16 + tid] = 0; kcCnt[s * 16 + tid] = 0; } }
  if constexpr (sizeof...(G) > 0) if (tid < 16) (gate.cnt, ...)[s * 16 + tid] = 0;
  if (nch > MAXCHUNK) { if (tid == 0) atomicOr(&ctr->err, ERR_CHUNKS); return; }
  const int Nc = chunk_prefix<NT>(cropCnt + chunk_off[s], nch, pre, sc);
  if (Nc == 0) return;
  const int nRingsAll = single_ring ? 1 : 16;
  // Entries per ring are only counted when needed: a scan with at most CAP crop survivors is first
  // gathered whole (all rings, one group); the count and the ring groups are the fallback when the
  // doubled end-point entries push it over the capacity.
  bool counted = false, whole = (Nc <= CAP);
  int group = 0;
  int r0 = 0;
  while (r0 < nRingsAll) {
    int r1 = r0, tot = 0;
    if (whole) {
      r1 = nRingsAll; tot = Nc;
    } else {
      if (!counted) {
        counted = true;
        if (tid < 16) ringCnt[tid] = 0;
        __syncthreads();
        for (int i = tid; i < Nc; i += NT) {
          const unsigned cd = cropMeta[piece_pos(pre, nch, i, base)] & 63u;
          if (cd & 32u) continue;
          const int r = single_ring ? 0 : (int)(cd & 15u);
          atomicAdd(&ringCnt[r], 1);
          if ((cd & 16u) && !single_ring) atomicAdd(&ringCnt[r + 1], 1);
        }
        __syncthreads();
        int big = 0;
        for (int r = 0; r < nRingsAll; r++) big = max(big, ringCnt[r]);
        if (big > CAP) {  // a single ring is larger than this instantiation's capacity
          if (tid == 0) {
            if (ovfList) ovfList[atomicAdd(ovfCount, 1)] = s;  // the next larger instantiation takes it
            else atomicOr(&ctr->err, ERR_RING_CAP);
          }
          return;
        }
      }
      // greedy run of consecutive rings that fits the shared-memory capacity
      while (r1 < nRingsAll && tot + ringCnt[r1] <= CAP) { tot += ringCnt[r1]; r1++; }
    }
    if (tot > 0) {
      // ---- gather the entries of rings [r0, r1) in original order ----
      int run = 0;
      for (int i0 = 0; i0 < Nc; i0 += NT) {
        const int i = i0 + tid;
        int take = 0, ra = 0, rb = -1;
        long long pp = 0;
        if (i < Nc) {
          pp = piece_pos(pre, nch, i, base);
          const unsigned cd = cropMeta[pp] & 63u;
          if (!(cd & 32u)) {
            ra = single_ring ? 0 : (int)(cd & 15u);
            if ((cd & 16u) && !single_ring) rb = ra + 1;
            const bool ina = (ra >= r0 && ra < r1), inb = (rb >= r0 && rb < r1);
            if (!ina && inb) { ra = rb; rb = -1; }
            if (!inb) rb = -1;
            take = (ina ? 1 : 0) + (inb ? 1 : 0);
          }
        }
        int t2;
        const int pos = block_excl_scan<NT>(take, &t2, sc);
        if (take && run + pos + take <= CAP) {  // the bound only bites on the uncounted attempt
          const float4 q = crop[pp];
          int e = run + pos;
          S.x[e] = q.x; S.y[e] = q.y; S.z[e] = q.z; S.gref[e] = (unsigned)pp; S.ring[e] = (unsigned char)(ra - r0);
          if (take == 2) {
            e++;
            S.x[e] = q.x; S.y[e] = q.y; S.z[e] = q.z; S.gref[e] = (unsigned)pp; S.ring[e] = (unsigned char)(rb - r0);
          }
        }
        run += t2;
      }
      __syncthreads();
      if (run > CAP) { whole = false; continue; }  // uncounted attempt did not fit: count, then go ring group by ring group
      __syncthreads();
      const int E = run;
      ClusterOut C;
      cluster_extract<NT>(S, E, P.tol_f, P.r2f_cluster, P.min_count, P.max_count, r1 - r0, BRUTE_PAIRS_RINGS, C);
      // ---- getCylinderSegments gate + centroid per cluster (src:282-325), one thread each ----
      int* sh = sc + 100;  // [0] = pool base, [1] = kc base
      int runG = 0, runM = 0;
      // pass 0 counts, pass 1 writes; with a single tile of clusters (the usual case) pass 1 reuses
      // the registers of pass 0 instead of walking the member lists again
      const bool oneTile = (C.nC <= NT);
      int ok = 0, size = 0, pg = 0, pm = 0;
      float4 cen = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int pass = 0; pass < 2; pass++) {
        int accG = 0, accM = 0;
        for (int i0 = 0; i0 < C.nC; i0 += NT) {
          const int i = i0 + tid;
          int tg = 0, tm = 0;
          if (pass == 0 || !oneTile) {
            ok = 0; size = 0;
            cen = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < C.nC) {
              const unsigned root = C.slotRoot[i];
              size = (int)C.cnt[root];
              const int st = C.slotStart[i];
              double sumx = 0.0, sumy = 0.0, sumz = 0.0;
              double minx = 1000.0, maxx = -1000.0, miny = 1000.0, maxy = -1000.0;
              for (int j = 0; j < size; j++) {
                const int e = C.mem[st + j];
                const double x = S.x[e], y = S.y[e], z = S.z[e];
                sumx += x; sumy += y; sumz += z;
                if (x < minx) minx = x;
                if (y < miny) miny = y;
                if (x > maxx) maxx = x;
                if (y > maxy) maxy = y;
              }
              const double ddx = maxx - minx, ddy = maxy - miny;
              const double diameter = sqrt(__dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy)));
              if constexpr (sizeof...(G) > 0)
                if (pass == 0 && fabs(diameter - P.two_radius_threshold) < (gate.eps, ...)) atomicAdd(&(gate.cnt, ...)[s * 16], 1u);
              if (diameter < P.two_radius_threshold) {
                ok = 1;
                cen.x = (float)(sumx / (double)size);
                cen.y = (float)(sumy / (double)size);
                cen.z = (float)(sumz / (double)size);
              }
            }
            pg = block_excl_scan<NT>(ok, &tg, sc);
            if (kcPool) pm = block_excl_scan<NT>(ok ? size : 0, &tm, sc);
          }
          if (pass == 1 && ok) {
            const int b = sh[0];
            if (b >= 0) {
              cen.w = crop[S.gref[C.slotRoot[i]]].w;  // intensity of indices[0] (src:320)
              kfPool[b + accG + pg] = cen;
            }
            if (kcPool && sh[1] >= 0) {
              const int st = C.slotStart[i];
              for (int j = 0; j < size; j++) kcPool[sh[1] + accM + pm + j] = crop[S.gref[C.mem[st + j]]];
            }
          }
          accG += tg; accM += tm;
        }
        if (pass == 0) {
          runG = accG; runM = accM;
          __syncthreads();
          if (tid == 0) {
            int b = -1, bc = -1;
            if (runG > 0) {
              b = atomicAdd(&ctr->kf_cursor, runG);
              if (b + runG > kfCap) { atomicOr(&ctr->err, ERR_KF_POOL); b = -1; }
            }
            if (kcPool && runM > 0) {
              bc = atomicAdd(&ctr->kc_cursor, runM);
              if (bc + runM > kcCap) { atomicOr(&ctr->err, ERR_KC_POOL); bc = -1; }
            }
            sh[0] = b; sh[1] = bc;
            kfBase[s * 16 + group] = max(b, 0);
            kfCnt[s * 16 + group] = (b >= 0) ? runG : 0;
            if (kcBase) { kcBase[s * 16 + group] = max(bc, 0); kcCnt[s * 16 + group] = (bc >= 0) ? runM : 0; }
          }
          __syncthreads();
          if (runG == 0) break;
        }
      }
      __syncthreads();
      group++;
    }
    r0 = r1;
  }
}

// scanList == nullptr: block b handles scan b and defers oversized scans to ovfList;
// otherwise the blocks loop over scanList[0 .. *nList) (the deferred scans).  gate...: nothing, or a GateCount.
template <int CAP, int NT, int MINB, bool GLOBAL, class... G>
__global__ void __launch_bounds__(NT, MINB) k_cluster_rings(
    const float4* __restrict__ crop, const unsigned* __restrict__ cropMeta,
    const int* __restrict__ cropCnt, const long long* __restrict__ scan_off,
    const int* __restrict__ chunk_off, DevParams P, int single_ring,
    float4* __restrict__ kfPool, int kfCap, int* __restrict__ kfBase, int* __restrict__ kfCnt,
    float4* __restrict__ kcPool, int kcCap, int* __restrict__ kcBase, int* __restrict__ kcCnt,
    DevCounters* __restrict__ ctr, const int* __restrict__ scanList, const int* __restrict__ nList,
    int* __restrict__ ovfList, int* __restrict__ ovfCount, unsigned char* __restrict__ slabs, G... gate) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ClusterSm S;
  if (GLOBAL) cluster_carve_global<CAP, NT>(slabs + (size_t)blockIdx.x * cluster_slab_bytes(CAP), smem_raw, S);
  else cluster_sm_carve<CAP, NT>(smem_raw, S);
  if (!scanList) {
    cluster_rings_scan<CAP, NT>(S, blockIdx.x, crop, cropMeta, cropCnt, scan_off, chunk_off, P, single_ring, kfPool, kfCap,
                            kfBase, kfCnt, kcPool, kcCap, kcBase, kcCnt, ctr, ovfList, ovfCount, gate...);
  } else {
    const int n = *nList;
    for (int i = blockIdx.x; i < n; i += gridDim.x) {
      __syncthreads();
      cluster_rings_scan<CAP, NT>(S, scanList[i], crop, cropMeta, cropCnt, scan_off, chunk_off, P, single_ring, kfPool, kfCap,
                              kfBase, kfCnt, kcPool, kcCap, kcBase, kcCnt, ctr, ovfList, ovfCount, gate...);
    }
  }
}

}  // namespace fe
#include "fe_ring_runs.cuh"
namespace fe {

// ============================================================================================
// K3 — cross-ring merge (src:205-257) for one scan per block; also the stage kernel behind
// fe_extract_clusters when `stage` != 0 (then it just reports the clusters of `crop`).
// ============================================================================================
template <int CAP, int NT>
__device__ void merge_keypoints_scan(
    ClusterSm& S, const int s, const float4* __restrict__ kfPool, const int* __restrict__ kfBase,
    const int* __restrict__ kfCnt, const DevParams& P, float4* __restrict__ kpPool, int kpCap,
    int* __restrict__ kpBase, int* __restrict__ kpCnt, DevCounters* __restrict__ ctr,
    int* __restrict__ ovfList, int* __restrict__ ovfCount) {
  const int tid = threadIdx.x;
  int* sc = S.misc + MAXCHUNK + 1;
  int* pre = S.misc;  // 17 prefix entries of the pieces
  if (tid == 0) {
    int run = 0;
    for (int g = 0; g < 16; g++) { pre[g] = run; run += kfCnt[s * 16 + g]; }
    pre[16] = run;
    kpBase[s] = 0; kpCnt[s] = 0;
  }
  __syncthreads();
  const int Kf = pre[16];
  if (Kf == 0) return;
  if (Kf > CAP) {
    if (tid == 0) {
      if (ovfList) ovfList[atomicAdd(ovfCount, 1)] = s;  // the next larger instantiation takes it
      else atomicOr(&ctr->err, ERR_MERGE_CAP);
    }
    return;
  }
  for (int i = tid; i < Kf; i += NT) {
    int g = 0;
    while (g < 15 && pre[g + 1] <= i) g++;
    const int src = kfBase[s * 16 + g] + (i - pre[g]);
    const float4 q = kfPool[src];
    S.x[i] = q.x; S.y[i] = q.y;
    // src:217 — z replaced by intensity*0.75*clusterRadiusThreshold/2 (double, narrowed to float)
    S.z[i] = (float)__ddiv_rn(__dmul_rn(__dmul_rn((double)q.w, 0.75), P.radius_threshold), 2.0);
    S.gref[i] = (unsigned)src;
    S.ring[i] = 0;
  }
  __syncthreads();
  ClusterOut C;
  cluster_extract<NT>(S, Kf, P.merge_tol_f, P.r2f_merge, P.min_channels, 16, 1, BRUTE_PAIRS_MERGE, C);
  if (C.nC == 0) return;
  int* sh = sc + 100;
  if (tid == 0) {
    int b = atomicAdd(&ctr->kp_cursor, C.nC);
    if (b + C.nC > kpCap) { atomicOr(&ctr->err, ERR_KP_POOL); b = -1; }
    sh[0] = b;
    kpBase[s] = max(b, 0);
    kpCnt[s] = (b >= 0) ? C.nC : 0;
  }
  __syncthreads();
  const int b = sh[0];
  if (b < 0) return;
  for (int i = tid; i < C.nC; i += NT) {
    const unsigned root = C.slotRoot[i];
    const int size = (int)C.cnt[root];
    const int st = C.slotStart[i];
    double sumx = 0.0, sumy = 0.0, sumz = 0.0;
    for (int j = 0; j < size; j++) {
      const int e = C.mem[st + j];
      sumx += (double)S.x[e];
      sumy += (double)S.y[e];
      sumz += (double)kfPool[S.gref[e]].z;  // the real z, restored at src:231-232
    }
    float4 kp;
    kp.x = (float)(sumx / (double)size);
    kp.y = (float)(sumy / (double)size);
    kp.z = (float)(sumz / (double)size);
    kp.w = kfPool[S.gref[root]].w;  // src:254
    kpPool[b + i] = kp;
  }
}

template <int CAP, int NT, int MINB, bool GLOBAL>
__global__ void __launch_bounds__(NT, MINB) k_merge_keypoints(
    const float4* __restrict__ kfPool, const int* __restrict__ kfBase, const int* __restrict__ kfCnt,
    DevParams P, float4* __restrict__ kpPool, int kpCap, int* __restrict__ kpBase,
    int* __restrict__ kpCnt, DevCounters* __restrict__ ctr, const int* __restrict__ scanList,
    const int* __restrict__ nList, int* __restrict__ ovfList, int* __restrict__ ovfCount,
    unsigned char* __restrict__ slabs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ClusterSm S;
  if (GLOBAL) cluster_carve_global<CAP, NT>(slabs + (size_t)blockIdx.x * cluster_slab_bytes(CAP), smem_raw, S);
  else cluster_sm_carve<CAP, NT>(smem_raw, S);
  if (!scanList) {
    merge_keypoints_scan<CAP, NT>(S, blockIdx.x, kfPool, kfBase, kfCnt, P, kpPool, kpCap, kpBase, kpCnt, ctr, ovfList, ovfCount);
  } else {
    const int n = *nList;
    for (int i = blockIdx.x; i < n; i += gridDim.x) {
      __syncthreads();
      merge_keypoints_scan<CAP, NT>(S, scanList[i], kfPool, kfBase, kfCnt, P, kpPool, kpCap, kpBase, kpCnt, ctr, ovfList, ovfCount);
    }
  }
}

// Stage kernel: plain EuclideanClusterExtraction of n points (one block), CSR result.
template <bool GLOBAL>
__global__ void __launch_bounds__(NT2, 1) k_extract_clusters_stage(
    const float4* __restrict__ pts, int n, float tol_f, float r2f, int minSz, int maxSz,
    int* __restrict__ offsets, int capClusters, int* __restrict__ indices, int* __restrict__ nOut,
    unsigned char* __restrict__ slabs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ClusterSm S;
  if (GLOBAL) cluster_carve_global<ECAP_G, NT2>(slabs, smem_raw, S);
  else cluster_sm_carve<ECAP_L, NT2>(smem_raw, S);
  const int tid = threadIdx.x;
  for (int i = tid; i < n; i += NT2) {
    const float4 q = pts[i];
    S.x[i] = q.x; S.y[i] = q.y; S.z[i] = q.z; S.gref[i] = (unsigned)i; S.ring[i] = 0;
  }
  __syncthreads();
  ClusterOut C;
  cluster_extract<NT2>(S, n, tol_f, r2f, minSz, maxSz, 1, BRUTE_PAIRS_RINGS, C);
  if (tid == 0) { nOut[0] = C.nC; offsets[0] = 0; }
  if (C.nC > capClusters) return;
  for (int i = tid; i < C.nC; i += NT2) {
    const int size = (int)C.cnt[C.slotRoot[i]];
    const int st = C.slotStart[i];
    offsets[i + 1] = st + size;
    for (int j = 0; j < size; j++) indices[st + j] = (int)C.mem[st + j];
  }
}

// ============================================================================================
// Keypoint CSR offsets (one block) and ordered copy of the keypoints out of the pool.
// ============================================================================================
__global__ void __launch_bounds__(1024) k_kp_offsets(const int* __restrict__ kpCnt, int n_scans,
                                                      int* __restrict__ kpOff, DevCounters* ctr) {
  __shared__ int sc[40];
  int run = 0;
  for (int s0 = 0; s0 < n_scans; s0 += 1024) {
    const int s = s0 + threadIdx.x;
    const int v = (s < n_scans) ? kpCnt[s] : 0;
    int tot;
    const int pos = block_excl_scan<1024>(v, &tot, sc);
    if (s < n_scans) kpOff[s] = run + pos;
    run += tot;
  }
  if (threadIdx.x == 0) { kpOff[n_scans] = run; ctr->kp_total = run; }
}

__device__ __forceinline__ int scan_of_keypoint(const int* __restrict__ kpOff, int n_scans, int g) {
  int lo = 0, hi = n_scans - 1;  // largest s with kpOff[s] <= g
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (kpOff[mid] <= g) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__global__ void k_kp_gather(const float4* __restrict__ kpPool, const int* __restrict__ kpBase,
                            const int* __restrict__ kpOff, int n_scans, float4* __restrict__ kpOut,
                            int* __restrict__ kpScan) {
  const int total = kpOff[n_scans];
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < total; g += gridDim.x * blockDim.x) {
    const int s = scan_of_keypoint(kpOff, n_scans, g);
    kpOut[g] = kpPool[kpBase[s] + (g - kpOff[s])];
    kpScan[g] = s;
  }
}

// Both steps in one launch for a call of at most 32 scans (one block; a warp copies a scan's keypoints).
__global__ void __launch_bounds__(1024) k_kp_offsets_gather_small(const int* __restrict__ kpCnt, int n_scans, int* __restrict__ kpOff,
                                                                   DevCounters* ctr, const float4* __restrict__ kpPool,
                                                                   const int* __restrict__ kpBase, float4* __restrict__ kpOut,
                                                                   int* __restrict__ kpScan) {
  __shared__ int sc[40];
  __shared__ int s_off[33];
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const int v = (t < n_scans) ? kpCnt[t] : 0;
  int tot;
  const int pos = block_excl_scan<1024>(v, &tot, sc);
  if (t < n_scans) { kpOff[t] = pos; s_off[t] = pos; }
  if (t == 0) { kpOff[n_scans] = tot; s_off[n_scans] = tot; ctr->kp_total = tot; }
  __syncthreads();
  if (w < n_scans) {
    const int o = s_off[w], n = s_off[w + 1] - o, b = kpBase[w];
    for (int i = lane; i < n; i += 32) { kpOut[o + i] = kpPool[b + i]; kpScan[o + i] = w; }
  }
}

// Concatenate chunk pieces (or pool pieces) of every scan into a dense CSR array.
__global__ void k_piece_counts(const int* __restrict__ cnt, const int* __restrict__ chunk_off,
                               int n_scans, int* __restrict__ perScan) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_scans) return;
  int t = 0;
  for (int c = chunk_off[s]; c < chunk_off[s + 1]; c++) t += cnt[c];
  perScan[s] = t;
}

__global__ void __launch_bounds__(256) k_gather_chunks(
    const float4* __restrict__ src, const int* __restrict__ cnt, const long long* __restrict__ scan_off,
    const int* __restrict__ chunk_off, const int* __restrict__ outOff, float4* __restrict__ dst) {
  // one block per scan; chunk after chunk
  const int s = blockIdx.x;
  long long o = outOff[s];
  const long long base = scan_off[s];
  const int c0 = chunk_off[s], c1 = chunk_off[s + 1];
  for (int c = c0; c < c1; c++) {
    const int n = cnt[c];
    for (int j = threadIdx.x; j < n; j += blockDim.x) dst[o + j] = src[base + (long long)(c - c0) * CH + j];
    o += n;
  }
}

__global__ void __launch_bounds__(256) k_gather_pool16(
    const float4* __restrict__ pool, const int* __restrict__ pBase, const int* __restrict__ pCnt,
    const int* __restrict__ outOff, float4* __restrict__ dst) {
  const int s = blockIdx.x;
  long long o = outOff[s];
  for (int g = 0; g < 16; g++) {
    const int n = pCnt[s * 16 + g], b = pBase[s * 16 + g];
    for (int j = threadIdx.x; j < n; j += blockDim.x) dst[o + j] = pool[b + j];
    o += n;
  }
}

// exclusive prefix of n counts (one block): off[0..n], off[n] = total
__global__ void __launch_bounds__(1024) k_offsets_scan(const int* __restrict__ cnt, int n, int* __restrict__ off) {
  __shared__ int sc[40];
  int run = 0;
  for (int s0 = 0; s0 < n; s0 += 1024) {
    const int s = s0 + threadIdx.x;
    const int v = (s < n) ? cnt[s] : 0;
    int tot;
    const int pos = block_excl_scan<1024>(v, &tot, sc);
    if (s < n) off[s] = run + pos;
    run += tot;
  }
  if (threadIdx.x == 0) off[n] = run;
}

__global__ void k_pool16_counts(const int* __restrict__ pCnt, int n_scans, int* __restrict__ perScan) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_scans) return;
  int t = 0;
  for (int g = 0; g < 16; g++) t += pCnt[s * 16 + g];
  perScan[s] = t;
}

// ============================================================================================
// K4a — 2-D cell grid of the descriptor search surface, one scan per block: radix sort of
// (cell key, source position) through global memory (L2-resident: a scan is a few hundred KB),
// then the sorted point array, its key array and a per-row start table.
// ============================================================================================
__device__ __forceinline__ int surf_cell(float v, float o, float inv, int n) {
  int c = (int)floorf((v - o) * inv);
  return max(0, min(c, n - 1));
}

struct SurfGlobalSm {
  int pre[MAXCHUNK + 1];
  int sc[40];
  unsigned wc[(NT2 / 32) * 257];
  unsigned rbase[256 + 32];
};

__device__ void surface_grid_scan_global(
    SurfGlobalSm& M, const int s, const float4* __restrict__ surf, const int* __restrict__ surfCnt,
    const long long* __restrict__ scan_off, const int* __restrict__ chunk_off, const DevParams& P,
    unsigned* __restrict__ keyA, unsigned* __restrict__ keyB, unsigned* __restrict__ valA,
    unsigned* __restrict__ valB, float4* __restrict__ sorted, unsigned* __restrict__ sortedKey,
    int* __restrict__ rowStart, int* __restrict__ surfN, DevCounters* __restrict__ ctr, int* __restrict__ rho) {
  int* pre = M.pre;
  int* sc = M.sc;
  unsigned* wc = M.wc;
  unsigned* rbase = M.rbase;
  const int tid = threadIdx.x;
  const long long base = scan_off[s];
  const int nch = chunk_off[s + 1] - chunk_off[s];
  int* rs = rowStart + (long long)s * (P.sg_ny + 1);
  if (nch > MAXCHUNK) { if (tid == 0) { atomicOr(&ctr->err, ERR_CHUNKS); surfN[s] = 0; } return; }
  const int n = chunk_prefix<NT2>(surfCnt + chunk_off[s], nch, pre, sc);
  if (tid == 0) surfN[s] = n;
  if (n == 0) {
    for (int r = tid; r <= P.sg_ny; r += NT2) rs[r] = 0;
    return;
  }
  unsigned* kA = keyA + base; unsigned* kB = keyB + base;
  unsigned* vA = valA + base; unsigned* vB = valB + base;
  for (int i = tid; i < n; i += NT2) rho[base + i] = 0;
  for (int i = tid; i < n; i += NT2) {
    const long long pp = piece_pos(pre, nch, i, base);
    const float4 q = surf[pp];
    const int cx = surf_cell(q.x, P.sx0, P.sg_inv, P.sg_nx), cy = surf_cell(q.y, P.sy0, P.sg_inv, P.sg_ny);
    kA[i] = ((unsigned)cy << P.sg_bx) | (unsigned)cx;
    vA[i] = (unsigned)(pp - base);
  }
  const int keybits = P.sg_bx + bits_for(P.sg_ny - 1);
  unsigned *kS = kA, *kT = kB, *vS = vA, *vT = vB;
  for (int shift = 0; shift < keybits; shift += 8) {
    unsigned* ki = kS; unsigned* ko = kT; unsigned* vi = vS; unsigned* vo = vT;
    block_radix_pass<NT2, unsigned>(
        n, [=](int i) { return (ki[i] >> shift) & 255u; },
        [=](int i, int pos) { ko[pos] = ki[i]; vo[pos] = vi[i]; }, wc, rbase);
    kS = ko; kT = ki; vS = vo; vT = vi;
  }
  __syncthreads();
  float4* so = sorted + base;
  unsigned* sk = sortedKey + base;
  for (int i = tid; i < n; i += NT2) {
    const unsigned k = kS[i];
    so[i] = surf[base + vS[i]];
    sk[i] = k;
    const int r = (int)(k >> P.sg_bx);
    const int rp = (i == 0) ? -1 : (int)(kS[i - 1] >> P.sg_bx);
    for (int rr = rp + 1; rr <= r; rr++) rs[rr] = i;
    if (i == n - 1) for (int rr = r + 1; rr <= P.sg_ny; rr++) rs[rr] = n;
  }
}


// Global-memory K4a.  scanList == nullptr: block b sorts scan b; otherwise the blocks loop over the
// scans the shared-memory instantiation deferred.
__global__ void __launch_bounds__(NT2, 2) k_surface_grid(
    const float4* __restrict__ surf, const int* __restrict__ surfCnt,
    const long long* __restrict__ scan_off, const int* __restrict__ chunk_off, DevParams P,
    unsigned* __restrict__ keyA, unsigned* __restrict__ keyB, unsigned* __restrict__ valA,
    unsigned* __restrict__ valB, float4* __restrict__ sorted, unsigned* __restrict__ sortedKey,
    int* __restrict__ rowStart, int* __restrict__ surfN, DevCounters* __restrict__ ctr,
    const int* __restrict__ scanList, const int* __restrict__ nList, int* __restrict__ tabOk, int* __restrict__ rho) {
  __shared__ SurfGlobalSm M;
  if (!scanList) {
    if (threadIdx.x == 0) tabOk[blockIdx.x] = 0;
    surface_grid_scan_global(M, blockIdx.x, surf, surfCnt, scan_off, chunk_off, P, keyA, keyB, valA, valB, sorted, sortedKey,
                             rowStart, surfN, ctr, rho);
  } else {
    const int n = *nList;
    for (int i = blockIdx.x; i < n; i += gridDim.x) {
      __syncthreads();
      if (threadIdx.x == 0) tabOk[scanList[i]] = 0;
      surface_grid_scan_global(M, scanList[i], surf, surfCnt, scan_off, chunk_off, P, keyA, keyB, valA, valB, sorted,
                               sortedKey, rowStart, surfN, ctr, rho);
    }
  }
}

// Shared-memory K4a: a counting sort by grid cell.  Nothing downstream depends on the order of the
// points inside a cell (K4b marks, K4c counts, K4d orders its records itself), so the sort is:
// count the points of every cell (16-bit counters, two per shared-memory word), exclusive-scan the
// cells (their starts; the row starts fall out of it), then scatter every point to the next free
// slot of its cell.  Two coalesced sweeps over the scan's surface pieces, no key/value ping-pong.
// Scans with more than 65,535 surface points (16-bit counters) are deferred to the radix kernel.
constexpr int NT_SURF = 512;           // threads of the counting-sort K4a (384 was measured: slower)
constexpr int SURF_MAX_CELLS = 57344;  // 112 KB of counters: 2 blocks / SM at the upper end

// The cell grid only ever serves the 3DSC stage, and that only looks at surface points within R of a
// keypoint (support) or within R + R/5 (density of the support points).  The kernel therefore runs after
// the keypoints are known and keeps only the points of HALO cells — cells a keypoint's box of half-width
// R + R/5 touches (a bit map in shared memory) — which is a few percent of a sparse scan.  Scans without
// keypoints are not read at all.  Halo cells are numbered in cell order (rank = bits set before the cell:
// a per-word prefix plus a popcount), and every halo cell is cut into NS z slabs: the counting sort runs
// over (rank, slab), so that a cell's points are grouped by slab and the density sweep (K4c) visits only
// the slabs its z window touches, while a row of cells over all slabs is still one contiguous span for
// the support sweeps (K4b, K4d).  NS = min(16, GRID_TAB_CAP / halo cells) per scan.
// Per-scan index in global memory (GridHdr): bit map | word prefix | NS, halo cells | slot table.
constexpr int GRID_TAB_CAP = 28672;     // (halo cell, slab) counters per scan: 56 KB of 16-bit counters in shared memory
constexpr int GRID_MAX_SLABS = 16;
constexpr int GRID_SLAB_MIN_POINTS = 20000;  // surface points of a scan from which its cells are cut into z slabs
__host__ __device__ constexpr long long grid_hdr_bytes(int ncells) {
  // bitmap words, word prefix (u16, one extra, padded to 4 B), 2 meta words, table (u16, TAB_CAP + 2)
  return (long long)((ncells + 31) / 32) * 4 + (long long)((((ncells + 31) / 32) + 2) / 2) * 4 + 8 + (long long)(GRID_TAB_CAP + 2) * 2;
}
constexpr size_t surf_cells_smem_bytes(int ncells) {
  return (size_t)((GRID_TAB_CAP + 2) / 2) * 4 + 64 + (size_t)((ncells + 31) / 32) * 4 + 16 + (size_t)((ncells + 31) / 32 + 2) * 2 + 16;
}

__device__ __forceinline__ int z_slab(float z, float zs0, float zs_scale, int ns) {
  const int l = (int)floorf((z - zs0) * zs_scale);
  return max(0, min(l, ns - 1));
}

template <int NTS>
__global__ void __launch_bounds__(NTS) k_surface_grid_cells(
    const float4* __restrict__ surf, const int* __restrict__ surfCnt,
    const long long* __restrict__ scan_off, const int* __restrict__ chunk_off, DevParams P,
    const float4* __restrict__ kpOut, const int* __restrict__ kpOff,
    float4* __restrict__ sorted, int* __restrict__ rho,
    int* __restrict__ surfN, DevCounters* __restrict__ ctr, int* __restrict__ ovfList,
    unsigned char* __restrict__ gridHdr, long long gridStride, int* __restrict__ tabOk) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int nx = P.sg_nx, ny = P.sg_ny, ncells = nx * ny, nbm = (ncells + 31) / 32;
  unsigned* cnts = (unsigned*)smem_raw;                   // packed pairs of 16-bit counters / cursors over (rank, slab)
  unsigned* halo = cnts + ((GRID_TAB_CAP + 2) / 2) + 16;  // one bit per cell
  unsigned short* wpre = (unsigned short*)(halo + nbm + 4);  // halo cells before every bit-map word
  __shared__ int sc[40];
  __shared__ int s_n, s_hc, s_hl;
  const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  constexpr int NW = NTS / 32;
  const long long base = scan_off[s];
  const int c0 = chunk_off[s];
  const int nch = chunk_off[s + 1] - c0;
  const int k0 = kpOff[s], k1 = kpOff[s + 1];
  if (tid == 0) s_hl = 0;
  if (k1 == k0) {  // no keypoint: nothing of this scan's surface is ever looked at
    if (tid == 0) { surfN[s] = 0; tabOk[s] = 1; }
    return;
  }
  // total surface points of the scan (the 16-bit slots hold at most 65,535 of them)
  {
    int v = 0;
    for (int c = tid; c < nch; c += NTS) v += surfCnt[c0 + c];
    int tot;
    block_excl_scan<NTS>(v, &tot, sc);
    if (tid == 0) s_n = tot;
  }
  for (int i = tid; i < nbm; i += NTS) halo[i] = 0u;
  __syncthreads();
  if (s_n > 65535) {
    if (tid == 0) { ovfList[atomicAdd(&ctr->ovf_surf, 1)] = s; tabOk[s] = 0; }
    return;
  }
  // (0) halo cells: a warp per keypoint, lanes over the cells of its box
  for (int k = k0 + w; k < k1; k += NW) {
    const float4 o = kpOut[k];
    if (!finite3(o.x, o.y, o.z)) continue;
    const int cx0 = surf_cell(o.x - P.halopad, P.sx0, P.sg_inv, nx), cx1 = surf_cell(o.x + P.halopad, P.sx0, P.sg_inv, nx);
    const int cy0 = surf_cell(o.y - P.halopad, P.sy0, P.sg_inv, ny), cy1 = surf_cell(o.y + P.halopad, P.sy0, P.sg_inv, ny);
    const int bw = cx1 - cx0 + 1, nb = bw * (cy1 - cy0 + 1);
    for (int t = lane; t < nb; t += 32) {
      const int cell = (cy0 + t / bw) * nx + cx0 + t % bw;
      atomicOr(&halo[cell >> 5], 1u << (cell & 31));
    }
  }
  __syncthreads();
  // (1) rank of every halo cell: exclusive prefix of the words' popcounts
  {
    int run = 0;
    for (int w0 = 0; w0 < nbm; w0 += NTS) {
      const int i = w0 + tid;
      const int v = (i < nbm) ? __popc(halo[i]) : 0;
      int tot;
      const int pos = block_excl_scan<NTS>(v, &tot, sc);
      if (i < nbm) wpre[i] = (unsigned short)(run + pos);
      run += tot;
    }
    if (tid == 0) { wpre[nbm] = (unsigned short)run; s_hc = run; }
  }
  __syncthreads();
  const int hc = s_hc;
  // z slabs pay when cell columns are long, i.e. for dense sensors (measured: 4x azimuth density, K4c 13.9 ->
  // 11.3 ms; at the VLP-16's own density the per-cell lookups cost what the skipped tests save)
  const int NS = (s_n >= GRID_SLAB_MIN_POINTS) ? max(1, min(GRID_MAX_SLABS, GRID_TAB_CAP / max(hc, 1))) : 1;
  if (hc > GRID_TAB_CAP) {  // more halo cells than counters: the radix kernel takes the scan
    if (tid == 0) { ovfList[atomicAdd(&ctr->ovf_surf, 1)] = s; tabOk[s] = 0; }
    return;
  }
  const int nslots = hc * NS, nwords = (nslots + 2) / 2;
  const float zscale = (float)NS * P.zs_inv_range;
  for (int i = tid; i < nwords; i += NTS) cnts[i] = 0u;
  __syncthreads();
  auto slot_of = [&](float x, float y, float z) -> int {  // (rank, slab) counter of a point, -1 outside the halo
    const int cell = surf_cell(y, P.sy0, P.sg_inv, ny) * nx + surf_cell(x, P.sx0, P.sg_inv, nx);
    const unsigned bits = halo[cell >> 5];
    if (!((bits >> (cell & 31)) & 1u)) return -1;
    const int rk = (int)wpre[cell >> 5] + __popc(bits & ((1u << (cell & 31)) - 1u));
    return rk * NS + z_slab(z, P.zs0, zscale, NS);
  };
  // (2) count: the survivors of a chunk are contiguous; the chunks are cut into runs of 128 points that
  //     are dealt to the warps, four 16-byte loads in flight per lane.  The halo points found (a few percent
  //     of a sparse scan) are also listed — (piece position, slot) pairs in the unused tail of the counter
  //     array — so that the scatter pass touches only them instead of streaming the surface a second time.
  unsigned* hlist = cnts + ((nwords + 3) & ~3);
  const int hlCap = max(0, ((GRID_TAB_CAP + 2) / 2 - ((nwords + 3) & ~3)) / 2);
  for (int it = w; it < nch * (CH / 128); it += NW) {
    const int c = it / (CH / 128);
    const int j1 = surfCnt[c0 + c];
    const float4* src = surf + base + (long long)c * CH;
    const int j = (it % (CH / 128)) * 128 + lane;
    if (j - lane >= j1) continue;
    float4 q[4];
#pragma unroll
    for (int k = 0; k < 4; k++) q[k] = (j + 32 * k < j1) ? src[j + 32 * k] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      int sl = -1;
      if (j + 32 * k < j1) sl = slot_of(q[k].x, q[k].y, q[k].z);
      if (sl >= 0) atomicAdd(&cnts[sl >> 1], (sl & 1) ? 65536u : 1u);
      const unsigned hm = __ballot_sync(FE_FULL, sl >= 0);
      if (hm) {
        int at = 0;
        if (lane == __ffs(hm) - 1) at = atomicAdd(&s_hl, __popc(hm));
        at = __shfl_sync(FE_FULL, at, __ffs(hm) - 1) + __popc(hm & lanemask_lt());
        if (sl >= 0 && at < hlCap) { hlist[2 * at] = (unsigned)(c * CH + j + 32 * k); hlist[2 * at + 1] = (unsigned)sl; }
      }
    }
  }
  __syncthreads();
  // (3) exclusive scan over the (rank, slab) counters in key order; every thread owns a run of whole words
  {
    const int per = (nwords + NTS - 1) / NTS;
    const int wb = min(tid * per, nwords), we = min(wb + per, nwords);
    int sum = 0;
    for (int i = wb; i < we; i++) { const unsigned v = cnts[i]; sum += (int)(v & 0xFFFFu) + (int)(v >> 16); }
    int tot;
    int run = block_excl_scan<NTS>(sum, &tot, sc);
    for (int i = wb; i < we; i++) {
      const unsigned v = cnts[i];
      const int lo = (int)(v & 0xFFFFu), hi = (int)(v >> 16);
      cnts[i] = (unsigned)run | ((unsigned)(run + lo) << 16);  // starts of the two slots
      run += lo + hi;
    }
    if (tid == 0) s_n = tot;  // halo points only
  }
  __syncthreads();
  const int n = s_n;
  if (tid == 0) { surfN[s] = n; tabOk[s] = 1; }
  // the scan's index for K4b-d: bit map, word prefix, NS / halo cells, and the table of slot starts — exactly
  // the packed words (low half = even slot; entry nslots, the end of the last slot, is n by construction
  // because the unused tail counters are zero)
  {
    unsigned* g = (unsigned*)(gridHdr + (long long)s * gridStride);
    for (int i = tid; i < nbm; i += NTS) g[i] = halo[i];
    unsigned* gp = g + nbm;
    const unsigned* wp32 = (const unsigned*)wpre;
    const int npw = (nbm + 2) / 2;
    for (int i = tid; i < npw; i += NTS) gp[i] = wp32[i];
    unsigned* gm = gp + npw;
    if (tid == 0) { gm[0] = (unsigned)NS; gm[1] = (unsigned)hc; }
    unsigned* gt = gm + 2;
    for (int i = tid; i < nwords; i += NTS) gt[i] = cnts[i];
  }
  for (int i = tid; i < n; i += NTS) rho[base + i] = 0;  // K4b marks, K4c counts: only these slots are ever used
  __syncthreads();
  if (n == 0) return;
  // (4) scatter: the start of a slot doubles as its cursor (it ends at the slot's end <= n <= 65535, so a
  //     16-bit half never carries into its neighbour); the order inside a slot is free
  float4* so = sorted + base;
  if (s_hl <= hlCap) {  // every halo point is listed
    const int nl = s_hl;
    for (int e = tid; e < nl; e += NTS) {
      const unsigned sl = hlist[2 * e + 1];
      const float4 q = surf[base + hlist[2 * e]];
      const unsigned old = atomicAdd(&cnts[sl >> 1], (sl & 1) ? 65536u : 1u);
      so[(sl & 1) ? (int)(old >> 16) : (int)(old & 0xFFFFu)] = q;
    }
    return;
  }
  for (int it = w; it < nch * (CH / 128); it += NW) {
    const int c = it / (CH / 128);
    const int j1 = surfCnt[c0 + c];
    const float4* src = surf + base + (long long)c * CH;
    const int j = (it % (CH / 128)) * 128 + lane;
    if (j - lane >= j1) continue;
    float4 q[4];
#pragma unroll
    for (int k = 0; k < 4; k++) q[k] = (j + 32 * k < j1) ? src[j + 32 * k] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (j + 32 * k < j1) {
        const int sl = slot_of(q[k].x, q[k].y, q[k].z);
        if (sl >= 0) {
          const unsigned old = atomicAdd(&cnts[sl >> 1], (sl & 1) ? 65536u : 1u);
          so[(sl & 1) ? (int)(old >> 16) : (int)(old & 0xFFFFu)] = q[k];
        }
      }
    }
  }
}

// How K4b-d find the sorted positions of a cell range: through the per-scan index that the counting-sort
// K4a publishes (bit map of halo cells, word prefix -> rank of a cell, table of (rank, slab) slot starts),
// or — for scans that went through the radix kernel — by binary search in the sorted keys inside the row.
struct SurfIndex {
  const unsigned* sortedKey;      // keys of the sorted points (CSR by scan); radix path only
  const int* rowStart;            // [scan][ny+1]; radix path only
  const unsigned char* gridHdr;   // [scan] GridHdr blobs, may be null (grid too large for the counting sort)
  long long gridStride;
  const int* tabOk;               // [scan] 1: the scan has a GridHdr
};

struct ScanGrid {                 // one scan's view of the index
  const unsigned* bm;             // halo bit map; null: radix path
  const unsigned short* wpre;
  const unsigned short* tab;
  int ns, hc, ncells;
  const unsigned* sk;
  const int* rs;
  int nx, bx;
  float zs0, zscale;
  __device__ __forceinline__ int rank_lb(int cell) const {  // halo cells with a smaller index
    if (cell >= ncells) return hc;
    const unsigned bits = bm[cell >> 5];
    return (int)wpre[cell >> 5] + __popc(bits & ((1u << (cell & 31)) - 1u));
  }
  // span of sorted positions of row r whose cell x is in [cx0, cx1], all slabs
  __device__ __forceinline__ void row_span(int r, int cx0, int cx1, int& b, int& e) const {
    if (bm) {
      b = (int)tab[rank_lb(r * nx + cx0) * ns];
      e = (int)tab[rank_lb(r * nx + cx1 + 1) * ns];  // cx1 + 1 may be the first cell of the next row: still "cells before it"
      return;
    }
    const int rb = rs[r], re = rs[r + 1];
    const unsigned klo = ((unsigned)r << bx) | (unsigned)cx0, khi = ((unsigned)r << bx) | (unsigned)cx1;
    int lo = rb, hi = re;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (sk[mid] < klo) lo = mid + 1; else hi = mid; }
    b = lo;
    hi = re;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (sk[mid] <= khi) lo = mid + 1; else hi = mid; }
    e = lo;
  }
  // span of one cell restricted to slabs [l0, l1] (index path only)
  __device__ __forceinline__ void cell_slabs(int cell, int l0, int l1, int& b, int& e) const {
    const unsigned bits = bm[cell >> 5];
    if (!((bits >> (cell & 31)) & 1u)) { b = e = 0; return; }
    const int rk = (int)wpre[cell >> 5] + __popc(bits & ((1u << (cell & 31)) - 1u));
    b = (int)tab[rk * ns + l0];
    e = (int)tab[rk * ns + l1 + 1];
  }
  // span of one cell restricted to the slabs that [zlo, zhi] touches (index path only)
  __device__ __forceinline__ void cell_slab_span(int cell, float zlo, float zhi, int& b, int& e) const {
    const unsigned bits = bm[cell >> 5];
    if (!((bits >> (cell & 31)) & 1u)) { b = e = 0; return; }
    const int rk = (int)wpre[cell >> 5] + __popc(bits & ((1u << (cell & 31)) - 1u));
    b = (int)tab[rk * ns + z_slab(zlo, zs0, zscale, ns)];
    e = (int)tab[rk * ns + z_slab(zhi, zs0, zscale, ns) + 1];
  }
};

__device__ __forceinline__ ScanGrid scan_grid(const SurfIndex& X, int s, long long base, const DevParams& P) {
  ScanGrid G;
  G.sk = X.sortedKey + base;
  G.rs = X.rowStart + (long long)s * (P.sg_ny + 1);
  G.nx = P.sg_nx; G.bx = P.sg_bx;
  G.bm = nullptr; G.wpre = nullptr; G.tab = nullptr; G.ns = 1; G.hc = 0; G.ncells = P.sg_nx * P.sg_ny;
  G.zs0 = P.zs0; G.zscale = P.zs_inv_range;
  if (X.gridHdr && X.tabOk[s]) {
    const int nbm = (P.sg_nx * P.sg_ny + 31) / 32;
    const unsigned* g = (const unsigned*)(X.gridHdr + (long long)s * X.gridStride);
    G.bm = g;
    G.wpre = (const unsigned short*)(g + nbm);
    const unsigned* gm = g + nbm + (nbm + 2) / 2;
    G.ns = (int)gm[0];
    G.hc = (int)gm[1];
    G.tab = (const unsigned short*)(gm + 2);
    G.zscale = (float)G.ns * P.zs_inv_range;
  }
  return G;
}

// ============================================================================================
// K4b — mark the surface points inside the search sphere of any keypoint (3dsc.hpp
// searchForNeighbors with search_radius_), count each keypoint's neighbours and hand their sorted
// positions to K4d: the list is collected in shared memory and copied to a slice of `nbrPool`
// reserved with one atomic (kpNbrOff[g] = first slot, or -1 when a warp found more than
// MARK_WCAP or the pool is full — K4d then finds the neighbours itself).
// rho[i] = -(scan+1) marks "density needed".  One block per keypoint, grid-stride.
// ============================================================================================
constexpr int KD_BATCH = 4;   // keypoints a block of the fast K4d instantiation takes per request
constexpr int DCAP = 1536;    // K4d: contributions per keypoint of the fast instantiation (256 threads, 5 blocks / SM)
constexpr int DCAP_M = 4096;  // of the medium instantiation (512 threads, 2 blocks / SM)
constexpr int DCAP_L = 8192;  // of the large instantiation (512 threads, 1 block / SM)
constexpr int MARK_WCAP = 512;            // list entries per warp (16 KB per block: 8 blocks / SM stay resident)
constexpr int MARK_LCAP = 8 * MARK_WCAP;  // longer lists: K4d's larger instantiations find the neighbours themselves

__global__ void __launch_bounds__(256) k_desc_mark(
    const float4* __restrict__ kpOut, const int* __restrict__ kpScan, const int* __restrict__ kpOff,
    int n_scans, const float4* __restrict__ sorted, SurfIndex X, const long long* __restrict__ scan_off, DevParams P,
    int* __restrict__ rho, int* __restrict__ kpNbr, unsigned* __restrict__ nbrPool, long long nbrCap,
    int* __restrict__ kpNbrOff, DevCounters* __restrict__ ctr) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned* s_list = (unsigned*)smem_raw;  // [8 warps][MARK_WCAP]: every warp lists what it finds, no atomics
  __shared__ int s_wcnt[8];
  __shared__ long long s_off;
  const int total = kpOff[n_scans];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned* mylist = s_list + w * MARK_WCAP;
  for (int g = blockIdx.x; g < total; g += gridDim.x) {
    const float4 o = kpOut[g];
    const int s = kpScan[g];
    int wcnt = 0;
    if (finite3(o.x, o.y, o.z)) {
      const long long base = scan_off[s];
      const float4* so = sorted + base;
      const ScanGrid G = scan_grid(X, s, base, P);
      const int cx0 = surf_cell(o.x - P.Rpad, P.sx0, P.sg_inv, P.sg_nx), cx1 = surf_cell(o.x + P.Rpad, P.sx0, P.sg_inv, P.sg_nx);
      const int cy0 = surf_cell(o.y - P.Rpad, P.sy0, P.sg_inv, P.sg_ny), cy1 = surf_cell(o.y + P.Rpad, P.sy0, P.sg_inv, P.sg_ny);
      for (int r = cy0 + w; r <= cy1; r += 8) {
        int b, e;
        G.row_span(r, cx0, cx1, b, e);
        for (int i0 = b; i0 < e; i0 += 32) {
          const int i = i0 + lane;
          bool isn = false;
          if (i < e) {
            const float4 q = so[i];
            isn = l2_simple(o.x, o.y, o.z, q.x, q.y, q.z) < P.R2f;
            if (isn) rho[base + i] = -(s + 1);
          }
          const unsigned m = __ballot_sync(FE_FULL, isn);
          const int pos = wcnt + __popc(m & lanemask_lt());
          if (isn && pos < MARK_WCAP) mylist[pos] = (unsigned)i;
          wcnt += __popc(m);
        }
      }
    }
    if (lane == 0) s_wcnt[w] = wcnt;
    __syncthreads();
    int n = 0, before = 0;
    bool fits = true;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const int c = s_wcnt[k];
      if (k < w) before += c;
      n += c;
      fits = fits && (c <= MARK_WCAP);
    }
    if (threadIdx.x == 0) {
      kpNbr[g] = n;
      long long off = -1;
      if (n > 0 && fits) {
        off = (long long)atomicAdd(&ctr->nbr_cursor, (unsigned long long)n);
        if (off + n > nbrCap) off = -1;
      }
      s_off = off;
      kpNbrOff[g] = (int)off;
    }
    __syncthreads();
    const long long off = s_off;
    if (off >= 0)
      for (int t = lane; t < wcnt; t += 32) nbrPool[off + before + t] = mylist[t];
  }
}

// Position of every keypoint among the keypoints of its scan that have neighbours: the index of its
// RNG draws (3dsc.hpp consumes three per keypoint that reaches the axis computation).
__global__ void __launch_bounds__(256) k_kp_rank(const int* __restrict__ kpScan, const int* __restrict__ kpOff, int n_scans,
                                                 const int* __restrict__ kpNbr, int* __restrict__ kpRank,
                                                 int* __restrict__ listM, int* __restrict__ listL, DevCounters* __restrict__ ctr) {
  const int total = kpOff[n_scans];
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total) return;
  int c = 0;
  for (int j = kpOff[kpScan[g]]; j < g; j++) c += (kpNbr[j] > 0) ? 1 : 0;
  kpRank[g] = c;
  // the few keypoints of K4d's larger instantiations, listed so that those do not have to look for them
  const int nb = kpNbr[g];
  if (nb > DCAP_M) listL[atomicAdd(&ctr->n_list_l, 1)] = g;
  else if (nb > DCAP) listM[atomicAdd(&ctr->n_list_m, 1)] = g;
}

// ============================================================================================
// K4c — local point density (3dsc.hpp: searchForNeighbors(point_density_radius_)), once per
// marked surface point instead of once per (keypoint, neighbour) as PCL does.
// ============================================================================================
// Blocks (scan, y) walk the scan's sorted (halo) points in tiles: the marked ones of a tile are
// compacted into a list (they stay in cell order, so neighbouring lanes share cells and their loads hit
// L1), then every thread takes one marked point and sweeps the three rows of cells its density sphere
// touches (contiguous spans, fixed trip counts).
constexpr int DENS_TILE = 1024;
__global__ void __launch_bounds__(256) k_density(
    const float4* __restrict__ sorted, SurfIndex X, const long long* __restrict__ scan_off, DevParams P,
    const int* __restrict__ surfN, int* __restrict__ rho, unsigned long long* __restrict__ tests) {
  __shared__ unsigned short s_list[DENS_TILE];
  __shared__ int s_wsum[8];
  const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int n = surfN[s];
  if (n == 0) return;
  const long long base = scan_off[s];
  const float4* so = sorted + base;
  int* rh = rho + base;
  const ScanGrid G = scan_grid(X, s, base, P);
  const int nx = P.sg_nx, ny = P.sg_ny;
  unsigned ntest = 0, nmark = 0;  // per thread: at most 65,535 candidates per marked point, a few marked points
  // blockIdx.y strides over the scan's tiles: dense scans are shared by several blocks
  for (int t0 = (int)blockIdx.y * DENS_TILE; t0 < n; t0 += (int)gridDim.y * DENS_TILE) {
    // marked points of the tile, in order
    int cntw = 0;
    unsigned mk[DENS_TILE / 256];
#pragma unroll
    for (int k = 0; k < DENS_TILE / 256; k++) {
      const int i = t0 + (w * (DENS_TILE / 256) + k) * 32 + lane;  // a warp owns DENS_TILE/8 consecutive points
      mk[k] = __ballot_sync(FE_FULL, i < n && rh[i] < 0);
      cntw += __popc(mk[k]);
    }
    __syncthreads();  // the previous tile's list is no longer read
    if (lane == 0) s_wsum[w] = cntw;
    __syncthreads();
    int off = 0, m = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) { if (k < w) off += s_wsum[k]; m += s_wsum[k]; }
#pragma unroll
    for (int k = 0; k < DENS_TILE / 256; k++) {
      if ((mk[k] >> lane) & 1u) s_list[off + __popc(mk[k] & lanemask_lt())] = (unsigned short)((w * (DENS_TILE / 256) + k) * 32 + lane);
      off += __popc(mk[k]);
    }
    __syncthreads();
    for (int tw = (tid & ~31); tw < m; tw += 256) {   // a warp takes 32 consecutive marked points
      const int t = tw + lane;
      const bool act = t < m;
      const int i = t0 + (int)s_list[act ? t : tw];
      const float4 p = so[i];
      // cells reached by the density radius (>= 1 cell each way; more only if the grid was capped)
      const int cx0 = surf_cell(p.x - P.rhopad, P.sx0, P.sg_inv, nx), cx1 = surf_cell(p.x + P.rhopad, P.sx0, P.sg_inv, nx);
      const int cy0 = surf_cell(p.y - P.rhopad, P.sy0, P.sg_inv, ny), cy1 = surf_cell(p.y + P.rhopad, P.sy0, P.sg_inv, ny);
      int cnt = 0;
      if (G.bm && G.ns > 1) {  // per cell, only the z slabs the density sphere reaches
        const float zlo = p.z - P.rhopad, zhi = p.z + P.rhopad;
        // The 32 points are consecutive in (cell, slab) order, so they mostly share their cell and their slabs:
        // the warp sweeps the UNION of their neighbourhoods together — every lane tests every candidate
        // (the exact predicate rejects what lies outside its own sphere), all loads are broadcasts, the
        // loops are uniform.  Only a warp that straddles distant cells falls back to per-lane sweeps.
        const int ux0 = __reduce_min_sync(FE_FULL, cx0), ux1 = __reduce_max_sync(FE_FULL, cx1);
        const int uy0 = __reduce_min_sync(FE_FULL, cy0), uy1 = __reduce_max_sync(FE_FULL, cy1);
        if ((ux1 - ux0 + 1) * (uy1 - uy0 + 1) <= 16) {
          const int l0 = __reduce_min_sync(FE_FULL, z_slab(zlo, G.zs0, G.zscale, G.ns));
          const int l1 = __reduce_max_sync(FE_FULL, z_slab(zhi, G.zs0, G.zscale, G.ns));
          for (int r = uy0; r <= uy1; r++)
            for (int c = ux0; c <= ux1; c++) {
              int b, e;
              G.cell_slabs(r * nx + c, l0, l1, b, e);
              for (int j = b; j < e; j++) {
                const float4 q = so[j];
                // FLANN evaluates dist(query, point): query = the neighbour whose density is wanted
                if (l2_simple(p.x, p.y, p.z, q.x, q.y, q.z) < P.rho2f) cnt++;
              }
              if (act) ntest += (unsigned)(e - b);
            }
        } else {
          for (int r = cy0; r <= cy1; r++)
            for (int c = cx0; c <= cx1; c++) {
              int b, e;
              G.cell_slab_span(r * nx + c, zlo, zhi, b, e);
              for (int j = b; j < e; j++) {
                const float4 q = so[j];
                if (l2_simple(p.x, p.y, p.z, q.x, q.y, q.z) < P.rho2f) cnt++;
              }
              if (act) ntest += (unsigned)(e - b);
            }
        }
      } else {
        for (int r = cy0; r <= cy1; r++) {
          int b, e;
          G.row_span(r, cx0, cx1, b, e);
          for (int j = b; j < e; j++) {
            const float4 q = so[j];
            if (l2_simple(p.x, p.y, p.z, q.x, q.y, q.z) < P.rho2f) cnt++;
          }
          if (act) ntest += (unsigned)(e - b);
        }
      }
      if (!act) continue;
      rh[i] = cnt;
      nmark++;
    }
  }
  if (tests) {  // work counters for the bench: marked points and distance tests
    unsigned long long a = ntest, b = nmark;
#pragma unroll
    for (int d = 16; d; d >>= 1) { a += __shfl_xor_sync(FE_FULL, a, d); b += __shfl_xor_sync(FE_FULL, b, d); }
    if (lane == 0 && b) { atomicAdd(&tests[0], a); atomicAdd(&tests[1], b); }
  }
}

// ============================================================================================
// K4d — the 1980-bin 3D shape context of one keypoint per block (3dsc.hpp computePoint).
// ============================================================================================
__device__ __forceinline__ float eigen_sum3(float a0, float a1, float a2) {
  return __fadd_rn(a0, __fadd_rn(a1, a2));  // Eigen's unrolled 3-term reduction: a0 + (a1 + a2)
}

constexpr size_t desc_smem_bytes(int cap, int nt) {
  return (size_t)cap * 24 + FE_DESC_LEN * 4 + 64 + 0 * nt;
}

// The angles a neighbour is binned by (3dsc.hpp computePoint): azimuth phi and elevation th in degrees.
// o = keypoint, q = surface point, (axx, axy, -0) = normalised x axis; pox, poy: q - o in x and y.
__device__ __forceinline__ void shape_context_angles(const float4 o, const float4 q, const float axx, const float axy,
                                                     const DevParams& P, float& phi, float& th, float& pox, float& poy) {
  const float axz = -0.0f;
  // pcl::geometry::project(neighbour, origin, normal=(0,0,1), proj); proj -= origin
  pox = __fsub_rn(q.x, o.x); poy = __fsub_rn(q.y, o.y);
  const float poz = __fsub_rn(q.z, o.z);
  const float lambda = eigen_sum3(__fmul_rn(0.0f, pox), __fmul_rn(0.0f, poy), __fmul_rn(1.0f, poz));
  float prx = __fsub_rn(__fsub_rn(q.x, __fmul_rn(lambda, 0.0f)), o.x);
  float pry = __fsub_rn(__fsub_rn(q.y, __fmul_rn(lambda, 0.0f)), o.y);
  float prz = __fsub_rn(__fsub_rn(q.z, __fmul_rn(lambda, 1.0f)), o.z);
  {  // Eigen 3.2 normalize(): multiply by 1/norm
    const float inv = __fdiv_rn(1.0f, __fsqrt_rn(eigen_sum3(__fmul_rn(prx, prx), __fmul_rn(pry, pry), __fmul_rn(prz, prz))));
    prx = __fmul_rn(prx, inv); pry = __fmul_rn(pry, inv); prz = __fmul_rn(prz, inv);
  }
  // cross = x_axis x proj
  const float crx = __fsub_rn(__fmul_rn(axy, prz), __fmul_rn(axz, pry));
  const float cry = __fsub_rn(__fmul_rn(axz, prx), __fmul_rn(axx, prz));
  const float crz = __fsub_rn(__fmul_rn(axx, pry), __fmul_rn(axy, prx));
  const float crn = __fsqrt_rn(eigen_sum3(__fmul_rn(crx, crx), __fmul_rn(cry, cry), __fmul_rn(crz, crz)));
  const float dt = eigen_sum3(__fmul_rn(axx, prx), __fmul_rn(axy, pry), __fmul_rn(axz, prz));
  // std::atan2(float, float) / acosf: the host libm's float routines.  angle_libm 0 (default): the fdlibm
  // algorithm of glibc <= 2.40, restated operation by operation (glibc_f32.h) — the same last bit as the
  // reference's x86-64 build, so a neighbour on a bin edge lands in the same bin; 1: correctly rounded
  // (evaluated in double, then narrowed), what glibc >= 2.41 (CORE-MATH) returns.
  phi = P.angle_libm ? (float)atan2((double)crn, (double)dt) : glibc::atan2f_fdlibm(crn, dt);
  phi = __fmul_rn(phi, 57.29578f);
  const float cdn = eigen_sum3(__fmul_rn(crx, 0.0f), __fmul_rn(cry, 0.0f), __fmul_rn(crz, 1.0f));
  phi = (cdn < 0.f) ? __fsub_rn(360.0f, phi) : phi;
  float nox = pox, noy = poy, noz = poz;
  {
    const float inv = __fdiv_rn(1.0f, __fsqrt_rn(eigen_sum3(__fmul_rn(nox, nox), __fmul_rn(noy, noy), __fmul_rn(noz, noz))));
    nox = __fmul_rn(nox, inv); noy = __fmul_rn(noy, inv); noz = __fmul_rn(noz, inv);
  }
  th = eigen_sum3(__fmul_rn(0.0f, nox), __fmul_rn(0.0f, noy), __fmul_rn(1.0f, noz));
  const float t1 = (-1.0f < th) ? th : -1.0f;  // std::max(-1.0f, theta)
  const float t2 = (t1 < 1.0f) ? t1 : 1.0f;    // std::min(1.0f, .)
  th = __fmul_rn(P.angle_libm ? (float)acos((double)t2) : glibc::acosf_fdlibm(t2), 57.29578f);
}

// One neighbour's contribution (3dsc.hpp computePoint, the body of the neighbour loop): bin and
// weight.  Returns false when PCL skips the neighbour.  o = keypoint, q = surface point,
// (axx, axy, -0) = normalised x axis, dens = local point density of q.
__device__ __forceinline__ bool shape_context_contribution(const float4 o, const float4 q, const float d2, const float axx,
                                                           const float axy, const DevParams& P, const float* __restrict__ lut,
                                                           const int dens, int& bin, float& wgt) {
  if (fabsf(d2 - 0.0f) < 1.17549435e-38f) return false;  // pcl::utils::equal(nn_dists, 0)
  if (dens <= 0) return false;
  const float rr = __fsqrt_rn(d2);
  float phi, th, pox, poy;
  shape_context_angles(o, q, axx, axy, P, phi, th, pox, poy);
  int j = 0, k = 0, l = 0;
#pragma unroll
  for (int a = 15; a >= 1; a--) if (rr <= P.radii[a]) j = a - 1;
#pragma unroll
  for (int a = 11; a >= 1; a--) if (th <= P.theta[a]) k = a - 1;
#pragma unroll
  for (int a = 12; a >= 1; a--) if (phi <= P.phi[a]) l = a - 1;
  bin = l * 165 + k * 15 + j;
  wgt = __fmul_rn(__fdiv_rn(1.0f, (float)dens), lut[bin]);
  return true;
}

// PCL adds the contributions of a keypoint in ascending (squared distance, point index) order
// (FLANN's sorted radius search), so a bin's float sum depends on that order.  Up to CAP
// contributions are therefore collected as (key, weight) records with
//   key = bin << 52 | float_bits(d2) << 20 | point index      (bin < 2048, index < 2^20)
// grouped by bin with a counting pass (the bin is the major key), ranked inside their bin by
// counting smaller keys (keys are unique) and summed bin by bin in that order, which makes the
// descriptor bit-identical to the sequential loop.
// Work layout per keypoint: one warp finds the spans of all grid rows the search sphere touches
// (one row per lane), every thread sweeps the flattened candidate range and the true neighbours are
// compacted into a list, so the expensive bin arithmetic runs on a dense list with no idle lanes.
// Three instantiations share the keypoints by neighbour count: (NB_MIN, CAP] each; the LAST one also
// takes keypoints beyond its CAP and handles their bins in groups that fit the workspace (one sweep of
// the candidates per group), so they are bit-identical too; only a single bin holding more than CAP
// contributions is summed with order-free float atomics (counted in DevCounters::desc_unordered).
template <int NT, int CAP, int NB_MIN, bool LAST, bool DYN>
__global__ void __launch_bounds__(NT) k_desc_hist(
    const float4* __restrict__ kpOut, const int* __restrict__ kpScan, const int* __restrict__ kpOff,
    int n_scans, const int* __restrict__ kpNbr, const float4* __restrict__ sorted, SurfIndex X,
    const long long* __restrict__ scan_off, DevParams P, const int* __restrict__ rho,
    const float* __restrict__ lut, const float2* __restrict__ axes, int axesCap,
    const unsigned* __restrict__ nbrPool, const int* __restrict__ kpNbrOff, const int* __restrict__ kpRank,
    const int* __restrict__ glist, const int* __restrict__ nlist, float* __restrict__ desc, int descStride, int descOff,
    DevCounters* __restrict__ ctr, int warpCap) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* keyA = (unsigned long long*)smem_raw;
  unsigned long long* keyB = keyA + CAP;
  float* wA = (float*)(keyB + CAP);
  float* wB = wA + CAP;
  float* hist = wB + CAP;
  int* binCnt = (int*)hist;  // the histogram's storage counts records per bin while they are collected
  unsigned* nbrList = (unsigned*)keyB;  // compacted neighbour positions (consumed before keyB is written)
  __shared__ int s_cnt, s_total;
  __shared__ int s_scan[40];
  __shared__ int s_spanB[32], s_spanS[33];
  const int total = kpOff[n_scans];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  // The fast instantiation takes the keypoints in batches of KD_BATCH from a device-wide cursor (their
  // cost varies with the neighbour count; equal static shares left the slowest block ~40 % behind);
  // the next batch is requested before the current one is worked on.  The larger instantiations
  // stride over the list of their keypoints that k_kp_rank made.
  __shared__ int s_next;
  int g0 = blockIdx.x, gstep = gridDim.x, glen = 1;
  if (DYN) {
    if (tid == 0) s_next = atomicAdd(&ctr->kd_cursor, KD_BATCH);
    __syncthreads();
    g0 = s_next; glen = KD_BATCH;
  }
  const int bound = DYN ? total : *nlist;
  while (g0 < bound) {
  int nxt = 0;
  if (DYN && tid == 0) nxt = atomicAdd(&ctr->kd_cursor, KD_BATCH);
  const int gend = min(g0 + glen, bound);
  for (int gi = g0; gi < gend; gi++) {
    const int g = DYN ? gi : glist[gi];
    float* out = desc + (long long)g * descStride + descOff;
    const int nb = kpNbr[g];
    if (!LAST && nb > CAP) continue;           // a larger instantiation's keypoint
    // warpCap = min(NB_MIN, what the host lets the warp kernel take: -1 for a handful of scans, where a block per
    // keypoint finishes sooner than a warp per keypoint)
    if (NB_MIN > 0 && nb <= warpCap && (nb == 0 || kpNbrOff[g] >= 0)) continue;  // the warp kernel's keypoint
    if (nb == 0) {  // no neighbour (or non-finite keypoint): descriptor is NaN (3dsc.hpp)
      for (int i = tid; i < FE_DESC_LEN; i += NT) out[i] = __int_as_float(0x7fc00000);
      continue;
    }
    const bool ordered = nb <= CAP;
    const int s = kpScan[g];
    // the RNG is consumed only by keypoints that have neighbours, in keypoint order (k_kp_rank)
    const int rank = kpRank[g];
    const int off = ordered ? kpNbrOff[g] : -1;  // >= 0: K4b left the neighbour list in nbrPool
    const float4 o = kpOut[g];
    const long long base = scan_off[s];
    for (int i = tid; i < FE_DESC_LEN; i += NT) hist[i] = 0.0f;
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    if (rank >= axesCap) {
      if (tid == 0) atomicOr(&ctr->err, ERR_AXIS_CAP);
      for (int i = tid; i < FE_DESC_LEN; i += NT) out[i] = __int_as_float(0x7fc00000);
      __syncthreads();
      continue;
    }
    const float2 ax = axes[rank];  // normalised x_axis = (ax.x, ax.y, -0)
    const float4* so = sorted + base;
    const ScanGrid G = scan_grid(X, s, base, P);
    const int* rh = rho + base;
    const int cx0 = surf_cell(o.x - P.Rpad, P.sx0, P.sg_inv, P.sg_nx), cx1 = surf_cell(o.x + P.Rpad, P.sx0, P.sg_inv, P.sg_nx);
    const int cy0 = surf_cell(o.y - P.Rpad, P.sy0, P.sg_inv, P.sg_ny), cy1 = surf_cell(o.y + P.Rpad, P.sy0, P.sg_inv, P.sg_ny);
    if (LAST && !ordered) {
      // More contributions than the sort workspace holds: the bins are handled in GROUPS of consecutive bins whose
      // contributions fit (counted first), one sweep of the candidates per group — so these keypoints, too, are summed
      // in PCL's order.  Only a single bin with more than CAP contributions is summed with order-free atomics.
      __shared__ int s_ge, s_base, s_nrec;
      __shared__ float s_acc;
      auto sweep = [&](auto&& fn) {  // fn(i, q, d2) for every neighbour of the keypoint
        for (int r0 = cy0; r0 <= cy1; r0 += 32) {
          __syncthreads();
          if (w == 0) {
            int b = 0, e = 0;
            if (r0 + lane <= cy1) G.row_span(r0 + lane, cx0, cx1, b, e);
            int inc = e - b;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
              const int t = __shfl_up_sync(FE_FULL, inc, d);
              if (lane >= d) inc += t;
            }
            s_spanB[lane] = b;
            s_spanS[lane] = inc - (e - b);
            if (lane == 31) { s_spanS[32] = inc; s_total = inc; }
          }
          __syncthreads();
          const int ncand = s_total;
          for (int t = tid; t < ncand; t += NT) {
            int r = 0;
#pragma unroll
            for (int k = 16; k; k >>= 1) if (r + k < 32 && s_spanS[r + k] <= t) r += k;
            const int i = s_spanB[r] + (t - s_spanS[r]);
            const float4 q = so[i];
            const float d2 = l2_simple(o.x, o.y, o.z, q.x, q.y, q.z);
            if (d2 < P.R2f) fn(i, q, d2);
          }
        }
        __syncthreads();
      };
      // (A) contributions per bin
      sweep([&](int i, const float4& q, float d2) {
        int bin; float wgt;
        if (shape_context_contribution(o, q, d2, ax.x, ax.y, P, lut, rh[i], bin, wgt)) atomicAdd(&binCnt[bin], 1);
      });
      // (B) exclusive prefix: binCnt[b] = first record of bin b
      {
        constexpr int PER = (FE_DESC_LEN + NT - 1) / NT;
        int loc[PER];
        int sum = 0;
#pragma unroll
        for (int k = 0; k < PER; k++) {
          const int bi = tid * PER + k;
          loc[k] = (bi < FE_DESC_LEN) ? binCnt[bi] : 0;
          sum += loc[k];
        }
        int tot;
        int run = block_excl_scan<NT>(sum, &tot, s_scan);
#pragma unroll
        for (int k = 0; k < PER; k++) {
          const int bi = tid * PER + k;
          if (bi < FE_DESC_LEN) binCnt[bi] = run;
          run += loc[k];
        }
        if (tid == 0) s_nrec = tot;
      }
      __syncthreads();
      const int nrec = s_nrec;
      bool anyUnordered = false;
      for (int gb = 0; gb < FE_DESC_LEN;) {
        if (tid == 0) {  // the group: bins [gb, ge) with at most CAP contributions (at least one bin)
          const int basep = binCnt[gb];
          int ge = gb + 1;
          while (ge < FE_DESC_LEN && ((ge + 1 < FE_DESC_LEN) ? binCnt[ge + 1] : nrec) - basep <= CAP) ge++;
          s_ge = ge; s_base = basep; s_acc = 0.0f;
        }
        __syncthreads();
        const int ge = s_ge, basep = s_base;
        const int gcount = ((ge < FE_DESC_LEN) ? binCnt[ge] : nrec) - basep;
        __syncthreads();
        if (gcount > CAP) {  // one bin alone exceeds the workspace: order-free
          anyUnordered = true;
          sweep([&](int i, const float4& q, float d2) {
            int bin; float wgt;
            if (shape_context_contribution(o, q, d2, ax.x, ax.y, P, lut, rh[i], bin, wgt) && bin == gb) atomicAdd(&s_acc, wgt);
          });
          if (tid == 0) out[gb] = s_acc;
        } else if (gcount > 0) {
          // records of the group, placed by bin as they are found (the bin's start doubles as its cursor)
          sweep([&](int i, const float4& q, float d2) {
            int bin; float wgt;
            if (shape_context_contribution(o, q, d2, ax.x, ax.y, P, lut, rh[i], bin, wgt) && bin >= gb && bin < ge) {
              const int pos = atomicAdd(&binCnt[bin], 1) - basep;
              keyB[pos] = ((unsigned long long)bin << 52) | ((unsigned long long)__float_as_uint(d2) << 20) |
                          (unsigned long long)((unsigned)__float_as_int(q.w) & 0xFFFFFu);
              wB[pos] = wgt;
            }
          });
          // rank inside every bin (binCnt[b] is now the END of bin b; bin gb starts at the group's base)
          for (int i = tid; i < gcount; i += NT) {
            const unsigned long long k = keyB[i];
            const int bin = (int)(k >> 52);
            const int b0 = (bin > gb ? binCnt[bin - 1] : basep) - basep, e0 = binCnt[bin] - basep;
            int smaller = 0;
            for (int t = b0; t < e0; t++) smaller += (keyB[t] < k) ? 1 : 0;
            keyA[b0 + smaller] = k;
            wA[b0 + smaller] = wB[i];
          }
          __syncthreads();
          for (int bin = gb + tid; bin < ge; bin += NT) {
            const int b0 = (bin > gb ? binCnt[bin - 1] : basep) - basep, e0 = binCnt[bin] - basep;
            float acc = 0.0f;
            for (int t = b0; t < e0; t++) acc = __fadd_rn(acc, wA[t]);
            out[bin] = acc;
          }
        } else {
          for (int bin = gb + tid; bin < ge; bin += NT) out[bin] = 0.0f;
        }
        __syncthreads();
        gb = ge;
      }
      if (anyUnordered && tid == 0) atomicAdd(&ctr->desc_unordered, 1);
      __syncthreads();
      continue;
    }
    for (int r0 = cy0; off < 0 && r0 <= cy1; r0 += 32) {  // at most ~12 rows: one pass
      if (w == 0) {
        int b = 0, e = 0;
        if (r0 + lane <= cy1) G.row_span(r0 + lane, cx0, cx1, b, e);
        int inc = e - b;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int t = __shfl_up_sync(FE_FULL, inc, d);
          if (lane >= d) inc += t;
        }
        s_spanB[lane] = b;
        s_spanS[lane] = inc - (e - b);
        if (lane == 31) { s_spanS[32] = inc; s_total = inc; }
      }
      __syncthreads();
      const int ncand = s_total;
      for (int t0 = 0; t0 < ncand; t0 += NT) {
        const int t = t0 + tid;
        bool isn = false;
        int i = 0;
        float d2 = 0.f;
        if (t < ncand) {
          int r = 0;
#pragma unroll
          for (int k = 16; k; k >>= 1) if (r + k < 32 && s_spanS[r + k] <= t) r += k;
          i = s_spanB[r] + (t - s_spanS[r]);
          const float4 q = so[i];
          d2 = l2_simple(o.x, o.y, o.z, q.x, q.y, q.z);
          isn = d2 < P.R2f;
          if (isn && !ordered) {  // beyond the capacity: order-free accumulation
            int bin; float wgt;
            if (shape_context_contribution(o, q, d2, ax.x, ax.y, P, lut, rh[i], bin, wgt)) atomicAdd(&hist[bin], wgt);
          }
        }
        if (ordered) {
          const unsigned m = __ballot_sync(FE_FULL, isn);
          int basePos = 0;
          if (lane == 0 && m) basePos = atomicAdd(&s_cnt, __popc(m));
          basePos = __shfl_sync(FE_FULL, basePos, 0);
          if (isn) nbrList[basePos + __popc(m & lanemask_lt())] = (unsigned)i;
        }
      }
      __syncthreads();
    }
    if (ordered) {
      const int nl = (off >= 0) ? nb : s_cnt;  // == nb
      __syncthreads();
      if (tid == 0) s_cnt = 0;
      __syncthreads();
      // dense pass over the neighbours: bin, weight, record
      for (int t = tid; t < nl; t += NT) {
        const int i = (off >= 0) ? (int)nbrPool[off + t] : (int)nbrList[t];
        const float4 q = so[i];
        const float d2 = l2_simple(o.x, o.y, o.z, q.x, q.y, q.z);
        int bin; float wgt;
        if (shape_context_contribution(o, q, d2, ax.x, ax.y, P, lut, rh[i], bin, wgt)) {
          // one slot reservation per warp-ful of contributions, not one atomic on the same word per lane
          const unsigned act = __activemask();
          const int leader = __ffs(act) - 1;
          int slot = 0;
          if (lane == leader) slot = atomicAdd(&s_cnt, __popc(act));
          slot = __shfl_sync(act, slot, leader) + __popc(act & lanemask_lt());
          keyA[slot] = ((unsigned long long)bin << 52) | ((unsigned long long)__float_as_uint(d2) << 20) |
                       (unsigned long long)((unsigned)__float_as_int(q.w) & 0xFFFFFu);
          wA[slot] = wgt;
          atomicAdd(&binCnt[bin], 1);
        }
      }
      __syncthreads();
      const int n = s_cnt;
      // (1) exclusive scan of the per-bin counts -> first slot of every bin
      {
        constexpr int PER = (FE_DESC_LEN + NT - 1) / NT;
        int loc[PER];
        int sum = 0;
#pragma unroll
        for (int k = 0; k < PER; k++) {
          const int bi = tid * PER + k;
          loc[k] = (bi < FE_DESC_LEN) ? binCnt[bi] : 0;
          sum += loc[k];
        }
        int tot;
        int run = block_excl_scan<NT>(sum, &tot, s_scan);
#pragma unroll
        for (int k = 0; k < PER; k++) {
          const int bi = tid * PER + k;
          if (bi < FE_DESC_LEN) binCnt[bi] = run;
          run += loc[k];
        }
      }
      __syncthreads();
      // (2) group the records by bin (order inside a bin still arbitrary)
      for (int i = tid; i < n; i += NT) {
        const unsigned long long k = keyA[i];
        const int pos = atomicAdd(&binCnt[(int)(k >> 52)], 1);
        keyB[pos] = k;
        wB[pos] = wA[i];
      }
      __syncthreads();
      // (3) rank every record inside its bin: position = bin start + number of smaller keys.  After (2) binCnt[b]
      //     is the END of bin b, so a bin's segment is [binCnt[b-1], binCnt[b]): fixed trip counts, no key decoding
      for (int i = tid; i < n; i += NT) {
        const unsigned long long k = keyB[i];
        const int bin = (int)(k >> 52);
        const int b0 = bin ? binCnt[bin - 1] : 0, e0 = binCnt[bin];
        int smaller = 0;
        for (int t = b0; t < e0; t++) smaller += (keyB[t] < k) ? 1 : 0;
        keyA[b0 + smaller] = k;
        wA[b0 + smaller] = wB[i];
      }
      // (4) sum every bin in order: a thread owns PER consecutive bins; their bounds are read before the sums
      //     overwrite the counters (hist shares their storage)
      {
        constexpr int PER = (FE_DESC_LEN + NT - 1) / NT;
        int bnd[PER + 1];
        bnd[0] = (tid * PER > 0 && tid * PER <= FE_DESC_LEN) ? binCnt[tid * PER - 1] : 0;
#pragma unroll
        for (int k = 0; k < PER; k++) {
          const int bi = tid * PER + k;
          bnd[k + 1] = (bi < FE_DESC_LEN) ? binCnt[bi] : n;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < PER; k++) {
          const int bi = tid * PER + k;
          if (bi < FE_DESC_LEN) {
            float acc = 0.0f;
            for (int t = bnd[k]; t < bnd[k + 1]; t++) acc = __fadd_rn(acc, wA[t]);
            hist[bi] = acc;
          }
        }
      }
      __syncthreads();
    }
    for (int i = tid; i < FE_DESC_LEN; i += NT) out[i] = hist[i];
    __syncthreads();
  }
  if (DYN) {
    __syncthreads();
    if (tid == 0) s_next = nxt;
    __syncthreads();
    g0 = s_next;
  } else {
    g0 += gstep;
  }
  }
}

// K4d for small neighbourhoods: ONE WARP per keypoint, no block barrier anywhere.  Keypoints with at most
// DW_CAP neighbours whose list K4b left in the pool (and those with none: NaN rows) are handed out to the
// warps of the grid from a device-wide cursor.  The warp computes every neighbour's (bin, weight), sorts
// the records by key = bin | d2 | index with a bitonic network in its own slice of shared memory, sums
// every bin's run in that order (PCL's order, bit-identical) and writes the 1980-float row as zeros plus
// the few non-zero bins.
constexpr int DW_CAP = 256;     // neighbours per keypoint of the warp kernel
constexpr int DW_WARPS = 8;
constexpr size_t desc_warp_smem_bytes() { return (size_t)DW_WARPS * DW_CAP * 12; }

// The same algorithm with a BLOCK of DW_CAP threads per keypoint (one listed neighbour per thread): what calls of a
// handful of scans use instead of the warp kernel — their few keypoints cannot fill the GPU with warps, and a block
// finishes one keypoint several times sooner than a warp does (latency, not throughput).
__global__ void __launch_bounds__(DW_CAP) k_desc_hist_small(
    const float4* __restrict__ kpOut, const int* __restrict__ kpScan, const int* __restrict__ kpOff,
    int n_scans, const int* __restrict__ kpNbr, const float4* __restrict__ sorted,
    const long long* __restrict__ scan_off, DevParams P, const int* __restrict__ rho,
    const float* __restrict__ lut, const float2* __restrict__ axes, int axesCap,
    const unsigned* __restrict__ nbrPool, const int* __restrict__ kpNbrOff, const int* __restrict__ kpRank,
    float* __restrict__ desc, int descStride, int descOff, DevCounters* __restrict__ ctr) {
  __shared__ unsigned long long key[DW_CAP];
  __shared__ float wgt[DW_CAP];
  __shared__ int s_g;
  const int tid = threadIdx.x;
  const int total = kpOff[n_scans];
  for (;;) {
    __syncthreads();  // the previous keypoint's records are no longer read
    if (tid == 0) s_g = atomicAdd(&ctr->kw_cursor, 1);
    __syncthreads();
    const int g = s_g;
    if (g >= total) break;
    const int nb = kpNbr[g];
    const int off = kpNbrOff[g];
    if (nb > DW_CAP || (nb > 0 && off < 0)) continue;  // the block kernels' keypoint
    float* out = desc + (long long)g * descStride + descOff;
    const int rank = (nb > 0) ? kpRank[g] : 0;
    if (nb == 0 || rank >= axesCap) {  // no neighbour (or non-finite keypoint): NaN row (3dsc.hpp)
      if (nb > 0 && tid == 0) atomicOr(&ctr->err, ERR_AXIS_CAP);
      for (int i = tid; i < FE_DESC_LEN; i += DW_CAP) out[i] = __int_as_float(0x7fc00000);
      continue;
    }
    const int s = kpScan[g];
    const float4 o = kpOut[g];
    const long long base = scan_off[s];
    const float4* so = sorted + base;
    const int* rh = rho + base;
    const float2 ax = axes[rank];
    int np2 = 32;
    while (np2 < nb) np2 <<= 1;
    // records: (bin | d2 | point index) keys, a neighbour without a contribution sorts to the end
    bool has = false;
    if (tid < np2) {
      unsigned long long k = ~0ull;
      float wv = 0.f;
      if (tid < nb) {
        const int i = (int)nbrPool[off + tid];
        const float4 q = so[i];
        const float d2 = l2_simple(o.x, o.y, o.z, q.x, q.y, q.z);
        int bin;
        has = shape_context_contribution(o, q, d2, ax.x, ax.y, P, lut, rh[i], bin, wv);
        if (has)
          k = ((unsigned long long)bin << 52) | ((unsigned long long)__float_as_uint(d2) << 20) |
              (unsigned long long)((unsigned)__float_as_int(q.w) & 0xFFFFFu);
        else
          wv = 0.f;
      }
      key[tid] = k; wgt[tid] = wv;
    }
    // the row's zeros go out while the records are sorted
    if ((((unsigned long long)out) & 15ull) == 0ull) {
      float4* o4 = reinterpret_cast<float4*>(out);
      for (int i = tid; i < FE_DESC_LEN / 4; i += DW_CAP) o4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
      for (int i = tid; i < FE_DESC_LEN; i += DW_CAP) out[i] = 0.0f;
    }
    const int n = __syncthreads_count(has);
    // bitonic sort of (key, weight), ascending
    for (int k2 = 2; k2 <= np2; k2 <<= 1) {
      for (int j = k2 >> 1; j > 0; j >>= 1) {
        if (tid < (np2 >> 1)) {
          const int i = ((tid & ~(j - 1)) << 1) | (tid & (j - 1));  // lower index of the pair
          const int l = i | j;
          const bool up = (i & k2) == 0;
          const unsigned long long a = key[i], b = key[l];
          if ((a > b) == up) {
            key[i] = b; key[l] = a;
            const float wa = wgt[i]; wgt[i] = wgt[l]; wgt[l] = wa;
          }
        }
        __syncthreads();
      }
    }
    // every bin's sum in key order (the barriers above order these stores after the zeros)
    if (tid < n) {
      const unsigned bin = (unsigned)(key[tid] >> 52);
      if (tid == 0 || (unsigned)(key[tid - 1] >> 52) != bin) {
        float acc = 0.0f;
        for (int t = tid; t < n && (unsigned)(key[t] >> 52) == bin; t++) acc = __fadd_rn(acc, wgt[t]);
        out[bin] = acc;
      }
    }
  }
}

__global__ void __launch_bounds__(DW_WARPS * 32) k_desc_hist_warp(
    const float4* __restrict__ kpOut, const int* __restrict__ kpScan, const int* __restrict__ kpOff,
    int n_scans, const int* __restrict__ kpNbr, const float4* __restrict__ sorted,
    const long long* __restrict__ scan_off, DevParams P, const int* __restrict__ rho,
    const float* __restrict__ lut, const float2* __restrict__ axes, int axesCap,
    const unsigned* __restrict__ nbrPool, const int* __restrict__ kpNbrOff, const int* __restrict__ kpRank,
    float* __restrict__ desc, int descStride, int descOff, DevCounters* __restrict__ ctr) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned long long* key = (unsigned long long*)smem_raw + (size_t)w * DW_CAP;
  float* wgt = (float*)((unsigned long long*)smem_raw + (size_t)DW_WARPS * DW_CAP) + (size_t)w * DW_CAP;
  const int total = kpOff[n_scans];
  for (;;) {
    int g = 0;
    if (lane == 0) g = atomicAdd(&ctr->kw_cursor, 1);
    g = __shfl_sync(FE_FULL, g, 0);
    if (g >= total) break;
    const int nb = kpNbr[g];
    const int off = kpNbrOff[g];
    if (nb > DW_CAP || (nb > 0 && off < 0)) continue;  // the block kernels' keypoint
    float* out = desc + (long long)g * descStride + descOff;
    const int rank = (nb > 0) ? kpRank[g] : 0;
    if (nb == 0 || rank >= axesCap) {  // no neighbour (or non-finite keypoint): NaN row (3dsc.hpp)
      if (nb > 0 && lane == 0) atomicOr(&ctr->err, ERR_AXIS_CAP);
      for (int i = lane; i < FE_DESC_LEN; i += 32) out[i] = __int_as_float(0x7fc00000);
      continue;
    }
    const int s = kpScan[g];
    const float4 o = kpOut[g];
    const long long base = scan_off[s];
    const float4* so = sorted + base;
    const int* rh = rho + base;
    const float2 ax = axes[rank];
    // records
    int n = 0;
    for (int t0 = 0; t0 < nb; t0 += 32) {
      const int t = t0 + lane;
      bool has = false;
      unsigned long long k = 0;
      float wv = 0.f;
      if (t < nb) {
        const int i = (int)nbrPool[off + t];
        const float4 q = so[i];
        const float d2 = l2_simple(o.x, o.y, o.z, q.x, q.y, q.z);
        int bin;
        has = shape_context_contribution(o, q, d2, ax.x, ax.y, P, lut, rh[i], bin, wv);
        k = ((unsigned long long)bin << 52) | ((unsigned long long)__float_as_uint(d2) << 20) |
            (unsigned long long)((unsigned)__float_as_int(q.w) & 0xFFFFFu);
      }
      const unsigned hm = __ballot_sync(FE_FULL, has);
      if (has) { const int slot = n + __popc(hm & lanemask_lt()); key[slot] = k; wgt[slot] = wv; }
      n += __popc(hm);
    }
    int np2 = 32;
    while (np2 < n) np2 <<= 1;
    for (int i = n + lane; i < np2; i += 32) { key[i] = ~0ull; wgt[i] = 0.f; }
    __syncwarp();
    // bitonic sort of (key, weight), ascending
    for (int k2 = 2; k2 <= np2; k2 <<= 1) {
      for (int j = k2 >> 1; j > 0; j >>= 1) {
        for (int t = lane; t < (np2 >> 1); t += 32) {
          const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));  // lower index of the pair
          const int l = i | j;
          const bool up = (i & k2) == 0;
          const unsigned long long a = key[i], b = key[l];
          if ((a > b) == up) {
            key[i] = b; key[l] = a;
            const float wa = wgt[i]; wgt[i] = wgt[l]; wgt[l] = wa;
          }
        }
        __syncwarp();
      }
    }
    // the row: zeros, then every bin's sum in key order
    {
      float4* o4 = reinterpret_cast<float4*>(out);  // rows are 16-byte aligned in both layouts? only when descStride/descOff allow
      if ((((unsigned long long)out) & 15ull) == 0ull) {
        for (int i = lane; i < FE_DESC_LEN / 4; i += 32) o4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      } else {
        for (int i = lane; i < FE_DESC_LEN; i += 32) out[i] = 0.0f;
      }
    }
    __syncwarp();
    for (int i = lane; i < n; i += 32) {
      const unsigned bin = (unsigned)(key[i] >> 52);
      if (i == 0 || (unsigned)(key[i - 1] >> 52) != bin) {
        float acc = 0.0f;
        for (int t = i; t < n && (unsigned)(key[t] >> 52) == bin; t++) acc = __fadd_rn(acc, wgt[t]);
        out[bin] = acc;
      }
    }
    __syncwarp();
  }
}

// Record output (fe_enable_record_output): everything of a pcl::PointDescriptor record
// (feature_extraction_node.h:35-53, filled by pcl::concatenateFields at src:119) that is not the
// descriptor itself — x, y, z, the unregistered pad float, intensity, rf[9] = 0, tail padding.
__global__ void __launch_bounds__(256) k_record_frame(const float4* __restrict__ kpOut, const int* __restrict__ kpOff, int n_scans,
                                                      float* __restrict__ rec, int stride, int descLen) {
  const int total = kpOff[n_scans];
  const int tail = stride - 5 - descLen;  // rf[9] + alignment padding
  const int per = 5 + tail;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < (long long)total * per;
       t += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(t / per), f = (int)(t % per);
    const float4 k = kpOut[g];
    float* r = rec + (long long)g * stride;
    if (f < 5) r[f] = (f == 0) ? k.x : (f == 1) ? k.y : (f == 2) ? k.z : (f == 3) ? 0.0f : k.w;
    else r[5 + descLen + (f - 5)] = 0.0f;
  }
}

// ============================================================================================
// Tolerance-boundary report (fe_enable_boundary_report) — audit kernels, not part of the hot path.
// BASELINE.json north_star: "points lying within 1e-6 m of a tolerance boundary reported
// separately".  Every radius predicate of the path is d2 < r2f in float; a pair is on the boundary
// when |sqrt((double)d2) - sqrt((double)r2f)| < eps.  bnd[FE_BOUNDARY_KINDS * scan + k] counts them per predicate:
//   0 ring clustering (src:269-276): unordered pairs of crop points sharing a ring
//   1 cross-ring merge (src:222-229): unordered pairs of ring centroids (pseudo z, src:217)
//   2 3DSC support radius (src:350): (keypoint, surface point) pairs
//   3 3DSC point-density radius (src:352): (marked surface point, surface point) pairs, the query
//     being every surface point inside some keypoint's sphere, once
// The oracle counts the same pairs in its own searches (feo_process_batch_boundary).
// ============================================================================================
struct BoundarySpec {
  double eps;
  double bdist[4];  // sqrt((double)r2f) of the four predicates
  float r2f[4];
  float win[4];     // float pre-filter on |d2 - r2f| that contains every boundary pair
};

__device__ __forceinline__ bool on_boundary(const BoundarySpec& B, int k, float d2) {
  if (!(fabsf(d2 - B.r2f[k]) <= B.win[k])) return false;
  return fabs(sqrt((double)d2) - B.bdist[k]) < B.eps;
}

constexpr int BND_TILE = 1024;

// one block per scan: all pairs of the scan's crop survivors (tiles of BND_TILE in shared memory)
__global__ void __launch_bounds__(256) k_boundary_rings(
    const float4* __restrict__ crop, const unsigned* __restrict__ cropMeta, const int* __restrict__ cropCnt,
    const long long* __restrict__ scan_off, const int* __restrict__ chunk_off, int single_ring, BoundarySpec B,
    unsigned long long* __restrict__ bnd) {
  __shared__ int pre[MAXCHUNK + 1];
  __shared__ int sc[40];
  __shared__ float4 tile[BND_TILE];
  const int s = blockIdx.x, tid = threadIdx.x;
  const long long base = scan_off[s];
  const int nch = chunk_off[s + 1] - chunk_off[s];
  if (nch > MAXCHUNK) return;
  const int Nc = chunk_prefix<256>(cropCnt + chunk_off[s], nch, pre, sc);
  unsigned long long cnt = 0;
  auto ring_mask = [&](unsigned cd) -> unsigned {
    if (cd & 32u) return 0u;
    if (single_ring) return 1u;
    const unsigned r = cd & 15u;
    return (1u << r) | ((cd & 16u) ? (1u << (r + 1)) : 0u);
  };
  for (int t0 = 0; t0 < Nc; t0 += BND_TILE) {
    __syncthreads();
    for (int j = tid; j < BND_TILE && t0 + j < Nc; j += 256) {
      const long long pp = piece_pos(pre, nch, t0 + j, base);
      float4 q = crop[pp];
      q.w = __uint_as_float(ring_mask(cropMeta[pp] & 63u));
      tile[j] = q;
    }
    __syncthreads();
    const int tn = min(BND_TILE, Nc - t0);
    for (int i = tid; i < t0 + tn; i += 256) {  // i < j, j inside the tile
      float4 p;
      if (i >= t0) p = tile[i - t0];
      else {
        const long long pp = piece_pos(pre, nch, i, base);
        p = crop[pp];
        p.w = __uint_as_float(ring_mask(cropMeta[pp] & 63u));
      }
      const unsigned mi = __float_as_uint(p.w);
      if (!mi) continue;
      for (int j = max(i + 1 - t0, 0); j < tn; j++) {
        const float4 q = tile[j];
        const unsigned both = mi & __float_as_uint(q.w);
        if (!both) continue;
        if (on_boundary(B, 0, l2_simple(p.x, p.y, p.z, q.x, q.y, q.z))) cnt += (unsigned)__popc(both);
      }
    }
  }
  if (cnt) atomicAdd(&bnd[FE_BOUNDARY_KINDS * s + 0], cnt);
}

// one block per scan: all pairs of the scan's ring centroids with the pseudo z of src:217
__global__ void __launch_bounds__(128) k_boundary_merge(const float4* __restrict__ kfPool, const int* __restrict__ kfBase,
                                                        const int* __restrict__ kfCnt, DevParams P, BoundarySpec B,
                                                        unsigned long long* __restrict__ bnd) {
  __shared__ int pre[17];
  const int s = blockIdx.x, tid = threadIdx.x;
  if (tid == 0) {
    int run = 0;
    for (int g = 0; g < 16; g++) { pre[g] = run; run += kfCnt[s * 16 + g]; }
    pre[16] = run;
  }
  __syncthreads();
  const int Kf = pre[16];
  auto load = [&](int i) -> float4 {
    int g = 0;
    while (g < 15 && pre[g + 1] <= i) g++;
    float4 q = kfPool[kfBase[s * 16 + g] + (i - pre[g])];
    q.z = (float)__ddiv_rn(__dmul_rn(__dmul_rn((double)q.w, 0.75), P.radius_threshold), 2.0);
    return q;
  };
  unsigned long long cnt = 0;
  for (int i = tid; i < Kf; i += 128) {
    const float4 p = load(i);
    for (int j = i + 1; j < Kf; j++) {
      const float4 q = load(j);
      if (on_boundary(B, 1, l2_simple(p.x, p.y, p.z, q.x, q.y, q.z))) cnt++;
    }
  }
  if (cnt) atomicAdd(&bnd[FE_BOUNDARY_KINDS * s + 1], cnt);
}

// keypoints against the search surface (slot 2): the sweep of K4b, widened by eps
__global__ void __launch_bounds__(256) k_boundary_support(
    const float4* __restrict__ kpOut, const int* __restrict__ kpScan, const int* __restrict__ kpOff, int n_scans,
    const float4* __restrict__ sorted, SurfIndex X, const long long* __restrict__ scan_off, DevParams P, BoundarySpec B,
    unsigned long long* __restrict__ bnd) {
  const int total = kpOff[n_scans];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int g = blockIdx.x; g < total; g += gridDim.x) {
    const float4 o = kpOut[g];
    const int s = kpScan[g];
    if (!finite3(o.x, o.y, o.z)) continue;
    const long long base = scan_off[s];
    const float4* so = sorted + base;
    const ScanGrid G = scan_grid(X, s, base, P);
    const int cx0 = surf_cell(o.x - P.Rpad, P.sx0, P.sg_inv, P.sg_nx), cx1 = surf_cell(o.x + P.Rpad, P.sx0, P.sg_inv, P.sg_nx);
    const int cy0 = surf_cell(o.y - P.Rpad, P.sy0, P.sg_inv, P.sg_ny), cy1 = surf_cell(o.y + P.Rpad, P.sy0, P.sg_inv, P.sg_ny);
    unsigned long long cnt = 0;
    for (int r = cy0 + w; r <= cy1; r += 8) {
      int b, e;
      G.row_span(r, cx0, cx1, b, e);
      for (int i = b + lane; i < e; i += 32) {
        const float4 q = so[i];
        if (on_boundary(B, 2, l2_simple(o.x, o.y, o.z, q.x, q.y, q.z))) cnt++;
      }
    }
    if (cnt) atomicAdd(&bnd[FE_BOUNDARY_KINDS * s + 2], cnt);
  }
}

// marked surface points against the surface (slot 3): the sweep of K4c over whole cell columns; one block per
// scan; runs while rho still holds the marks that K4b left
__global__ void __launch_bounds__(256) k_boundary_density(
    const float4* __restrict__ sorted, SurfIndex X, const long long* __restrict__ scan_off, DevParams P, const int* __restrict__ surfN,
    const int* __restrict__ rho, BoundarySpec B, unsigned long long* __restrict__ bnd) {
  const int s = blockIdx.x;
  const int n = surfN[s];
  const long long base = scan_off[s];
  const float4* so = sorted + base;
  const ScanGrid G = scan_grid(X, s, base, P);
  unsigned long long cnt = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    if (rho[base + i] >= 0) continue;
    const float4 p = so[i];
    const int cx0 = surf_cell(p.x - P.rhopad, P.sx0, P.sg_inv, P.sg_nx), cx1 = surf_cell(p.x + P.rhopad, P.sx0, P.sg_inv, P.sg_nx);
    const int cy0 = surf_cell(p.y - P.rhopad, P.sy0, P.sg_inv, P.sg_ny), cy1 = surf_cell(p.y + P.rhopad, P.sy0, P.sg_inv, P.sg_ny);
    for (int r = cy0; r <= cy1; r++) {
      int b, e;
      G.row_span(r, cx0, cx1, b, e);
      for (int j = b; j < e; j++) {
        const float4 q = so[j];
        if (on_boundary(B, 3, l2_simple(p.x, p.y, p.z, q.x, q.y, q.z))) cnt++;
      }
    }
  }
  if (cnt) atomicAdd(&bnd[FE_BOUNDARY_KINDS * s + 3], cnt);
}

// ---- kinds 4-9 (fe_enable_boundary_report_all): the threshold decisions in metres or degrees that are not radius
// predicates.  Margins are evaluated in double with + - * / sqrt only (no FMA: -fmad=false), in the order of
// include/fe_b200.h, so the oracle's counts agree to the last pair.  bnd[FE_BOUNDARY_KINDS * scan + k] counts kind k. ----
constexpr double BND_DEG = 0.017453292519943295;  // pi / 180

// kinds 4 (crop box) and 5 (ring-window ends): one block per K1 chunk, K1's decode, levelling and crop again
template <bool RAW>
__global__ void __launch_bounds__(256) k_boundary_crop_ring(const float4* __restrict__ pts, const int4* __restrict__ chunkTab,
                                                            const float* __restrict__ rot, DevParams P, RawLayout L, double eps,
                                                            unsigned long long* __restrict__ bnd) {
  const int4 ct = __ldg(chunkTab + blockIdx.x);
  const int s = ct.x, nIn = ct.y & 4095;
  const long long base = (long long)(((unsigned long long)(unsigned)ct.w << 32) | (unsigned)ct.z);
  float m[9];
#pragma unroll
  for (int i = 0; i < 9; i++) m[i] = rot[s * 9 + i];
  const double lo[3] = {(double)P.xmin, (double)P.ymin, (double)P.zmin}, hi[3] = {(double)P.xmax, (double)P.ymax, (double)P.zmax};
  unsigned nCrop = 0, nRing = 0;
  for (int j0 = 0; j0 < nIn; j0 += 256) {  // warp-uniform trip count: the sums below take the full warp
    const int j = j0 + threadIdx.x;
    if (j >= nIn) continue;
    float4 p;
    if (RAW) {
      const unsigned char* rec = L.raw + (base + j) * (long long)L.stride;
      p = make_float4(load_f32_any(rec + L.xo), load_f32_any(rec + L.yo), load_f32_any(rec + L.zo), 0.0f);
    } else {
      p = __ldg(pts + base + j);
    }
    const float3 l = level_xyz(m, p);
    const float4 q = make_float4(l.x, l.y, l.z, 0.0f);
    if (!finite3(q.x, q.y, q.z)) continue;
    const double v[3] = {(double)q.x, (double)q.y, (double)q.z};
    bool inside = true, near = false;
#pragma unroll
    for (int a = 0; a < 3; a++) {
      inside = inside && v[a] > lo[a] - eps && v[a] < hi[a] + eps;
      near = near || fabs(v[a] - lo[a]) < eps || fabs(v[a] - hi[a]) < eps;
    }
    if (inside && near) nCrop++;
    if (!crop_keeps(P, q)) continue;
    const float el = elevation_deg(p.x, p.y, p.z);
    if (!isfinite(el)) continue;
    const double range = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(v[0], v[0]), __dmul_rn(v[1], v[1])), __dmul_rn(v[2], v[2])));
    double dmin = fabs((double)el + 16.0);
    for (int e = -14; e <= 16; e += 2) dmin = fmin(dmin, fabs((double)el - (double)e));
    if (__dmul_rn(range, __dmul_rn(dmin, BND_DEG)) < eps) nRing++;
  }
  __syncwarp();
  nCrop = __reduce_add_sync(FE_FULL, nCrop);
  nRing = __reduce_add_sync(FE_FULL, nRing);
  if ((threadIdx.x & 31) == 0) {
    if (nCrop) atomicAdd(&bnd[FE_BOUNDARY_KINDS * s + 4], (unsigned long long)nCrop);
    if (nRing) atomicAdd(&bnd[FE_BOUNDARY_KINDS * s + 5], (unsigned long long)nRing);
  }
}

// kind 6: the per-ring counts the GateCount instantiations of K2 left, summed per scan
__global__ void __launch_bounds__(256) k_boundary_gate_sum(const unsigned* __restrict__ gate, int n_scans,
                                                           unsigned long long* __restrict__ bnd) {
  const int s = blockIdx.x * 256 + threadIdx.x;
  if (s >= n_scans) return;
  unsigned t = 0;
  for (int r = 0; r < 16; r++) t += gate[s * 16 + r];
  bnd[FE_BOUNDARY_KINDS * s + 6] = t;
}

// kinds 7-9 (3DSC radial shells, elevation and azimuth edges): the (keypoint, neighbour) pairs K4d bins — the sweep of
// K4b, the angles of shape_context_angles with the keypoint's x axis
__global__ void __launch_bounds__(256) k_boundary_bins(
    const float4* __restrict__ kpOut, const int* __restrict__ kpScan, const int* __restrict__ kpOff, int n_scans,
    const float4* __restrict__ sorted, SurfIndex X, const long long* __restrict__ scan_off, DevParams P,
    const float2* __restrict__ axes, int axesCap, const int* __restrict__ kpRank, double eps,
    unsigned long long* __restrict__ bnd) {
  const int total = kpOff[n_scans];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int g = blockIdx.x; g < total; g += gridDim.x) {
    const float4 o = kpOut[g];
    const int s = kpScan[g];
    const int rank = kpRank[g];
    if (!finite3(o.x, o.y, o.z) || rank >= axesCap) continue;  // no bins (K4d reports the axis overflow)
    const float2 ax = axes[rank];
    const long long base = scan_off[s];
    const float4* so = sorted + base;
    const ScanGrid G = scan_grid(X, s, base, P);
    const int cx0 = surf_cell(o.x - P.Rpad, P.sx0, P.sg_inv, P.sg_nx), cx1 = surf_cell(o.x + P.Rpad, P.sx0, P.sg_inv, P.sg_nx);
    const int cy0 = surf_cell(o.y - P.Rpad, P.sy0, P.sg_inv, P.sg_ny), cy1 = surf_cell(o.y + P.Rpad, P.sy0, P.sg_inv, P.sg_ny);
    unsigned long long nRad = 0, nEl = 0, nAz = 0;
    for (int r = cy0 + w; r <= cy1; r += 8) {
      int b, e;
      G.row_span(r, cx0, cx1, b, e);
      for (int i = b + lane; i < e; i += 32) {
        const float4 q = so[i];
        const float d2 = l2_simple(o.x, o.y, o.z, q.x, q.y, q.z);
        if (!(d2 < P.R2f) || fabsf(d2 - 0.0f) < 1.17549435e-38f) continue;  // not a neighbour; pcl::utils::equal(d2, 0)
        const float rr = __fsqrt_rn(d2);
        float phi, th, pox, poy;
        shape_context_angles(o, q, ax.x, ax.y, P, phi, th, pox, poy);
        double dr = fabs((double)rr - (double)P.radii[1]), dt = fabs((double)th - (double)P.theta[1]);
        double dp = fabs((double)phi - (double)P.phi[0]);
        for (int a = 2; a <= 14; a++) dr = fmin(dr, fabs((double)rr - (double)P.radii[a]));
        for (int a = 2; a <= 10; a++) dt = fmin(dt, fabs((double)th - (double)P.theta[a]));
        for (int a = 1; a <= 12; a++) dp = fmin(dp, fabs((double)phi - (double)P.phi[a]));
        const double rho = sqrt(__dadd_rn(__dmul_rn((double)pox, (double)pox), __dmul_rn((double)poy, (double)poy)));
        if (dr < eps) nRad++;
        if (__dmul_rn((double)rr, __dmul_rn(dt, BND_DEG)) < eps) nEl++;
        // straight above or below the keypoint (rho = 0, phi NaN): any horizontal move picks the azimuth bin
        if (rho == 0.0 || __dmul_rn(rho, __dmul_rn(dp, BND_DEG)) < eps) nAz++;
      }
    }
    if (nRad) atomicAdd(&bnd[FE_BOUNDARY_KINDS * s + 7], nRad);
    if (nEl) atomicAdd(&bnd[FE_BOUNDARY_KINDS * s + 8], nEl);
    if (nAz) atomicAdd(&bnd[FE_BOUNDARY_KINDS * s + 9], nAz);
  }
}

// test hook: the device's fdlibm restatement (glibc_f32.h) element-wise; op 0 atan2f(a,b), 1 acosf(a), 2 atanf(a)
__global__ void k_debug_libm_f32(int op, const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = op == 0 ? glibc::atan2f_fdlibm(a[i], b[i]) : op == 1 ? glibc::acosf_fdlibm(a[i]) : glibc::atanf_fdlibm(a[i]);
}

}  // namespace fe
