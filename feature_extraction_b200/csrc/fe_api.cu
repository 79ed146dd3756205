// fe_api.cu — host side of libfe_b200.so: context, parameter derivation, sub-batch pipeline and
// the C-ABI of include/fe_b200.h.  No CPU fallback anywhere: every entry point that computes
// launches the kernels of fe_kernels.cuh.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <thread>
#include <vector>

#include "fe_kernels.cuh"
#include "fe_loop.h"
#include "fe_match.h"
#include "fe_odometry.h"
#include "fe_register.h"

using namespace fe;

#define FE_VERSION "fe_b200 0.1 (sm_100a)"

namespace {

// Small sub-batches (a single scan per callback is how the reference runs, src:72) are launch-bound: ~17 dependent
// launches.  Their whole chain — staging copies, kernels, result copies — is captured once per shape into a CUDA
// graph and replayed (fe_process_batch, sub-batches of at most GRAPH_MAX_SCANS scans).
constexpr int GRAPH_MAX_SCANS = 16;
static_assert(GRAPH_MAX_SCANS <= 32, "k_kp_offsets_gather_small gives every scan a warp of one 1024-thread block");

// What one enqueue of the pipeline computes (enqueue_pipeline).  The slot keeps the sub-batch in flight, so that
// lean_rerun_if_deferred can run it again and the stats hooks can read its shape.
struct SubBatch {
  const float4* pts = nullptr;  // device input: a slot's d_pts or the caller's array (fe_process_batch_device)
  int nscans = 0;
  int64_t npts = 0;
  int nch = 0;                  // K1 chunks of the staged scans
  int k1flags = 0;
  bool desc = false, wantKc = false;
  RawLayout lay = {nullptr, 0, 0, 0, 0};
  bool lean = false;            // first instantiation of every stage only (see enqueue_subbatch)
};

// A captured graph replays the launches of one SubBatch: the record plus whatever else the host code of
// enqueue_pipeline branches on.  npts is left out: it enters through `by` and through nch (no chunks, no points);
// every setting of the context that changes the launches bumps `epoch`.
struct GraphKey {
  SubBatch sb;
  int by;        // density_blocks_per_scan: K4c's grid
  bool bigScan;  // a scan of more than 65,535 points: launch_surface_grid adds the radix kernel
  int bnd;       // boundary report: 0 off, 4 radius kinds (k_boundary_*), FE_BOUNDARY_KINDS all kinds
  int epoch;
  bool operator==(const GraphKey& o) const {
    const SubBatch &a = sb, &b = o.sb;
    return a.pts == b.pts && a.nscans == b.nscans && a.nch == b.nch && a.k1flags == b.k1flags && a.desc == b.desc &&
           a.wantKc == b.wantKc && a.lay.raw == b.lay.raw && a.lay.stride == b.lay.stride && a.lay.xo == b.lay.xo &&
           a.lay.yo == b.lay.yo && a.lay.zo == b.lay.zo && a.lean == b.lean && by == o.by && bigScan == o.bigScan &&
           bnd == o.bnd && epoch == o.epoch;
  }
};
struct GraphEntry {
  GraphKey key;
  cudaGraphExec_t exec = nullptr;  // null: the shape has been seen once (run eagerly, so that every lazy init is done)
  int64_t launches = 0;
};

// A device buffer and a pinned buffer carved by one layout (Carve).  A slot has one per group of its arrays.  A match,
// register, odometry or loop-closure call has one of its own, whose results come first at the same offsets in both, so that one copy
// brings them back; the pinned buffer ends with the tables the call uploads, at their device offsets too.
struct Workspace {
  unsigned char* d = nullptr;
  int64_t dCap = 0;  // bytes
  unsigned char* h = nullptr;
  int64_t hCap = 0;
};

// A typed array at a byte offset of a Workspace buffer.
template <class T>
struct Span {
  int64_t off;
  T* in(unsigned char* base) const { return (T*)(base + off); }
};

// Hands out consecutive `align`-byte-aligned Spans; `bytes` is the running total.
struct Carve {
  int64_t align = 16;
  int64_t bytes = 0;
  template <class T>
  Span<T> take(int64_t n) {
    const Span<T> s{bytes};
    bytes = (bytes + n * (int64_t)sizeof(T) + align - 1) & ~(align - 1);
    return s;
  }
};

// The groups of a slot's arrays, one per lifetime (slot_arrays lists each group's arrays).  Opening a slot (open_slot)
// makes its stream and events only; ensure_group allocates a group in full when a call first needs it.
enum Group { CORE, POINTS, FULL, CLOUDS, REPORT, GRID, NGROUPS };

// Rule: no array that a captured graph can name is moved or freed before the slot is destroyed (free_slot).  A group
// is allocated once, in full, and never grown.  GraphKey depends on this: a replay finds every array where the
// capture saw it.  The context's pinned result buffers may grow (grow_pinned): they are copied into outside any graph.
struct Slot {
  cudaStream_t stream = nullptr;
  SubBatch sb;  // the sub-batch in flight (or the last one)
  std::vector<GraphEntry> graphs;
  Workspace group[NGROUPS];
  int64_t capPts = 0;
  int capScans = 0, capChunks = 0;
  int64_t capKp = 0;
  int capKf = 0, capKc = 0;
  // device
  float4 *d_pts = nullptr, *d_surf = nullptr, *d_crop = nullptr, *d_sorted = nullptr, *d_full = nullptr;
  float4* d_ringPts = nullptr;  // K2: the crop survivors bucketed by ring (CSR like the input)
  unsigned *d_cropMeta = nullptr, *d_keyA = nullptr, *d_keyB = nullptr, *d_valA = nullptr, *d_valB = nullptr, *d_sortedKey = nullptr;
  int* d_rho = nullptr;
  long long* d_scan_off = nullptr;
  int *d_chunk_off = nullptr, *d_surfCnt = nullptr, *d_cropCnt = nullptr;
  float* d_rot = nullptr;
  int *d_kfBase = nullptr, *d_kfCnt = nullptr, *d_kcBase = nullptr, *d_kcCnt = nullptr;
  int *d_kpBase = nullptr, *d_kpCnt = nullptr, *d_kpOff = nullptr, *d_kpScan = nullptr, *d_kpNbr = nullptr;
  int *d_kpNbrOff = nullptr, *d_kpRank = nullptr;  // K4b -> K4d: slice of the neighbour pool (d_keyA), RNG rank
  int *d_kpListM = nullptr, *d_kpListL = nullptr;  // keypoints of K4d's medium / large instantiation
  int *d_rowStart = nullptr, *d_surfN = nullptr, *d_perScan = nullptr, *d_outOff = nullptr;
  int *d_perScan2 = nullptr, *d_outOff2 = nullptr;   // cloud outputs: ~keypoint_cloud counts / offsets
  float4* d_gather2 = nullptr;
  int *h_cloudOff = nullptr, *h_kcOff = nullptr;     // pinned: per-scan offsets of the two cloud outputs of the sub-batch
  unsigned char* d_gridHdr = nullptr;  // per-scan index of the halo cell grid (bit map, word prefix, slot table)
  int* d_tabOk = nullptr;
  int *d_ringBase = nullptr, *d_ovfRuns = nullptr, *d_scanFlag = nullptr;  // K2: ring segment offsets per scan, rings for the wide run kernel
  int *d_ovfRings = nullptr, *d_ovfRings2 = nullptr, *d_ovfMerge = nullptr, *d_ovfMerge2 = nullptr, *d_ovfSurf = nullptr;
  unsigned char* d_slabs = nullptr;
  float4 *d_kfPool = nullptr, *d_kcPool = nullptr, *d_kpPool = nullptr, *d_kpOut = nullptr, *d_gather = nullptr;
  float* d_desc = nullptr;
  DevCounters* d_ctr = nullptr;
  unsigned long long *d_boundary = nullptr, *h_boundary = nullptr;  // tolerance-boundary report: [scan][FE_BOUNDARY_KINDS] counts
  unsigned* d_gate = nullptr;  // kind 6 per (scan, ring) as the K2 kernels leave it (GateCount)
  // pinned host mirrors
  long long* h_scan_off = nullptr;
  int* h_chunk_off = nullptr;
  int4* d_chunkTab = nullptr;  // k_chunk_table, per chunk: scan, (chunk of scan << 12) | points, first point lo, hi
  float* h_rot = nullptr;
  DevCounters* h_ctr = nullptr;
  int* h_kpOff = nullptr;
  int* h_perScan = nullptr;
  cudaEvent_t evDone = nullptr, evT0 = nullptr, evT1 = nullptr;
  int64_t maxScanPts = 0;  // largest scan of the staged sub-batch
  int firstScan = 0;       // where the sub-batch in flight goes in the call's results
  bool busy = false;
  // stage timing
  std::vector<cudaEvent_t> ev;
  std::vector<const char*> evName;
  int nev = 0;
};

}  // namespace

struct fe_ctx {
  int device = 0;
  fe_params_t params;
  DevParams dp;
  fe_limits_t lim;
  Slot slot[2];
  float* d_lut = nullptr;
  float2* d_axes = nullptr;
  int axesCap = 0;
  bool cloudOutputs = false;
  int leanHold = 0;           // sub-batches for which the lean chain stays off after one had to be run again
  int64_t leanReruns = 0;
  bool stageTiming = false;   // serialise the stages and time each with CUDA events (fe_enable_stage_timing)
  bool gridClustering = false;  // fe_debug_force_grid_clustering: K2 through the grid-based kernels only
  bool recordOutput = false;  // descriptors leave as FE_RECORD_FLOATS-float PointDescriptor records
  int numSms = 148;           // cudaDevAttrMultiProcessorCount of the context's device (grids are sized in resident waves)
  int epoch = 0;              // bumped by every setting that changes what a captured graph would do
  bool useGraphs = true;      // fe_debug_enable_graphs
  int64_t graphReplays = 0;
  int angleLibm = 0;          // fe_set_angle_libm
  double bndEps = 0.0;        // boundary report: the decisions within bndEps of their threshold are counted
  int bndKinds = 0;           // ... of kinds 0-3 (4, fe_enable_boundary_report), 0-9 (FE_BOUNDARY_KINDS, _all) or none (0)
  std::vector<int64_t> bndCounts;     // [scan][4] of the last batch call
  std::vector<int64_t> bndCountsAll;  // [scan][FE_BOUNDARY_KINDS] of the last batch call (all kinds enabled)
  // results (host, pinned, grown on demand)
  std::vector<int64_t> kpOffsets;
  fe_point_t* h_kp = nullptr;
  float* h_desc = nullptr;
  int64_t capResKp = 0, capResDesc = 0;
  // optional cloud outputs of the last host batch call (fe_enable_cloud_outputs): CSR by scan, pinned
  std::vector<int64_t> cloudOff, kcOff;
  fe_point_t *h_cloud = nullptr, *h_kc = nullptr;
  int64_t capCloud = 0, capKcRes = 0, cloudRun = 0, kcRun = 0;
  // stage times of the last device call
  std::vector<const char*> stName;
  std::vector<float> stMs;
  int64_t launches = 0;
  // fe_match_descriptors*, fe_register_matches*, fe_odometry* and fe_loop_closures*: a workspace per family, so that a
  // call leaves the last batch call's results and the other families' results alone (fe_register_matches_device and
  // fe_odometry_device may read `best` straight out of matchWs)
  Workspace matchWs, regWs, odoWs, loopWs;
  bool matchAttrs = false;
  std::string err;
};

namespace {

#define CK(call)                                                                       \
  do {                                                                                 \
    cudaError_t e_ = (call);                                                           \
    if (e_ != cudaSuccess) {                                                           \
      char b_[512];                                                                    \
      snprintf(b_, sizeof b_, "%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
      ctx->err = b_;                                                                   \
      return FE_ERR_CUDA;                                                              \
    }                                                                                  \
  } while (0)

int fail(fe_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->err = msg;
  return code;
}

// wait for whatever the two slots have in flight
int sync_slots(fe_ctx* ctx) {
  for (Slot& s : ctx->slot) if (s.stream) CK(cudaStreamSynchronize(s.stream));
  return FE_OK;
}

// scans [pts, ...) of a batch call: K1 runs every stage, K4 whenever the parameters ask for descriptors
SubBatch batch_subbatch(const fe_ctx* ctx, const float4* pts, int nscans) {
  SubBatch sb;
  sb.pts = pts;
  sb.nscans = nscans;
  sb.desc = ctx->params.estimate_descriptors != 0;
  sb.k1flags = F_ELEV | F_ROT | F_CROP | F_RING | (sb.desc ? F_SURF : 0);
  return sb;
}

// ---- parameter derivation (host, float/double exactly as PCL narrows them) ------------------

float radius_sq_as_flann_sees_it(double radius) { return (float)(radius * radius); }

// pcl::ShapeContext3DEstimation::initCompute (3dsc.hpp): bin edges and the 1/cbrt(volume) table
void shape_context_tables(double R, double rmin, float radii[16], float theta[12], float phi[13], float* lut) {
  const int NA = 12, NE = 11, NR = 15;
  const float az_step = 360.0f / (float)NA, el_step = 180.0f / (float)NE;
  for (int j = 0; j <= NR; j++)
    radii[j] = (float)exp(log(rmin) + (((float)j / (float)NR) * log(R / rmin)));
  for (int k = 0; k <= NE; k++) theta[k] = (float)k * el_step;
  for (int l = 0; l <= NA; l++) phi[l] = (float)l * az_step;
  const float d2r = 0.017453293f;
  const float dphi = phi[1] * d2r - phi[0] * d2r;
  const float third = 1.0f / 3.0f;
  for (int j = 0; j < NR; j++) {
    const float dr = (radii[j + 1] * radii[j + 1] * radii[j + 1] / 3.0f) - (radii[j] * radii[j] * radii[j] / 3.0f);
    for (int k = 0; k < NE; k++) {
      const float dth = cosf(theta[k] * d2r) - cosf(theta[k + 1] * d2r);
      const float V = dphi * dth * dr;
      for (int l = 0; l < NA; l++) lut[l * NE * NR + k * NR + j] = 1.0f / powf(V, third);
    }
  }
}

// Eigen 3.2 AngleAxisf(pitch, Y) * AngleAxisf(roll, X) -> rotation matrix (row-major 3x3)
void leveling_matrix(double roll, double pitch, float m[9]) {
  const float hp = 0.5f * (float)pitch, hr = 0.5f * (float)roll;
  // quaternions (w, x, y, z)
  const float aw = cosf(hp), ax = 0.0f * sinf(hp), ay = 1.0f * sinf(hp), az = 0.0f * sinf(hp);
  const float bw = cosf(hr), bx = 1.0f * sinf(hr), by = 0.0f * sinf(hr), bz = 0.0f * sinf(hr);
  const float w = aw * bw - ax * bx - ay * by - az * bz;
  const float x = aw * bx + ax * bw + ay * bz - az * by;
  const float y = aw * by + ay * bw + az * bx - ax * bz;
  const float z = aw * bz + az * bw + ax * by - ay * bx;
  const float tx = 2.0f * x, ty = 2.0f * y, tz = 2.0f * z;
  const float twx = tx * w, twy = ty * w, twz = tz * w;
  const float txx = tx * x, txy = ty * x, txz = tz * x;
  const float tyy = ty * y, tyz = tz * y, tzz = tz * z;
  float R[9];
  R[0] = 1.0f - (tyy + tzz); R[1] = txy - twz;          R[2] = txz + twy;
  R[3] = txy + twz;          R[4] = 1.0f - (txx + tzz); R[5] = tyz - twx;
  R[6] = txz - twy;          R[7] = tyz + twx;          R[8] = 1.0f - (txx + tyy);
  // Affine3f::Identity().rotate(q): Identity.linear() * R, 3-term sums as a0 + (a1 + a2)
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      const float i0 = (i == 0) ? 1.0f : 0.0f, i1 = (i == 1) ? 1.0f : 0.0f, i2 = (i == 2) ? 1.0f : 0.0f;
      m[i * 3 + j] = i0 * R[j] + (i1 * R[3 + j] + i2 * R[6 + j]);
    }
}

int bits_for_host(int v) { int b = 0; while (v > 0) { b++; v >>= 1; } return b; }

// cells of the descriptor grid along x and along y at most: surface_grid clamps to it, and the GRID group's row starts
// are sized by it
constexpr int SURF_GRID_MAX = 2048;

// surface keep-box and 2-D grid for keypoints known to lie inside [x0,x1]x[y0,y1]x[z0,z1]
void surface_grid(DevParams& dp, double R, float x0, float x1, float y0, float y1, float z0, float z1) {
  const double rrho = R / 5.0;
  const float reach = (float)((R + rrho) * 1.001 + 1e-3);
  dp.sx0 = x0 - reach; dp.sx1 = x1 + reach;
  dp.sy0 = y0 - reach; dp.sy1 = y1 + reach;
  dp.sz0 = z0 - reach; dp.sz1 = z1 + reach;
  float cell = (float)(rrho * 1.001);
  if (!(cell > 1e-6f)) cell = 1e-6f;
  const float ex = dp.sx1 - dp.sx0, ey = dp.sy1 - dp.sy0;
  const float maxdim = (float)(SURF_GRID_MAX - 1);
  if (ex / cell > maxdim) cell = ex / maxdim;
  if (ey / cell > maxdim) cell = ey / maxdim;
  dp.sg_inv = 1.0f / cell;
  dp.sg_nx = std::max(1, std::min(SURF_GRID_MAX, (int)floorf(ex * dp.sg_inv) + 1));
  dp.sg_ny = std::max(1, std::min(SURF_GRID_MAX, (int)floorf(ey * dp.sg_inv) + 1));
  dp.sg_bx = std::max(1, bits_for_host(dp.sg_nx - 1));
  dp.Rpad = (float)(R * 1.0001 + 1e-6);
  dp.rhopad = (float)(rrho * 1.0001 + 1e-6);
  dp.halopad = (float)((R + rrho) * 1.0002 + 4e-6);
  dp.zs0 = z0 - (float)(2.0 * rrho);  // z slabs of the cell grid: uniform over the keypoints' z range grown by 2 R/5, clamped outside
  dp.zs_inv_range = 1.0f / std::max((z1 + (float)(2.0 * rrho)) - dp.zs0, 1e-3f);
}

int derive_params(fe_ctx* ctx, const fe_params_t& p) {
  if (!(p.descriptor_radius > 0.0) || !(p.cluster_tolerance > 0.0) || !(p.cluster_radius_threshold > 0.0))
    return fail(ctx, FE_ERR_INVALID, "cluster_tolerance, cluster_radius_threshold and descriptor_radius must be > 0");
  DevParams& dp = ctx->dp;
  memset(&dp, 0, sizeof dp);
  dp.xmin = (float)p.x_min; dp.xmax = (float)p.x_max;
  dp.ymin = (float)p.y_min; dp.ymax = (float)p.y_max;
  dp.zmin = (float)p.z_min; dp.zmax = (float)p.z_max;
  dp.tol_f = (float)p.cluster_tolerance;
  dp.r2f_cluster = radius_sq_as_flann_sees_it((double)dp.tol_f);
  dp.min_count = p.cluster_min_count;
  dp.max_count = p.cluster_max_count;
  dp.two_radius_threshold = 2 * p.cluster_radius_threshold;
  dp.radius_threshold = p.cluster_radius_threshold;
  dp.merge_tol_f = (float)p.cluster_radius_threshold;
  dp.r2f_merge = radius_sq_as_flann_sees_it((double)dp.merge_tol_f);
  dp.min_channels = p.number_detection_channels;
  dp.R2f = radius_sq_as_flann_sees_it(p.descriptor_radius);
  dp.rho2f = radius_sq_as_flann_sees_it(p.descriptor_radius / 5.0);
  dp.estimate_descriptors = p.estimate_descriptors;
  dp.angle_libm = ctx->angleLibm;
  std::vector<float> lut(FE_DESC_LEN);
  shape_context_tables(p.descriptor_radius, p.descriptor_radius / 10.0, dp.radii, dp.theta, dp.phi, lut.data());
  surface_grid(dp, p.descriptor_radius, dp.xmin, dp.xmax, dp.ymin, dp.ymax, dp.zmin, dp.zmax);
  CK(cudaMemcpy(ctx->d_lut, lut.data(), FE_DESC_LEN * sizeof(float), cudaMemcpyHostToDevice));
  ctx->params = p;
  return FE_OK;
}

// ---- slot allocation ---------------------------------------------------------------------------

template <class T>
cudaError_t dalloc(T** p, size_t n) { return cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T)); }
template <class T>
cudaError_t halloc(T** p, size_t n) { return cudaHostAlloc((void**)p, std::max<size_t>(n, 1) * sizeof(T), cudaHostAllocDefault); }

void free_ws(Workspace& w) {
  if (w.d) cudaFree(w.d);
  if (w.h) cudaFreeHost(w.h);
  w = Workspace();
}

void free_slot(Slot& s) {
  for (Workspace& w : s.group) free_ws(w);
  for (cudaEvent_t e : s.ev) if (e) cudaEventDestroy(e);
  for (GraphEntry& g : s.graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  if (s.evDone) cudaEventDestroy(s.evDone);
  if (s.evT0) cudaEventDestroy(s.evT0);
  if (s.evT1) cudaEventDestroy(s.evT1);
  if (s.stream) cudaStreamDestroy(s.stream);
  s = Slot();
}

// A slot's stream, its events and its capacities, nothing else.  The stream is made last: a slot with a stream is open.
int open_slot(fe_ctx* ctx, Slot& s) {
  if (s.stream) return FE_OK;
  const fe_limits_t& L = ctx->lim;
  s.capPts = L.max_points_per_call;
  s.capScans = L.max_scans_per_call;
  s.capChunks = (int)(s.capPts / CH) + s.capScans + 1;
  s.capKp = L.max_keypoints_per_call;
  s.capKf = (int)L.max_ring_clusters_per_call;
  s.capKc = (int)std::min<int64_t>(s.capPts, 1 << 26);
  s.ev.assign(24, nullptr);
  s.evName.assign(24, "");
  cudaError_t e = cudaEventCreateWithFlags(&s.evDone, cudaEventDisableTiming);
  for (cudaEvent_t* t : {&s.evT0, &s.evT1}) if (e == cudaSuccess) e = cudaEventCreate(t);
  for (cudaEvent_t& t : s.ev) if (e == cudaSuccess) e = cudaEventCreate(&t);
  cudaStream_t stream = nullptr;
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    free_slot(s);
    cudaGetLastError();
    return fail(ctx, FE_ERR_CUDA, std::string("opening a slot: ") + cudaGetErrorString(e));
  }
  s.stream = stream;
  return FE_OK;
}

// Lays out one group of a slot's arrays at 256 bytes, the alignment cudaMalloc gives: without bases it only adds up
// the bytes of the device and the pinned buffer; with them it also points the slot's arrays into the buffers.
struct GroupCarve {
  Carve d{256}, h{256};
  unsigned char *dBase = nullptr, *hBase = nullptr;
  template <class T>
  void dev(T*& p, int64_t n) { const Span<T> a = d.take<T>(n); if (dBase) p = a.in(dBase); }
  template <class T>
  void pin(T*& p, int64_t n) { const Span<T> a = h.take<T>(n); if (hBase) p = a.in(hBase); }
};

// Every array of the slot's group g, with its element count: the one list that sizes the group and sets its pointers.
void slot_arrays(Slot& s, Group g, GroupCarve& c) {
  const int64_t np = s.capPts, ns = s.capScans, nkp = s.capKp;
  switch (g) {
    case CORE:  // everything the pipeline sizes from the limits
      c.dev(s.d_surf, np); c.dev(s.d_crop, np); c.dev(s.d_sorted, np); c.dev(s.d_ringPts, np);
      c.dev(s.d_cropMeta, np); c.dev(s.d_keyA, np); c.dev(s.d_keyB, np);
      c.dev(s.d_valA, np); c.dev(s.d_valB, np); c.dev(s.d_sortedKey, np);
      c.dev(s.d_rho, np);
      c.dev(s.d_scan_off, ns + 1); c.dev(s.d_chunk_off, ns + 1);
      c.dev(s.d_surfCnt, s.capChunks); c.dev(s.d_cropCnt, s.capChunks);
      c.dev(s.d_chunkTab, s.capChunks);
      c.dev(s.d_rot, ns * 9);
      c.dev(s.d_kfBase, ns * 16); c.dev(s.d_kfCnt, ns * 16);
      c.dev(s.d_kcBase, ns * 16); c.dev(s.d_kcCnt, ns * 16);
      c.dev(s.d_kpBase, ns); c.dev(s.d_kpCnt, ns); c.dev(s.d_kpOff, ns + 1);
      c.dev(s.d_kpScan, nkp); c.dev(s.d_kpNbr, nkp);
      c.dev(s.d_kpNbrOff, nkp); c.dev(s.d_kpRank, nkp);
      c.dev(s.d_kpListM, nkp); c.dev(s.d_kpListL, nkp);
      c.dev(s.d_surfN, ns); c.dev(s.d_perScan, ns); c.dev(s.d_outOff, ns + 1); c.dev(s.d_tabOk, ns);
      c.dev(s.d_ringBase, ns * 17); c.dev(s.d_ovfRuns, ns * 16); c.dev(s.d_scanFlag, ns);
      c.dev(s.d_ovfRings, ns); c.dev(s.d_ovfRings2, ns); c.dev(s.d_ovfMerge, ns); c.dev(s.d_ovfMerge2, ns);
      c.dev(s.d_ovfSurf, ns);
      c.dev(s.d_slabs, (int64_t)NGLOBAL * cluster_slab_bytes(ECAP_G));
      c.dev(s.d_kfPool, s.capKf); c.dev(s.d_kpPool, nkp); c.dev(s.d_kpOut, nkp);
      c.dev(s.d_desc, nkp * FE_RECORD_FLOATS);  // room for either output layout
      c.dev(s.d_ctr, 1);
      c.pin(s.h_scan_off, ns + 1); c.pin(s.h_chunk_off, ns + 1); c.pin(s.h_rot, ns * 9);
      c.pin(s.h_ctr, 1); c.pin(s.h_kpOff, ns + 1); c.pin(s.h_perScan, ns + 1);
      break;
    case POINTS:  // host points staged for the pipeline (fe_process_batch_device reads the caller's array instead)
      c.dev(s.d_pts, np);
      break;
    case FULL:  // fe_get_elevation_angles, fe_rotate_cloud
      c.dev(s.d_full, np);
      break;
    case CLOUDS:  // the two cloud outputs and the keypoint_cloud pool
      c.dev(s.d_kcPool, s.capKc); c.dev(s.d_gather, np); c.dev(s.d_gather2, s.capKc);
      c.dev(s.d_perScan2, ns); c.dev(s.d_outOff2, ns + 1);
      c.pin(s.h_cloudOff, ns + 1); c.pin(s.h_kcOff, ns + 1);
      break;
    case REPORT:  // the boundary report
      c.dev(s.d_boundary, ns * FE_BOUNDARY_KINDS); c.dev(s.d_gate, ns * 16);
      c.pin(s.h_boundary, ns * FE_BOUNDARY_KINDS);
      break;
    case GRID:  // rows of every grid surface_grid can make; headers of every grid the counting sort takes
      c.dev(s.d_rowStart, ns * (SURF_GRID_MAX + 1)); c.dev(s.d_gridHdr, ns * grid_hdr_bytes(SURF_MAX_CELLS));
      break;
    case NGROUPS: break;
  }
}

// Allocates group g of an open slot, once and in full.  Its arrays are set only when both of its buffers exist; on a
// failure nothing is held, the CUDA error is cleared (a later launch check must not report it) and the next call tries
// again.
int ensure_group(fe_ctx* ctx, Slot& s, Group g) {
  Workspace& w = s.group[g];
  if (w.d) return FE_OK;  // every group has device arrays
  GroupCarve c;
  slot_arrays(s, g, c);
  unsigned char *d = nullptr, *h = nullptr;
  cudaError_t e = cudaMalloc((void**)&d, (size_t)c.d.bytes);
  if (e == cudaSuccess && c.h.bytes > 0) {
    e = cudaHostAlloc((void**)&h, (size_t)c.h.bytes, cudaHostAllocDefault);
    if (e != cudaSuccess) cudaFree(d);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    char b[160];
    snprintf(b, sizeof b, "slot arrays of %lld device and %lld pinned bytes: %s", (long long)c.d.bytes, (long long)c.h.bytes,
             cudaGetErrorString(e));
    return fail(ctx, FE_ERR_CUDA, b);
  }
  w = Workspace{d, c.d.bytes, h, c.h.bytes};
  GroupCarve set;
  set.dBase = d;
  set.hBase = h;
  slot_arrays(s, g, set);
  return FE_OK;
}

// Opens the slot and allocates `groups` in the order given.
int ensure_slot(fe_ctx* ctx, Slot& s, std::initializer_list<Group> groups) {
  int st = open_slot(ctx, s);
  for (Group g : groups)
    if (st == FE_OK) st = ensure_group(ctx, s, g);
  return st;
}

void mark(fe_ctx* ctx, Slot& s, const char* name) {
  if (ctx->stageTiming && s.nev < (int)s.ev.size()) {
    cudaEventRecord(s.ev[s.nev], s.stream);
    s.evName[s.nev] = name;
    s.nev++;
  }
}

std::string err_bits(int e) {
  std::string m;
  if (e & ERR_RING_CAP) m += "one ring of a scan holds more cluster entries than the shared-memory capacity; ";
  if (e & ERR_KF_POOL) m += "ring-centroid pool exhausted (raise max_ring_clusters_per_call); ";
  if (e & ERR_KP_POOL) m += "keypoint pool exhausted (raise max_keypoints_per_call); ";
  if (e & ERR_MERGE_CAP) m += "a scan has more ring centroids than the merge capacity; ";
  if (e & ERR_AXIS_CAP) m += "a scan has more keypoints than precomputed 3DSC axes; ";
  if (e & ERR_CHUNKS) m += "a scan has more points than the per-scan kernels index; ";
  if (e & ERR_KC_POOL) m += "keypoint_cloud pool exhausted; ";
  return m;
}

// the device copies of the arrays stage_scans left in the pinned mirrors (the same addresses every call, so the
// copies can live inside a captured graph)
int stage_scans_copy(fe_ctx* ctx, Slot& s, int nscans, bool deferRot) {
  CK(cudaMemcpyAsync(s.d_scan_off, s.h_scan_off, (nscans + 1) * sizeof(long long), cudaMemcpyHostToDevice, s.stream));
  CK(cudaMemcpyAsync(s.d_chunk_off, s.h_chunk_off, (nscans + 1) * sizeof(int), cudaMemcpyHostToDevice, s.stream));
  if (s.h_chunk_off[nscans] > 0) {  // K1's chunk -> scan table, built where the offsets just landed
    k_chunk_table<<<(nscans + 7) / 8, 256, 0, s.stream>>>(s.d_scan_off, s.d_chunk_off, nscans, s.d_chunkTab);
    ctx->launches++;
  }
  if (!deferRot) CK(cudaMemcpyAsync(s.d_rot, s.h_rot, (size_t)nscans * 9 * sizeof(float), cudaMemcpyHostToDevice, s.stream));
  return FE_OK;
}

// Host-side staging of the small per-scan arrays of a sub-batch into the pinned mirrors.  offs are absolute offsets
// of the caller's array; the device sees offsets relative to the first point of the sub-batch.
int stage_scans(fe_ctx* ctx, Slot& s, const int64_t* offs, const double* rp, int nscans, int64_t* nptsOut, int* nchOut,
                bool deferRot = false) {
  // the pinned mirrors hold capScans(+1) entries: check before the first write
  if (nscans > s.capScans) return fail(ctx, FE_ERR_CAPACITY, "sub-batch exceeds max_scans_per_call");
  const int64_t o0 = offs[0];
  if (o0 < 0) return fail(ctx, FE_ERR_INVALID, "scan_offsets must not be negative");
  if (offs[nscans] - o0 > s.capPts) return fail(ctx, FE_ERR_CAPACITY, "sub-batch exceeds max_points_per_call");
  int nch = 0;
  s.maxScanPts = 0;
  for (int i = 0; i < nscans; i++) {
    const int64_t n = offs[i + 1] - offs[i];
    if (n < 0) return fail(ctx, FE_ERR_INVALID, "scan_offsets must be non-decreasing");
    s.maxScanPts = std::max(s.maxScanPts, n);
    s.h_scan_off[i] = (long long)(offs[i] - o0);
    s.h_chunk_off[i] = nch;
    const int64_t nc = (n + CH - 1) / CH;
    if (nc > (int64_t)s.capChunks - nch) return fail(ctx, FE_ERR_CAPACITY, "sub-batch exceeds the chunk capacity");
    if (nc >= (1 << 20)) return fail(ctx, FE_ERR_CAPACITY, "a scan of more than 2^31 points");  // k_chunk_table packs (chunk << 12) | points
    nch += (int)nc;
    if (deferRot) continue;  // enqueue_pipeline computes the matrices range by range (lateRp)
    if (rp) leveling_matrix(rp[2 * i], rp[2 * i + 1], s.h_rot + 9 * i);
    else { float* m = s.h_rot + 9 * i; for (int k = 0; k < 9; k++) m[k] = (k % 4 == 0) ? 1.0f : 0.0f; }
  }
  s.h_scan_off[nscans] = (long long)(offs[nscans] - o0);
  s.h_chunk_off[nscans] = nch;
  *nptsOut = offs[nscans] - o0;
  *nchOut = nch;
  if (nch > s.capChunks) return fail(ctx, FE_ERR_CAPACITY, "sub-batch exceeds the chunk capacity");
  return FE_OK;
}

SurfIndex surf_index(const DevParams& P, const Slot& s) {
  const int64_t ncells = (int64_t)P.sg_nx * P.sg_ny;
  SurfIndex X;
  X.sortedKey = s.d_sortedKey;
  X.rowStart = s.d_rowStart;
  X.gridHdr = (ncells <= SURF_MAX_CELLS) ? s.d_gridHdr : nullptr;
  X.gridStride = grid_hdr_bytes((int)ncells);
  X.tabOk = s.d_tabOk;
  return X;
}

const size_t kClusterSmem = cluster_smem_bytes(ECAP, NTF);
const size_t kClusterSmemL = cluster_smem_bytes(ECAP_L, NT2);
const size_t kClusterSmemL2 = cluster_smem_bytes(ECAP_L, NTL);
const size_t kClusterSmemM = cluster_smem_bytes(ECAP_M, NTM);

int set_kernel_attrs(fe_ctx* ctx) {
  CK(cudaFuncSetAttribute(k_cluster_rings<ECAP, NTF, 4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kClusterSmem));
  CK(cudaFuncSetAttribute(k_ring_runs<NW_RR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RingRunsSmT<RW>)));
  CK(cudaFuncSetAttribute(k_ring_runs<NW_RR_SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RingRunsSmT<RW, NW_RR_SMALL>)));
  CK(cudaFuncSetAttribute(k_ring_runs_wide<>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(NW_RR * sizeof(RunBufT<RW2>))));
  CK(cudaFuncSetAttribute(k_cluster_rings<ECAP_L, NTL, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kClusterSmemL2));
  CK(cudaFuncSetAttribute(k_merge_keypoints<ECAP_M, NTM, 8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kClusterSmemM));
  CK(cudaFuncSetAttribute(k_merge_keypoints<ECAP_L, NT2, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kClusterSmemL));
  CK(cudaFuncSetAttribute(k_extract_clusters_stage<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kClusterSmemL));
  CK(cudaFuncSetAttribute(k_desc_hist_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)desc_warp_smem_bytes()));
  CK(cudaFuncSetAttribute(k_desc_hist<256, DCAP, DW_CAP, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)desc_smem_bytes(DCAP, 256)));
  CK(cudaFuncSetAttribute(k_desc_hist<512, DCAP_M, DCAP, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)desc_smem_bytes(DCAP_M, 512)));
  CK(cudaFuncSetAttribute(k_desc_hist<512, DCAP_L, DCAP_M, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)desc_smem_bytes(DCAP_L, 512)));
  CK(cudaFuncSetAttribute(k_surface_grid_cells<NT_SURF>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)surf_cells_smem_bytes(SURF_MAX_CELLS)));
  // the boundary report's K2 instantiations (kind 6).  Named after every other kernel: the order in which the host
  // code first names the kernels is the order the compiler meets them, and the kernels above compile as they did
  // before these existed only in this order.
  CK(cudaFuncSetAttribute(k_cluster_rings<ECAP, NTF, 4, false, GateCount>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kClusterSmem));
  CK(cudaFuncSetAttribute(k_ring_runs<NW_RR, GateCount>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RingRunsSmT<RW>)));
  CK(cudaFuncSetAttribute(k_ring_runs<NW_RR_SMALL, GateCount>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)sizeof(RingRunsSmT<RW, NW_RR_SMALL>)));
  CK(cudaFuncSetAttribute(k_ring_runs_wide<GateCount>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(NW_RR * sizeof(RunBufT<RW2>))));
  CK(cudaFuncSetAttribute(k_cluster_rings<ECAP_L, NT2, 1, false, GateCount>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kClusterSmemL));
  return FE_OK;
}

// K4d: three instantiations split the keypoints by neighbour count (smaller footprint = more blocks / SM)
void launch_desc_hist(fe_ctx* ctx, Slot& s, int nscans, const DevParams& P, int gridKp, bool records, bool lean = false) {
  const int descStride = records ? FE_RECORD_FLOATS : FE_DESC_LEN, descOff = records ? 5 : 0;
  // the blocks stride over the keypoints with equal shares: grids of exactly one resident wave
  static const int perSm = []() {  // initialised once, also when fe_multi's threads get here together
    int v = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, k_desc_hist<256, DCAP, DW_CAP, false, true>, 256, desc_smem_bytes(DCAP, 256)) != cudaSuccess) v = 4;
    return v;
  }();
  // A handful of scans (the reference's one scan per callback) has too few keypoints to fill the GPU with warps:
  // there the same algorithm runs with a block per keypoint (k_desc_hist_small), several times shorter per keypoint.
  const int warpCap = DW_CAP;
  if (nscans <= GRAPH_MAX_SCANS) {
    k_desc_hist_small<<<std::min(gridKp, ctx->numSms * 4), DW_CAP, 0, s.stream>>>(
        s.d_kpOut, s.d_kpScan, s.d_kpOff, nscans, s.d_kpNbr, s.d_sorted, s.d_scan_off, P, s.d_rho, ctx->d_lut, ctx->d_axes, ctx->axesCap,
        s.d_keyA, s.d_kpNbrOff, s.d_kpRank, s.d_desc, descStride, descOff, s.d_ctr);
    ctx->launches++;
  } else {  // keypoints with at most DW_CAP listed neighbours (and the empty ones): a warp each
    static const int perSmW = []() {
      int v = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, k_desc_hist_warp, DW_WARPS * 32, desc_warp_smem_bytes()) != cudaSuccess) v = 2;
      return v;
    }();
    const int nsm = ctx->numSms;
    k_desc_hist_warp<<<nsm * std::max(perSmW, 1), DW_WARPS * 32, desc_warp_smem_bytes(), s.stream>>>(
        s.d_kpOut, s.d_kpScan, s.d_kpOff, nscans, s.d_kpNbr, s.d_sorted, s.d_scan_off, P, s.d_rho, ctx->d_lut, ctx->d_axes, ctx->axesCap,
        s.d_keyA, s.d_kpNbrOff, s.d_kpRank, s.d_desc, descStride, descOff, s.d_ctr);
    ctx->launches++;
  }
  // glist / nlist: the keypoints the previous instantiation listed for this one (null: every keypoint)
  auto hist = [&](auto kernel, int grid, int nt, size_t smem, const int* glist, const int* nlist) {
    kernel<<<grid, nt, smem, s.stream>>>(s.d_kpOut, s.d_kpScan, s.d_kpOff, nscans, s.d_kpNbr, s.d_sorted, surf_index(P, s),
                                         s.d_scan_off, P, s.d_rho, ctx->d_lut, ctx->d_axes, ctx->axesCap, s.d_keyA, s.d_kpNbrOff,
                                         s.d_kpRank, glist, nlist, s.d_desc, descStride, descOff, s.d_ctr, warpCap);
    ctx->launches++;
  };
  hist(k_desc_hist<256, DCAP, DW_CAP, false, true>, std::min(gridKp, ctx->numSms * std::max(perSm, 1)), 256,
       desc_smem_bytes(DCAP, 256), nullptr, nullptr);
  if (!lean) {  // lean: keypoints listed for the two larger instantiations make the caller run the sub-batch again
    hist(k_desc_hist<512, DCAP_M, DCAP, false, false>, std::min(gridKp, ctx->numSms * 2), 512, desc_smem_bytes(DCAP_M, 512),
         s.d_kpListM, &s.d_ctr->n_list_m);
    hist(k_desc_hist<512, DCAP_L, DCAP_M, true, false>, std::min(gridKp, ctx->numSms), 512, desc_smem_bytes(DCAP_L, 512),
         s.d_kpListL, &s.d_ctr->n_list_l);
  }
  if (records) {
    k_record_frame<<<ctx->numSms * 2, 256, 0, s.stream>>>(s.d_kpOut, s.d_kpOff, nscans, s.d_desc, descStride, FE_DESC_LEN);
    ctx->launches++;
  }
}

// K4b: mark + count + neighbour lists (the pool is d_keyA, idle once K4a is done), then the RNG ranks.
void launch_desc_mark(fe_ctx* ctx, Slot& s, int nscans, const DevParams& P, int gridKp) {
  const long long nbrCap = (long long)std::min<int64_t>(s.capPts, 0x7fffffff - MARK_LCAP);
  // the blocks stride over the keypoints with equal shares: a grid of exactly one resident wave
  static const int perSm = []() {
    int v = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, k_desc_mark, 256, MARK_LCAP * sizeof(unsigned)) != cudaSuccess) v = 4;
    return v;
  }();
  gridKp = std::min(gridKp, ctx->numSms * std::max(perSm, 1));
  k_desc_mark<<<gridKp, 256, MARK_LCAP * sizeof(unsigned), s.stream>>>(s.d_kpOut, s.d_kpScan, s.d_kpOff, nscans, s.d_sorted,
                                                                       surf_index(P, s), s.d_scan_off, P, s.d_rho, s.d_kpNbr,
                                                                       s.d_keyA, nbrCap, s.d_kpNbrOff, s.d_ctr);
  k_kp_rank<<<(int)((s.capKp + 255) / 256), 256, 0, s.stream>>>(s.d_kpScan, s.d_kpOff, nscans, s.d_kpNbr, s.d_kpRank, s.d_kpListM, s.d_kpListL, s.d_ctr);
  ctx->launches += 2;
}

// K4a: counting sort by cell in shared memory for scans that fit (<= 65,535 surface points, grid <=
// SURF_MAX_CELLS cells), radix sort through global memory for the deferred rest.
void launch_surface_grid(fe_ctx* ctx, Slot& s, int nscans, const DevParams& P) {
  const int ncells = P.sg_nx * P.sg_ny;
  if (ncells <= SURF_MAX_CELLS) {
    k_surface_grid_cells<NT_SURF><<<nscans, NT_SURF, surf_cells_smem_bytes(ncells), s.stream>>>(
        s.d_surf, s.d_surfCnt, s.d_scan_off, s.d_chunk_off, P, s.d_kpOut, s.d_kpOff, s.d_sorted, s.d_rho,
        s.d_surfN, s.d_ctr, s.d_ovfSurf, s.d_gridHdr, grid_hdr_bytes(ncells), s.d_tabOk);
    ctx->launches++;
    // the radix kernel only takes scans the counting sort defers: more than 65,535 surface points or more halo
    // cells than counters — impossible when every scan is small and the grid has no more cells than counters
    if (s.maxScanPts <= 65535 && ncells <= GRID_TAB_CAP) return;
    k_surface_grid<<<std::min(nscans, ctx->numSms * 2), NT2, 0, s.stream>>>(s.d_surf, s.d_surfCnt, s.d_scan_off, s.d_chunk_off, P, s.d_keyA,
                                                                   s.d_keyB, s.d_valA, s.d_valB, s.d_sorted, s.d_sortedKey,
                                                                   s.d_rowStart, s.d_surfN, s.d_ctr, s.d_ovfSurf, &s.d_ctr->ovf_surf,
                                                                   s.d_tabOk, s.d_rho);
  } else {
    k_surface_grid<<<nscans, NT2, 0, s.stream>>>(s.d_surf, s.d_surfCnt, s.d_scan_off, s.d_chunk_off, P, s.d_keyA, s.d_keyB, s.d_valA,
                                                 s.d_valB, s.d_sorted, s.d_sortedKey, s.d_rowStart, s.d_surfN, s.d_ctr, nullptr, nullptr,
                                                 s.d_tabOk, s.d_rho);
  }
  ctx->launches++;
}

// blocks per scan of K4c: about one per 8k points of an average scan (a dense scan's halo is tens of tiles)
int density_blocks_per_scan(int nscans, int64_t npts) {
  return (int)std::max<int64_t>(1, std::min<int64_t>(16, npts / std::max(nscans, 1) / 8192 + 1));
}

void launch_density(fe_ctx* ctx, Slot& s, int nscans, const DevParams& P, int64_t npts) {
  if (nscans <= 0) return;
  const int by = density_blocks_per_scan(nscans, npts);
  k_density<<<dim3((unsigned)nscans, (unsigned)by), 256, 0, s.stream>>>(s.d_sorted, surf_index(P, s), s.d_scan_off, P, s.d_surfN, s.d_rho, s.d_ctr->dens_work);
  ctx->launches++;
}

// K2 + K3 for `nscans` scans: the 2-blocks-per-SM instantiation first, then the large one over
// whatever scans it deferred (an immediate exit when there are none).
// gate...: nothing, or the GateCount with which the K2 instantiations count kind 6 of the boundary report
// (fe_enable_boundary_report_all)
template <class... G>
void launch_clustering(fe_ctx* ctx, Slot& s, int nscans, bool singleRing, bool wantKc, bool merge, bool marks = false, bool lean = false,
                       G... gate) {
  // Every stage is a chain of instantiations: the fast one takes all scans and defers those that do
  // not fit its shared memory to a list; the large shared-memory one takes that list; what does not
  // fit there either goes to the instantiation whose per-entry arrays live in global memory.
  const DevParams& P = ctx->dp;
  const int gridL = std::min(nscans, ctx->numSms), gridG = std::min(nscans, NGLOBAL);
  const size_t smemG = cluster_smem_bytes_global(NT2);
  // K2's large instantiation counting kind 6 runs 512 threads, not NTL: a second caller of the 1024-thread cluster
  // helpers changes how k_cluster_rings<ECAP_L, NTL> compiles (the capacity is the same, hence the same deferrals
  // and clusters)
  constexpr int ntL = sizeof...(G) > 0 ? NT2 : NTL;
  int* ovfR = &s.d_ctr->ovf_rings;
  int* ovfR2 = &s.d_ctr->ovf_rings2;
  int* ovfM = &s.d_ctr->ovf_merge;
  int* ovfM2 = &s.d_ctr->ovf_merge2;
  float4* kc = wantKc ? s.d_kcPool : nullptr;
  int* kcB = wantKc ? s.d_kcBase : nullptr;
  int* kcC = wantKc ? s.d_kcCnt : nullptr;
  const int sr = singleRing ? 1 : 0;
  // inList / inN: the scans the previous instantiation deferred to this one (null: every scan); outList / outN: where
  // this one defers what it cannot take (null: the last of the chain); slabs: per-entry arrays in global memory
  auto k2 = [&](auto kernel, int grid, int nt, size_t smem, const int* inList, const int* inN, int* outList, int* outN,
                unsigned char* slabs) {
    kernel<<<grid, nt, smem, s.stream>>>(s.d_crop, s.d_cropMeta, s.d_cropCnt, s.d_scan_off, s.d_chunk_off, P, sr, s.d_kfPool,
                                         s.capKf, s.d_kfBase, s.d_kfCnt, kc, s.capKc, kcB, kcC, s.d_ctr, inList, inN, outList,
                                         outN, slabs, gate...);
    ctx->launches++;
  };
  auto k3 = [&](auto kernel, int grid, int nt, size_t smem, const int* inList, const int* inN, int* outList, int* outN,
                unsigned char* slabs) {
    kernel<<<grid, nt, smem, s.stream>>>(s.d_kfPool, s.d_kfBase, s.d_kfCnt, P, s.d_kpPool, (int)s.capKp, s.d_kpBase, s.d_kpCnt,
                                         s.d_ctr, inList, inN, outList, outN, slabs);
    ctx->launches++;
  };
  // K2: the run-based kernel takes every scan; what it cannot handle (a ring with more than RW runs — unordered
  // input — or more ring entries than the scan's scratch slot) goes down the chain of grid-based instantiations.
  if (ctx->gridClustering) {
    k2(k_cluster_rings<ECAP, NTF, 4, false, G...>, nscans, NTF, kClusterSmem, nullptr, nullptr, s.d_ovfRings, ovfR, nullptr);
  } else {
    auto rr = [&](auto kernel, int nt, size_t smem) {
      kernel<<<nscans, nt, smem, s.stream>>>(s.d_crop, s.d_cropMeta, s.d_cropCnt, s.d_scan_off, s.d_chunk_off, P, sr, s.d_ringPts,
                                             s.d_ringBase, s.d_kfPool, s.capKf, s.d_kfBase, s.d_kfCnt, kc, s.capKc, kcB, kcC, s.d_ctr,
                                             s.d_ovfRuns, &s.d_ctr->ovf_runs, s.d_scanFlag, s.d_ovfRings, ovfR, gate...);
      ctx->launches++;
    };
    if (nscans <= GRAPH_MAX_SCANS)  // a handful of scans: a warp for each of a scan's 16 rings at once (latency, not throughput)
      rr(k_ring_runs<NW_RR_SMALL, G...>, NW_RR_SMALL * 32, sizeof(RingRunsSmT<RW, NW_RR_SMALL>));
    else
      rr(k_ring_runs<NW_RR, G...>, NT_RR, sizeof(RingRunsSmT<RW>));
    if (!lean) {
      k_ring_runs_wide<G...><<<std::min(nscans * 4, ctx->numSms * 7), NT_RR, NW_RR * sizeof(RunBufT<RW2>), s.stream>>>(
          s.d_scan_off, P, s.d_ringPts, s.d_ringBase, s.d_kfPool, s.capKf, s.d_kfBase, s.d_kfCnt, kc, s.capKc, kcB, kcC, s.d_ctr,
          s.d_ovfRuns, &s.d_ctr->ovf_runs, s.d_scanFlag, s.d_ovfRings, ovfR, gate...);
      ctx->launches++;
    }
  }
  // lean: the fallback instantiations are left out; whatever the first kernel deferred shows in the counters and the
  // caller runs the sub-batch again with the whole chain
  if (!lean) {
    k2(k_cluster_rings<ECAP_L, ntL, 1, false, G...>, gridL, ntL, cluster_smem_bytes(ECAP_L, ntL), s.d_ovfRings, ovfR, s.d_ovfRings2,
       ovfR2, nullptr);
    k2(k_cluster_rings<ECAP_G, NT2, 1, true, G...>, gridG, NT2, smemG, s.d_ovfRings2, ovfR2, nullptr, nullptr, s.d_slabs);
  }
  if (marks) mark(ctx, s, "K2 ring clusters");
  if (merge) {
    k3(k_merge_keypoints<ECAP_M, NTM, 8, false>, nscans, NTM, kClusterSmemM, nullptr, nullptr, s.d_ovfMerge, ovfM, nullptr);
    if (!lean) {
      k3(k_merge_keypoints<ECAP_L, NT2, 1, false>, gridL, NT2, kClusterSmemL, s.d_ovfMerge, ovfM, s.d_ovfMerge2, ovfM2, nullptr);
      k3(k_merge_keypoints<ECAP_G, NT2, 1, true>, gridG, NT2, smemG, s.d_ovfMerge2, ovfM2, nullptr, nullptr, s.d_slabs);
    }
  }
}


// fe_enable_boundary_report: the four radius predicates of the path and the float pre-filter windows
BoundarySpec boundary_spec(const fe_ctx* ctx) {
  BoundarySpec B;
  B.eps = ctx->bndEps;
  const float r2[4] = {ctx->dp.r2f_cluster, ctx->dp.r2f_merge, ctx->dp.R2f, ctx->dp.rho2f};
  for (int k = 0; k < 4; k++) {
    B.r2f[k] = r2[k];
    B.bdist[k] = sqrt((double)r2[k]);
    B.win[k] = (float)(B.eps * (2.0 * B.bdist[k] + B.eps) * 1.01 + (double)r2[k] * 1e-6);
  }
  return B;
}

// Enqueue the kernels of the slot's sub-batch s.sb, K1 to K4d, and the copies of its counters, keypoint offsets and
// boundary counts to the pinned mirrors; its scan offsets must be on the device already (stage_scans_copy).  With
// `lateRp` the levelling matrices are computed here, interleaved with K1.  recordDone: record the slot's evDone.
int enqueue_pipeline(fe_ctx* ctx, Slot& s, const double* lateRp, bool recordDone) {
  const DevParams& P = ctx->dp;
  const SubBatch& sb = s.sb;
  const int nscans = sb.nscans;
  s.nev = 0;
  mark(ctx, s, "begin");
  CK(cudaMemsetAsync(s.d_ctr, 0, sizeof(DevCounters), s.stream));
  if (sb.nch > 0) {
    // With `lateRp` the levelling matrices (two sincos and a quaternion product per scan on the host,
    // ~0.4 ms for 10 k scans) are not staged yet: they are computed range by range — an eighth, an
    // eighth, a quarter, a half of the scans — and K1 is launched per range, so that all but the first
    // eighth of that host work runs while the GPU is already busy.  (16 equal ranges were measured:
    // slower, the per-range copy and launch calls starve the GPU.)
    const int cuts[5] = {0, nscans / 8, nscans / 4, nscans / 2, nscans};
    const int nparts = lateRp ? 4 : 1;
    for (int part = 0; part < nparts; part++) {
      const int a = lateRp ? cuts[part] : 0, b = lateRp ? cuts[part + 1] : nscans;
      if (b <= a) continue;
      if (lateRp) {
        for (int i = a; i < b; i++) leveling_matrix(lateRp[2 * i], lateRp[2 * i + 1], s.h_rot + 9 * i);
        CK(cudaMemcpyAsync(s.d_rot + 9 * (size_t)a, s.h_rot + 9 * (size_t)a, (size_t)(b - a) * 9 * sizeof(float), cudaMemcpyHostToDevice, s.stream));
        // stage times: whatever the GPU waited for the host goes to its own line, not to K1
        if (part == 0) { s.nev = 0; mark(ctx, s, "begin"); } else mark(ctx, s, "host: levelling matrices");
      }
      const int ca = s.h_chunk_off[a], cb = s.h_chunk_off[b];
      if (cb <= ca) continue;
      if (sb.lay.raw)
        k_level_crop_ring<true, true><<<cb - ca, 256, 0, s.stream>>>(sb.pts, s.d_chunkTab, s.d_rot, P, sb.k1flags,
                                                               s.d_surf, s.d_surfCnt, s.d_crop, s.d_cropMeta, s.d_cropCnt, nullptr, sb.lay, ca);
      else
        k_level_crop_ring<false, true><<<cb - ca, 256, 0, s.stream>>>(sb.pts, s.d_chunkTab, s.d_rot, P, sb.k1flags,
                                                                s.d_surf, s.d_surfCnt, s.d_crop, s.d_cropMeta, s.d_cropCnt, nullptr, sb.lay, ca);
      ctx->launches++;
      if (lateRp && part + 1 < nparts) mark(ctx, s, "K1 level+crop+ring");
    }
  }
  mark(ctx, s, "K1 level+crop+ring");
  const int kinds = nscans > 0 ? ctx->bndKinds : 0;  // of the boundary report: 0, 4 or FE_BOUNDARY_KINDS
  const bool allKinds = kinds == FE_BOUNDARY_KINDS;
  const BoundarySpec B = boundary_spec(ctx);
  if (kinds) {
    CK(cudaMemsetAsync(s.d_boundary, 0, (size_t)nscans * FE_BOUNDARY_KINDS * sizeof(unsigned long long), s.stream));
    k_boundary_rings<<<nscans, 256, 0, s.stream>>>(s.d_crop, s.d_cropMeta, s.d_cropCnt, s.d_scan_off, s.d_chunk_off, 0, B, s.d_boundary);
    ctx->launches++;
  }
  if (allKinds) {
    CK(cudaMemsetAsync(s.d_gate, 0, (size_t)nscans * 16 * sizeof(unsigned), s.stream));
    const int nch = s.h_chunk_off[nscans];  // every chunk of the sub-batch: the matrices of all of them are staged by now
    if (nch > 0) {
      if (sb.lay.raw) k_boundary_crop_ring<true><<<nch, 256, 0, s.stream>>>(sb.pts, s.d_chunkTab, s.d_rot, P, sb.lay, B.eps, s.d_boundary);
      else k_boundary_crop_ring<false><<<nch, 256, 0, s.stream>>>(sb.pts, s.d_chunkTab, s.d_rot, P, sb.lay, B.eps, s.d_boundary);
      ctx->launches++;
    }
  }
  if (allKinds) launch_clustering(ctx, s, nscans, false, sb.wantKc, true, true, sb.lean, GateCount{B.eps, s.d_gate});
  else launch_clustering(ctx, s, nscans, false, sb.wantKc, true, true, sb.lean);
  mark(ctx, s, "K3 merge keypoints");
  if (kinds) {
    k_boundary_merge<<<nscans, 128, 0, s.stream>>>(s.d_kfPool, s.d_kfBase, s.d_kfCnt, P, B, s.d_boundary);
    ctx->launches++;
  }
  if (allKinds) {
    k_boundary_gate_sum<<<(nscans + 255) / 256, 256, 0, s.stream>>>(s.d_gate, nscans, s.d_boundary);
    ctx->launches++;
  }
  if (nscans <= GRAPH_MAX_SCANS) {  // a handful of scans: offsets and ordered copy in one launch
    k_kp_offsets_gather_small<<<1, 1024, 0, s.stream>>>(s.d_kpCnt, nscans, s.d_kpOff, s.d_ctr, s.d_kpPool, s.d_kpBase, s.d_kpOut, s.d_kpScan);
    ctx->launches++;
  } else {
    k_kp_offsets<<<1, 1024, 0, s.stream>>>(s.d_kpCnt, nscans, s.d_kpOff, s.d_ctr);
    k_kp_gather<<<std::max(1, std::min(1024, (nscans * 8 + 255) / 256)), 256, 0, s.stream>>>(s.d_kpPool, s.d_kpBase, s.d_kpOff, nscans,
                                                                                              s.d_kpOut, s.d_kpScan);
    ctx->launches += 2;
  }
  mark(ctx, s, "keypoint CSR");
  if (sb.desc) {
    // K4a runs after the keypoints are known: it only keeps the surface points a keypoint can reach
    launch_surface_grid(ctx, s, nscans, P);
    mark(ctx, s, "K4a surface grid");
    const int gridKp = ctx->numSms * 8;
    launch_desc_mark(ctx, s, nscans, P, gridKp);
    mark(ctx, s, "K4b mark neighbours");
    if (kinds) {  // before K4c turns the marks in rho into densities
      k_boundary_support<<<ctx->numSms * 4, 256, 0, s.stream>>>(s.d_kpOut, s.d_kpScan, s.d_kpOff, nscans, s.d_sorted, surf_index(P, s),
                                                         s.d_scan_off, P, B, s.d_boundary);
      if (sb.npts > 0)
        k_boundary_density<<<nscans, 256, 0, s.stream>>>(s.d_sorted, surf_index(P, s), s.d_scan_off, P, s.d_surfN, s.d_rho, B,
                                                         s.d_boundary);
      ctx->launches += 2;
    }
    if (allKinds) {
      k_boundary_bins<<<ctx->numSms * 4, 256, 0, s.stream>>>(s.d_kpOut, s.d_kpScan, s.d_kpOff, nscans, s.d_sorted, surf_index(P, s),
                                                             s.d_scan_off, P, ctx->d_axes, ctx->axesCap, s.d_kpRank, B.eps, s.d_boundary);
      ctx->launches++;
    }
    launch_density(ctx, s, nscans, P, sb.npts);
    mark(ctx, s, "K4c density");
    launch_desc_hist(ctx, s, nscans, P, gridKp, ctx->recordOutput, sb.lean);
    mark(ctx, s, "K4d shape context");
  }
  if (sb.wantKc && ctx->cloudOutputs && nscans > 0) {
    // ~cloud (src:137-139) and ~keypoint_cloud (src:133-135): per-scan counts, offsets and the ordered gather all
    // on the device; the host only learns the offsets (finalize_subbatch then copies the dense arrays out)
    const int gb = (nscans + 255) / 256;
    k_piece_counts<<<gb, 256, 0, s.stream>>>(s.d_cropCnt, s.d_chunk_off, nscans, s.d_perScan);
    k_offsets_scan<<<1, 1024, 0, s.stream>>>(s.d_perScan, nscans, s.d_outOff);
    k_gather_chunks<<<nscans, 256, 0, s.stream>>>(s.d_crop, s.d_cropCnt, s.d_scan_off, s.d_chunk_off, s.d_outOff, s.d_gather);
    k_pool16_counts<<<gb, 256, 0, s.stream>>>(s.d_kcCnt, nscans, s.d_perScan2);
    k_offsets_scan<<<1, 1024, 0, s.stream>>>(s.d_perScan2, nscans, s.d_outOff2);
    k_gather_pool16<<<nscans, 256, 0, s.stream>>>(s.d_kcPool, s.d_kcBase, s.d_kcCnt, s.d_outOff2, s.d_gather2);
    ctx->launches += 6;
    CK(cudaMemcpyAsync(s.h_cloudOff, s.d_outOff, (size_t)(nscans + 1) * sizeof(int), cudaMemcpyDeviceToHost, s.stream));
    CK(cudaMemcpyAsync(s.h_kcOff, s.d_outOff2, (size_t)(nscans + 1) * sizeof(int), cudaMemcpyDeviceToHost, s.stream));
  }
  CK(cudaMemcpyAsync(s.h_ctr, s.d_ctr, sizeof(DevCounters), cudaMemcpyDeviceToHost, s.stream));
  CK(cudaMemcpyAsync(s.h_kpOff, s.d_kpOff, (size_t)(nscans + 1) * sizeof(int), cudaMemcpyDeviceToHost, s.stream));
  if (kinds)
    CK(cudaMemcpyAsync(s.h_boundary, s.d_boundary, (size_t)nscans * FE_BOUNDARY_KINDS * sizeof(unsigned long long),
                       cudaMemcpyDeviceToHost, s.stream));
  if (recordDone) CK(cudaEventRecord(s.evDone, s.stream));
  CK(cudaGetLastError());
  return FE_OK;
}

void collect_times(fe_ctx* ctx, Slot& s) {
  ctx->stName.clear();
  ctx->stMs.clear();
  for (int i = 1; i < s.nev; i++) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, s.ev[i - 1], s.ev[i]) == cudaSuccess) {
      ctx->stName.push_back(s.evName[i]);
      ctx->stMs.push_back(ms);
    }
  }
}

// Grow the pinned result buffer *buf of *cap records of `rec` elements to hold `need` records (half as many again, at
// least minCap), keeping its first `keep` records.  A sub-batch in flight may still be copying into the old buffer:
// both slots are drained first.
template <class T>
int grow_pinned(fe_ctx* ctx, T** buf, int64_t* cap, int64_t need, int64_t minCap, int64_t keep, size_t rec = 1) {
  if (need <= *cap) return FE_OK;
  int st = sync_slots(ctx);
  if (st) return st;
  const int64_t ncap = std::max<int64_t>(need * 3 / 2, minCap);
  T* nb = nullptr;
  CK(halloc(&nb, (size_t)ncap * rec));
  if (*buf) { memcpy(nb, *buf, (size_t)keep * rec * sizeof(T)); cudaFreeHost(*buf); }
  *buf = nb;
  *cap = ncap;
  return FE_OK;
}

// The sub-batch ran the lean chain (first instantiation of every stage only, see enqueue_subbatch).  Anything one of
// them deferred to a fallback kernel is in the counters: run the sub-batch again, eagerly, with the whole chain (its
// points and staged offsets are still where they were), and keep the lean chain off for a while — inputs that defer
// once (unordered clouds, very large descriptor radii) usually keep doing so.  Call after the slot's evDone.
int lean_rerun_if_deferred(fe_ctx* ctx, Slot& s) {
  if (!s.sb.lean) return FE_OK;
  s.sb.lean = false;
  const DevCounters& c = *s.h_ctr;
  if (c.err || !(c.ovf_runs | c.ovf_rings | c.ovf_rings2 | c.ovf_merge | c.ovf_merge2 | c.n_list_m | c.n_list_l)) return FE_OK;
  ctx->leanHold = 256;
  ctx->leanReruns++;
  int st = enqueue_pipeline(ctx, s, nullptr, true);
  if (st) return st;
  CK(cudaEventSynchronize(s.evDone));
  return FE_OK;
}

// Enqueue `sb`, whose offsets stage_scans left in the slot's pinned mirrors, and record the slot's evDone; `upload`:
// `bytes` of host points to copy to the slot's d_pts first (none: the points are on the device).  A large sub-batch
// runs eagerly.  One of at most GRAPH_MAX_SCANS scans is captured into a CUDA graph per GraphKey (on its second
// sighting) and replayed from then on.  Lean chain: a handful of scans almost never needs a fallback instantiation,
// and seven kernels that only find that out cost more than a tenth of a single scan's latency; they are left out and
// lean_rerun_if_deferred repairs the rare miss.
int enqueue_subbatch(fe_ctx* ctx, Slot& s, const SubBatch& sb, const double* lateRp, const void* upload = nullptr,
                     size_t bytes = 0) {
  // every group the pipeline may need is allocated before it is enqueued, so never while a capture runs
  int st = sb.desc ? ensure_group(ctx, s, GRID) : FE_OK;
  if (st == FE_OK && ctx->bndKinds) st = ensure_group(ctx, s, REPORT);
  if (st == FE_OK && sb.wantKc) st = ensure_group(ctx, s, CLOUDS);
  if (st) return st;
  s.sb = sb;
  s.sb.lean = false;
  if (lateRp || !ctx->useGraphs || ctx->stageTiming || sb.nscans > GRAPH_MAX_SCANS) {
    // offsets and chunk table ahead of the points: with the points first, 10k scans through fe_process_batch took
    // 49 instead of 43 ms on a B200 (1,000 W)
    st = stage_scans_copy(ctx, s, sb.nscans, lateRp != nullptr);
    if (st) return st;
    if (bytes) CK(cudaMemcpyAsync(s.d_pts, upload, bytes, cudaMemcpyHostToDevice, s.stream));
    return enqueue_pipeline(ctx, s, lateRp, true);
  }
  if (bytes) CK(cudaMemcpyAsync(s.d_pts, upload, bytes, cudaMemcpyHostToDevice, s.stream));
  s.sb.lean = ctx->leanHold == 0;
  if (ctx->leanHold > 0) ctx->leanHold--;
  const GraphKey key = {s.sb, density_blocks_per_scan(sb.nscans, sb.npts), s.maxScanPts > 65535, ctx->bndKinds, ctx->epoch};
  GraphEntry* ge = nullptr;
  for (GraphEntry& g : s.graphs) if (g.key == key) { ge = &g; break; }
  if (ge && ge->exec) {  // replay
    CK(cudaGraphLaunch(ge->exec, s.stream));
    ctx->launches += ge->launches;
    ctx->graphReplays++;
  } else if (!ge) {      // first sighting of the shape: eager, so that every lazily initialised piece exists
    st = stage_scans_copy(ctx, s, sb.nscans, false);
    if (st) return st;
    st = enqueue_pipeline(ctx, s, nullptr, false);
    if (st) return st;
    if (s.graphs.size() >= 16) {  // drop the oldest shape
      if (s.graphs[0].exec) cudaGraphExecDestroy(s.graphs[0].exec);
      s.graphs.erase(s.graphs.begin());
    }
    GraphEntry e; e.key = key;
    s.graphs.push_back(e);
  } else {               // second sighting: capture, instantiate, launch
    const int64_t l0 = ctx->launches;
    CK(cudaStreamBeginCapture(s.stream, cudaStreamCaptureModeThreadLocal));
    st = stage_scans_copy(ctx, s, sb.nscans, false);
    if (st == FE_OK) st = enqueue_pipeline(ctx, s, nullptr, false);
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(s.stream, &graph);
    if (st) { if (graph) cudaGraphDestroy(graph); return st; }
    if (ce != cudaSuccess) return fail(ctx, FE_ERR_CUDA, std::string("graph capture: ") + cudaGetErrorString(ce));
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ci = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ci != cudaSuccess) return fail(ctx, FE_ERR_CUDA, std::string("graph instantiate: ") + cudaGetErrorString(ci));
    ge->exec = exec;
    ge->launches = ctx->launches - l0;
    CK(cudaGraphLaunch(exec, s.stream));
    ctx->graphReplays++;
  }
  CK(cudaEventRecord(s.evDone, s.stream));
  return FE_OK;
}

// Wait for the sub-batch in `s`, run it again in full if its lean chain deferred anything, check its error word, and
// write its keypoint offsets (plus kpBase) and boundary counts at scan s.firstScan of the call's results.
int complete_subbatch(fe_ctx* ctx, Slot& s, int64_t kpBase) {
  CK(cudaEventSynchronize(s.evDone));
  int st = lean_rerun_if_deferred(ctx, s);
  if (st) return st;
  if (s.h_ctr->err) return fail(ctx, FE_ERR_CAPACITY, err_bits(s.h_ctr->err));
  const int ns = s.sb.nscans;
  for (int i = 0; i <= ns; i++) ctx->kpOffsets[s.firstScan + i] = kpBase + s.h_kpOff[i];
  if (ctx->bndKinds && s.h_boundary)
    for (int i = 0; i < ns; i++) {
      const unsigned long long* row = s.h_boundary + (size_t)i * FE_BOUNDARY_KINDS;
      const size_t scan = (size_t)s.firstScan + i;
      std::copy(row, row + 4, &ctx->bndCounts[scan * 4]);
      if (ctx->bndKinds == FE_BOUNDARY_KINDS) std::copy(row, row + FE_BOUNDARY_KINDS, &ctx->bndCountsAll[scan * FE_BOUNDARY_KINDS]);
    }
  return FE_OK;
}

// complete the sub-batch in `s` (if any) and append its results to the host call's pinned result buffers
int finalize_subbatch(fe_ctx* ctx, Slot& s, int64_t& kpRun) {
  if (!s.busy) return FE_OK;
  s.busy = false;
  int st = complete_subbatch(ctx, s, kpRun);
  if (st) return st;
  const int ns = s.sb.nscans;
  const int K = s.h_kpOff[ns];
  st = grow_pinned(ctx, &ctx->h_kp, &ctx->capResKp, kpRun + K, 4096, kpRun);
  if (st) return st;
  if (s.sb.desc) {
    st = grow_pinned(ctx, &ctx->h_desc, &ctx->capResDesc, kpRun + K, 4096, kpRun, FE_RECORD_FLOATS);
    if (st) return st;
  }
  if (K > 0) {
    CK(cudaMemcpyAsync(ctx->h_kp + kpRun, s.d_kpOut, (size_t)K * sizeof(float4), cudaMemcpyDeviceToHost, s.stream));
    const size_t dl = ctx->recordOutput ? FE_RECORD_FLOATS : FE_DESC_LEN;
    if (s.sb.desc) CK(cudaMemcpyAsync(ctx->h_desc + kpRun * dl, s.d_desc, (size_t)K * dl * sizeof(float), cudaMemcpyDeviceToHost, s.stream));
  }
  kpRun += K;
  if (ctx->cloudOutputs && s.h_cloudOff) {  // the two optional clouds, gathered on the device by enqueue_pipeline
    const int64_t tc = s.h_cloudOff[ns], tk = s.h_kcOff[ns];
    st = grow_pinned(ctx, &ctx->h_cloud, &ctx->capCloud, ctx->cloudRun + tc, 1 << 16, ctx->cloudRun);
    if (st) return st;
    st = grow_pinned(ctx, &ctx->h_kc, &ctx->capKcRes, ctx->kcRun + tk, 1 << 16, ctx->kcRun);
    if (st) return st;
    for (int i = 0; i <= ns; i++) {
      ctx->cloudOff[s.firstScan + i] = ctx->cloudRun + s.h_cloudOff[i];
      ctx->kcOff[s.firstScan + i] = ctx->kcRun + s.h_kcOff[i];
    }
    if (tc > 0) CK(cudaMemcpyAsync(ctx->h_cloud + ctx->cloudRun, s.d_gather, (size_t)tc * sizeof(float4), cudaMemcpyDeviceToHost, s.stream));
    if (tk > 0) CK(cudaMemcpyAsync(ctx->h_kc + ctx->kcRun, s.d_gather2, (size_t)tk * sizeof(float4), cudaMemcpyDeviceToHost, s.stream));
    ctx->cloudRun += tc;
    ctx->kcRun += tk;
  }
  return FE_OK;
}

int gather_to_host(fe_ctx* ctx, Slot& s, int nscans, bool chunks, const float4* src, const int* cnt, const int* pBase,
                   std::vector<int64_t>& offOut, std::vector<fe_point_t>& ptsOut) {
  if (chunks) k_piece_counts<<<(nscans + 255) / 256, 256, 0, s.stream>>>(cnt, s.d_chunk_off, nscans, s.d_perScan);
  else k_pool16_counts<<<(nscans + 255) / 256, 256, 0, s.stream>>>(cnt, nscans, s.d_perScan);
  ctx->launches++;
  CK(cudaMemcpyAsync(s.h_perScan, s.d_perScan, (size_t)nscans * sizeof(int), cudaMemcpyDeviceToHost, s.stream));
  CK(cudaStreamSynchronize(s.stream));
  offOut.assign(nscans + 1, 0);
  std::vector<int> off32(nscans + 1, 0);
  for (int i = 0; i < nscans; i++) { offOut[i + 1] = offOut[i] + s.h_perScan[i]; off32[i + 1] = (int)offOut[i + 1]; }
  const int64_t tot = offOut[nscans];
  ptsOut.resize((size_t)tot);
  if (tot == 0) return FE_OK;
  if (tot > s.capPts) return fail(ctx, FE_ERR_CAPACITY, "cloud output exceeds max_points_per_call");
  CK(cudaMemcpyAsync(s.d_outOff, off32.data(), (size_t)(nscans + 1) * sizeof(int), cudaMemcpyHostToDevice, s.stream));
  if (chunks) k_gather_chunks<<<nscans, 256, 0, s.stream>>>(src, cnt, s.d_scan_off, s.d_chunk_off, s.d_outOff, s.d_gather);
  else k_gather_pool16<<<nscans, 256, 0, s.stream>>>(src, pBase, cnt, s.d_outOff, s.d_gather);
  ctx->launches++;
  CK(cudaMemcpyAsync(ptsOut.data(), s.d_gather, (size_t)tot * sizeof(float4), cudaMemcpyDeviceToHost, s.stream));
  CK(cudaStreamSynchronize(s.stream));
  return FE_OK;
}

// A host batch call that fails half-way leaves sub-batches in flight on the two slots.  Whatever the
// exit path, both streams are drained and the slots marked idle, so the next call on the context starts
// clean instead of finalising a stale sub-batch into its own result arrays.
struct SlotDrain {
  fe_ctx* ctx;
  bool ok = false;
  explicit SlotDrain(fe_ctx* c) : ctx(c) { drain(); }
  ~SlotDrain() { if (!ok) drain(); }
  void drain() {
    for (int k = 0; k < 2; k++) {
      Slot& s = ctx->slot[k];
      if (s.stream) cudaStreamSynchronize(s.stream);
      s.busy = false;
    }
  }
};

}  // namespace

// ================================================================================================
extern "C" {

const char* fe_version(void) { return FE_VERSION; }

void fe_params_node_default(fe_params_t* p) {
  p->x_min = 0.0; p->x_max = 75.0;
  p->y_min = -30.0; p->y_max = 30.0;
  p->z_min = -1.5; p->z_max = 5.0;
  p->cluster_tolerance = 0.65;
  p->cluster_min_count = 5;
  p->cluster_max_count = 50;
  p->cluster_radius_threshold = 0.15;
  p->number_detection_channels = 1;
  p->estimate_descriptors = 1;
  p->descriptor_radius = 2.5;
}

void fe_params_launch_playback(fe_params_t* p) {
  fe_params_node_default(p);
  p->x_max = 100.0;
  p->y_min = -50.0; p->y_max = 50.0;
  p->z_max = 4.0;
  p->cluster_tolerance = 1.0;
  p->cluster_min_count = 1;
  p->cluster_max_count = 1000;
  p->cluster_radius_threshold = 0.2;
  p->number_detection_channels = 2;
}

int fe_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

void* fe_host_alloc(int64_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, (size_t)std::max<int64_t>(bytes, 1), cudaHostAllocDefault) != cudaSuccess) return nullptr;
  return p;
}

void fe_host_free(void* p) { if (p) cudaFreeHost(p); }

const char* fe_last_error(const fe_ctx_t* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int fe_create(int device, const fe_params_t* params, const fe_limits_t* limits, fe_ctx_t** out) {
  if (!out || !params) return FE_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return FE_ERR_NO_DEVICE;  // no CPU fallback
  if (device < 0 || device >= n) return FE_ERR_INVALID;
  fe_ctx* ctx = new fe_ctx();
  ctx->device = device;
  fe_limits_t L = {0, 0, 0, 0};
  if (limits) L = *limits;
  if (L.max_points_per_call <= 0) L.max_points_per_call = 32LL << 20;
  if (L.max_scans_per_call <= 0) L.max_scans_per_call = 2048;
  if (L.max_keypoints_per_call <= 0) L.max_keypoints_per_call = 64 << 10;
  if (L.max_ring_clusters_per_call <= 0) L.max_ring_clusters_per_call = 1 << 20;
  if (L.max_points_per_call >= (1LL << 32) - CH) { delete ctx; return FE_ERR_INVALID; }
  ctx->lim = L;
  auto bail = [&](int code) { fe_destroy(ctx); return code; };
  if (cudaSetDevice(device) != cudaSuccess) return bail(FE_ERR_CUDA);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return bail(FE_ERR_CUDA);
  if (prop.major != 10) return bail(FE_ERR_NO_DEVICE);  // built for sm_100a only
  ctx->numSms = std::max(prop.multiProcessorCount, 1);
  if (cudaMalloc((void**)&ctx->d_lut, FE_DESC_LEN * sizeof(float)) != cudaSuccess) return bail(FE_ERR_CUDA);
  // 3DSC x-axes: boost::uniform_01<mt19937>(12345) draws 3k..3k+2 -> (x0, x1, -0) normalised
  ctx->axesCap = 1 << 16;
  {
    std::vector<float2> ax(ctx->axesCap);
    std::mt19937 gen(12345u);
    for (int k = 0; k < ctx->axesCap; k++) {
      const float u0 = (float)((double)gen() * (1.0 / 4294967296.0));
      const float u1 = (float)((double)gen() * (1.0 / 4294967296.0));
      (void)gen();  // the third draw is overwritten by -(n.x*x0 + n.y*x1)/n.z = -0
      const float z = -(0.0f * u0 + 0.0f * u1) / 1.0f;
      const float inv = 1.0f / sqrtf(u0 * u0 + (u1 * u1 + z * z));
      ax[k].x = u0 * inv;
      ax[k].y = u1 * inv;
    }
    if (cudaMalloc((void**)&ctx->d_axes, ax.size() * sizeof(float2)) != cudaSuccess) return bail(FE_ERR_CUDA);
    if (cudaMemcpy(ctx->d_axes, ax.data(), ax.size() * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess) return bail(FE_ERR_CUDA);
  }
  int st = derive_params(ctx, *params);
  if (st) { fe_destroy(ctx); return st; }
  st = set_kernel_attrs(ctx);
  if (st) { fe_destroy(ctx); return st; }
  *out = ctx;
  return FE_OK;
}

int fe_set_params(fe_ctx_t* ctx, const fe_params_t* params) {
  if (!ctx || !params) return FE_ERR_INVALID;
  cudaSetDevice(ctx->device);
  sync_slots(ctx);
  ctx->epoch++;
  return derive_params(ctx, *params);
}

void fe_destroy(fe_ctx_t* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  for (int k = 0; k < 2; k++) free_slot(ctx->slot[k]);
  if (ctx->d_lut) cudaFree(ctx->d_lut);
  if (ctx->d_axes) cudaFree(ctx->d_axes);
  if (ctx->h_kp) cudaFreeHost(ctx->h_kp);
  if (ctx->h_desc) cudaFreeHost(ctx->h_desc);
  if (ctx->h_cloud) cudaFreeHost(ctx->h_cloud);
  if (ctx->h_kc) cudaFreeHost(ctx->h_kc);
  for (Workspace* w : {&ctx->matchWs, &ctx->regWs, &ctx->odoWs, &ctx->loopWs}) free_ws(*w);
  delete ctx;
}

int fe_enable_cloud_outputs(fe_ctx_t* ctx, int32_t enable) {
  if (!ctx) return FE_ERR_INVALID;
  ctx->cloudOutputs = enable != 0;
  ctx->epoch++;
  return FE_OK;
}

int fe_enable_stage_timing(fe_ctx_t* ctx, int32_t enable) {
  if (!ctx) return FE_ERR_INVALID;
  if (int st = sync_slots(ctx)) return st;
  ctx->stageTiming = enable != 0;
  ctx->epoch++;
  return FE_OK;
}

int fe_enable_record_output(fe_ctx_t* ctx, int32_t enable) {
  if (!ctx) return FE_ERR_INVALID;
  if (int st = sync_slots(ctx)) return st;
  ctx->recordOutput = enable != 0;
  ctx->epoch++;
  return FE_OK;
}

int fe_set_angle_libm(fe_ctx_t* ctx, int32_t mode) {
  if (!ctx || (mode != FE_LIBM_FDLIBM && mode != FE_LIBM_CORRECTLY_ROUNDED)) return FE_ERR_INVALID;
  if (int st = sync_slots(ctx)) return st;
  ctx->angleLibm = mode;
  ctx->dp.angle_libm = mode;
  ctx->epoch++;
  return FE_OK;
}

static int enable_boundary_report(fe_ctx_t* ctx, double eps_m, bool all) {
  if (!ctx || !(eps_m == eps_m)) return FE_ERR_INVALID;
  if (int st = sync_slots(ctx)) return st;
  ctx->bndEps = eps_m > 0.0 ? eps_m : 0.0;
  ctx->bndKinds = eps_m > 0.0 ? (all ? FE_BOUNDARY_KINDS : 4) : 0;
  ctx->bndCounts.clear();
  ctx->bndCountsAll.clear();
  ctx->epoch++;
  return FE_OK;
}

int fe_enable_boundary_report(fe_ctx_t* ctx, double eps_m) { return enable_boundary_report(ctx, eps_m, false); }

int fe_enable_boundary_report_all(fe_ctx_t* ctx, double eps_m) { return enable_boundary_report(ctx, eps_m, true); }

int fe_get_boundary_report(fe_ctx_t* ctx, const int64_t** counts, int32_t* n_scans) {
  if (!ctx || !counts || !n_scans) return FE_ERR_INVALID;
  if (!ctx->bndKinds) return fail(ctx, FE_ERR_INVALID, "boundary report not enabled (fe_enable_boundary_report)");
  *counts = ctx->bndCounts.data();
  *n_scans = (int32_t)(ctx->bndCounts.size() / 4);
  return FE_OK;
}

int fe_get_boundary_report_all(fe_ctx_t* ctx, const int64_t** counts, int32_t* n_scans) {
  if (!ctx || !counts || !n_scans) return FE_ERR_INVALID;
  if (ctx->bndKinds != FE_BOUNDARY_KINDS)
    return fail(ctx, FE_ERR_INVALID, "boundary report of all kinds not enabled (fe_enable_boundary_report_all)");
  *counts = ctx->bndCountsAll.data();
  *n_scans = (int32_t)(ctx->bndCountsAll.size() / FE_BOUNDARY_KINDS);
  return FE_OK;
}

int fe_debug_libm_f32(fe_ctx_t* ctx, int32_t op, const float* a, const float* b, float* out, int64_t n) {
  if (!ctx || op < 0 || op > 2 || n < 0 || (n > 0 && (!a || !out || (op == 0 && !b)))) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  if (n == 0) return FE_OK;
  float *da = nullptr, *db = nullptr, *dout = nullptr;
  auto done = [&](int code) { cudaFree(da); cudaFree(db); cudaFree(dout); return code; };
  if (cudaMalloc((void**)&da, (size_t)n * 4) != cudaSuccess || cudaMalloc((void**)&db, (size_t)n * 4) != cudaSuccess ||
      cudaMalloc((void**)&dout, (size_t)n * 4) != cudaSuccess)
    return done(fail(ctx, FE_ERR_CUDA, "fe_debug_libm_f32: out of device memory"));
  cudaMemcpy(da, a, (size_t)n * 4, cudaMemcpyHostToDevice);
  if (op == 0) cudaMemcpy(db, b, (size_t)n * 4, cudaMemcpyHostToDevice);
  k_debug_libm_f32<<<ctx->numSms * 8, 256>>>(op, da, db, dout, (long long)n);
  ctx->launches++;
  if (cudaMemcpy(out, dout, (size_t)n * 4, cudaMemcpyDeviceToHost) != cudaSuccess)
    return done(fail(ctx, FE_ERR_CUDA, std::string("fe_debug_libm_f32: ") + cudaGetErrorString(cudaGetLastError())));
  return done(FE_OK);
}

int fe_get_cloud_outputs(fe_ctx_t* ctx, const int64_t** cloud_offsets, const fe_point_t** cloud,
                         const int64_t** kpcloud_offsets, const fe_point_t** keypoint_cloud) {
  if (!ctx) return FE_ERR_INVALID;
  if (ctx->cloudOff.empty()) return fail(ctx, FE_ERR_INVALID, "no cloud outputs recorded (fe_enable_cloud_outputs before fe_process_batch)");
  if (cloud_offsets) *cloud_offsets = ctx->cloudOff.data();
  if (cloud) *cloud = ctx->h_cloud;
  if (kpcloud_offsets) *kpcloud_offsets = ctx->kcOff.data();
  if (keypoint_cloud) *keypoint_cloud = ctx->h_kc;
  return FE_OK;
}

int fe_get_stage_times(fe_ctx_t* ctx, int32_t cap, const char** names, float* ms, int32_t* n) {
  if (!ctx || !n || cap < 0 || (cap > 0 && (!names || !ms))) return FE_ERR_INVALID;
  const int m = std::min<int>(cap, (int)ctx->stName.size());
  for (int i = 0; i < m; i++) { names[i] = ctx->stName[i]; ms[i] = ctx->stMs[i]; }
  *n = m;
  return FE_OK;
}

// ---- the fused path ------------------------------------------------------------------------------

static int process_batch_host(fe_ctx_t* ctx, const unsigned char* points, int stride, int xo, int yo, int zo, bool isFloat4,
                              const int64_t* scan_offsets, const double* roll_pitch, int32_t n_scans, fe_batch_result_t* out) {
  if (!ctx || !out || n_scans < 0 || (n_scans > 0 && (!scan_offsets || !roll_pitch))) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  ctx->err.clear();
  if (n_scans > 0 && scan_offsets[0] < 0) return fail(ctx, FE_ERR_INVALID, "scan_offsets must not be negative");
  SlotDrain guard(ctx);
  const bool desc = ctx->params.estimate_descriptors != 0;
  const int64_t launches0 = ctx->launches;
  ctx->kpOffsets.assign((size_t)n_scans + 1, 0);
  ctx->bndCounts.assign(ctx->bndKinds ? (size_t)n_scans * 4 : 0, 0);
  ctx->bndCountsAll.assign(ctx->bndKinds == FE_BOUNDARY_KINDS ? (size_t)n_scans * FE_BOUNDARY_KINDS : 0, 0);
  ctx->cloudOff.clear(); ctx->kcOff.clear();
  ctx->cloudRun = ctx->kcRun = 0;
  if (ctx->cloudOutputs) { ctx->cloudOff.assign((size_t)n_scans + 1, 0); ctx->kcOff.assign((size_t)n_scans + 1, 0); }
  int64_t kpRun = 0;
  int first = 0, cur = 0;
  int nsub = 0;
  while (first < n_scans) {
    Slot& s = ctx->slot[cur];
    int st = ensure_slot(ctx, s, {CORE, POINTS});
    if (st) return st;
    // previous sub-batch of this slot must have been finalised (its device buffers are reused)
    st = finalize_subbatch(ctx, s, kpRun);
    if (st) return st;
    // greedy sub-batch
    int last = first;
    int64_t npts = 0;
    while (last < n_scans && (last - first) < s.capScans) {
      const int64_t n = scan_offsets[last + 1] - scan_offsets[last];
      if (n < 0) return fail(ctx, FE_ERR_INVALID, "scan_offsets must be non-decreasing");
      if (n > FE_MAX_SCAN_POINTS) return fail(ctx, FE_ERR_CAPACITY, "a scan of more than 2^20 points");
      if (n > s.capPts || n * stride > s.capPts * 16) return fail(ctx, FE_ERR_CAPACITY, "a single scan exceeds max_points_per_call");
      if (npts + n > s.capPts || (npts + n) * stride > s.capPts * 16) break;
      npts += n;
      last++;
    }
    SubBatch sb = batch_subbatch(ctx, s.d_pts, last - first);
    sb.wantKc = ctx->cloudOutputs;
    sb.lay = RawLayout{isFloat4 ? nullptr : (const unsigned char*)s.d_pts, stride, xo, yo, zo};
    st = stage_scans(ctx, s, scan_offsets + first, roll_pitch + 2 * first, sb.nscans, &sb.npts, &sb.nch);
    if (st) return st;
    st = enqueue_subbatch(ctx, s, sb, nullptr, points + scan_offsets[first] * (int64_t)stride, (size_t)npts * (size_t)stride);
    if (st) return st;
    s.busy = true; s.firstScan = first;
    nsub++;
    // the other slot's sub-batch was enqueued earlier: finalise it while this one runs
    Slot& o = ctx->slot[cur ^ 1];
    if (o.busy) { st = finalize_subbatch(ctx, o, kpRun); if (st) return st; }
    first = last;
    cur ^= 1;
  }
  // drain in submission order
  for (int k = 0; k < 2; k++) {
    Slot& s = ctx->slot[cur ^ k];  // cur now points at the older one
    int st = finalize_subbatch(ctx, s, kpRun);
    if (st) return st;
  }
  if (int st = sync_slots(ctx)) return st;
  if (nsub == 1) collect_times(ctx, ctx->slot[0]);
  out->n_scans = n_scans;
  out->n_keypoints = kpRun;
  out->keypoint_offsets = ctx->kpOffsets.data();
  out->keypoints = ctx->h_kp;
  out->descriptors = desc ? ctx->h_desc : nullptr;
  out->on_device = 0;
  out->gpu_launches = ctx->launches - launches0;
  guard.ok = true;
  return FE_OK;
}

int fe_process_batch(fe_ctx_t* ctx, const fe_point_t* points, const int64_t* scan_offsets,
                     const double* roll_pitch, int32_t n_scans, fe_batch_result_t* out) {
  return process_batch_host(ctx, (const unsigned char*)points, 16, 0, 4, 8, true, scan_offsets, roll_pitch, n_scans, out);
}

int fe_process_batch_layout(fe_ctx_t* ctx, const void* points, const fe_point_layout_t* layout,
                            const int64_t* scan_offsets, const double* roll_pitch, int32_t n_scans,
                            fe_batch_result_t* out) {
  if (!ctx || !layout) return FE_ERR_INVALID;
  const fe_point_layout_t& L = *layout;
  if (L.stride < 12 || L.stride > 4096 || L.x_off < 0 || L.y_off < 0 || L.z_off < 0 || L.x_off + 4 > L.stride ||
      L.y_off + 4 > L.stride || L.z_off + 4 > L.stride)
    return fail(ctx, FE_ERR_INVALID, "fe_point_layout: need 12 <= stride <= 4096 and x/y/z floats inside the record");
  return process_batch_host(ctx, (const unsigned char*)points, L.stride, L.x_off, L.y_off, L.z_off, false, scan_offsets,
                            roll_pitch, n_scans, out);
}

// tf::Matrix3x3(quat).getRPY(tmproll, pitch, yaw) as imuCallback uses it (src:60-65)
int fe_imu_to_roll_pitch(const double q[4], int32_t cloud_leveling, double* roll, double* pitch) {
  if (!q || !roll || !pitch) return FE_ERR_INVALID;
  if (!cloud_leveling) { *roll = 0.0; *pitch = 0.0; return FE_OK; }  // src:66-69
  const double x = q[0], y = q[1], z = q[2], w = q[3];
  // Matrix3x3::setRotation
  const double d = x * x + y * y + z * z + w * w;
  const double s = 2.0 / d;
  const double xs = x * s, ys = y * s;
  const double wx = w * xs, wy = w * ys;
  const double xx = x * xs, xz = x * (z * s);
  const double yy = y * ys, yz = y * (z * s);
  const double m20 = xz - wy, m21 = yz + wx, m22 = 1.0 - (xx + yy);
  // Matrix3x3::getEulerYPR, solution 1
  double tmproll, p;
  if (fabs(m20) >= 1.0) {
    const double delta = atan2(m21, m22);
    p = (m20 < 0.0) ? 3.14159265358979323846 / 2.0 : -3.14159265358979323846 / 2.0;
    tmproll = delta;
  } else {
    p = -asin(m20);
    tmproll = atan2(m21 / cos(p), m22 / cos(p));
  }
  *roll = tmproll - 3.14159265358979323846;  // src:65
  *pitch = p;
  return FE_OK;
}

int fe_process_batch_device(fe_ctx_t* ctx, const fe_point_t* d_points, const int64_t* scan_offsets,
                            const double* roll_pitch, int32_t n_scans, fe_batch_result_t* out) {
  if (!ctx || !out || n_scans < 0 || (n_scans > 0 && (!scan_offsets || !roll_pitch || !d_points))) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  ctx->err.clear();
  if (n_scans > 0 && scan_offsets[0] < 0) return fail(ctx, FE_ERR_INVALID, "scan_offsets must not be negative");
  const bool desc = ctx->params.estimate_descriptors != 0;
  const int64_t launches0 = ctx->launches;
  Slot& s = ctx->slot[0];
  int st = ensure_slot(ctx, s, {CORE});
  if (st) return st;
  for (int i = 0; i < n_scans; i++)
    if (scan_offsets[i + 1] - scan_offsets[i] > FE_MAX_SCAN_POINTS) return fail(ctx, FE_ERR_CAPACITY, "a scan of more than 2^20 points");
  ctx->kpOffsets.assign((size_t)n_scans + 1, 0);
  if (n_scans > 0) {
    // 2048 scans and more: the levelling matrices are computed while K1 runs (enqueue_pipeline)
    const double* lateRp = n_scans >= 2048 ? roll_pitch : nullptr;
    // the input's address is part of the graph key: a replay reads the same address
    SubBatch sb = batch_subbatch(ctx, (const float4*)d_points + scan_offsets[0], n_scans);
    st = stage_scans(ctx, s, scan_offsets, roll_pitch, n_scans, &sb.npts, &sb.nch, lateRp != nullptr);
    if (st) return st;
    st = enqueue_subbatch(ctx, s, sb, lateRp);
    if (st) return st;
    ctx->bndCounts.assign(ctx->bndKinds ? (size_t)n_scans * 4 : 0, 0);
    ctx->bndCountsAll.assign(ctx->bndKinds == FE_BOUNDARY_KINDS ? (size_t)n_scans * FE_BOUNDARY_KINDS : 0, 0);
    s.firstScan = 0;
    st = complete_subbatch(ctx, s, 0);
    if (st) return st;
    collect_times(ctx, s);
  }
  out->n_scans = n_scans;
  out->n_keypoints = ctx->kpOffsets[n_scans];
  out->keypoint_offsets = ctx->kpOffsets.data();
  out->keypoints = (const fe_point_t*)s.d_kpOut;
  out->descriptors = desc ? s.d_desc : nullptr;
  out->on_device = 1;
  out->gpu_launches = ctx->launches - launches0;
  return FE_OK;
}

int fe_timer_begin(fe_ctx_t* ctx) {
  if (!ctx) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int st = open_slot(ctx, ctx->slot[0]);
  if (st) return st;
  CK(cudaEventRecord(ctx->slot[0].evT0, ctx->slot[0].stream));
  return FE_OK;
}

int fe_timer_end(fe_ctx_t* ctx, float* elapsed_ms) {
  if (!ctx || !elapsed_ms || !ctx->slot[0].stream) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventRecord(ctx->slot[0].evT1, ctx->slot[0].stream));
  CK(cudaEventSynchronize(ctx->slot[0].evT1));
  CK(cudaEventElapsedTime(elapsed_ms, ctx->slot[0].evT0, ctx->slot[0].evT1));
  return FE_OK;
}

int fe_get_batch_stats(fe_ctx_t* ctx, int64_t out[10]) {
  if (!ctx || !out || !ctx->slot[0].h_ctr) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  Slot& s = ctx->slot[0];
  CK(cudaStreamSynchronize(s.stream));
  for (int i = 0; i < 10; i++) out[i] = 0;
  out[0] = s.sb.npts;
  std::vector<int> a((size_t)std::max(s.sb.nch, 1)), b((size_t)std::max(s.sb.nch, 1));
  if (s.sb.nch > 0) {
    CK(cudaMemcpy(a.data(), s.d_surfCnt, (size_t)s.sb.nch * sizeof(int), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(b.data(), s.d_cropCnt, (size_t)s.sb.nch * sizeof(int), cudaMemcpyDeviceToHost));
    for (int i = 0; i < s.sb.nch; i++) { out[1] += a[i]; out[2] += b[i]; }
  }
  if (s.sb.nscans > 0) {
    std::vector<int> kf((size_t)s.sb.nscans * 16);
    CK(cudaMemcpy(kf.data(), s.d_kfCnt, kf.size() * sizeof(int), cudaMemcpyDeviceToHost));
    for (int v : kf) out[3] += v;
    const int K = s.h_kpOff[s.sb.nscans];
    out[4] = K;
    if (K > 0 && ctx->params.estimate_descriptors) {
      std::vector<int> nb((size_t)K);
      CK(cudaMemcpy(nb.data(), s.d_kpNbr, (size_t)K * sizeof(int), cudaMemcpyDeviceToHost));
      for (int v : nb) out[5] += v;
    }
  }
  out[6] = s.h_ctr->ovf_rings;  // (of which ovf_rings2 went on to the large instantiation)
  out[7] = s.h_ctr->ovf_merge;
  out[8] = s.h_ctr->ovf_surf;
  out[9] = s.h_ctr->desc_unordered;
  return FE_OK;
}

int fe_download(fe_ctx_t* ctx, void* host_dst, const void* device_src, int64_t bytes) {
  if (!ctx || bytes < 0 || (bytes > 0 && (!host_dst || !device_src))) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  if (bytes > 0) CK(cudaMemcpy(host_dst, device_src, (size_t)bytes, cudaMemcpyDeviceToHost));
  return FE_OK;
}

}  // extern "C"

// ---- descriptor matching (fe_match.cu) -----------------------------------------------------------------

namespace {

template <class T>
int grow_device(fe_ctx* ctx, T** buf, int64_t* cap, int64_t need) {
  if (need <= *cap) return FE_OK;
  if (*buf) { CK(cudaFree(*buf)); *buf = nullptr; *cap = 0; }
  const int64_t ncap = need + need / 2;
  CK(dalloc(buf, (size_t)ncap));
  *cap = ncap;
  return FE_OK;
}

// What a match, register, odometry or loop-closure call does once its arguments have passed: clear the last error, select the
// context's device and hand out slot 0's stream (the slot is opened; none of its arrays are allocated).
int begin_call(fe_ctx* ctx, cudaStream_t* stream) {
  ctx->err.clear();
  CK(cudaSetDevice(ctx->device));
  int st = open_slot(ctx, ctx->slot[0]);
  if (st) return st;
  *stream = ctx->slot[0].stream;
  return FE_OK;
}

// The host variant's upload: elements [first, first + n) of the caller's array p to dst, which p then points at.
template <class T>
int upload(fe_ctx* ctx, const T*& p, T* dst, int64_t first, int64_t n, cudaStream_t stream) {
  if (n > 0) CK(cudaMemcpyAsync(dst, p + first, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, stream));
  p = dst;
  return FE_OK;
}

const char* check_offsets(const int64_t* o, int32_t G) {
  if (o[0] < 0) return "negative entry";
  for (int32_t g = 0; g < G; g++)
    if (o[g + 1] < o[g]) return "decreasing entries";
  return nullptr;
}

// The group checks of the match and register calls: n_groups, both offset arrays, rows on a side whose arrays are
// missing (haveQ / haveR false; qName / rName name them) and the 2^31 query rows.  Sets the row counts *nQ and *nR.
int check_groups(fe_ctx* ctx, int32_t G, const int64_t* qo, const int64_t* ro, bool haveQ, const char* qName, bool haveR,
                 const char* rName, int64_t* nQ, int64_t* nR) {
  if (G < 0) return fail(ctx, FE_ERR_INVALID, "n_groups must not be negative");
  if (!qo || !ro) return fail(ctx, FE_ERR_INVALID, "query_offsets and ref_offsets need n_groups + 1 entries");
  if (const char* e = check_offsets(qo, G)) return fail(ctx, FE_ERR_INVALID, std::string("query_offsets: ") + e);
  if (const char* e = check_offsets(ro, G)) return fail(ctx, FE_ERR_INVALID, std::string("ref_offsets: ") + e);
  *nQ = qo[G] - qo[0];
  *nR = ro[G] - ro[0];
  if (*nQ > 0 && !haveQ) return fail(ctx, FE_ERR_INVALID, std::string(qName) + " is NULL but there are query rows");
  if (*nR > 0 && !haveR) return fail(ctx, FE_ERR_INVALID, std::string(rName) + " is NULL but there are reference rows");
  if (*nQ >= (1LL << 31)) return fail(ctx, FE_ERR_INVALID, "more than 2^31 - 1 query rows");
  return FE_OK;
}

// both entry points: rows q / r are device memory (onDevice) or host memory to upload
int match_descriptors(fe_ctx* ctx, const float* q, int64_t qStride, const int64_t* qo, const float* r, int64_t rStride,
                      const int64_t* ro, int32_t G, fe_match_result_t* out, bool onDevice) {
  if (!ctx || !out) return FE_ERR_INVALID;
  if (qStride < FE_DESC_LEN || rStride < FE_DESC_LEN) return fail(ctx, FE_ERR_INVALID, "a row stride is below FE_DESC_LEN");
  int64_t nQ, nR;
  if (int st = check_groups(ctx, G, qo, ro, q, "query", r, "ref", &nQ, &nR)) return st;
  cudaStream_t stream;
  if (int st = begin_call(ctx, &stream)) return st;

  // the work items (fe_match.h): per group, reference segment outer and query tile inner, so that the warps running at
  // one time share a segment of reference rows in L2
  const int64_t QT = fe_match::ITEM_QUERIES, RS = fe_match::ITEM_REFS;
  int64_t nItems = 0;
  for (int32_t g = 0; g < G; g++) {
    const int64_t nq = qo[g + 1] - qo[g], nr = ro[g + 1] - ro[g];
    if (nq > 0) nItems += ((nq + QT - 1) / QT) * std::max<int64_t>((nr + RS - 1) / RS, 1);
  }
  if (nItems >= (1LL << 31)) return fail(ctx, FE_ERR_INVALID, "too many query tiles x reference segments");
  Workspace& ws = ctx->matchWs;
  Carve c;  // results (best at 0: fe_match_device_best) | items (uploaded) | partials and rows (device only)
  const Span<int64_t> best = c.take<int64_t>(nQ);
  const Span<float> dist2 = c.take<float>(nQ), second = c.take<float>(nQ);
  const Span<int32_t> shift = c.take<int32_t>(nQ);
  const int64_t resBytes = c.bytes;
  const Span<fe_match::Item> items = c.take<fe_match::Item>(nItems);
  const int64_t hostBytes = c.bytes;
  int st = grow_pinned(ctx, &ws.h, &ws.hCap, hostBytes, 4096, 0);
  if (st) return st;
  out->n_queries = nQ;
  out->best = best.in(ws.h);
  out->dist2 = dist2.in(ws.h);
  out->second_dist2 = second.in(ws.h);
  out->shift = shift.in(ws.h);
  if (nQ == 0) return FE_OK;

  int64_t nPart = 0, k = 0;
  fe_match::Item* hItems = items.in(ws.h);
  for (int32_t g = 0; g < G; g++) {
    const int64_t nq = qo[g + 1] - qo[g], nr = ro[g + 1] - ro[g];
    if (nq == 0) continue;
    const int64_t nseg = std::max<int64_t>((nr + RS - 1) / RS, 1);
    for (int64_t sg = 0; sg < nseg; sg++)
      for (int64_t t = 0; t < nq; t += QT) {
        fe_match::Item& I = hItems[k++];
        I.q0 = qo[g] + t;
        I.r0 = ro[g] + sg * RS;
        I.out = qo[g] + t - qo[0];
        I.part = nseg > 1 ? nPart + t * nseg : 0;
        I.nq = (int32_t)std::min(QT, nq - t);
        I.nr = (int32_t)std::min(RS, nr - sg * RS);
        I.nseg = (int32_t)nseg;
        I.seg = (int32_t)sg;
      }
    if (nseg > 1) nPart += nq * nseg;
  }
  const Span<fe_match::Partial> part = c.take<fe_match::Partial>(nPart);
  // the host variant's rows [qo[0], qo[G]) and [ro[0], ro[G]); the last row of a side ends FE_DESC_LEN floats in
  const int64_t qf = onDevice ? 0 : (nQ - 1) * qStride + FE_DESC_LEN, rf = onDevice || nR == 0 ? 0 : (nR - 1) * rStride + FE_DESC_LEN;
  const Span<float> qRows = c.take<float>(qf), rRows = c.take<float>(rf);
  if ((st = grow_device(ctx, &ws.d, &ws.dCap, c.bytes))) return st;

  if (!ctx->matchAttrs) {
    CK(fe_match::set_attributes());
    ctx->matchAttrs = true;
  }
  int64_t qBias = 0, rBias = 0;
  if (!onDevice) {
    if ((st = upload(ctx, q, qRows.in(ws.d), qo[0] * qStride, qf, stream))) return st;
    if ((st = upload(ctx, r, rRows.in(ws.d), ro[0] * rStride, rf, stream))) return st;
    qBias = qo[0];
    rBias = ro[0];
  }
  CK(cudaMemcpyAsync(ws.d + resBytes, ws.h + resBytes, (size_t)(hostBytes - resBytes), cudaMemcpyHostToDevice, stream));
  fe_match::Result res;
  res.best = (long long*)best.in(ws.d);
  res.dist2 = dist2.in(ws.d);
  res.second = second.in(ws.d);
  res.shift = shift.in(ws.d);
  CK(fe_match::launch(q, qStride, qBias, r, rStride, rBias, items.in(ws.d), (int)nItems, nPart > 0, part.in(ws.d), res,
                      stream));
  ctx->launches += nPart > 0 ? 2 : 1;
  CK(cudaMemcpyAsync(ws.h, ws.d, (size_t)resBytes, cudaMemcpyDeviceToHost, stream));
  CK(cudaStreamSynchronize(stream));
  return FE_OK;
}

}  // namespace

extern "C" {

int fe_match_descriptors(fe_ctx_t* ctx, const float* query, int64_t query_stride, const int64_t* query_offsets,
                         const float* ref, int64_t ref_stride, const int64_t* ref_offsets, int32_t n_groups,
                         fe_match_result_t* out) {
  return match_descriptors(ctx, query, query_stride, query_offsets, ref, ref_stride, ref_offsets, n_groups, out, false);
}

int fe_match_descriptors_device(fe_ctx_t* ctx, const float* query, int64_t query_stride, const int64_t* query_offsets,
                                const float* ref, int64_t ref_stride, const int64_t* ref_offsets, int32_t n_groups,
                                fe_match_result_t* out) {
  return match_descriptors(ctx, query, query_stride, query_offsets, ref, ref_stride, ref_offsets, n_groups, out, true);
}

int fe_match_device_best(fe_ctx_t* ctx, const int64_t** best) {
  if (!ctx || !best) return FE_ERR_INVALID;
  if (!ctx->matchWs.d) return fail(ctx, FE_ERR_INVALID, "no match call has run on this context");
  *best = (const int64_t*)ctx->matchWs.d;  // match_descriptors carves `best` at offset 0
  return FE_OK;
}

void fe_register_params_default(fe_register_params_t* p) {
  if (!p) return;
  p->inlier_radius = 0.5;
  p->min_separation = 1.0;
  p->max_hypotheses = 512;
  p->min_inliers = 16;
  p->refine_iterations = 4;
}

}  // extern "C"

// ---- registration (fe_register.cu) -----------------------------------------------------------------------

namespace {

// the parameter checks of the register and odometry calls, and the kernel's form of the parameters
int register_params(fe_ctx* ctx, const fe_register_params_t* prm, fe_register::Params* kp) {
  if (!prm) return fail(ctx, FE_ERR_INVALID, "params is NULL");
  const fe_register_params_t p = *prm;
  if (!(std::isfinite(p.inlier_radius) && p.inlier_radius > 0.0))
    return fail(ctx, FE_ERR_INVALID, "inlier_radius must be finite and > 0");
  if (!(std::isfinite(p.min_separation) && p.min_separation > 0.0))
    return fail(ctx, FE_ERR_INVALID, "min_separation must be finite and > 0");
  if (p.max_hypotheses < 1 || p.max_hypotheses > 65536) return fail(ctx, FE_ERR_INVALID, "max_hypotheses must be in [1, 65536]");
  if (p.min_inliers < 1) return fail(ctx, FE_ERR_INVALID, "min_inliers must be >= 1");
  if (p.refine_iterations < 0 || p.refine_iterations > 1000)
    return fail(ctx, FE_ERR_INVALID, "refine_iterations must be in [0, 1000]");
  kp->r2 = p.inlier_radius * p.inlier_radius;
  kp->sep2 = p.min_separation * p.min_separation;
  kp->twoR = 2.0 * p.inlier_radius;
  kp->maxH = p.max_hypotheses;
  kp->minInliers = p.min_inliers;
  kp->refine = p.refine_iterations;
  return FE_OK;
}

// both entry points: keypoints and `best` are device memory (onDevice) or host memory to upload
int register_matches(fe_ctx* ctx, const fe_point_t* q, const fe_point_t* r, const int64_t* best, const int64_t* qo,
                     const int64_t* ro, int32_t G, const fe_register_params_t* prm, fe_register_result_t* out,
                     bool onDevice) {
  if (!ctx || !out) return FE_ERR_INVALID;
  fe_register::Params kp;
  if (int st = register_params(ctx, prm, &kp)) return st;
  int64_t nQ, nR;
  if (int st = check_groups(ctx, G, qo, ro, q && best, "query_kp or best", r, "ref_kp", &nQ, &nR)) return st;
  for (int32_t g = 0; g < G; g++)  // so that h * P of the hypothesis map fits 64 bits (P < 2^47, h < 2^16)
    if (qo[g + 1] - qo[g] >= (1LL << 24)) return fail(ctx, FE_ERR_INVALID, "a group has 2^24 or more query rows");
  if (!onDevice)
    for (int32_t g = 0; g < G; g++)
      for (int64_t k = qo[g]; k < qo[g + 1]; k++) {
        const int64_t b = best[k - qo[0]];
        if (b != -1 && (b < ro[g] || b >= ro[g + 1]))
          return fail(ctx, FE_ERR_INVALID, "best[" + std::to_string(k - qo[0]) + "] is neither -1 nor a reference row of its group");
      }
  cudaStream_t stream;
  if (int st = begin_call(ctx, &stream)) return st;

  Workspace& ws = ctx->regWs;
  Carve c;  // results | query then reference offsets (uploaded) | scratch and the host variant's rows (device only)
  const Span<double> pose = c.take<double>(4 * (int64_t)G), rms = c.take<double>(G);
  const Span<int64_t> assoc = c.take<int64_t>(nQ);
  const Span<int32_t> nInl = c.take<int32_t>(G), nHyp = c.take<int32_t>(G), status = c.take<int32_t>(G);
  const Span<int32_t> err = c.take<int32_t>(1);  // the device's error flag
  const int64_t resBytes = c.bytes;
  const Span<int64_t> offs = c.take<int64_t>(2 * ((int64_t)G + 1));
  const int64_t hostBytes = c.bytes;
  const Span<long long> assocNew = c.take<long long>(nQ);
  const Span<double> d2Cur = c.take<double>(nQ), d2New = c.take<double>(nQ);
  const Span<int32_t> corr = c.take<int32_t>(nQ);
  const int64_t nUp = onDevice ? 0 : 1;  // the host variant's rows [qo[0], qo[G]) and [ro[0], ro[G]), and `best`
  const Span<fe_point_t> qRows = c.take<fe_point_t>(nUp * nQ), rRows = c.take<fe_point_t>(nUp * nR);
  const Span<int64_t> bestRows = c.take<int64_t>(nUp * nQ);
  int st = grow_pinned(ctx, &ws.h, &ws.hCap, hostBytes, 4096, 0);
  if (st) return st;
  out->n_groups = G;
  out->n_queries = nQ;
  out->pose = pose.in(ws.h);
  out->rms = rms.in(ws.h);
  out->assoc = assoc.in(ws.h);
  out->n_inliers = nInl.in(ws.h);
  out->n_hypotheses = nHyp.in(ws.h);
  out->status = status.in(ws.h);
  if (G == 0) return FE_OK;

  if ((st = grow_device(ctx, &ws.d, &ws.dCap, c.bytes))) return st;
  memcpy(offs.in(ws.h), qo, (size_t)(G + 1) * sizeof(int64_t));
  memcpy(offs.in(ws.h) + G + 1, ro, (size_t)(G + 1) * sizeof(int64_t));
  int64_t qBias = 0, rBias = 0;
  if (!onDevice) {
    if ((st = upload(ctx, q, qRows.in(ws.d), qo[0], nQ, stream))) return st;
    if ((st = upload(ctx, best, bestRows.in(ws.d), 0, nQ, stream))) return st;
    if ((st = upload(ctx, r, rRows.in(ws.d), ro[0], nR, stream))) return st;
    qBias = qo[0];
    rBias = ro[0];
  }
  CK(cudaMemcpyAsync(ws.d + resBytes, ws.h + resBytes, (size_t)(hostBytes - resBytes), cudaMemcpyHostToDevice, stream));
  CK(cudaMemsetAsync(err.in(ws.d), 0, sizeof(int32_t), stream));
  fe_register::Out o;
  o.pose = pose.in(ws.d);
  o.rms = rms.in(ws.d);
  o.assoc = (long long*)assoc.in(ws.d);
  o.nInl = nInl.in(ws.d);
  o.nHyp = nHyp.in(ws.d);
  o.status = status.in(ws.d);
  o.err = err.in(ws.d);
  fe_register::Scratch sc;
  sc.assocNew = assocNew.in(ws.d);
  sc.d2Cur = d2Cur.in(ws.d);
  sc.d2New = d2New.in(ws.d);
  sc.corr = corr.in(ws.d);
  CK(fe_register::launch(q, qBias, r, rBias, (const long long*)best, offs.in(ws.d), offs.in(ws.d) + G + 1, G, kp, o, sc,
                         stream));
  ctx->launches += 1;
  CK(cudaMemcpyAsync(ws.h, ws.d, (size_t)resBytes, cudaMemcpyDeviceToHost, stream));
  CK(cudaStreamSynchronize(stream));
  if (*err.in(ws.h)) return fail(ctx, FE_ERR_INVALID, "an entry of best is neither -1 nor a reference row of its group");
  return FE_OK;
}

}  // namespace

extern "C" {

int fe_register_matches(fe_ctx_t* ctx, const fe_point_t* query_kp, const fe_point_t* ref_kp, const int64_t* best,
                        const int64_t* query_offsets, const int64_t* ref_offsets, int32_t n_groups,
                        const fe_register_params_t* params, fe_register_result_t* out) {
  return register_matches(ctx, query_kp, ref_kp, best, query_offsets, ref_offsets, n_groups, params, out, false);
}

int fe_register_matches_device(fe_ctx_t* ctx, const fe_point_t* query_kp, const fe_point_t* ref_kp, const int64_t* best,
                               const int64_t* query_offsets, const int64_t* ref_offsets, int32_t n_groups,
                               const fe_register_params_t* params, fe_register_result_t* out) {
  return register_matches(ctx, query_kp, ref_kp, best, query_offsets, ref_offsets, n_groups, params, out, true);
}

}  // extern "C"

// ---- odometry (fe_odometry.cu) -------------------------------------------------------------------------

namespace {

// both entry points: keypoints and `best` are device memory (onDevice) or host memory to upload
int odometry(fe_ctx* ctx, const fe_point_t* kp, const int64_t* ko, int32_t B, const int64_t* best, const int64_t* so,
             int32_t S, int32_t W, const fe_register_params_t* prm, fe_odometry_result_t* out, bool onDevice) {
  if (!ctx || !out) return FE_ERR_INVALID;
  fe_register::Params rp;
  if (int st = register_params(ctx, prm, &rp)) return st;
  if (B < 0 || S < 0) return fail(ctx, FE_ERR_INVALID, "n_scans and n_sequences must not be negative");
  if (!ko || !so) return fail(ctx, FE_ERR_INVALID, "keypoint_offsets and sequence_offsets need n_scans + 1 and n_sequences + 1 entries");
  if (W < 1 || W > 64) return fail(ctx, FE_ERR_INVALID, "window must be in [1, 64]");
  if (const char* e = check_offsets(ko, B)) return fail(ctx, FE_ERR_INVALID, std::string("keypoint_offsets: ") + e);
  if (const char* e = check_offsets(so, S)) return fail(ctx, FE_ERR_INVALID, std::string("sequence_offsets: ") + e);
  if (so[0] != 0 || so[S] != B) return fail(ctx, FE_ERR_INVALID, "sequence_offsets must run from 0 to n_scans");
  for (int32_t b = 0; b < B; b++)
    if (ko[b + 1] - ko[b] >= (1LL << 24)) return fail(ctx, FE_ERR_INVALID, "a scan has 2^24 or more keypoints");
  const int64_t nRows = ko[B] - ko[0];
  if (nRows >= (1LL << 31)) return fail(ctx, FE_ERR_INVALID, "more than 2^31 - 1 keypoint rows");

  // the steps: sequences with a scan t, each with a slot for its largest window
  std::vector<fe_odo::Step> steps;
  std::vector<fe_odo::Item> items;
  std::vector<int64_t> offs;
  int64_t maxQ = 1, maxR = 1, maxN = 1, bestRows = 0;
  for (int64_t t = 1;; t++) {
    fe_odo::Step st;
    st.item0 = (int64_t)items.size();
    st.offs0 = (int64_t)offs.size();
    for (int32_t q = 0; q < S; q++)
      if (so[q + 1] - so[q] > t) items.push_back({(int)(so[q] + t), (int)so[q]});
    st.n = (int)((int64_t)items.size() - st.item0);
    if (st.n == 0) break;
    offs.resize(offs.size() + 2 * (size_t)(2 * st.n + 1));
    int64_t* qo = offs.data() + st.offs0;
    int64_t* ro = qo + 2 * st.n + 1;
    qo[0] = ro[0] = 0;
    for (int i = 0; i < st.n; i++) {
      const int s = items[(size_t)(st.item0 + i)].scan;
      const int64_t nq = ko[s + 1] - ko[s], slot = ko[s] - ko[s - std::min<int64_t>(W, t)];
      qo[2 * i + 1] = qo[2 * i + 2] = qo[2 * i] + nq;
      ro[2 * i + 1] = ro[2 * i + 2] = ro[2 * i] + slot;  // ro[2i + 1] is the device's to write
      bestRows += nq;
    }
    maxQ = std::max(maxQ, qo[2 * st.n]);
    maxR = std::max(maxR, ro[2 * st.n]);
    maxN = std::max<int64_t>(maxN, st.n);
    steps.push_back(st);
  }
  if (bestRows > 0 && !best) return fail(ctx, FE_ERR_INVALID, "best is NULL but there are scans to register");
  if (!steps.empty() && nRows > 0 && !kp) return fail(ctx, FE_ERR_INVALID, "kp is NULL but there are keypoints");
  if (!onDevice)
    for (const fe_odo::Item& it : items)
      for (int64_t k = ko[it.scan]; k < ko[it.scan + 1]; k++) {
        const int64_t b = best[k - ko[1]];
        if (b != -1 && (b < ko[it.scan - 1] || b >= ko[it.scan]))
          return fail(ctx, FE_ERR_INVALID, "best[" + std::to_string(k - ko[1]) + "] is neither -1 nor a row of the previous scan");
      }
  cudaStream_t stream;
  if (int st = begin_call(ctx, &stream)) return st;

  Workspace& ws = ctx->odoWs;
  Carve c;  // results | tables (uploaded) | the steps' work buffers and the host variant's rows (device only)
  const Span<double> pose = c.take<double>(4 * (int64_t)B), motion = c.take<double>(4 * (int64_t)B), rms = c.take<double>(B);
  const Span<int64_t> assoc = c.take<int64_t>(nRows);
  const Span<int32_t> source = c.take<int32_t>(B), status = c.take<int32_t>(B), nInl = c.take<int32_t>(B);
  const Span<int32_t> nHyp = c.take<int32_t>(B), err = c.take<int32_t>(1);  // err: the device's error flag
  const int64_t resBytes = c.bytes;
  const Span<int64_t> tKo = c.take<int64_t>((int64_t)B + 1), tSo = c.take<int64_t>((int64_t)S + 1);
  const Span<int64_t> tOffs = c.take<int64_t>((int64_t)offs.size());
  const Span<fe_odo::Item> tItems = c.take<fe_odo::Item>((int64_t)items.size());
  const int64_t hostBytes = c.bytes;
  // sized for the largest step
  const int64_t maxG = 2 * maxN;
  const Span<fe_point_t> wQ = c.take<fe_point_t>(maxQ), wR = c.take<fe_point_t>(maxR);
  const Span<long long> wBest = c.take<long long>(maxQ), wAssoc = c.take<long long>(maxQ);
  const Span<long long> wAssocNew = c.take<long long>(maxQ);
  const Span<double> wD2Cur = c.take<double>(maxQ), wD2New = c.take<double>(maxQ);
  const Span<int64_t> wWinLo = c.take<int64_t>(maxN);
  const Span<double> wPose = c.take<double>(4 * maxG), wRms = c.take<double>(maxG);
  const Span<int32_t> wCorr = c.take<int32_t>(maxQ), wNInl = c.take<int32_t>(maxG), wNHyp = c.take<int32_t>(maxG);
  const Span<int32_t> wStatus = c.take<int32_t>(maxG);
  // the host variant's rows [ko[0], ko[B]) and the `best` entries of the scans that are registered
  const int64_t nBest = onDevice || bestRows == 0 || B < 2 ? 0 : ko[B] - ko[1];
  const Span<fe_point_t> kpRows = c.take<fe_point_t>(onDevice ? 0 : nRows);
  const Span<int64_t> bestUp = c.take<int64_t>(nBest);
  int st = grow_pinned(ctx, &ws.h, &ws.hCap, hostBytes, 4096, 0);
  if (st) return st;
  out->n_scans = B;
  out->n_rows = nRows;
  out->pose = pose.in(ws.h);
  out->motion = motion.in(ws.h);
  out->rms = rms.in(ws.h);
  out->assoc = assoc.in(ws.h);
  out->source = source.in(ws.h);
  out->status = status.in(ws.h);
  out->n_inliers = nInl.in(ws.h);
  out->n_hypotheses = nHyp.in(ws.h);
  out->gpu_launches = 0;
  if (B == 0) return FE_OK;

  if ((st = grow_device(ctx, &ws.d, &ws.dCap, c.bytes))) return st;
  memcpy(tKo.in(ws.h), ko, 8 * ((size_t)B + 1));
  memcpy(tSo.in(ws.h), so, 8 * ((size_t)S + 1));
  if (!offs.empty()) memcpy(tOffs.in(ws.h), offs.data(), 8 * offs.size());
  if (!items.empty()) memcpy(tItems.in(ws.h), items.data(), sizeof(fe_odo::Item) * items.size());
  CK(cudaMemcpyAsync(ws.d + resBytes, ws.h + resBytes, (size_t)(hostBytes - resBytes), cudaMemcpyHostToDevice, stream));
  fe_odo::Tables T;
  T.ko = tKo.in(ws.d);
  T.so = tSo.in(ws.d);
  T.offs = tOffs.in(ws.d);
  T.items = tItems.in(ws.d);
  fe_odo::Out o;
  o.pose = pose.in(ws.d);
  o.motion = motion.in(ws.d);
  o.rms = rms.in(ws.d);
  o.assoc = (long long*)assoc.in(ws.d);
  o.source = source.in(ws.d);
  o.status = status.in(ws.d);
  o.nInl = nInl.in(ws.d);
  o.nHyp = nHyp.in(ws.d);
  o.err = err.in(ws.d);
  fe_odo::Work w;
  w.q = wQ.in(ws.d);
  w.r = wR.in(ws.d);
  w.best = wBest.in(ws.d);
  w.winLo = wWinLo.in(ws.d);
  w.reg.pose = wPose.in(ws.d);
  w.reg.rms = wRms.in(ws.d);
  w.reg.assoc = wAssoc.in(ws.d);
  w.reg.nInl = wNInl.in(ws.d);
  w.reg.nHyp = wNHyp.in(ws.d);
  w.reg.status = wStatus.in(ws.d);
  w.reg.err = o.err;
  w.scratch.corr = wCorr.in(ws.d);
  w.scratch.assocNew = wAssocNew.in(ws.d);
  w.scratch.d2Cur = wD2Cur.in(ws.d);
  w.scratch.d2New = wD2New.in(ws.d);

  int64_t kpBias = 0;
  if (!onDevice) {
    if ((st = upload(ctx, kp, kpRows.in(ws.d), ko[0], nRows, stream))) return st;
    if ((st = upload(ctx, best, bestUp.in(ws.d), 0, nBest, stream))) return st;
    kpBias = ko[0];
  }
  CK(cudaMemsetAsync(o.err, 0, sizeof(int32_t), stream));
  CK(fe_odo::run(kp, kpBias, (const long long*)best, S, W, steps, T, w, o, rp, stream));
  const int64_t launches = S > 0 ? 1 + 3 * (int64_t)steps.size() : 0;
  ctx->launches += launches;
  out->gpu_launches = launches;
  CK(cudaMemcpyAsync(ws.h, ws.d, (size_t)resBytes, cudaMemcpyDeviceToHost, stream));
  CK(cudaStreamSynchronize(stream));
  if (*err.in(ws.h)) return fail(ctx, FE_ERR_INVALID, "an entry of best is neither -1 nor a row of the previous scan");
  return FE_OK;
}

}  // namespace

extern "C" {

int fe_odometry(fe_ctx_t* ctx, const fe_point_t* kp, const int64_t* keypoint_offsets, int32_t n_scans, const int64_t* best,
                const int64_t* sequence_offsets, int32_t n_sequences, int32_t window, const fe_register_params_t* params,
                fe_odometry_result_t* out) {
  return odometry(ctx, kp, keypoint_offsets, n_scans, best, sequence_offsets, n_sequences, window, params, out, false);
}

int fe_odometry_device(fe_ctx_t* ctx, const fe_point_t* kp, const int64_t* keypoint_offsets, int32_t n_scans,
                       const int64_t* best, const int64_t* sequence_offsets, int32_t n_sequences, int32_t window,
                       const fe_register_params_t* params, fe_odometry_result_t* out) {
  return odometry(ctx, kp, keypoint_offsets, n_scans, best, sequence_offsets, n_sequences, window, params, out, true);
}

}  // extern "C"

// ---- loop closures (fe_loop.cu) ------------------------------------------------------------------------------

namespace {

// both entry points: keypoints and descriptor rows are device memory (onDevice) or host memory to upload
int loop_closures(fe_ctx* ctx, const fe_point_t* kp, const float* desc, int64_t stride, const int64_t* ko, int32_t B,
                  const int64_t* so, int32_t S, const fe_loop_params_t* lp, const fe_register_params_t* prm,
                  fe_loop_result_t* out, bool onDevice) {
  if (!ctx || !out) return FE_ERR_INVALID;
  fe_register::Params rp;
  if (int st = register_params(ctx, prm, &rp)) return st;
  if (!lp) return fail(ctx, FE_ERR_INVALID, "loop_params is NULL");
  const int K = lp->candidates, gap = lp->min_gap;
  if (K < 1 || K > fe_loop::MAX_CANDIDATES) return fail(ctx, FE_ERR_INVALID, "candidates must be in [1, 16]");
  if (gap < 1) return fail(ctx, FE_ERR_INVALID, "min_gap must be >= 1");
  if (stride < FE_DESC_LEN) return fail(ctx, FE_ERR_INVALID, "the descriptor row stride is below FE_DESC_LEN");
  if (B < 0 || S < 0) return fail(ctx, FE_ERR_INVALID, "n_scans and n_sequences must not be negative");
  if (!ko || !so) return fail(ctx, FE_ERR_INVALID, "keypoint_offsets and sequence_offsets need n_scans + 1 and n_sequences + 1 entries");
  if (const char* e = check_offsets(ko, B)) return fail(ctx, FE_ERR_INVALID, std::string("keypoint_offsets: ") + e);
  if (const char* e = check_offsets(so, S)) return fail(ctx, FE_ERR_INVALID, std::string("sequence_offsets: ") + e);
  if (so[0] != 0 || so[S] != B) return fail(ctx, FE_ERR_INVALID, "sequence_offsets must run from 0 to n_scans");
  for (int32_t b = 0; b < B; b++)
    if (ko[b + 1] - ko[b] >= (1LL << 24)) return fail(ctx, FE_ERR_INVALID, "a scan has 2^24 or more keypoints");
  const int64_t nRows = ko[B] - ko[0];
  if (nRows >= (1LL << 31)) return fail(ctx, FE_ERR_INVALID, "more than 2^31 - 1 keypoint rows");
  if (nRows > 0 && (!kp || !desc)) return fail(ctx, FE_ERR_INVALID, "kp or desc is NULL but there are keypoints");

  // the tables: eligible scans, retrieval items (scan t against its database, segment outer as match_descriptors lays
  // them out), and K verification slots per eligible scan, sized for the largest scan of its sequence
  const int64_t QT = fe_match::ITEM_QUERIES, RS = fe_match::ITEM_REFS;
  std::vector<int> elig((size_t)B, -1);
  std::vector<fe_loop::Scan> scans;
  std::vector<fe_loop::Slot> slots;
  std::vector<fe_match::Item> items1, items2;
  std::vector<int64_t> qo{0}, ro{0};
  int64_t nPart1 = 0, nPart2 = 0, nQ = 0, nR = 0;
  auto tile_items = [&](std::vector<fe_match::Item>& items, int64_t q0, int64_t nq, int64_t r0, int64_t nr, int64_t nseg,
                        int64_t out0, int64_t* nPart) {
    for (int64_t sg = 0; sg < nseg; sg++)
      for (int64_t t = 0; t < nq; t += QT) {
        fe_match::Item I;
        I.q0 = q0 + t;
        I.r0 = r0 + sg * RS;
        I.out = out0 + t;
        I.part = nseg > 1 ? *nPart + t * nseg : 0;
        I.nq = (int32_t)std::min(QT, nq - t);
        I.nr = (int32_t)std::max<int64_t>(0, std::min(RS, nr - sg * RS));
        I.nseg = (int32_t)nseg;
        I.seg = (int32_t)sg;
        items.push_back(I);
      }
    if (nseg > 1) *nPart += nq * nseg;
  };
  for (int32_t q = 0; q < S; q++) {
    int64_t cap = 0;
    for (int64_t s = so[q]; s < so[q + 1]; s++) cap = std::max(cap, ko[s + 1] - ko[s]);
    const int64_t nseg2 = std::max<int64_t>((cap + RS - 1) / RS, 1);
    for (int64_t s = so[q] + gap; s < so[q + 1]; s++) {
      elig[(size_t)s] = (int)scans.size();
      scans.push_back({(int)s, (int)so[q]});
      const int64_t nq = ko[s + 1] - ko[s], nr = ko[s - gap + 1] - ko[so[q]];
      tile_items(items1, ko[s], nq, ko[so[q]], nr, std::max<int64_t>((nr + RS - 1) / RS, 1), ko[s] - ko[0], &nPart1);
      for (int k = 0; k < K; k++) {
        fe_loop::Slot sl;
        sl.q0 = nQ;
        sl.r0 = nR;
        sl.cap = cap;
        sl.item0 = (int64_t)items2.size();
        sl.tiles = (int32_t)((nq + QT - 1) / QT);
        sl.nseg = (int32_t)nseg2;
        slots.push_back(sl);
        tile_items(items2, ko[s], nq, 0, 0, nseg2, nQ, &nPart2);  // r0 and nr are k_loop_place's to write
        nQ += nq;
        qo.push_back(nQ);
        qo.push_back(nQ);
        ro.push_back(nR);  // the start of the slot's unused tail: k_loop_place writes it
        nR += cap;
        ro.push_back(nR);
      }
    }
  }
  const int E = (int)scans.size(), nSlots = (int)slots.size();
  if ((int64_t)items1.size() >= (1LL << 31) || (int64_t)items2.size() >= (1LL << 31))
    return fail(ctx, FE_ERR_INVALID, "too many query tiles x reference segments");
  cudaStream_t stream;
  if (int st = begin_call(ctx, &stream)) return st;

  Workspace& ws = ctx->loopWs;
  const int64_t BK = (int64_t)B * K, G = 2 * (int64_t)nSlots;
  Carve c;  // results | tables (uploaded) | retrieval, slots, registration and the host variant's rows (device only)
  const Span<double> pose = c.take<double>(4 * (int64_t)B), rms = c.take<double>(B);
  const Span<double> cPose = c.take<double>(4 * BK), cRms = c.take<double>(BK);
  const Span<int64_t> assoc = c.take<int64_t>(nRows);
  const Span<int32_t> loop = c.take<int32_t>(B), loopScan = c.take<int32_t>(B), nInl = c.take<int32_t>(B);
  const Span<int32_t> nHyp = c.take<int32_t>(B), cScan = c.take<int32_t>(BK), cVotes = c.take<int32_t>(BK);
  const Span<int32_t> cStatus = c.take<int32_t>(BK), cInl = c.take<int32_t>(BK), cHyp = c.take<int32_t>(BK);
  const int64_t resBytes = c.bytes;
  const Span<int64_t> tKo = c.take<int64_t>((int64_t)B + 1);
  const Span<int32_t> tElig = c.take<int32_t>(B);
  const Span<fe_loop::Scan> tScans = c.take<fe_loop::Scan>(E);
  const Span<fe_loop::Slot> tSlots = c.take<fe_loop::Slot>(nSlots);
  const Span<fe_match::Item> tItems1 = c.take<fe_match::Item>((int64_t)items1.size());
  const Span<fe_match::Item> tItems2 = c.take<fe_match::Item>((int64_t)items2.size());
  const Span<int64_t> tQo = c.take<int64_t>((int64_t)qo.size()), tRo = c.take<int64_t>((int64_t)ro.size());
  const int64_t hostBytes = c.bytes;
  const Span<int64_t> best1 = c.take<int64_t>(nRows);
  const Span<int32_t> shift1 = c.take<int32_t>(nRows), voteScan = c.take<int32_t>(nRows);
  const Span<float> dist1 = c.take<float>(nRows), second1 = c.take<float>(nRows);
  const Span<uint64_t> voteKey = c.take<uint64_t>(nRows);
  const Span<fe_match::Partial> part1 = c.take<fe_match::Partial>(nPart1), part2 = c.take<fe_match::Partial>(nPart2);
  const Span<fe_point_t> wQ = c.take<fe_point_t>(nQ), wR = c.take<fe_point_t>(nR);
  const Span<int64_t> best2 = c.take<int64_t>(nQ), slotBest = c.take<int64_t>(nQ);
  const Span<int32_t> shift2 = c.take<int32_t>(nQ);
  const Span<float> dist2 = c.take<float>(nQ), second2 = c.take<float>(nQ);
  const Span<double> gPose = c.take<double>(4 * G), gRms = c.take<double>(G);
  const Span<int64_t> gAssoc = c.take<int64_t>(nQ), gAssocNew = c.take<int64_t>(nQ);
  const Span<double> gD2Cur = c.take<double>(nQ), gD2New = c.take<double>(nQ);
  const Span<int32_t> gNInl = c.take<int32_t>(G), gNHyp = c.take<int32_t>(G), gStatus = c.take<int32_t>(G);
  const Span<int32_t> gCorr = c.take<int32_t>(nQ), gErr = c.take<int32_t>(1);
  // the host variant's rows [ko[0], ko[B]); the last descriptor row ends FE_DESC_LEN floats in
  const int64_t df = onDevice || nRows == 0 ? 0 : (nRows - 1) * stride + FE_DESC_LEN;
  const Span<fe_point_t> kpRows = c.take<fe_point_t>(onDevice ? 0 : nRows);
  const Span<float> descRows = c.take<float>(df);
  int st = grow_pinned(ctx, &ws.h, &ws.hCap, hostBytes, 4096, 0);
  if (st) return st;
  out->n_scans = B;
  out->candidates = K;
  out->n_rows = nRows;
  out->loop = loop.in(ws.h);
  out->loop_scan = loopScan.in(ws.h);
  out->pose = pose.in(ws.h);
  out->rms = rms.in(ws.h);
  out->n_inliers = nInl.in(ws.h);
  out->n_hypotheses = nHyp.in(ws.h);
  out->cand_scan = cScan.in(ws.h);
  out->cand_votes = cVotes.in(ws.h);
  out->cand_status = cStatus.in(ws.h);
  out->cand_inliers = cInl.in(ws.h);
  out->cand_hypotheses = cHyp.in(ws.h);
  out->cand_rms = cRms.in(ws.h);
  out->cand_pose = cPose.in(ws.h);
  out->assoc = assoc.in(ws.h);
  out->gpu_launches = 0;
  if (B == 0) return FE_OK;

  if ((st = grow_device(ctx, &ws.d, &ws.dCap, c.bytes))) return st;
  memcpy(tKo.in(ws.h), ko, 8 * ((size_t)B + 1));
  memcpy(tElig.in(ws.h), elig.data(), 4 * (size_t)B);
  if (E) memcpy(tScans.in(ws.h), scans.data(), sizeof(fe_loop::Scan) * scans.size());
  if (nSlots) memcpy(tSlots.in(ws.h), slots.data(), sizeof(fe_loop::Slot) * slots.size());
  if (!items1.empty()) memcpy(tItems1.in(ws.h), items1.data(), sizeof(fe_match::Item) * items1.size());
  if (!items2.empty()) memcpy(tItems2.in(ws.h), items2.data(), sizeof(fe_match::Item) * items2.size());
  memcpy(tQo.in(ws.h), qo.data(), 8 * qo.size());
  memcpy(tRo.in(ws.h), ro.data(), 8 * ro.size());
  CK(cudaMemcpyAsync(ws.d + resBytes, ws.h + resBytes, (size_t)(hostBytes - resBytes), cudaMemcpyHostToDevice, stream));
  int64_t bias = 0;
  if (!onDevice) {
    if ((st = upload(ctx, kp, kpRows.in(ws.d), ko[0], nRows, stream))) return st;
    if ((st = upload(ctx, desc, descRows.in(ws.d), ko[0] * stride, df, stream))) return st;
    bias = ko[0];
  }
  if (!ctx->matchAttrs) {
    CK(fe_match::set_attributes());
    ctx->matchAttrs = true;
  }
  fe_loop::Tables T;
  T.ko = tKo.in(ws.d);
  T.elig = tElig.in(ws.d);
  T.scans = tScans.in(ws.d);
  T.slots = tSlots.in(ws.d);
  T.items = tItems2.in(ws.d);
  T.qo = tQo.in(ws.d);
  T.ro = tRo.in(ws.d);
  fe_loop::Out o;
  o.loop = loop.in(ws.d);
  o.loopScan = loopScan.in(ws.d);
  o.nInl = nInl.in(ws.d);
  o.nHyp = nHyp.in(ws.d);
  o.pose = pose.in(ws.d);
  o.rms = rms.in(ws.d);
  o.cScan = cScan.in(ws.d);
  o.cVotes = cVotes.in(ws.d);
  o.cStatus = cStatus.in(ws.d);
  o.cInl = cInl.in(ws.d);
  o.cHyp = cHyp.in(ws.d);
  o.cRms = cRms.in(ws.d);
  o.cPose = cPose.in(ws.d);
  o.assoc = (long long*)assoc.in(ws.d);
  fe_loop::Work w;
  w.best1 = (const long long*)best1.in(ws.d);
  w.voteScan = voteScan.in(ws.d);
  w.voteKey = (unsigned long long*)voteKey.in(ws.d);
  w.q = wQ.in(ws.d);
  w.r = wR.in(ws.d);
  w.best2 = (long long*)best2.in(ws.d);
  w.slotBest = (long long*)slotBest.in(ws.d);
  w.reg.pose = gPose.in(ws.d);
  w.reg.rms = gRms.in(ws.d);
  w.reg.assoc = (long long*)gAssoc.in(ws.d);
  w.reg.nInl = gNInl.in(ws.d);
  w.reg.nHyp = gNHyp.in(ws.d);
  w.reg.status = gStatus.in(ws.d);
  w.reg.err = gErr.in(ws.d);
  w.scratch.corr = gCorr.in(ws.d);
  w.scratch.assocNew = (long long*)gAssocNew.in(ws.d);
  w.scratch.d2Cur = gD2Cur.in(ws.d);
  w.scratch.d2New = gD2New.in(ws.d);
  fe_match::Result r1, r2;
  r1.best = (long long*)best1.in(ws.d);
  r1.shift = shift1.in(ws.d);
  r1.dist2 = dist1.in(ws.d);
  r1.second = second1.in(ws.d);
  r2.best = w.best2;
  r2.shift = shift2.in(ws.d);
  r2.dist2 = dist2.in(ws.d);
  r2.second = second2.in(ws.d);

  // retrieval, votes, slots, verification matching, remap, registration, choice: one stream, no round trip
  int64_t launches = 0;
  const int n1 = (int)items1.size(), n2 = (int)items2.size();
  CK(fe_match::launch(desc, stride, bias, desc, stride, bias, tItems1.in(ws.d), n1, nPart1 > 0, part1.in(ws.d), r1, stream));
  launches += n1 ? (nPart1 > 0 ? 2 : 1) : 0;
  CK(fe_loop::vote(E, K, gap, T, w, o, stream));
  CK(fe_loop::place(kp, bias, nSlots, K, T, w, o, stream));
  CK(fe_match::launch(desc, stride, bias, desc, stride, bias, T.items, n2, nPart2 > 0, part2.in(ws.d), r2, stream));
  launches += n2 ? (nPart2 > 0 ? 2 : 1) : 0;
  CK(fe_loop::remap(nSlots, K, T, w, o, stream));
  if (nSlots > 0) {
    CK(cudaMemsetAsync(w.reg.err, 0, sizeof(int32_t), stream));
    CK(fe_register::launch(w.q, 0, w.r, 0, w.slotBest, T.qo, T.ro, (int)G, rp, w.reg, w.scratch, stream));
  }
  CK(fe_loop::select(B, K, T, w, o, stream));
  launches += (E > 0) + 3 * (nSlots > 0) + 1;
  ctx->launches += launches;
  out->gpu_launches = launches;
  CK(cudaMemcpyAsync(ws.h, ws.d, (size_t)resBytes, cudaMemcpyDeviceToHost, stream));
  CK(cudaStreamSynchronize(stream));
  return FE_OK;
}

}  // namespace

extern "C" {

void fe_loop_params_default(fe_loop_params_t* p) {
  if (!p) return;
  p->min_gap = FE_LOOP_MIN_GAP_DEFAULT;
  p->candidates = FE_LOOP_CANDIDATES_DEFAULT;
}

int fe_loop_closures(fe_ctx_t* ctx, const fe_point_t* kp, const float* desc, int64_t desc_stride,
                     const int64_t* keypoint_offsets, int32_t n_scans, const int64_t* sequence_offsets,
                     int32_t n_sequences, const fe_loop_params_t* loop_params, const fe_register_params_t* params,
                     fe_loop_result_t* out) {
  return loop_closures(ctx, kp, desc, desc_stride, keypoint_offsets, n_scans, sequence_offsets, n_sequences, loop_params,
                       params, out, false);
}

int fe_loop_closures_device(fe_ctx_t* ctx, const fe_point_t* kp, const float* desc, int64_t desc_stride,
                            const int64_t* keypoint_offsets, int32_t n_scans, const int64_t* sequence_offsets,
                            int32_t n_sequences, const fe_loop_params_t* loop_params,
                            const fe_register_params_t* params, fe_loop_result_t* out) {
  return loop_closures(ctx, kp, desc, desc_stride, keypoint_offsets, n_scans, sequence_offsets, n_sequences, loop_params,
                       params, out, true);
}

// ---- one entry point per reference function ----------------------------------------------------------

// Upload a one-scan cloud and run K1 on it with `flags` and the parameters P, levelled by rp = {roll, pitch} (null:
// the identity).  K1 compacts its survivors into the chunk pieces; with fullOut it also writes every point, transformed
// in place, to s.d_full (group FULL), which is copied to fullOut before this returns.
static int scan_k1(fe_ctx* ctx, Slot& s, const DevParams& P, const fe_point_t* in, int64_t n, int flags,
                   const double* rp = nullptr, fe_point_t* fullOut = nullptr) {
  int64_t offs[2] = {0, n};
  int64_t npts; int nch;
  int st = stage_scans(ctx, s, offs, rp, 1, &npts, &nch);
  if (st == FE_OK) st = stage_scans_copy(ctx, s, 1, false);
  if (st) return st;
  if (n > 0) CK(cudaMemcpyAsync(s.d_pts, in, (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, s.stream));
  if (nch > 0) {
    k_level_crop_ring<false, false><<<nch, 256, 0, s.stream>>>(s.d_pts, s.d_chunkTab, s.d_rot, P, flags, s.d_surf, s.d_surfCnt,
                                                               s.d_crop, s.d_cropMeta, s.d_cropCnt, fullOut ? s.d_full : nullptr,
                                                               RawLayout{nullptr, 0, 0, 0, 0}, 0);
    ctx->launches++;
  }
  CK(cudaGetLastError());
  if (fullOut) {
    CK(cudaMemcpyAsync(fullOut, s.d_full, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, s.stream));
    CK(cudaStreamSynchronize(s.stream));
  }
  return FE_OK;
}

int fe_get_elevation_angles(fe_ctx_t* ctx, fe_point_t* cloud, int64_t n) {
  if (!ctx || (n > 0 && !cloud) || n < 0) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int st = ensure_slot(ctx, ctx->slot[0], {CORE, POINTS, FULL});
  if (st || n == 0) return st;
  const double rp[2] = {0.0, 0.0};
  return scan_k1(ctx, ctx->slot[0], ctx->dp, cloud, n, F_ELEV, rp, cloud);
}

int fe_rotate_cloud(fe_ctx_t* ctx, fe_point_t* cloud, int64_t n, double roll, double pitch) {
  if (!ctx || (n > 0 && !cloud) || n < 0) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int st = ensure_slot(ctx, ctx->slot[0], {CORE, POINTS, FULL});
  if (st || n == 0) return st;
  const double rp[2] = {roll, pitch};
  return scan_k1(ctx, ctx->slot[0], ctx->dp, cloud, n, F_ROT, rp, cloud);
}

int fe_rotation_matrix(double roll, double pitch, float m[9]) {
  if (!m) return FE_ERR_INVALID;
  leveling_matrix(roll, pitch, m);
  return FE_OK;
}

static int copy_points_out(fe_ctx* ctx, const std::vector<fe_point_t>& v, fe_point_t* out, int64_t cap, int64_t* n_out) {
  if (n_out) *n_out = (int64_t)v.size();
  if (!out) return FE_OK;
  if ((int64_t)v.size() > cap) return fail(ctx, FE_ERR_CAPACITY, "output buffer too small");
  if (!v.empty()) memcpy(out, v.data(), v.size() * sizeof(fe_point_t));
  return FE_OK;
}

int fe_filter_cloud(fe_ctx_t* ctx, const fe_point_t* in, int64_t n, fe_point_t* out, int64_t cap, int64_t* n_out) {
  if (!ctx || n < 0 || (n > 0 && !in)) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  if (n_out) *n_out = 0;
  if (n == 0) return FE_OK;
  Slot& s = ctx->slot[0];
  int st = ensure_slot(ctx, s, {CORE, POINTS, CLOUDS});
  if (st) return st;
  st = scan_k1(ctx, s, ctx->dp, in, n, F_CROP);
  if (st) return st;
  std::vector<int64_t> off;
  std::vector<fe_point_t> pts;
  st = gather_to_host(ctx, s, 1, true, s.d_crop, s.d_cropCnt, nullptr, off, pts);
  if (st) return st;
  return copy_points_out(ctx, pts, out, cap, n_out);
}

int fe_extract_clusters(fe_ctx_t* ctx, const fe_point_t* cloud, int64_t n, double tolerance,
                        int32_t min_size, int32_t max_size, int32_t* cluster_offsets,
                        int32_t cap_clusters, int32_t* indices, int64_t cap_indices, int32_t* n_clusters) {
  if (!ctx || n < 0 || (n > 0 && !cloud) || !n_clusters || !cluster_offsets) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  *n_clusters = 0;
  cluster_offsets[0] = 0;
  if (n == 0) return FE_OK;
  if (n > ECAP_G) return fail(ctx, FE_ERR_CAPACITY, "fe_extract_clusters: more than 65535 points");
  if (!(tolerance > 0.0)) return fail(ctx, FE_ERR_INVALID, "tolerance must be > 0");
  Slot& s = ctx->slot[0];
  int st = ensure_slot(ctx, s, {CORE, POINTS});
  if (st) return st;
  if (n > s.capPts) return fail(ctx, FE_ERR_CAPACITY, "fe_extract_clusters: more points than max_points_per_call");
  CK(cudaMemcpyAsync(s.d_pts, cloud, (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, s.stream));
  const float tol_f = (float)tolerance;
  const float r2f = radius_sq_as_flann_sees_it((double)tol_f);
  int* d_off = (int*)s.d_keyA;
  int* d_idx = (int*)s.d_keyB;
  int* d_n = (int*)s.d_valA;
  if (n <= ECAP_L)
    k_extract_clusters_stage<false><<<1, NT2, kClusterSmemL, s.stream>>>(s.d_pts, (int)n, tol_f, r2f, min_size, max_size, d_off, (int)n,
                                                                         d_idx, d_n, nullptr);
  else
    k_extract_clusters_stage<true><<<1, NT2, cluster_smem_bytes_global(NT2), s.stream>>>(s.d_pts, (int)n, tol_f, r2f, min_size, max_size,
                                                                                          d_off, (int)n, d_idx, d_n, s.d_slabs);
  ctx->launches++;
  CK(cudaGetLastError());
  int nc = 0;
  CK(cudaMemcpyAsync(&nc, d_n, sizeof(int), cudaMemcpyDeviceToHost, s.stream));
  CK(cudaStreamSynchronize(s.stream));
  *n_clusters = nc;
  if (nc > cap_clusters) return fail(ctx, FE_ERR_CAPACITY, "cluster_offsets too small");
  std::vector<int> off(nc + 1);
  CK(cudaMemcpy(off.data(), d_off, (size_t)(nc + 1) * sizeof(int), cudaMemcpyDeviceToHost));
  memcpy(cluster_offsets, off.data(), (size_t)(nc + 1) * sizeof(int));
  if (off[nc] > cap_indices) return fail(ctx, FE_ERR_CAPACITY, "indices too small");
  if (off[nc] > 0 && indices) CK(cudaMemcpy(indices, d_idx, (size_t)off[nc] * sizeof(int), cudaMemcpyDeviceToHost));
  return FE_OK;
}

static int stage_keypoints(fe_ctx* ctx, const fe_point_t* cloud, int64_t n, bool singleRing, bool merge,
                           fe_point_t* kp, int64_t capKp, int64_t* nKp, fe_point_t* kc, int64_t capKc, int64_t* nKc) {
  if (nKp) *nKp = 0;
  if (nKc) *nKc = 0;
  if (n == 0) return FE_OK;
  Slot& s = ctx->slot[0];
  int st = ensure_slot(ctx, s, {CORE, POINTS, CLOUDS});
  if (st) return st;
  st = scan_k1(ctx, s, ctx->dp, cloud, n, singleRing ? 0 : F_RING);
  if (st) return st;
  CK(cudaMemsetAsync(s.d_ctr, 0, sizeof(DevCounters), s.stream));
  launch_clustering(ctx, s, 1, singleRing, true, merge);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(s.h_ctr, s.d_ctr, sizeof(DevCounters), cudaMemcpyDeviceToHost, s.stream));
  CK(cudaStreamSynchronize(s.stream));
  if (s.h_ctr->err) return fail(ctx, FE_ERR_CAPACITY, err_bits(s.h_ctr->err));
  std::vector<int64_t> off;
  std::vector<fe_point_t> pts;
  if (merge) {
    int base = 0, cnt = 0;
    CK(cudaMemcpy(&base, s.d_kpBase, sizeof(int), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&cnt, s.d_kpCnt, sizeof(int), cudaMemcpyDeviceToHost));
    pts.resize(cnt);
    if (cnt) CK(cudaMemcpy(pts.data(), s.d_kpPool + base, (size_t)cnt * sizeof(float4), cudaMemcpyDeviceToHost));
  } else {
    st = gather_to_host(ctx, s, 1, false, s.d_kfPool, s.d_kfCnt, s.d_kfBase, off, pts);
    if (st) return st;
  }
  st = copy_points_out(ctx, pts, kp, capKp, nKp);
  if (st) return st;
  st = gather_to_host(ctx, s, 1, false, s.d_kcPool, s.d_kcCnt, s.d_kcBase, off, pts);
  if (st) return st;
  return copy_points_out(ctx, pts, kc, capKc, nKc);
}

int fe_get_cylinder_segments(fe_ctx_t* ctx, const fe_point_t* ring_cloud, int64_t n, fe_point_t* centroids,
                             int64_t cap_centroids, int64_t* n_centroids, fe_point_t* cluster_cloud,
                             int64_t cap_cloud, int64_t* n_cloud) {
  if (!ctx || n < 0 || (n > 0 && !ring_cloud)) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  return stage_keypoints(ctx, ring_cloud, n, true, false, centroids, cap_centroids, n_centroids, cluster_cloud, cap_cloud, n_cloud);
}

int fe_estimate_keypoints(fe_ctx_t* ctx, const fe_point_t* cloud, int64_t n, fe_point_t* keypoints,
                          int64_t cap_keypoints, int64_t* n_keypoints, fe_point_t* keypoint_cloud,
                          int64_t cap_cloud, int64_t* n_cloud) {
  if (!ctx || n < 0 || (n > 0 && !cloud)) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  return stage_keypoints(ctx, cloud, n, false, true, keypoints, cap_keypoints, n_keypoints, keypoint_cloud, cap_cloud, n_cloud);
}

int fe_estimate_descriptors(fe_ctx_t* ctx, const fe_point_t* cloud_full, int64_t n, const fe_point_t* keypoints,
                            int64_t k, float* descriptors) {
  if (!ctx || n < 0 || k < 0 || (n > 0 && !cloud_full) || (k > 0 && (!keypoints || !descriptors))) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  if (k == 0) return FE_OK;  // src:331-332
  Slot& s = ctx->slot[0];
  int st = ensure_slot(ctx, s, {CORE, POINTS, GRID});
  if (st) return st;
  if (k > s.capKp) return fail(ctx, FE_ERR_CAPACITY, "more keypoints than max_keypoints_per_call");
  // the 3DSC order key holds a point's index in 20 bits (include/fe_b200.h, per-scan limits)
  if (n > FE_MAX_SCAN_POINTS) return fail(ctx, FE_ERR_CAPACITY, "a cloud of more than 2^20 points");
  // the search surface only matters around the keypoints: grid over their bounding box
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int64_t i = 0; i < k; i++) {
    const float v[3] = {keypoints[i].x, keypoints[i].y, keypoints[i].z};
    if (!std::isfinite(v[0]) || !std::isfinite(v[1]) || !std::isfinite(v[2])) continue;
    for (int d = 0; d < 3; d++) { lo[d] = std::min(lo[d], v[d]); hi[d] = std::max(hi[d], v[d]); }
  }
  if (!(lo[0] <= hi[0])) { for (int d = 0; d < 3; d++) { lo[d] = 0.f; hi[d] = 0.f; } }
  DevParams P = ctx->dp;
  surface_grid(P, ctx->params.descriptor_radius, lo[0], hi[0], lo[1], hi[1], lo[2], hi[2]);
  st = scan_k1(ctx, s, P, cloud_full, n, F_SURF);  // n == 0: one empty scan
  if (st) return st;
  cudaStream_t q = s.stream;
  std::vector<int> kpOff = {0, (int)k};
  std::vector<int> kpScan((size_t)k, 0);
  if (cudaMemsetAsync(s.d_ctr, 0, sizeof(DevCounters), q) != cudaSuccess ||
      cudaMemcpyAsync(s.d_kpOff, kpOff.data(), 2 * sizeof(int), cudaMemcpyHostToDevice, q) != cudaSuccess ||
      cudaMemcpyAsync(s.d_kpScan, kpScan.data(), (size_t)k * sizeof(int), cudaMemcpyHostToDevice, q) != cudaSuccess ||
      cudaMemcpyAsync(s.d_kpOut, keypoints, (size_t)k * sizeof(float4), cudaMemcpyHostToDevice, q) != cudaSuccess)
    return fail(ctx, FE_ERR_CUDA, "staging of the descriptor inputs failed");
  launch_surface_grid(ctx, s, 1, P);
  launch_desc_mark(ctx, s, 1, P, ctx->numSms * 4);
  launch_density(ctx, s, 1, P, n);
  launch_desc_hist(ctx, s, 1, P, ctx->numSms * 4, false);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(s.h_ctr, s.d_ctr, sizeof(DevCounters), cudaMemcpyDeviceToHost, q));
  CK(cudaMemcpyAsync(descriptors, s.d_desc, (size_t)k * FE_DESC_LEN * sizeof(float), cudaMemcpyDeviceToHost, q));
  CK(cudaStreamSynchronize(q));
  if (s.h_ctr->err) return fail(ctx, FE_ERR_CAPACITY, err_bits(s.h_ctr->err));
  return FE_OK;
}

int fe_pack_point_descriptors(const fe_point_t* keypoints, const float* descriptors, int64_t k, float* records) {
  if (k < 0 || (k > 0 && (!keypoints || !descriptors || !records))) return FE_ERR_INVALID;
  for (int64_t i = 0; i < k; i++) {
    float* r = records + i * FE_RECORD_FLOATS;
    memset(r, 0, FE_RECORD_FLOATS * sizeof(float));
    // PCL_ADD_POINT4D: x,y,z + one pad float (not a registered field: stays value-initialised 0)
    r[0] = keypoints[i].x; r[1] = keypoints[i].y; r[2] = keypoints[i].z;
    r[4] = keypoints[i].intensity;
    memcpy(r + 5, descriptors + i * FE_DESC_LEN, FE_DESC_LEN * sizeof(float));
    // rf[9] at r + 5 + 1980 stays zero (3dsc.hpp zeroes it); 2 floats of tail padding (EIGEN_ALIGN16)
  }
  return FE_OK;
}

// ---- scan-parallel sharding over several GPUs in one process -----------------------------------------
struct fe_multi {
  std::vector<fe_ctx_t*> ctx;
  std::vector<int64_t> kpOffsets;
  bool cloudOutputs = false;
  std::vector<int64_t> cloudOff, kcOff;
  std::vector<fe_point_t> cloudPts, kcPts;
  fe_point_t* kp = nullptr;   // gathered results: plain malloc'd buffers grown on demand (no zero fill)
  float* desc = nullptr;
  int64_t capKp = 0, capDesc = 0;
  std::string err;
};

int fe_multi_create(const int32_t* devices, int32_t n_devices, const fe_params_t* params,
                    const fe_limits_t* limits, fe_multi_t** out) {
  if (!out || !devices || n_devices < 1 || !params) return FE_ERR_INVALID;
  *out = nullptr;
  fe_multi* m = new fe_multi();
  for (int g = 0; g < n_devices; g++) {
    fe_ctx_t* c = nullptr;
    const int st = fe_create(devices[g], params, limits, &c);
    if (st != FE_OK) { fe_multi_destroy(m); return st; }
    m->ctx.push_back(c);
  }
  *out = m;
  return FE_OK;
}

int fe_multi_enable_record_output(fe_multi_t* m, int32_t enable) {
  if (!m) return FE_ERR_INVALID;
  for (fe_ctx_t* c : m->ctx) {
    const int st = fe_enable_record_output(c, enable);
    if (st) return st;
  }
  return FE_OK;
}

int fe_multi_enable_cloud_outputs(fe_multi_t* m, int32_t enable) {
  if (!m) return FE_ERR_INVALID;
  for (fe_ctx_t* c : m->ctx) {
    const int st = fe_enable_cloud_outputs(c, enable);
    if (st) return st;
  }
  m->cloudOutputs = enable != 0;
  return FE_OK;
}

int fe_multi_get_cloud_outputs(fe_multi_t* m, const int64_t** cloud_offsets, const fe_point_t** cloud,
                               const int64_t** kpcloud_offsets, const fe_point_t** keypoint_cloud) {
  if (!m) return FE_ERR_INVALID;
  if (m->cloudOff.empty()) { m->err = "no cloud outputs recorded (fe_multi_enable_cloud_outputs before fe_multi_process_batch)"; return FE_ERR_INVALID; }
  if (cloud_offsets) *cloud_offsets = m->cloudOff.data();
  if (cloud) *cloud = m->cloudPts.data();
  if (kpcloud_offsets) *kpcloud_offsets = m->kcOff.data();
  if (keypoint_cloud) *keypoint_cloud = m->kcPts.data();
  return FE_OK;
}

void fe_multi_destroy(fe_multi_t* m) {
  if (!m) return;
  for (fe_ctx_t* c : m->ctx) fe_destroy(c);
  free(m->kp);
  free(m->desc);
  delete m;
}

const char* fe_multi_last_error(const fe_multi_t* m) { return m ? m->err.c_str() : "null context"; }

int fe_multi_process_batch(fe_multi_t* m, const fe_point_t* points, const int64_t* scan_offsets,
                           const double* roll_pitch, int32_t n_scans, fe_batch_result_t* out) {
  if (!m || !out || n_scans < 0 || (n_scans > 0 && (!scan_offsets || !roll_pitch))) return FE_ERR_INVALID;
  const int G = (int)m->ctx.size();
  m->err.clear();
  std::vector<fe_batch_result_t> res(G);
  std::vector<int> status(G, FE_OK);
  std::vector<int> lo(G + 1);
  for (int g = 0; g <= G; g++) lo[g] = (int)(((int64_t)n_scans * g) / G);
  {  // one host thread per GPU: its shard through fe_process_batch (absolute offsets into `points`)
    std::vector<std::thread> th;
    for (int g = 0; g < G; g++)
      th.emplace_back([&, g]() {
        status[g] = fe_process_batch(m->ctx[g], points, scan_offsets + lo[g], roll_pitch ? roll_pitch + 2 * (int64_t)lo[g] : nullptr,
                                     lo[g + 1] - lo[g], &res[g]);
      });
    for (auto& t : th) t.join();
  }
  for (int g = 0; g < G; g++)
    if (status[g] != FE_OK) {
      m->err = std::string("device shard ") + std::to_string(g) + ": " + fe_last_error(m->ctx[g]);
      return status[g];
    }
  // host-side gather in scan order
  std::vector<int64_t> kbase(G + 1, 0);
  for (int g = 0; g < G; g++) kbase[g + 1] = kbase[g] + res[g].n_keypoints;
  const int64_t K = kbase[G];
  const bool desc = m->ctx[0]->params.estimate_descriptors != 0;
  const size_t dl = m->ctx[0]->recordOutput ? FE_RECORD_FLOATS : FE_DESC_LEN;
  m->kpOffsets.assign((size_t)n_scans + 1, 0);
  if (K > m->capKp) {
    free(m->kp);
    m->capKp = K + K / 2 + 1024;
    m->kp = (fe_point_t*)malloc((size_t)m->capKp * sizeof(fe_point_t));
    if (!m->kp) { m->capKp = 0; m->err = "out of host memory"; return FE_ERR_CAPACITY; }
  }
  if (desc && K > m->capDesc) {
    free(m->desc);
    m->capDesc = K + K / 2 + 1024;
    m->desc = (float*)malloc((size_t)m->capDesc * FE_RECORD_FLOATS * sizeof(float));
    if (!m->desc) { m->capDesc = 0; m->err = "out of host memory"; return FE_ERR_CAPACITY; }
  }
  {
    std::vector<std::thread> th;
    for (int g = 0; g < G; g++)
      th.emplace_back([&, g]() {
        const int ns = lo[g + 1] - lo[g];
        for (int i = 0; i <= ns; i++) m->kpOffsets[lo[g] + i] = kbase[g] + res[g].keypoint_offsets[i];
        if (res[g].n_keypoints > 0) {
          memcpy(m->kp + kbase[g], res[g].keypoints, (size_t)res[g].n_keypoints * sizeof(fe_point_t));
          if (desc) memcpy(m->desc + kbase[g] * dl, res[g].descriptors, (size_t)res[g].n_keypoints * dl * sizeof(float));
        }
      });
    for (auto& t : th) t.join();
  }
  m->cloudOff.clear(); m->kcOff.clear();
  if (m->cloudOutputs) {  // the shards' ~cloud / ~keypoint_cloud concatenated in scan order
    m->cloudOff.assign((size_t)n_scans + 1, 0); m->kcOff.assign((size_t)n_scans + 1, 0);
    m->cloudPts.clear(); m->kcPts.clear();
    for (int g = 0; g < G; g++) {
      const int ns = lo[g + 1] - lo[g];
      if (ns == 0) continue;
      const int64_t *co = nullptr, *ko = nullptr;
      const fe_point_t *cp = nullptr, *kp2 = nullptr;
      const int st = fe_get_cloud_outputs(m->ctx[g], &co, &cp, &ko, &kp2);
      if (st != FE_OK) { m->err = std::string("device shard ") + std::to_string(g) + ": " + fe_last_error(m->ctx[g]); return st; }
      const int64_t cb = (int64_t)m->cloudPts.size(), kb = (int64_t)m->kcPts.size();
      for (int i = 0; i <= ns; i++) { m->cloudOff[lo[g] + i] = cb + co[i]; m->kcOff[lo[g] + i] = kb + ko[i]; }
      m->cloudPts.insert(m->cloudPts.end(), cp, cp + co[ns]);
      m->kcPts.insert(m->kcPts.end(), kp2, kp2 + ko[ns]);
    }
  }
  out->n_scans = n_scans;
  out->n_keypoints = K;
  out->keypoint_offsets = m->kpOffsets.data();
  out->keypoints = m->kp;
  out->descriptors = desc ? m->desc : nullptr;
  out->on_device = 0;
  out->gpu_launches = 0;
  for (int g = 0; g < G; g++) out->gpu_launches += res[g].gpu_launches;
  return FE_OK;
}

// bench hook: work of the 3DSC density stage of the last device call: out = {distance tests, marked surface points
// (distinct points inside some keypoint's support sphere), halo points kept by the cell grid}
int fe_debug_density_work(fe_ctx_t* ctx, int64_t out[3]) {
  if (!ctx || !out || !ctx->slot[0].h_ctr) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  Slot& s = ctx->slot[0];
  CK(cudaStreamSynchronize(s.stream));
  out[0] = (int64_t)s.h_ctr->dens_work[0];
  out[1] = (int64_t)s.h_ctr->dens_work[1];
  out[2] = 0;
  if (s.sb.nscans > 0 && ctx->params.estimate_descriptors) {
    std::vector<int> sn((size_t)s.sb.nscans);
    CK(cudaMemcpy(sn.data(), s.d_surfN, sn.size() * sizeof(int), cudaMemcpyDeviceToHost));
    for (int v : sn) out[2] += v;
  }
  return FE_OK;
}

// bench hook: bare pinned-host -> device copies of `bytes` from `host` into the context's staging buffer, chunk after
// chunk on one stream, timed with CUDA events — the ceiling the host entry points can reach on this box
int fe_debug_h2d_probe(fe_ctx_t* ctx, const void* host, int64_t bytes, float* ms) {
  if (!ctx || !host || bytes < 0 || !ms) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  Slot& s = ctx->slot[0];
  int st = ensure_slot(ctx, s, {POINTS});
  if (st) return st;
  const int64_t chunk = s.capPts * (int64_t)sizeof(float4);
  CK(cudaStreamSynchronize(s.stream));
  CK(cudaEventRecord(s.evT0, s.stream));
  for (int64_t off = 0; off < bytes; off += chunk)
    CK(cudaMemcpyAsync(s.d_pts, (const char*)host + off, (size_t)std::min(chunk, bytes - off), cudaMemcpyHostToDevice, s.stream));
  CK(cudaEventRecord(s.evT1, s.stream));
  CK(cudaEventSynchronize(s.evT1));
  CK(cudaEventElapsedTime(ms, s.evT0, s.evT1));
  return FE_OK;
}

// debug / test hook: run K2 through the grid-based kernels only (the general fallback of the run-based kernel), so
// that tests can cross-check the two algorithms against each other and against the oracle
int fe_debug_force_grid_clustering(fe_ctx_t* ctx, int32_t enable) {
  if (!ctx) return FE_ERR_INVALID;
  if (int st = sync_slots(ctx)) return st;
  ctx->gridClustering = enable != 0;
  ctx->epoch++;
  return FE_OK;
}

// debug / test hook: switch the CUDA-graph replay of small sub-batches off (eager launches) or on; out[0] (nullable)
// receives the number of graph replays so far
int fe_debug_enable_graphs(fe_ctx_t* ctx, int32_t enable, int64_t* replays) {
  if (!ctx) return FE_ERR_INVALID;
  ctx->useGraphs = enable != 0;
  if (replays) *replays = ctx->graphReplays;
  return FE_OK;
}

// debug / test hook: how many small sub-batches had to be run again with the whole chain of fallback kernels
int fe_debug_lean_reruns(fe_ctx_t* ctx, int64_t* reruns) {
  if (!ctx || !reruns) return FE_ERR_INVALID;
  *reruns = ctx->leanReruns;
  return FE_OK;
}

// debug / test hook: keypoints_full (src:205), i.e. estimateKeypoints before the cross-ring merge
int fe_debug_keypoints_full(fe_ctx_t* ctx, const fe_point_t* cloud, int64_t n, fe_point_t* kf, int64_t cap, int64_t* n_kf) {
  if (!ctx || n < 0 || (n > 0 && !cloud)) return FE_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  return stage_keypoints(ctx, cloud, n, false, false, kf, cap, n_kf, nullptr, 0, nullptr);
}

// debug / test hook: the cluster order PCL's final std::sort leaves, from the replay the kernels use
void fe_debug_sort_replay(const int32_t* sizes, int32_t n, int32_t* order_out) {
  std::vector<int> ids(n);
  for (int i = 0; i < n; i++) ids[i] = i;
  fe::pcl_cluster_order(ids.data(), n, [=](int id) { return sizes[id]; });
  for (int i = 0; i < n; i++) order_out[i] = ids[i];
}

}  // extern "C"
