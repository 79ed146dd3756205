/*
 * fe_b200.h — C-ABI of the B200-native per-scan keypoint pipeline.
 *
 * Drop-in boundary for the span of `cloudCallback` between
 * src/feature_extraction_node.cpp:83 (after PointCloud2 -> pcl conversion) and :117
 * (before publishing) of GAVLab/feature_extraction.  ROS / PointCloud2 I/O stays on the
 * host and is not part of this library.
 *
 * Everything behind these entry points runs as hand-written sm_100a CUDA kernels.  There is
 * NO CPU fallback: fe_create() fails when no CUDA device is usable.
 *
 * Conventions
 *   - plain C types only; no exceptions cross the boundary; every call returns an fe_status.
 *   - a context (fe_ctx_t) is bound to one GPU; it is NOT thread-safe; distinct contexts are
 *     independent (one per GPU for scan-parallel sharding).  The reference is single-threaded
 *     and serial per scan (ros::spin, src:386).
 *   - empty in -> empty out is not an error (src:209-210, 234-235, 263-264, 278-279, 331-332).
 *   - capacity overflow is FE_ERR_CAPACITY, never silent truncation.
 */
#ifndef FE_B200_H_
#define FE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FE_DESC_LEN 1980          /* pcl::ShapeContext1980: 12 az x 11 el x 15 rad          */
#define FE_RECORD_FLOATS 1996     /* pcl::PointDescriptor, feature_extraction_node.h:35-42:  */
                                  /* x,y,z,pad | intensity | descriptor[1980] | rf[9] -> 7976 B, 16-aligned 7984 B */
#define FE_NUM_RINGS 16           /* hard-coded channel loop, src:195                        */

typedef enum fe_status {
  FE_OK = 0,
  FE_ERR_INVALID = 1,       /* bad argument                                              */
  FE_ERR_CUDA = 2,          /* CUDA runtime error (see fe_last_error)                    */
  FE_ERR_CAPACITY = 3,      /* an output or workspace capacity would be exceeded         */
  FE_ERR_NO_DEVICE = 4,     /* no usable CUDA device: there is no CPU fallback           */
  FE_ERR_UNSUPPORTED = 5
} fe_status;

/* pcl::PointXYZI as the reference uses it (feature_extraction_node.h:66) minus PCL's padding:
 * 16 bytes, `intensity` carries the elevation angle in degrees after getElevationAngles. */
typedef struct fe_point {
  float x, y, z, intensity;
} fe_point_t;

/* The ROS parameters read in the constructor, src:9-34, with the member types of
 * feature_extraction_node.h:115-127.  `cloud_leveling` is applied by the caller (pass roll =
 * pitch = 0, as imuCallback does at src:66-69). */
typedef struct fe_params {
  double x_min, x_max;                /* src:14-15 */
  double y_min, y_max;                /* src:16-17 */
  double z_min, z_max;                /* src:18-19 */
  double cluster_tolerance;           /* src:24 */
  int32_t cluster_min_count;          /* src:25 */
  int32_t cluster_max_count;          /* src:26 */
  double cluster_radius_threshold;    /* src:27 */
  int32_t number_detection_channels;  /* src:28 */
  int32_t estimate_descriptors;       /* src:33 (bool) */
  double descriptor_radius;           /* src:34 */
} fe_params_t;

/* Workspace capacities of a context.  0 = library default. */
typedef struct fe_limits {
  int64_t max_points_per_call;     /* points staged on the device per sub-batch            */
  int32_t max_scans_per_call;      /* scans per sub-batch                                  */
  int64_t max_keypoints_per_call;  /* keypoints (and descriptors) per sub-batch            */
  int64_t max_ring_clusters_per_call; /* ring-level centroids (keypoints_full, src:205)    */
} fe_limits_t;

typedef struct fe_ctx fe_ctx_t;

/* ---- parameter presets ------------------------------------------------------------------ */
void fe_params_node_default(fe_params_t* p);     /* constructor defaults, src:9-34            */
void fe_params_launch_playback(fe_params_t* p);  /* launch/keypoint_playback.launch:17-33     */

/* ---- lifecycle --------------------------------------------------------------------------- */
const char* fe_version(void);
int fe_create(int device, const fe_params_t* params, const fe_limits_t* limits, fe_ctx_t** out);
int fe_set_params(fe_ctx_t* ctx, const fe_params_t* params);
void fe_destroy(fe_ctx_t* ctx);
const char* fe_last_error(const fe_ctx_t* ctx);
int fe_device_count(void);

/* Pinned host memory helpers (optional; any host pointer is accepted by the batch call, pinned
 * memory lets the H2D/D2H copies overlap the kernels). */
void* fe_host_alloc(int64_t bytes);
void fe_host_free(void* p);

/* ---- the fused path: cloudCallback, src:83-117 ------------------------------------------- */

typedef struct fe_batch_result {
  int32_t n_scans;
  int64_t n_keypoints;
  const int64_t* keypoint_offsets; /* host, n_scans+1 (CSR by scan)                         */
  const fe_point_t* keypoints;     /* n_keypoints x {x,y,z,el_deg}  (~keypoints, src:131)   */
  const float* descriptors;        /* n_keypoints x 1980 (NULL if estimate_descriptors==0)  */
  int32_t on_device;               /* 1: keypoints/descriptors are device pointers          */
  int64_t gpu_launches;            /* kernels launched by this call                         */
} fe_batch_result_t;

/* points/scan_offsets/roll_pitch are HOST buffers.  Scan s owns points
 * [scan_offsets[s], scan_offsets[s+1]); roll_pitch[2s], roll_pitch[2s+1] are the IMU roll and
 * pitch in radians as imuCallback leaves them (src:63-65).  Results are context-owned host
 * memory, valid until the next call on this context. */
int fe_process_batch(fe_ctx_t* ctx, const fe_point_t* points, const int64_t* scan_offsets,
                     const double* roll_pitch, int32_t n_scans, fe_batch_result_t* out);

/* Layout of the caller's point records (sensor_msgs/PointCloud2 point_step and field offsets, or any
 * array of structs): x, y, z are little-endian 32-bit floats at byte offsets x_off, y_off, z_off of
 * records `stride` bytes apart.  The input intensity is never read: getElevationAngles overwrites it
 * (src:154).  Examples: {16,0,4,8} fe_point_t; {12,0,4,8} packed xyz; {32,0,4,8} pcl::PointXYZI as
 * it sits in a pcl::PointCloud; {22,0,4,8} / {32,0,4,8} Velodyne PointCloud2 data (src:79-81). */
typedef struct fe_point_layout {
  int32_t stride, x_off, y_off, z_off;
} fe_point_layout_t;

/* fe_process_batch for records of any layout: `points` is the HOST byte buffer, scan_offsets count
 * records.  The records are copied to the device as they are and decoded by the first kernel. */
int fe_process_batch_layout(fe_ctx_t* ctx, const void* points, const fe_point_layout_t* layout,
                            const int64_t* scan_offsets, const double* roll_pitch, int32_t n_scans,
                            fe_batch_result_t* out);

/* imuCallback, src:57-70: orientation quaternion {x,y,z,w} -> the roll/pitch the node keeps
 * (tf::Matrix3x3(quat).getRPY, roll = tmproll - pi; both 0 when cloud_leveling is false). */
int fe_imu_to_roll_pitch(const double quat_xyzw[4], int32_t cloud_leveling, double* roll, double* pitch);

/* Same, but `d_points` is already resident in device memory and the results stay on the
 * device (keypoint_offsets is still host memory).  Must fit one sub-batch.
 * Calls of a handful of scans (<= 16; also through fe_process_batch) are replayed from a CUDA graph
 * captured the second time a shape is seen — here the shape includes `d_points`, so a caller that
 * keeps refilling the same device buffer gets the replay.  Results do not depend on the route. */
int fe_process_batch_device(fe_ctx_t* ctx, const fe_point_t* d_points,
                            const int64_t* scan_offsets, const double* roll_pitch,
                            int32_t n_scans, fe_batch_result_t* out);

/* ---- scan-parallel sharding over several GPUs of one box, in one process (SURVEY.md 8e) -------- */
/* Scans are independent (src:72-145 reads no cross-scan state): GPU g of G takes the contiguous scan
 * range [g*B/G, (g+1)*B/G), one host thread and one context per GPU, and the per-GPU results are
 * concatenated on the host in scan order.  No collective is involved. */
typedef struct fe_multi fe_multi_t;
int fe_multi_create(const int32_t* devices, int32_t n_devices, const fe_params_t* params,
                    const fe_limits_t* limits, fe_multi_t** out);
int fe_multi_process_batch(fe_multi_t* m, const fe_point_t* points, const int64_t* scan_offsets,
                           const double* roll_pitch, int32_t n_scans, fe_batch_result_t* out);
void fe_multi_destroy(fe_multi_t* m);
const char* fe_multi_last_error(const fe_multi_t* m);

/* Copy `bytes` of a device-resident result (fe_process_batch_device) to host memory. */
int fe_download(fe_ctx_t* ctx, void* host_dst, const void* device_src, int64_t bytes);

/* Optional extra outputs of the last fe_process_batch() / fe_process_batch_layout() (any number of
 * sub-batches): ~keypoint_cloud (src:133-135, the points of every gated ring cluster in the order
 * src:323 appends them) and ~cloud (src:137-139, the cropped cloud), CSR by scan, gathered on the device
 * and copied into context-owned pinned memory (valid until the next call).  Enabled with
 * fe_enable_cloud_outputs(ctx, 1) before the call; fe_multi_* concatenates the shards' outputs. */
int fe_enable_cloud_outputs(fe_ctx_t* ctx, int32_t enable);
int fe_get_cloud_outputs(fe_ctx_t* ctx, const int64_t** cloud_offsets, const fe_point_t** cloud,
                         const int64_t** kpcloud_offsets, const fe_point_t** keypoint_cloud);
int fe_multi_enable_cloud_outputs(fe_multi_t* m, int32_t enable);
int fe_multi_get_cloud_outputs(fe_multi_t* m, const int64_t** cloud_offsets, const fe_point_t** cloud,
                               const int64_t** kpcloud_offsets, const fe_point_t** keypoint_cloud);

/* Record output — pcl::concatenateFields(*keypoints, *descriptors, *pt_descriptors) at src:119 done
 * on the device: when enabled, `descriptors` of every following result (fe_process_batch,
 * fe_process_batch_layout, fe_process_batch_device, fe_multi_process_batch) points to n_keypoints
 * records of FE_RECORD_FLOATS floats in the layout of pcl::PointDescriptor
 * (feature_extraction_node.h:35-53): x, y, z, 0 | intensity | descriptor[1980] | rf[9] = 0 | padding —
 * what fe_pack_point_descriptors() would build on the host, ready to be published as ~features.
 * `keypoints` is filled as before.  With estimate_descriptors == 0 there are no descriptors and hence no
 * records (the reference publishes ~features only inside `if (descriptorEstimation)`, src:112-124): the
 * setting is kept but has no effect. */
int fe_enable_record_output(fe_ctx_t* ctx, int32_t enable);
int fe_multi_enable_record_output(fe_multi_t* m, int32_t enable);

/* Which float libm the 3DSC angles follow.  pcl::ShapeContext3DEstimation::computePoint (3dsc.hpp,
 * called at src:353) bins a neighbour by rad2deg(atan2(float, float)) and rad2deg(acosf(float)), i.e. by
 * the last bit of the host libm's atan2f / acosf.  FE_LIBM_FDLIBM (default): the fdlibm float routines
 * of glibc <= 2.40 restated on the device operation by operation (csrc/glibc_f32.h) — bit-identical to
 * the reference's x86-64 build and to this image's glibc 2.39.  FE_LIBM_CORRECTLY_ROUNDED: what
 * glibc >= 2.41 (CORE-MATH) returns. */
#define FE_LIBM_FDLIBM 0
#define FE_LIBM_CORRECTLY_ROUNDED 1
int fe_set_angle_libm(fe_ctx_t* ctx, int32_t mode);

/* Tolerance-boundary report (BASELINE.json north_star: "points lying within 1e-6 m of a tolerance
 * boundary reported separately").  Every radius predicate of the path is d2 < r2f evaluated in float
 * (FLANN L2_Simple; r2f = (float)(radius*radius)); a point pair is ON THE BOUNDARY of a predicate when
 * |sqrt((double)d2) - sqrt((double)r2f)| < eps_m.  After fe_enable_boundary_report(ctx, eps_m > 0) every
 * batch call also counts those pairs per scan — audit kernels next to the pipeline, slower — and
 * fe_get_boundary_report returns n_scans x 4 counts of the last call:
 *   [0] ring clustering, src:269-276: unordered pairs of cropped points of one ring (a point on a ring
 *       window's end value belongs to two rings, src:200-202, and counts in both)
 *   [1] cross-ring merge, src:222-229: unordered pairs of ring centroids with the pseudo z of src:217
 *   [2] 3DSC support radius, src:350: (keypoint, surface point) pairs
 *   [3] 3DSC point-density radius, src:352: (neighbour, surface point) pairs, the neighbour being every
 *       surface point inside some keypoint's support sphere, counted once
 * A scan with all four counts 0 has no decision within eps_m of flipping; the CPU oracle counts the same
 * pairs (feo_process_batch_boundary) and tools/parity_campaign.py prints both.  eps_m <= 0 disables. */
int fe_enable_boundary_report(fe_ctx_t* ctx, double eps_m);
int fe_get_boundary_report(fe_ctx_t* ctx, const int64_t** counts, int32_t* n_scans);

/* The same report over every threshold decision of the path in metres or degrees.  After
 * fe_enable_boundary_report_all(ctx, eps_m > 0) every batch call counts kinds 0-9 and
 * fe_get_boundary_report_all returns n_scans x FE_BOUNDARY_KINDS counts of the last call (FE_ERR_INVALID unless
 * the report was enabled with _all); fe_get_boundary_report still returns the n_scans x 4 of kinds 0-3.  A margin
 * is evaluated in IEEE double with + - * / sqrt only, in the order written here (no FMA), so the CPU oracle gets
 * the same count to the last pair.  DEG = 0.017453292519943295 (pi/180 as a double); "within eps" is < eps_m.
 *   [0-3] as above
 *   [4] crop box, src:169-183: points of the levelled full cloud with finite x, y, z such that, with
 *       lo_a = (double)(float)min_a, hi_a = (double)(float)max_a and v_a = (double) the levelled coordinate, every
 *       axis has lo_a - eps < v_a < hi_a + eps and some axis has |v_a - lo_a| < eps or |v_a - hi_a| < eps
 *   [5] ring-window ends, src:195-202: crop survivors with a finite elevation el (float, degrees);
 *       range = sqrt(((double)x*x + (double)y*y) + (double)z*z) of the cropped levelled point, counted once when
 *       range * (min over e = -16, -14, ..., 16 of |(double)el - e| * DEG) < eps
 *   [6] cluster diameter gate, src:314-316: ring clusters (every ring) that passed the size gate, counted when
 *       |diameter - 2 * cluster_radius_threshold| < eps, diameter being the double each side computes: sqrt on the
 *       device, pow(., 0.5) in the oracle.  The two differ by at most an ulp, so at eps >= 1e-9 m the counts agree.
 *   [7] 3DSC radial shells (3dsc.hpp, called at src:350-353): (keypoint, neighbour) pairs that reach the binning
 *       (finite keypoint, d2 < (float)R^2, d2 not pcl::utils::equal to 0); r = sqrtf(d2) as binned, counted when
 *       min over a = 1..14 of |(double)r - (double)radii[a]| < eps (radii[15] is kind 2's sphere)
 *   [8] 3DSC elevation edges: the same pairs, counted when (double)r * (min over a = 1..10 of
 *       |(double)theta - (double)theta_div[a]| * DEG) < eps, theta the float angle as binned
 *   [9] 3DSC azimuth edges: the same pairs; pox, poy = the float differences q - o in x and y,
 *       rho = sqrt((double)pox*pox + (double)poy*poy); counted when rho == 0 (straight above or below the keypoint)
 *       or rho * (min over a = 0..12 of |(double)phi - (double)phi_div[a]| * DEG) < eps (0 and 360 deg both: that
 *       half-plane separates bin 0 from bin 11)
 * With FE_LIBM_CORRECTLY_ROUNDED, kinds 8 and 9 are counted on the angles the device bins with.  The batch routes
 * all fill the report (fe_process_batch, fe_process_batch_layout, fe_process_batch_device, any number of
 * sub-batches); fe_multi_* has none.  eps_m <= 0 disables the report. */
#define FE_BOUNDARY_KINDS 10
int fe_enable_boundary_report_all(fe_ctx_t* ctx, double eps_m);
int fe_get_boundary_report_all(fe_ctx_t* ctx, const int64_t** counts, int32_t* n_scans);

/* ---- descriptor matching: the step downstream of ~features ---------------------------------- */
/* 3DSC descriptors of one pole seen from two scans have their 12 azimuth blocks rotated against each other by an
 * unknown amount: the x axis of a descriptor comes from the mt19937 draws of the keypoint's position in the output
 * order, and levelling removes roll and pitch but not yaw.  The matcher therefore compares two descriptors by the
 * minimum over the 12 azimuth rotations (Frome et al., ECCV 2004), evaluated to the last bit as follows.
 *
 * Rows.  A descriptor row is FE_DESC_LEN = 1980 floats, bin (l, k, j) at [l*165 + k*15 + j] (l azimuth, k elevation,
 * j radial), and row i starts i * stride floats after row 0.  stride = FE_DESC_LEN for plain bins; for the records of
 * fe_enable_record_output, stride = FE_RECORD_FLOATS and the row pointer is the record base + 5 floats.
 *
 * Distance.  For a query row a, a reference row b and a shift s in [0, 12):
 *   P(la, lb) = the chain over m = 0..164 ascending of  acc = 0.0f;  t = a[la*165+m] - b[lb*165+m];  acc = fmaf(t, t, acc)
 *   d_s(a, b) = 0.0f;  for l = 0..11 ascending:  d_s = d_s + P(l, (l + s) mod 12)        (float adds)
 * fmaf is the correctly rounded fused multiply-add, every other operation a separate IEEE float operation.  So if
 * b[((l+s) mod 12)*165 + m] == a[l*165 + m] for every l and m, d_s(a, b) == 0.
 *
 * Groups.  query_offsets[0..n_groups] and ref_offsets[0..n_groups] are host arrays of row indices, non-decreasing
 * and not negative.  Query rows [qo[g], qo[g+1]) are compared with reference rows [ro[g], ro[g+1]) and with nothing
 * else.  Output row i belongs to query row qo[0] + i: n_queries = qo[G] - qo[0].  One scan against a map is one
 * group; scan s against scan s-1 of one batch result is qo = keypoint_offsets + 1, ro = keypoint_offsets, G = B - 1.
 *
 * Per query, over the candidates (r, s) of its group (r the absolute reference row index):
 *   best, shift   the candidate with the smallest d_s; a candidate replaces the current best only if its d_s is
 *                 smaller (the current value starts at +inf), ties go to the lower r, then to the lower s; a NaN
 *                 distance never wins (so the all-NaN rows of zero-neighbour keypoints never match)
 *   dist2         d_s of the best candidate
 *   second_dist2  the smallest per-row minimum over the group's other reference rows (for a ratio test); equal to
 *                 dist2 when another row ties the best
 * A query without a winning candidate, e.g. every query of a group without reference rows, gets best = -1,
 * shift = -1, dist2 = second_dist2 = +inf.
 *
 * Results are context-owned pinned host memory, valid until the next match call.  A match call leaves the results of
 * the last batch call alone, device pointers of fe_process_batch_device included, so one can process, match on the
 * returned `descriptors` and read both.  FE_ERR_INVALID (the context stays usable) when a stride is below
 * FE_DESC_LEN, an offsets array decreases or has a negative entry, n_groups < 0, or a row pointer is NULL while its
 * side has rows.  n_groups = 0 and empty groups are not errors. */
typedef struct fe_match_result {
  int64_t n_queries;
  const int64_t* best;         /* n_queries: absolute reference row index, -1 = none */
  const int32_t* shift;        /* n_queries: s of the best candidate, -1 = none       */
  const float* dist2;          /* n_queries */
  const float* second_dist2;   /* n_queries */
} fe_match_result_t;

/* Rows in host memory: only rows [qo[0], qo[G]) and [ro[0], ro[G]) are uploaded. */
int fe_match_descriptors(fe_ctx_t* ctx, const float* query, int64_t query_stride, const int64_t* query_offsets,
                         const float* ref, int64_t ref_stride, const int64_t* ref_offsets, int32_t n_groups,
                         fe_match_result_t* out);
/* Rows already in device memory, e.g. the `descriptors` of fe_process_batch_device.  Runs on the context's stream,
 * behind whatever a batch call queued there: no synchronisation is needed in between. */
int fe_match_descriptors_device(fe_ctx_t* ctx, const float* query, int64_t query_stride, const int64_t* query_offsets,
                                const float* ref, int64_t ref_stride, const int64_t* ref_offsets, int32_t n_groups,
                                fe_match_result_t* out);

/* ---- registration: the planar motion between two scans from their matched keypoints ----------------------------- */
/* Levelling removes roll and pitch, so the motion between two scans is planar: a yaw and an xy translation (keypoint z
 * is the mean height of the visible ring centroids and depends on range; it is not used).  Descriptor matches propose
 * motions, two at a time; every query keypoint of the group votes on each, descriptor or not.  The motion is evaluated
 * to the last bit as follows.
 *
 * Arithmetic.  IEEE double with + - * / sqrt only, each operation rounded on its own (no FMA), in the order written;
 * |x| is exact.  Positions are the x, y floats of fe_point_t keypoints widened to double: p_k of query row k, r_j of
 * reference row j.
 *
 * Inputs.  Query and reference keypoints addressed by absolute row index; best[i] for query row qo[0] + i, the
 * absolute reference row of the group or -1 (fe_match_result_t.best as a match call returns it); query_offsets,
 * ref_offsets and n_groups as in the match call that produced `best`.
 *
 * Correspondences of group g: its query rows k with best >= 0, numbered 0 .. n_c - 1 in ascending row order; q_a is the
 * position of the reference row best of correspondence a.  Pairs (a, b), a < b, are numbered a*n_c - a*(a+1)/2 +
 * (b - a - 1); there are P = n_c*(n_c-1)/2.  With H = min(P, max_hypotheses), hypothesis h in [0, H) is pair
 * floor(h*P / H) (64-bit integers): every pair when P <= H, else H evenly spaced ones.  No random numbers.
 *
 * Motion of a hypothesis (a, b): u = p_b - p_a, v = q_b - q_a, lu = ux*ux + uy*uy, lv = vx*vx + vy*vy.  Rejected when
 * lu < sep2 or lv < sep2 (sep2 = min_separation*min_separation) or |sqrt(lu) - sqrt(lv)| >= 2*inlier_radius (a rigid
 * motion preserves distances).  Otherwise nn = sqrt(lu*lv), c = (ux*vx + uy*vy)/nn, s = (ux*vy - uy*vx)/nn,
 * mp = (p_a + p_b)*0.5 and mq = (q_a + q_b)*0.5 per coordinate, tx = mqx - (c*mpx - s*mpy), ty = mqy - (s*mpx + c*mpy).
 * A motion (c, s, tx, ty) maps a query position to w = ((c*px - s*py) + tx, (s*px + c*py) + ty), in the reference
 * scan's levelled frame.
 *
 * Evaluation of a motion.  Every query row k of the group, best = -1 included, visits the group's reference rows j in
 * ascending order with d = w - r_j, d2 = dx*dx + dy*dy, and takes j when d2 is below its current value, which starts at
 * r2 = inlier_radius*inlier_radius.  A row that took one is an inlier: assoc_k = the last j taken, d2_k its d2 (so the
 * nearest reference row, the lower row on ties, when it lies within the radius); otherwise assoc_k = -1.  Two query rows
 * may share a reference row.  The score is the number of inliers.  The winning hypothesis has the highest score, then
 * the lowest h.
 *
 * Refinement, at most refine_iterations rounds, from the winner's motion and evaluation.  A round stops the refinement
 * when there are fewer than 2 inliers.  Otherwise, with the inliers (k, assoc_k) in ascending k and every sum formed
 * sequentially in that order from 0.0, m their number: mp = (sum p_k) / m, mq = (sum r_assoc_k) / m per coordinate,
 * A = sum((pkx - mpx)*(qx - mqx) + (pky - mpy)*(qy - mqy)), B = sum((pkx - mpx)*(qy - mqy) - (pky - mpy)*(qx - mqx))
 * with q = r_assoc_k, n = sqrt(A*A + B*B).  It stops when n == 0; else the new motion is c = A/n, s = B/n and t as
 * above, and it is evaluated.  A lower score stops the refinement with the old motion kept; otherwise the new motion
 * and evaluation replace the old, and the refinement stops if no assoc_k changed.
 *
 * Outputs per group: pose = (c, s, tx, ty) of the final motion (yaw = atan2(s, c) is the caller's: no libm enters the
 * contract); n_inliers = its score; n_hypotheses = the hypotheses not rejected; rms = sqrt(sum d2_k / n_inliers) over
 * the final inliers in ascending k, 0 without inliers; status 0 when no hypothesis survived (pose = (1, 0, 0, 0),
 * everything else 0, every assoc -1), 1 when n_inliers < min_inliers, 2 = registered.  Per query row: assoc under the
 * final motion, the absolute reference row or -1.
 *
 * Cost: H*n_q*n_r distance tests per group (n_q, n_r its query and reference rows) plus n_q*n_r per refinement round,
 * each about ten double operations; one warp scores a group, one hypothesis per lane.  A scan against a map of 10^5
 * rows with 512 hypotheses is 10^9 tests on a single warp: split such a map into tiles near the scan.
 *
 * Results are context-owned pinned host memory, valid until the next register call; a register call leaves the results
 * of the last batch and match calls alone.  FE_ERR_INVALID (the context stays usable) when an offsets array decreases
 * or has a negative entry, n_groups < 0, a group has 2^24 or more query rows, a keypoint or `best` pointer is NULL
 * while its side has rows, an entry of `best` is neither -1 nor a reference row of its group, or a parameter is out of
 * range: inlier_radius and min_separation finite and > 0, max_hypotheses in [1, 65536], min_inliers >= 1,
 * refine_iterations in [0, 1000].  Empty groups and n_groups = 0 are not errors. */
typedef struct fe_register_params {
  double inlier_radius;       /* m: a mapped query keypoint this close to a reference keypoint is an inlier */
  double min_separation;      /* m: both matches of a hypothesis at least this far apart, in either scan   */
  int32_t max_hypotheses;     /* H at most this many pairs                                                  */
  int32_t min_inliers;        /* status 2 from this many inliers                                            */
  int32_t refine_iterations;  /* least-squares rounds over the inliers                                      */
} fe_register_params_t;

/* 0.5 m, 1.0 m, 512, 16, 4.  min_inliers = 16 is the least count at which no registered pair of the sequence
 * evaluation (DESIGN.md §13) is off by more than 0.5 m or 2 deg: a jittered pole lattice turned by 90 deg, or a
 * symmetric handful of poles turned by 180 deg, scores up to 15 inliers. */
void fe_register_params_default(fe_register_params_t* p);

typedef struct fe_register_result {
  int32_t n_groups;
  int64_t n_queries;
  const double* pose;           /* n_groups x {c, s, tx, ty}                         */
  const double* rms;            /* n_groups                                          */
  const int32_t* n_inliers;     /* n_groups                                          */
  const int32_t* n_hypotheses;  /* n_groups                                          */
  const int32_t* status;        /* n_groups: 0 no hypothesis, 1 too few inliers, 2 ok */
  const int64_t* assoc;         /* n_queries: absolute reference row, -1 = none      */
} fe_register_result_t;

/* Keypoints and `best` in host memory: only rows [qo[0], qo[G]) and [ro[0], ro[G]) are uploaded. */
int fe_register_matches(fe_ctx_t* ctx, const fe_point_t* query_kp, const fe_point_t* ref_kp, const int64_t* best,
                        const int64_t* query_offsets, const int64_t* ref_offsets, int32_t n_groups,
                        const fe_register_params_t* params, fe_register_result_t* out);
/* Keypoints (e.g. those of fe_process_batch_device) and `best` (fe_match_device_best) in device memory.  Runs on the
 * context's stream behind the batch and match calls, with no synchronisation in between.  `best` is checked on the
 * device: a bad entry makes the call return FE_ERR_INVALID after the kernel. */
int fe_register_matches_device(fe_ctx_t* ctx, const fe_point_t* query_kp, const fe_point_t* ref_kp, const int64_t* best,
                               const int64_t* query_offsets, const int64_t* ref_offsets, int32_t n_groups,
                               const fe_register_params_t* params, fe_register_result_t* out);
/* Device address of the `best` array of the last match call (n_queries entries, valid until the next match call), for
 * fe_register_matches_device.  FE_ERR_INVALID before the first match call. */
int fe_match_device_best(fe_ctx_t* ctx, const int64_t** best);

/* CUDA-event stopwatch on the context's stream (the stream every kernel of
 * fe_process_batch_device is launched on): begin, run any number of calls, end -> elapsed ms. */
int fe_timer_begin(fe_ctx_t* ctx);
int fe_timer_end(fe_ctx_t* ctx, float* elapsed_ms);

/* Work counters of the last fe_process_batch_device call (for roofline arithmetic):
 * out[0..9] = points, surface points kept, cropped points, ring clusters (keypoints_full),
 * keypoints, sum of 3DSC neighbours, scans deferred to the large K2, to the large K3, to the
 * global-memory K4a, keypoints whose descriptor was summed out of PCL's order (a single bin with
 * more than 8192 contributions; larger neighbourhoods are otherwise handled exactly, in bin groups). */
int fe_get_batch_stats(fe_ctx_t* ctx, int64_t out[10]);

/* Per-kernel CUDA-event times (ms) of the last device call; names are static strings.  Only collected
 * after fe_enable_stage_timing(ctx, 1) (an event pair around every stage; CUDA-graph replay is
 * bypassed while it is on). */
int fe_enable_stage_timing(fe_ctx_t* ctx, int32_t enable);
int fe_get_stage_times(fe_ctx_t* ctx, int32_t cap, const char** names, float* ms, int32_t* n);

/* ---- one entry point per reference function (host buffers, synchronous) ------------------ */

/* getElevationAngles, src:147-156: overwrites intensity with the elevation angle (deg). */
int fe_get_elevation_angles(fe_ctx_t* ctx, fe_point_t* cloud, int64_t n);

/* rotateCloud, src:159-167 (pcl::transformPointCloud with
 * AngleAxisf(pitch,Y)*AngleAxisf(roll,X)); in place, intensity carried through. */
int fe_rotate_cloud(fe_ctx_t* ctx, fe_point_t* cloud, int64_t n, double roll, double pitch);

/* The 3x3 float rotation rotateCloud applies (row-major), for inspection. */
int fe_rotation_matrix(double roll, double pitch, float m[9]);

/* filterCloud, src:169-183 (three pcl::PassThrough passes): stable crop. */
int fe_filter_cloud(fe_ctx_t* ctx, const fe_point_t* in, int64_t n, fe_point_t* out,
                    int64_t cap, int64_t* n_out);

/* pcl::EuclideanClusterExtraction::extract as called at src:222-229 and src:269-276.
 * cluster c owns indices[cluster_offsets[c] .. cluster_offsets[c+1]) (ascending), clusters in
 * PCL's output order. */
int fe_extract_clusters(fe_ctx_t* ctx, const fe_point_t* cloud, int64_t n, double tolerance,
                        int32_t min_size, int32_t max_size, int32_t* cluster_offsets,
                        int32_t cap_clusters, int32_t* indices, int64_t cap_indices,
                        int32_t* n_clusters);

/* getCylinderSegments, src:261-327: one ring's cloud -> gated centroids + their points. */
int fe_get_cylinder_segments(fe_ctx_t* ctx, const fe_point_t* ring_cloud, int64_t n,
                             fe_point_t* centroids, int64_t cap_centroids, int64_t* n_centroids,
                             fe_point_t* cluster_cloud, int64_t cap_cloud, int64_t* n_cloud);

/* estimateKeypoints, src:185-259: cropped cloud (intensity = elevation) -> keypoints and
 * keypoint_cloud. */
int fe_estimate_keypoints(fe_ctx_t* ctx, const fe_point_t* cloud, int64_t n,
                          fe_point_t* keypoints, int64_t cap_keypoints, int64_t* n_keypoints,
                          fe_point_t* keypoint_cloud, int64_t cap_cloud, int64_t* n_cloud);

/* estimateDescriptors, src:329-355: pcl::ShapeContext3DEstimation of `keypoints` against the
 * search surface `cloud_full`; descriptors is k x 1980 floats. */
int fe_estimate_descriptors(fe_ctx_t* ctx, const fe_point_t* cloud_full, int64_t n,
                            const fe_point_t* keypoints, int64_t k, float* descriptors);

/* concatenateFields, src:119 / feature_extraction_node.h:35-53: pack k keypoints and their
 * descriptors into pcl::PointDescriptor records of FE_RECORD_FLOATS floats (rf zeroed). */
int fe_pack_point_descriptors(const fe_point_t* keypoints, const float* descriptors, int64_t k,
                              float* records);

#ifdef __cplusplus
}
#endif
#endif /* FE_B200_H_ */
