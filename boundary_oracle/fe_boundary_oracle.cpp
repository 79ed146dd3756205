// fe_boundary_oracle.cpp — the CPU oracle's side of the tolerance-boundary report over all ten kinds
// (include/fe_b200.h, fe_enable_boundary_report_all).  TEST INFRASTRUCTURE ONLY, like the oracle it builds on.
//
// oracle/fe_oracle.cpp is compiled into this translation unit unchanged: kinds 0-3 are its own counts
// (process_scan with a boundary eps), and kinds 4-9 are evaluated on its intermediate results where it makes
// each decision — the levelled full cloud of the crop (src:169-183), the cropped cloud the ring windows select
// from (src:195-202), the clusters get_cylinder_segments gates (src:314-316) and the neighbour loop of
// estimate_descriptors after the pcl::utils::equal skip (3dsc.hpp via src:350-353).  Margins use + - * / sqrt in
// double in the order the header gives (built with -ffp-contract=off), so the device's counts must agree exactly.
#include "../oracle/fe_oracle.cpp"

namespace {

const double DEG = 0.017453292519943295;  // pi / 180

// [4] crop box: inside the box grown by eps and within eps of one of its six float limits
int64_t count_crop(const fe_params_t& P, const std::vector<P4>& cloud_full, double eps) {
  const double lo[3] = {(double)(float)P.x_min, (double)(float)P.y_min, (double)(float)P.z_min};
  const double hi[3] = {(double)(float)P.x_max, (double)(float)P.y_max, (double)(float)P.z_max};
  int64_t n = 0;
  for (const P4& p : cloud_full) {
    if (!std::isfinite(p.x) || !std::isfinite(p.y) || !std::isfinite(p.z)) continue;
    const double v[3] = {(double)p.x, (double)p.y, (double)p.z};
    bool inside = true, near = false;
    for (int a = 0; a < 3; a++) {
      inside = inside && v[a] > lo[a] - eps && v[a] < hi[a] + eps;
      near = near || fabs(v[a] - lo[a]) < eps || fabs(v[a] - hi[a]) < eps;
    }
    if (inside && near) n++;
  }
  return n;
}

// [5] ring-window ends: the 17 distinct float limits -16, -14, ..., 16 of src:200-201, as an arc length
int64_t count_ring_windows(const std::vector<P4>& cloud, double eps) {
  int64_t n = 0;
  for (const P4& p : cloud) {
    const float el = p.intensity;
    if (!std::isfinite(el)) continue;
    const double x = p.x, y = p.y, z = p.z;
    const double range = sqrt((x * x + y * y) + z * z);
    double dmin = fabs((double)el + 16.0);
    for (int e = -14; e <= 16; e += 2) dmin = std::min(dmin, fabs((double)el - (double)e));
    if (range * (dmin * DEG) < eps) n++;
  }
  return n;
}

// [6] the diameter gate of every cluster get_cylinder_segments sees, ring by ring as estimate_keypoints runs it
int64_t count_gate(const fe_params_t& P, const std::vector<P4>& cloud, bool use_tree, double eps) {
  int64_t n = 0;
  for (int i = 0; i < 16; ++i) {
    const double ch = (i - 7) * 2 - 1;  // src:200
    std::vector<P4> channel, centroids, cluster_cloud;
    pass_through(cloud, FI, ch - 1.0, ch + 1.0, channel);
    Clusters clusters;
    get_cylinder_segments(P, channel, use_tree, centroids, cluster_cloud, &clusters);
    for (const std::vector<int>& c : clusters) {
      double minx = 1000.0, maxx = -1000.0, miny = 1000.0, maxy = -1000.0;  // src:289-290
      for (int idx : c) {
        const double x = channel[idx].x, y = channel[idx].y;
        if (x < minx) minx = x;
        if (y < miny) miny = y;
        if (x > maxx) maxx = x;
        if (y > maxy) maxy = y;
      }
      const double diameter = pow(pow(maxx - minx, 2) + pow(maxy - miny, 2), 0.5);  // src:314
      if (fabs(diameter - 2 * P.cluster_radius_threshold) < eps) n++;
    }
  }
  return n;
}

// [7-9] the bin edges of every (keypoint, neighbour) pair estimate_descriptors bins: its loop, angle for angle
void count_bins(const fe_params_t& P, const std::vector<P4>& cloud, const std::vector<P4>& keypoints, bool use_tree,
                double eps, int64_t out[3]) {
  if (keypoints.empty()) return;
  const V3 normal = v3(0.0f, 0.0f, 1.0f);
  ShapeContextTables T;
  sc3d_init_compute(P.descriptor_radius, P.descriptor_radius / 10.0, T);
  const float R2f = radius_sq_float(P.descriptor_radius);
  Searcher tree;
  tree.set_input(cloud.data(), (int)cloud.size(), use_tree, /*sorted=*/true);
  std::mt19937 rng_alg(12345u);
  auto rnd = [&]() -> double { return (double)rng_alg() * (1.0 / 4294967296.0); };
  std::vector<Hit> nn;
  for (const P4& in : keypoints) {
    if (!std::isfinite(in.x) || !std::isfinite(in.y) || !std::isfinite(in.z)) continue;
    const size_t neighb_cnt = (size_t)tree.radius(in, R2f, nn);
    if (neighb_cnt == 0) continue;
    const V3 origin = v3(in.x, in.y, in.z);
    V3 x_axis;  // the normal is (0, 0, 1): estimate_descriptors' first branch
    x_axis.x = static_cast<float>(rnd());
    x_axis.y = static_cast<float>(rnd());
    x_axis.z = static_cast<float>(rnd());
    x_axis.z = -(normal.x * x_axis.x + normal.y * x_axis.y) / normal.z;
    eigen32_normalize(x_axis);
    for (size_t ne = 0; ne < neighb_cnt; ne++) {
      if (pcl_utils_equal(nn[ne].d2, 0.0f)) continue;
      const P4& nbp = cloud[nn[ne].idx];
      const V3 neighbour = v3(nbp.x, nbp.y, nbp.z);
      const float r = sqrtf(nn[ne].d2);
      const V3 po = sub(neighbour, origin);
      const float lambda = eigen_dot(normal, po);
      V3 proj = v3(neighbour.x - lambda * normal.x, neighbour.y - lambda * normal.y, neighbour.z - lambda * normal.z);
      proj = sub(proj, origin);
      eigen32_normalize(proj);
      const V3 cross = eigen_cross(x_axis, proj);
      float phi = pcl_rad2deg(atan2f(eigen_norm(cross), eigen_dot(x_axis, proj)));
      phi = eigen_dot(cross, normal) < 0.f ? (360.0f - phi) : phi;
      V3 no = sub(neighbour, origin);
      eigen32_normalize(no);
      float theta = eigen_dot(normal, no);
      theta = pcl_rad2deg(acosf(std::min(1.0f, std::max(-1.0f, theta))));
      double dr = fabs((double)r - (double)T.radii[1]), dt = fabs((double)theta - (double)T.theta[1]);
      double dp = fabs((double)phi - (double)T.phi[0]);
      for (int a = 2; a <= 14; a++) dr = std::min(dr, fabs((double)r - (double)T.radii[a]));
      for (int a = 2; a <= 10; a++) dt = std::min(dt, fabs((double)theta - (double)T.theta[a]));
      for (int a = 1; a <= 12; a++) dp = std::min(dp, fabs((double)phi - (double)T.phi[a]));
      const double rho = sqrt((double)po.x * po.x + (double)po.y * po.y);
      if (dr < eps) out[0]++;
      if ((double)r * (dt * DEG) < eps) out[1]++;
      if (rho == 0.0 || rho * (dp * DEG) < eps) out[2]++;  // straight above or below: any horizontal move decides
    }
  }
}

void count_scan(const fe_params_t& P, const P4* pts, int64_t n, double roll, double pitch, bool use_tree, double eps,
                int64_t out[FE_BOUNDARY_KINDS]) {
  ScanResult R;
  process_scan(P, pts, n, roll, pitch, use_tree, false, R, eps);  // kinds 0-3, the clouds and the keypoints
  for (int k = 0; k < 4; k++) out[k] = R.bnd.n[k];
  out[4] = count_crop(P, R.cloud_full, eps);
  out[5] = count_ring_windows(R.cloud, eps);
  out[6] = count_gate(P, R.cloud, use_tree, eps);
  out[7] = out[8] = out[9] = 0;
  if (P.estimate_descriptors) count_bins(P, R.cloud_full, R.keypoints, use_tree, eps, out + 7);
}

}  // namespace

extern "C" {

// boundary_counts[FE_BOUNDARY_KINDS * s + k] = the count of kind k of scan s within eps_m (include/fe_b200.h).
// mode: 0 = brute force, 1 = KD-tree (the oracle's two search back ends).
int feo_process_batch_boundary_all(const fe_params_t* P, const fe_point_t* points, const int64_t* scan_offsets,
                                   const double* roll_pitch, int32_t n_scans, int32_t mode, int32_t n_threads,
                                   double eps_m, int64_t* boundary_counts) {
  if (!P || n_scans < 0 || (n_scans > 0 && (!points || !scan_offsets || !roll_pitch || !boundary_counts))) return FE_ERR_INVALID;
  if (n_threads < 1) n_threads = 1;
  std::atomic<int> next(0);
  auto worker = [&]() {
    for (;;) {
      const int s = next.fetch_add(1);
      if (s >= n_scans) break;
      count_scan(*P, points + scan_offsets[s], scan_offsets[s + 1] - scan_offsets[s], roll_pitch[2 * s],
                 roll_pitch[2 * s + 1], mode == 1, eps_m, boundary_counts + (size_t)FE_BOUNDARY_KINDS * s);
    }
  };
  if (n_threads == 1) worker();
  else {
    std::vector<std::thread> th;
    for (int t = 0; t < n_threads; t++) th.emplace_back(worker);
    for (auto& t : th) t.join();
  }
  return FE_OK;
}

}  // extern "C"
