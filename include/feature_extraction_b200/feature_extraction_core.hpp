// feature_extraction_core.hpp — C++ host-side mirror of the reference's FeatureExtractionNode for
// the per-scan path (reference include/feature_extraction/feature_extraction_node.h:58-132,
// src/feature_extraction_node.cpp:147-355), header-only over the C-ABI of fe_b200.h.
//
// Same member-function names, parameter members and early-return behaviour as the reference; the
// pcl::PointCloud<pcl::PointXYZI>::Ptr arguments become std::vector<fe_point_t> (x, y, z,
// intensity), because PCL/ROS types are the host shell's business, not this library's.
// Every method runs sm_100a kernels through libfe_b200.so; there is no CPU fallback.
#ifndef FEATURE_EXTRACTION_B200_CORE_HPP_
#define FEATURE_EXTRACTION_B200_CORE_HPP_

#include <stdexcept>
#include <string>
#include <vector>

#include "../fe_b200.h"

namespace feature_extraction_b200 {

typedef fe_point_t Point;                 // pcl::PointXYZI            (.h:66)
typedef std::vector<Point> PointCloud;    // pcl::PointCloud<Point>    (.h:67)
typedef std::vector<float> DescriptorCloud;  // K x 1980 floats: pcl::PointCloud<pcl::ShapeContext1980> (.h:75-76)
typedef std::vector<std::vector<int> > IndicesClusters;  // std::vector<pcl::PointIndices> (.h:63)

class FeatureExtractionCore {
 public:
  // -- the class variables of feature_extraction_node.h:115-127 ---------------------------------
  double zMin, zMax, xMin, xMax, yMin, yMax;
  double roll, pitch;
  bool levelCloud;
  double clusterTolerance;
  int clusterMinCount;
  int clusterMaxCount;
  double clusterRadiusThreshold;
  int detectionChannelThreshold;
  double descriptorRadius;
  bool descriptorEstimation;

  // constructor defaults of src:9-34 (roll/pitch start at 0: the reference leaves them
  // uninitialised until the first IMU message, SURVEY.md §3.1)
  explicit FeatureExtractionCore(int device = 0) : ctx_(nullptr), device_(device) {
    fe_params_t p;
    fe_params_node_default(&p);
    fromParams(p);
    levelCloud = true;
    roll = pitch = 0.0;
    check(fe_create(device_, &p, nullptr, &ctx_), "fe_create");
    applied_ = p;
  }
  ~FeatureExtractionCore() { fe_destroy(ctx_); }
  FeatureExtractionCore(const FeatureExtractionCore&) = delete;
  FeatureExtractionCore& operator=(const FeatureExtractionCore&) = delete;

  // imuCallback, src:57-70, minus the tf quaternion -> RPY conversion (host shell)
  void setImuRollPitch(double tmproll, double imuPitch) {
    if (levelCloud) { roll = tmproll - 3.14159265358979323846; pitch = imuPitch; }
    else { roll = 0.0; pitch = 0.0; }
  }

  void getElevationAngles(PointCloud& cloud) {  // src:147-156
    sync();
    check(fe_get_elevation_angles(ctx_, cloud.data(), (int64_t)cloud.size()), "getElevationAngles");
  }
  void rotateCloud(PointCloud& cloud) {  // src:159-167
    sync();
    check(fe_rotate_cloud(ctx_, cloud.data(), (int64_t)cloud.size(), roll, pitch), "rotateCloud");
  }
  void filterCloud(PointCloud& cloud) {  // src:169-183 (in place, like the reference)
    sync();
    PointCloud out(cloud.size());
    int64_t n = 0;
    check(fe_filter_cloud(ctx_, cloud.data(), (int64_t)cloud.size(), out.data(), (int64_t)out.size(), &n), "filterCloud");
    out.resize((size_t)n);
    cloud.swap(out);
  }
  // pcl::EuclideanClusterExtraction as configured at src:269-276 / 222-229
  void extractClusters(const PointCloud& cloud, double tolerance, int minSize, int maxSize, IndicesClusters& clusters) {
    sync();
    clusters.clear();
    std::vector<int32_t> offs(cloud.size() + 2), idx(cloud.size() + 1);
    int32_t nc = 0;
    check(fe_extract_clusters(ctx_, cloud.data(), (int64_t)cloud.size(), tolerance, minSize, maxSize, offs.data(),
                              (int32_t)cloud.size() + 1, idx.data(), (int64_t)idx.size(), &nc), "extractClusters");
    for (int c = 0; c < nc; c++) clusters.push_back(std::vector<int>(idx.begin() + offs[c], idx.begin() + offs[c + 1]));
  }
  void getCylinderSegments(const PointCloud& cloud, PointCloud& keypoints, PointCloud& keypoint_cloud) {  // src:261-327
    sync();
    if (cloud.size() <= 0) return;
    PointCloud kp(cloud.size()), kc(cloud.size());
    int64_t n1 = 0, n2 = 0;
    check(fe_get_cylinder_segments(ctx_, cloud.data(), (int64_t)cloud.size(), kp.data(), (int64_t)kp.size(), &n1,
                                   kc.data(), (int64_t)kc.size(), &n2), "getCylinderSegments");
    keypoints.insert(keypoints.end(), kp.begin(), kp.begin() + n1);
    keypoint_cloud.insert(keypoint_cloud.end(), kc.begin(), kc.begin() + n2);
  }
  void estimateKeypoints(const PointCloud& cloud, PointCloud& keypoints, PointCloud& keypoint_cloud) {  // src:185-259
    sync();
    PointCloud kp(2 * cloud.size() + 1), kc(2 * cloud.size() + 1);
    int64_t n1 = 0, n2 = 0;
    check(fe_estimate_keypoints(ctx_, cloud.data(), (int64_t)cloud.size(), kp.data(), (int64_t)kp.size(), &n1,
                                kc.data(), (int64_t)kc.size(), &n2), "estimateKeypoints");
    keypoints.insert(keypoints.end(), kp.begin(), kp.begin() + n1);
    keypoint_cloud.insert(keypoint_cloud.end(), kc.begin(), kc.begin() + n2);
  }
  void estimateDescriptors(const PointCloud& cloud, const PointCloud& keypoints, DescriptorCloud& descriptors) {  // src:329-355
    sync();
    if (keypoints.size() <= 0) return;
    descriptors.assign(keypoints.size() * (size_t)FE_DESC_LEN, 0.0f);
    check(fe_estimate_descriptors(ctx_, cloud.data(), (int64_t)cloud.size(), keypoints.data(), (int64_t)keypoints.size(),
                                  descriptors.data()), "estimateDescriptors");
  }

  // The span of cloudCallback between src:83 and src:117 for one scan, fused on the device.
  // `cloud_full` is the converted PointCloud2 (sensor frame); outputs as the reference publishes.
  void processScan(const PointCloud& cloud_full, PointCloud& keypoints, DescriptorCloud& descriptors) {
    sync();
    const int64_t offs[2] = {0, (int64_t)cloud_full.size()};
    const double rp[2] = {roll, pitch};
    fe_batch_result_t r;
    check(fe_process_batch(ctx_, cloud_full.data(), offs, rp, 1, &r), "processScan");
    keypoints.assign(r.keypoints, r.keypoints + r.n_keypoints);
    descriptors.clear();
    if (r.descriptors) descriptors.assign(r.descriptors, r.descriptors + r.n_keypoints * FE_DESC_LEN);
  }

  // As processScan, but the ~features message body leaves the device finished: one
  // FE_RECORD_FLOATS-float pcl::PointDescriptor record per keypoint (concatenateFields, src:119).
  void processScanRecords(const PointCloud& cloud_full, PointCloud& keypoints, std::vector<float>& pt_descriptors) {
    sync();
    check(fe_enable_record_output(ctx_, 1), "processScanRecords");
    const int64_t offs[2] = {0, (int64_t)cloud_full.size()};
    const double rp[2] = {roll, pitch};
    fe_batch_result_t r;
    const int st = fe_process_batch(ctx_, cloud_full.data(), offs, rp, 1, &r);
    fe_enable_record_output(ctx_, 0);
    check(st, "processScanRecords");
    keypoints.assign(r.keypoints, r.keypoints + r.n_keypoints);
    pt_descriptors.clear();
    if (r.descriptors) pt_descriptors.assign(r.descriptors, r.descriptors + r.n_keypoints * FE_RECORD_FLOATS);
  }

  // The planar motion of scan `query` against scan `reference` (fe_register_matches, one group): `best` as the match
  // call returned it for these keypoints, one entry per query keypoint.  pose = {c, s, tx, ty} maps query xy into the
  // reference scan's levelled frame; returns the status (0 no hypothesis, 1 too few inliers, 2 registered).
  int registerMatches(const PointCloud& query, const PointCloud& reference, const std::vector<int64_t>& best,
                      double pose[4], int* nInliers = nullptr, const fe_register_params_t* params = nullptr) {
    if (best.size() != query.size()) throw std::runtime_error("registerMatches: best needs one entry per query keypoint");
    fe_register_params_t p;
    fe_register_params_default(&p);
    const int64_t qo[2] = {0, (int64_t)query.size()};
    const int64_t ro[2] = {0, (int64_t)reference.size()};
    fe_register_result_t r;
    check(fe_register_matches(ctx_, query.data(), reference.data(), best.data(), qo, ro, 1, params ? params : &p, &r),
          "registerMatches");
    for (int i = 0; i < 4; i++) pose[i] = r.pose[i];
    if (nInliers) *nInliers = r.n_inliers[0];
    return r.status[0];
  }

  // Poses of one sequence of scans (fe_odometry, one sequence): `keypoints` concatenated in scan order with
  // keypointOffsets (n_scans + 1 entries), `best` as the match call returned it for scan s against s - 1 (one entry per
  // keypoint from keypointOffsets[1]).  poses gets n_scans x {c, s, tx, ty}, scan xy into the first scan's frame;
  // sources (if given) 0 first scan, 1 registered, 2 predicted.
  void odometry(const PointCloud& keypoints, const std::vector<int64_t>& keypointOffsets, const std::vector<int64_t>& best,
                std::vector<double>& poses, std::vector<int32_t>* sources = nullptr, int window = FE_ODOMETRY_WINDOW_DEFAULT,
                const fe_register_params_t* params = nullptr) {
    if (keypointOffsets.empty()) throw std::runtime_error("odometry: keypointOffsets needs n_scans + 1 entries");
    const int32_t B = (int32_t)keypointOffsets.size() - 1;
    if (keypointOffsets[B] > (int64_t)keypoints.size()) throw std::runtime_error("odometry: keypointOffsets exceed the keypoints");
    if ((int64_t)best.size() != (B >= 2 ? keypointOffsets[B] - keypointOffsets[1] : 0))
      throw std::runtime_error("odometry: best needs one entry per keypoint from keypointOffsets[1]");
    fe_register_params_t p;
    fe_register_params_default(&p);
    const int64_t so[2] = {0, B};
    fe_odometry_result_t r;
    check(fe_odometry(ctx_, keypoints.data(), keypointOffsets.data(), B, best.data(), so, 1, window, params ? params : &p, &r),
          "odometry");
    poses.assign(r.pose, r.pose + 4 * (int64_t)B);
    if (sources) sources->assign(r.source, r.source + B);
  }

  // Loop closures of one sequence of scans (fe_loop_closures, one sequence): `keypoints` and `descriptors`
  // (FE_DESC_LEN floats a keypoint) concatenated in scan order with keypointOffsets (n_scans + 1 entries).  loopScans
  // gets, per scan, the earlier scan it sees again or -1; poses n_scans x {c, s, tx, ty}, scan xy into that scan's
  // frame ((1, 0, 0, 0) without a loop).
  void loopClosures(const PointCloud& keypoints, const std::vector<float>& descriptors,
                    const std::vector<int64_t>& keypointOffsets, std::vector<int32_t>& loopScans, std::vector<double>& poses,
                    const fe_loop_params_t* loopParams = nullptr, const fe_register_params_t* params = nullptr) {
    if (keypointOffsets.empty()) throw std::runtime_error("loopClosures: keypointOffsets needs n_scans + 1 entries");
    const int32_t B = (int32_t)keypointOffsets.size() - 1;
    if (keypointOffsets[B] > (int64_t)keypoints.size() || keypointOffsets[B] * FE_DESC_LEN > (int64_t)descriptors.size())
      throw std::runtime_error("loopClosures: keypointOffsets exceed the keypoints or descriptors");
    fe_register_params_t p;
    fe_register_params_default(&p);
    fe_loop_params_t lp;
    fe_loop_params_default(&lp);
    const int64_t so[2] = {0, B};
    fe_loop_result_t r;
    check(fe_loop_closures(ctx_, keypoints.data(), descriptors.data(), FE_DESC_LEN, keypointOffsets.data(), B, so, 1,
                           loopParams ? loopParams : &lp, params ? params : &p, &r),
          "loopClosures");
    loopScans.assign(r.loop_scan, r.loop_scan + B);
    poses.assign(r.pose, r.pose + 4 * (int64_t)B);
  }

  fe_ctx_t* context() { return ctx_; }

 private:
  fe_ctx_t* ctx_;
  int device_;
  fe_params_t applied_;

  void fromParams(const fe_params_t& p) {
    xMin = p.x_min; xMax = p.x_max; yMin = p.y_min; yMax = p.y_max; zMin = p.z_min; zMax = p.z_max;
    clusterTolerance = p.cluster_tolerance; clusterMinCount = p.cluster_min_count; clusterMaxCount = p.cluster_max_count;
    clusterRadiusThreshold = p.cluster_radius_threshold; detectionChannelThreshold = p.number_detection_channels;
    descriptorEstimation = p.estimate_descriptors != 0; descriptorRadius = p.descriptor_radius;
  }
  fe_params_t toParams() const {
    fe_params_t p;
    p.x_min = xMin; p.x_max = xMax; p.y_min = yMin; p.y_max = yMax; p.z_min = zMin; p.z_max = zMax;
    p.cluster_tolerance = clusterTolerance; p.cluster_min_count = clusterMinCount; p.cluster_max_count = clusterMaxCount;
    p.cluster_radius_threshold = clusterRadiusThreshold; p.number_detection_channels = detectionChannelThreshold;
    p.estimate_descriptors = descriptorEstimation ? 1 : 0; p.descriptor_radius = descriptorRadius;
    return p;
  }
  // push changed members to the device-side parameter block (the reference reads members directly)
  void sync() {
    const fe_params_t p = toParams();
    if (p.x_min != applied_.x_min || p.x_max != applied_.x_max || p.y_min != applied_.y_min || p.y_max != applied_.y_max ||
        p.z_min != applied_.z_min || p.z_max != applied_.z_max || p.cluster_tolerance != applied_.cluster_tolerance ||
        p.cluster_min_count != applied_.cluster_min_count || p.cluster_max_count != applied_.cluster_max_count ||
        p.cluster_radius_threshold != applied_.cluster_radius_threshold ||
        p.number_detection_channels != applied_.number_detection_channels ||
        p.estimate_descriptors != applied_.estimate_descriptors || p.descriptor_radius != applied_.descriptor_radius) {
      check(fe_set_params(ctx_, &p), "fe_set_params");
      applied_ = p;
    }
  }
  void check(int st, const char* what) {
    if (st != FE_OK) throw std::runtime_error(std::string(what) + ": " + (ctx_ ? fe_last_error(ctx_) : "fe_b200 error ") + " (status " + std::to_string(st) + ")");
  }
};

}  // namespace feature_extraction_b200
#endif
