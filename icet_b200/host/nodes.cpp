// icet_b200/host/nodes.cpp -- host side of include/icet_nodes.h: the reference's ROS callbacks
// (src/odometry.cpp:38-168, src/simpleMapMaker.cpp:78-240) reduced to what the host still has to do: hand the cloud
// to the device, draw the map sample, read the published values back.
#include "icet_nodes.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <numeric>

namespace {
void check(int rc) {
  if (rc < 0) throw std::runtime_error(std::string("ICET node: ") + icet_b200_last_error());
}
}  // namespace

OdometryNode::OdometryNode(int max_points, float minD, int run_length, int numBinsPhi, int numBinsTheta, int device)
    : OdometryNode(max_points, minD, run_length, numBinsPhi, numBinsTheta, device, true, 0.f, 0.f) {}

OdometryNode::OdometryNode(int max_points, float minD, int run_length, int numBinsPhi, int numBinsTheta, int device,
                           bool chain, float trans_thresh, float rot_thresh) {
  X0.resize(6);
  X0.setZero();                      // odometry.cpp:28-29
  X_homo = Eigen::MatrixXf::Zero(4, 4);
  for (int k = 0; k < 4; k++) X_homo(k, k) = 1.f;  // Matrix4f::Identity(), odometry.cpp:184
  check(icet_b200_create(device, &ctx_));
  icet_b200_params p;
  std::memset(&p, 0, sizeof(p));
  p.runlen = run_length;
  p.bins_phi = numBinsPhi;
  p.bins_theta = numBinsTheta;
  p.n = 25;
  p.thresh = 0.1f;
  p.buff = 0.1f;
  icet_b200_odometry_params op;
  std::memset(&op, 0, sizeof(op));
  op.min_range = minD;
  op.chain_x0 = chain ? 1 : 0;
  op.rate_hz = 10.f;                 // "assumes 10Hz LIDAR sensor", odometry.cpp:133
  op.guard_trans = trans_thresh;
  op.guard_rot = rot_thresh;
  const int rc = icet_b200_node_create(ctx_, &p, &op, max_points, nullptr, nullptr, &node_);
  if (rc < 0) {
    const std::string msg = std::string("ICET node: ") + icet_b200_last_error();
    icet_b200_destroy(ctx_);
    ctx_ = nullptr;
    throw std::runtime_error(msg);
  }
}

OdometryNode::~OdometryNode() {
  if (node_) icet_b200_node_destroy(node_);
  if (ctx_) icet_b200_destroy(ctx_);
}

bool OdometryNode::pointcloudCallback(const Eigen::MatrixXf& pcl_matrix, NodeOutput* out) {
  frameCount++;
  if (pcl_matrix.rows() > 0 && pcl_matrix.cols() != 3) throw std::runtime_error("ICET node: cloud must be N x 3");
  icet_b200_result res;
  icet_b200_pose pose;
  const int n = (int)pcl_matrix.rows();
  // Eigen::MatrixXf is column-major: data() is the x | y | z plane layout of the C ABI
  const int rc = icet_b200_node_push(node_, pcl_matrix.data(), n, n, &res, &pose);
  check(rc);
  if (rc == 0) return false;
  for (int k = 0; k < 6; k++) X0[k] = res.X[k];
  for (int a = 0; a < 4; a++)
    for (int b = 0; b < 4; b++) X_homo(a, b) = pose.X_homo[4 * a + b];
  if (!out) return true;
  out->X.resize(6);
  out->pred_stds.resize(6);
  for (int k = 0; k < 6; k++) {
    out->X[k] = pose.X[k];
    out->pred_stds[k] = res.pred_stds[k];
    out->twist[k] = pose.twist[k];
  }
  out->X_homo = X_homo;
  for (int k = 0; k < 3; k++) out->position[k] = pose.position[k];
  for (int k = 0; k < 4; k++) out->orientation[k] = pose.orientation[k];
  for (int k = 0; k < 36; k++) out->covariance[k] = 0.0;                        // odometry.cpp:122-125
  for (int k = 0; k < 6; k++) out->covariance[7 * k] = pose.covariance_diag[k];  // :126-131
  out->points = pose.n_points;
  out->guarded = pose.guarded != 0;
  return true;
}

icet_b200_keyframe_policy KeyframeOdometryNode::defaultPolicy() {
  icet_b200_keyframe_policy kp;
  std::memset(&kp, 0, sizeof(kp));
  kp.max_trans = 1.f;
  kp.max_rot = 0.1f;
  kp.min_overlap = 0.5f;
  kp.max_interval = 10;
  return kp;
}

KeyframeOdometryNode::KeyframeOdometryNode(int max_points, float minD, int run_length, int numBinsPhi, int numBinsTheta,
                                           const icet_b200_keyframe_policy* policy, int device, int map_keyframes) {
  X_homo = Eigen::MatrixXf::Zero(4, 4);
  for (int k = 0; k < 4; k++) X_homo(k, k) = 1.f;
  check(icet_b200_create(device, &ctx_));
  icet_b200_params p;
  std::memset(&p, 0, sizeof(p));
  p.runlen = run_length;
  p.bins_phi = numBinsPhi;
  p.bins_theta = numBinsTheta;
  p.n = 25;
  p.thresh = 0.1f;
  p.buff = 0.1f;
  icet_b200_odometry_params op;
  std::memset(&op, 0, sizeof(op));
  op.min_range = minD;
  op.chain_x0 = 1;
  op.rate_hz = 10.f;
  const icet_b200_keyframe_policy kp = policy ? *policy : defaultPolicy();
  const int rc = map_keyframes == 0
                     ? icet_b200_kfnode_create(ctx_, &p, &op, &kp, max_points, nullptr, nullptr, &node_)
                     : icet_b200_kfnode_create_local_map(ctx_, &p, &op, &kp, map_keyframes, max_points, nullptr,
                                                         nullptr, &node_);
  if (rc < 0) {
    const std::string msg = std::string("ICET node: ") + icet_b200_last_error();
    icet_b200_destroy(ctx_);
    ctx_ = nullptr;
    throw std::runtime_error(msg);
  }
}

KeyframeOdometryNode::~KeyframeOdometryNode() {
  if (node_) icet_b200_kfnode_destroy(node_);
  if (ctx_) icet_b200_destroy(ctx_);
}

Eigen::MatrixXf KeyframeOdometryNode::localMap() {
  int32_t n = 0;
  check(icet_b200_kfnode_local_map_host(node_, nullptr, 0, &n));
  Eigen::MatrixXf out(n, 3);
  if (n > 0) check(icet_b200_kfnode_local_map_host(node_, out.data(), n, &n));
  return out;
}

bool KeyframeOdometryNode::pointcloudCallback(const Eigen::MatrixXf& pcl_matrix, NodeOutput* out, KeyframeInfo* info) {
  frameCount++;
  if (pcl_matrix.rows() > 0 && pcl_matrix.cols() != 3) throw std::runtime_error("ICET node: cloud must be N x 3");
  icet_b200_result res;
  icet_b200_pose pose;
  icet_b200_kf_info ki;
  const int n = (int)pcl_matrix.rows();
  const int rc = icet_b200_kfnode_push(node_, pcl_matrix.data(), n, n, &res, &pose, &ki);
  check(rc);
  if (rc == 0) return false;
  for (int a = 0; a < 4; a++)
    for (int b = 0; b < 4; b++) X_homo(a, b) = pose.X_homo[4 * a + b];
  if (info) {
    info->keyframe = ki.keyframe;
    info->promoted = ki.promoted != 0;
    info->reason = ki.reason;
    for (int k = 0; k < 6; k++) info->x0[k] = ki.x0[k];
  }
  if (!out) return true;
  out->X.resize(6);
  out->pred_stds.resize(6);
  for (int k = 0; k < 6; k++) {
    out->X[k] = pose.X[k];
    out->pred_stds[k] = res.pred_stds[k];
    out->twist[k] = pose.twist[k];
  }
  out->X_homo = X_homo;
  for (int k = 0; k < 3; k++) out->position[k] = pose.position[k];
  for (int k = 0; k < 4; k++) out->orientation[k] = pose.orientation[k];
  for (int k = 0; k < 36; k++) out->covariance[k] = 0.0;
  for (int k = 0; k < 6; k++) out->covariance[7 * k] = pose.covariance_diag[k];
  out->points = pose.n_points;
  out->guarded = false;
  return true;
}

MapMakerNode::MapMakerNode(int max_points, int map_size, int downsampleSize, int device)
    : OdometryNode(max_points, 0.2f, 12, 24, 75, device, false, 0.3f, 0.3f), map_size_(map_size),
      downsampleSize_(downsampleSize) {
  check(icet_b200_map_create(ctx_, map_size, &q_));
}

MapMakerNode::~MapMakerNode() {
  if (q_) icet_b200_map_destroy(q_);
}

bool MapMakerNode::pointcloudCallback(const Eigen::MatrixXf& pcl_matrix, NodeOutput* out) {
  NodeOutput tmp;
  NodeOutput* o = out ? out : &tmp;
  if (!OdometryNode::pointcloudCallback(pcl_matrix, o)) return false;
  for (int k = 0; k < 6; k++) X0[k] = 0.f;  // simpleMapMaker.cpp:124
  // downsample pcl_matrix before passing it to the map queue (simpleMapMaker.cpp:149-159): shuffle 0..rows-1 with
  // the node's generator and keep the first downsampleSize (clipped to the rows that exist)
  const std::size_t originalSize = (std::size_t)o->points;
  std::vector<int> indices(originalSize);
  std::iota(indices.begin(), indices.end(), 0);
  std::shuffle(indices.begin(), indices.end(), gen);
  indices.resize(std::min<std::size_t>((std::size_t)downsampleSize_, originalSize));
  lastSample = indices;
  const float* scan = nullptr;
  const int32_t* n_dev = nullptr;
  int32_t ld = 0;
  check(icet_b200_node_current_scan(node_, &scan, &n_dev, &ld));
  const icet_b200_result* res_dev = nullptr;
  check(icet_b200_node_last_result(node_, &res_dev));
  // q.add_new_scan(downsampledMatrix, trans, rot_mat) with trans / rot_mat from the guarded X (:128-160)
  check(icet_b200_map_add_scan_device(q_, scan, (int32_t)originalSize, ld, n_dev, indices.data(), (int32_t)indices.size(),
                                      res_dev->X, trans_thresh, rot_thresh));
  return true;
}

Eigen::MatrixXf MapMakerNode::getQueue() {
  std::vector<float> planes((std::size_t)3 * map_size_);
  int32_t rows = 0;
  check(icet_b200_map_get(q_, planes.data(), map_size_, &rows));
  Eigen::MatrixXf m(rows, 3);
  for (int c = 0; c < 3; c++)
    for (int i = 0; i < rows; i++) m(i, c) = planes[(std::size_t)c * map_size_ + i];
  return m;
}

// ---------------------------------------------------------------------------------------------------------------------
ScanMatcherNode::ScanMatcherNode(int max_points, int run_length, int numBinsPhi, int numBinsTheta, int device)
    : OdometryNode(max_points, -1.f, run_length, numBinsPhi, numBinsTheta, device, false, 0.f, 0.f) {
  snailTrail = Eigen::MatrixXf::Zero(1, 3);  // scanMatcher.cpp:25-26
}

ScanMatcherNode::~ScanMatcherNode() {}

bool ScanMatcherNode::pointcloudCallback(const Eigen::MatrixXf& pcl_matrix, NodeOutput* out) {
  if (pcl_matrix.rows() == 0) return false;  // "Received an empty point cloud" (:41-44)
  NodeOutput tmp;
  NodeOutput* o = out ? out : &tmp;
  if (!OdometryNode::pointcloudCallback(pcl_matrix, o)) return false;  // first cloud (:47-51)
  for (int k = 0; k < 6; k++) X0[k] = 0.f;                              // :58-62
  const int n = (int)pcl_matrix.rows();
  const float* scan = nullptr;
  const int32_t* n_dev = nullptr;
  int32_t ld = 0;
  check(icet_b200_node_current_scan(node_, &scan, &n_dev, &ld));
  const icet_b200_result* res_dev = nullptr;
  check(icet_b200_node_last_result(node_, &res_dev));
  // scan2_in_scan1_frame = (pcl_matrix * rot_mat.inverse()).rowwise() - trans   (:73)
  // Eigen::MatrixXf is column-major: data() is the plane layout the C ABI writes
  scan2_in_scan1_frame.resize(n, 3);
  check(icet_b200_transform_cloud(ctx_, scan, n, ld, res_dev->X, 0, scan2_in_scan1_frame.data(), n));
  // snail trail (:76-80): a handful of rows, on the host like the reference.  rot_mat.inverse() by cofactors.
  const float phi = o->X[3], th = o->X[4], psi = o->X[5];
  const float sph = std::sin(phi), cph = std::cos(phi), sth = std::sin(th), cth = std::cos(th), sps = std::sin(psi),
              cps = std::cos(psi);
  const float R[9] = {cth * cps, sps * cph + sph * sth * cps, sph * sps - sth * cph * cps,
                      -sps * cth, cph * cps - sph * sth * sps, sph * cps + sth * sps * cph,
                      sth, -sph * cth, cph * cth};  // utils::R, src/utils.cpp:144-152
  float Ri[9];
  {
    const float c00 = R[4] * R[8] - R[5] * R[7], c10 = R[5] * R[6] - R[3] * R[8], c20 = R[3] * R[7] - R[4] * R[6];
    const float id = 1.0f / (c00 * R[0] + c10 * R[1] + c20 * R[2]);
    Ri[0] = c00 * id; Ri[3] = c10 * id; Ri[6] = c20 * id;
    Ri[1] = (R[2] * R[7] - R[1] * R[8]) * id; Ri[4] = (R[0] * R[8] - R[2] * R[6]) * id; Ri[7] = (R[1] * R[6] - R[0] * R[7]) * id;
    Ri[2] = (R[1] * R[5] - R[2] * R[4]) * id; Ri[5] = (R[2] * R[3] - R[0] * R[5]) * id; Ri[8] = (R[0] * R[4] - R[1] * R[3]) * id;
  }
  const long rows = snailTrail.rows();
  Eigen::MatrixXf next = Eigen::MatrixXf::Zero(rows + 1, 3);
  for (long i = 0; i < rows; i++)
    for (int c = 0; c < 3; c++)
      next(i, c) = snailTrail(i, 0) * Ri[c] + snailTrail(i, 1) * Ri[3 + c] + snailTrail(i, 2) * Ri[6 + c] - o->X[c];
  snailTrail = next;  // new row (0, 0, 0) appended (:77-80)
  return true;
}
