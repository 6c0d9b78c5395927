/*
 * include/icet_nodes.h -- the reference's two ROS nodes without ROS, over the C ABI (include/icet_b200.h,
 * "callers either side of the path"; SURVEY.md 8f rows N1, N2).
 *
 *   OdometryNode::pointcloudCallback   reference src/odometry.cpp:38-168
 *   MapMakerNode::pointcloudCallback   reference src/simpleMapMaker.cpp:78-240   (+ EigenQueue, :18-58)
 *   ScanMatcherNode::pointcloudCallback reference src/scanMatcher.cpp:30-112
 *
 * A ROS wrapper only has to convert sensor_msgs::PointCloud2 to the Eigen::MatrixXf the reference's
 * convertPCLtoEigen produces (odometry.cpp:186-192) and to copy the fields of NodeOutput into nav_msgs::Odometry /
 * geometry_msgs::TransformStamped (odometry.cpp:104-157).  Everything between -- min-range filter, registration,
 * seeding of the next registration, pose accumulation, map re-expression -- runs on the GPU; prev_pcl_matrix, X0 and
 * X_homo live in device memory.
 */
#ifndef ICET_NODES_H
#define ICET_NODES_H

#include <Eigen/Dense>
#include <random>
#include <stdexcept>
#include <string>
#include <vector>

#include "icet_b200.h"

struct NodeOutput {
  Eigen::VectorXf X;          // it.X          (after the divergence guard for MapMakerNode)
  Eigen::VectorXf pred_stds;  // it.pred_stds
  Eigen::MatrixXf X_homo;     // 4 x 4 accumulated transform
  float position[3];          // odom.pose.pose.position           odometry.cpp:110-112
  float orientation[4];       // quaternion x, y, z, w             odometry.cpp:114-119
  double covariance[36];      // odom.pose.covariance              odometry.cpp:122-131
  float twist[6];             // odom.twist.twist linear|angular   odometry.cpp:134-139
  int points;                 // rows of the filtered current scan
  bool guarded;               // simpleMapMaker.cpp:128-137 fired
};

class OdometryNode {
 public:
  // the constants of the reference node: minD = 2 (:57), run_length = 7, 24 x 75 bins (:73-75)
  explicit OdometryNode(int max_points = 262144, float minD = 2.f, int run_length = 7, int numBinsPhi = 24,
                        int numBinsTheta = 75, int device = 0);
  ~OdometryNode();
  OdometryNode(const OdometryNode&) = delete;
  OdometryNode& operator=(const OdometryNode&) = delete;
  // returns false for the very first cloud (it only becomes prev_pcl_matrix, odometry.cpp:47-52)
  bool pointcloudCallback(const Eigen::MatrixXf& pcl_matrix, NodeOutput* out);

  Eigen::VectorXf X0;      // seed of the next registration (odometry.cpp:82), host copy
  Eigen::MatrixXf X_homo;  // host copy of the accumulated transform
  int frameCount = 0;

 protected:
  OdometryNode(int max_points, float minD, int run_length, int numBinsPhi, int numBinsTheta, int device, bool chain,
               float trans_thresh, float rot_thresh);
  icet_b200_ctx* ctx_ = nullptr;
  icet_b200_node* node_ = nullptr;
};

class ScanMatcherNode : public OdometryNode {
 public:
  // src/scanMatcher.cpp:18-150: clouds as they come (no range filter), X0 = 0 (:58-62), run_length 7, 24 x 75 bins
  explicit ScanMatcherNode(int max_points = 262144, int run_length = 7, int numBinsPhi = 24, int numBinsTheta = 75,
                           int device = 0);
  ~ScanMatcherNode();
  // returns false for an empty cloud (:41-44) and for the first cloud (:47-51); otherwise fills out->X and
  // scan2_in_scan1_frame = (pcl_matrix * rot_mat.inverse()).rowwise() - trans (:73), computed on the device
  bool pointcloudCallback(const Eigen::MatrixXf& pcl_matrix, NodeOutput* out);
  Eigen::MatrixXf scan2_in_scan1_frame;  // N x 3
  Eigen::MatrixXf snailTrail;            // (:25-26, :76-80) grows by one row per registration
};

// Keyframe odometry (include/icet_b200.h "keyframe odometry", DESIGN.md §13): every filtered scan is registered against
// the node's current keyframe; the device decides after each registration whether the scan becomes the next keyframe.
struct KeyframeInfo {
  int keyframe;   // frame index of the keyframe the scan was registered against
  bool promoted;  // the scan is the keyframe of the next one
  int reason;     // ICET_B200_KF_* bits
  float x0[6];    // the seed the registration started from
};

class KeyframeOdometryNode {
 public:
  // the odometry node's constants (minD = 2, run_length = 7, 24 x 75 bins, 10 Hz twist, chained seeds) and a policy
  // (NULL: defaultPolicy()).  map_keyframes = M in 1 .. 16: scan 1 of every registration is the local map of the last M
  // keyframes (icet_b200_kfnode_create_local_map, DESIGN.md §14); 0: the keyframe alone.
  explicit KeyframeOdometryNode(int max_points = 262144, float minD = 2.f, int run_length = 7, int numBinsPhi = 24,
                                int numBinsTheta = 75, const icet_b200_keyframe_policy* policy = nullptr, int device = 0,
                                int map_keyframes = 0);
  ~KeyframeOdometryNode();
  KeyframeOdometryNode(const KeyframeOdometryNode&) = delete;
  KeyframeOdometryNode& operator=(const KeyframeOdometryNode&) = delete;
  // returns false for the very first cloud (it becomes keyframe 0); out->X is X relative to the keyframe
  bool pointcloudCallback(const Eigen::MatrixXf& pcl_matrix, NodeOutput* out, KeyframeInfo* info = nullptr);
  static icet_b200_keyframe_policy defaultPolicy();  // 1 m, 0.1 rad, overlap 0.5, 10 scans (DESIGN.md §13)
  Eigen::MatrixXf localMap();  // N x 3: scan 1 of the next registration (the keyframe cloud when map_keyframes = 0)

  Eigen::MatrixXf X_homo;  // host copy of the pose of the last scan
  int frameCount = 0;

 private:
  icet_b200_ctx* ctx_ = nullptr;
  icet_b200_kfnode* node_ = nullptr;
};

class MapMakerNode : public OdometryNode {
 public:
  // minD = 0.2 (:100), run_length = 12 (:115), X0 = 0 every time (:124), thresholds 0.3 / 0.3 (:241-242),
  // 600 000-point queue (:62), 2000-row sample (:150)
  explicit MapMakerNode(int max_points = 262144, int map_size = 600000, int downsampleSize = 2000, int device = 0);
  ~MapMakerNode();
  bool pointcloudCallback(const Eigen::MatrixXf& pcl_matrix, NodeOutput* out);
  Eigen::MatrixXf getQueue();  // EigenQueue::getQueue (:44-51): N x 3, oldest row first
  std::vector<int> lastSample; // the rows of the current scan that went into the map

 private:
  icet_b200_map* q_ = nullptr;
  int map_size_, downsampleSize_;
  float rot_thresh = 0.3f, trans_thresh = 0.3f;  // simpleMapMaker.cpp:241-242
  std::mt19937 gen;                              // default-seeded, like the reference's member (:258)
};

#endif
