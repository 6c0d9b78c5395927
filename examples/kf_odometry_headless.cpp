// examples/kf_odometry_headless.cpp -- replays a recorded sequence through the keyframe odometry node
// (include/icet_nodes.h KeyframeOdometryNode), printing the pose and keyframe decision of every scan.
//
// usage: kf_odometry_headless points_per_scan file.f32 [max_trans max_rot min_overlap max_interval [map_keyframes]]
//   file.f32: consecutive scans, each the x | y | z planes of points_per_scan float32 values.
//   map_keyframes: register against the local map of the last M keyframes (DESIGN.md §14); also prints its rows.
#include <cstdio>
#include <fstream>
#include <string>

#include "icet_nodes.h"

int main(int argc, char** argv) {
  if (argc != 3 && argc != 7 && argc != 8) {
    std::fprintf(stderr, "usage: %s points_per_scan file.f32 [max_trans max_rot min_overlap max_interval [map_keyframes]]\n",
                 argv[0]);
    return 2;
  }
  const long n = std::stol(argv[1]);
  std::ifstream f(argv[2], std::ios::binary | std::ios::ate);
  if (!f) { std::fprintf(stderr, "cannot open %s\n", argv[2]); return 2; }
  const long nscans = (long)f.tellg() / (12 * n);
  f.seekg(0);
  icet_b200_keyframe_policy kp = KeyframeOdometryNode::defaultPolicy();
  if (argc >= 7) {
    kp.max_trans = std::stof(argv[3]);
    kp.max_rot = std::stof(argv[4]);
    kp.min_overlap = std::stof(argv[5]);
    kp.max_interval = std::stoi(argv[6]);
  }
  const int map_keyframes = argc == 8 ? std::stoi(argv[7]) : 0;
  try {
    KeyframeOdometryNode node((int)n, 2.f, 7, 24, 75, &kp, 0, map_keyframes);
    for (long k = 0; k < nscans; k++) {
      Eigen::MatrixXf cloud(n, 3);
      f.read(reinterpret_cast<char*>(cloud.data()), n * 12);
      NodeOutput o;
      KeyframeInfo ki;
      if (!node.pointcloudCallback(cloud, &o, &ki)) continue;
      std::printf("POSE %ld X [%.9g, %.9g, %.9g, %.9g, %.9g, %.9g] pos [%.9g, %.9g, %.9g] quat [%.9g, %.9g, %.9g, %.9g] "
                  "points %d keyframe %d promoted %d reason %d\n", k, o.X[0], o.X[1], o.X[2], o.X[3], o.X[4], o.X[5],
                  o.position[0], o.position[1], o.position[2], o.orientation[0], o.orientation[1], o.orientation[2],
                  o.orientation[3], o.points, ki.keyframe, (int)ki.promoted, ki.reason);
      if (map_keyframes > 0) std::printf("MAP %ld rows %ld\n", k, (long)node.localMap().rows());
    }
  } catch (const std::exception& e) {
    std::fprintf(stderr, "node failed: %s\n", e.what());
    return 1;
  }
  return 0;
}
