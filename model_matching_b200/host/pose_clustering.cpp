// pose_clustering.cpp -- restatement of the reference's src/pose_clustering.cpp:5-122.
#include "pose_clustering.hpp"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <iostream>
#include <stdexcept>
#include <string>

#include "../../include/stocs_b200.h"
#include "../csrc/stocs_pose_math.h"

namespace clustering {

// src/pose_clustering.cpp:5-72.  The arithmetic is csrc/stocs_pose_math.h, which the clustering
// kernels (csrc/cluster.cu) share: IEEE operations in a fixed order and pinned atan2 / asin instead of
// libm, so that the host loop and the GPU keep the same clusters.
void get_pose_diff(const Eigen::Matrix4f& test_pose, const Eigen::Matrix4f& base_pose, const Eigen::Vector3f& sym_info,
                   float& mean_rotation_error, float& translation_error) {
  const float sym[3] = {sym_info(0), sym_info(1), sym_info(2)};
  stocsm::pose_diff(test_pose.data(), base_pose.data(), sym, &mean_rotation_error, &translation_error);
}

// src/pose_clustering.cpp:79-122
void greedy_clustering(std::vector<PoseCandidate*>& hypotheses_set, float acceptable_fraction, float best_score,
                       int maximum_pose_count, float min_distance, float min_angle, Eigen::Vector3f sym_info,
                       std::vector<PoseCandidate*>& clustered_hypotheses_set) {
  clustered_hypotheses_set.clear();
  std::vector<PoseCandidate*> pruned;
  for (auto pose_it : hypotheses_set)
    if (pose_it->lcp > acceptable_fraction * best_score) pruned.push_back(pose_it);
  // std::sort in the reference (order among equal scores unspecified); stable here
  std::stable_sort(pruned.begin(), pruned.end(), [](PoseCandidate* a, PoseCandidate* b) { return a->lcp > b->lcp; });
  for (auto candidate_it : pruned) {
    bool inValid = false;
    for (auto cluster_it : clustered_hypotheses_set) {
      float mean_rotation_error, translation_error;
      get_pose_diff(candidate_it->transform, cluster_it->transform, sym_info, mean_rotation_error, translation_error);
      if (mean_rotation_error < min_angle && translation_error < min_distance) { inValid = true; break; }
    }
    if (inValid == false) clustered_hypotheses_set.push_back(candidate_it);
    if ((int)clustered_hypotheses_set.size() > maximum_pose_count) break;
  }
}

// reference src/pose_clustering.cpp:123-141.  PCL's ICP loop runs on the device
// (stocs_b200_icp_point_to_plane); the context is created on first use and lives for the process.
void point_to_plane_icp(PCLPointCloud::Ptr segment_cloud, PCLPointCloud::Ptr model_cloud, Eigen::Matrix4f& offset_transform) {
  static stocs_b200_ctx* ctx = nullptr;
  if (!ctx) {
    const char* dev = getenv("STOCS_DEVICE");
    if (stocs_b200_create(&ctx, dev ? atoi(dev) : 0) != 0) {
      ctx = nullptr;  // create leaves *out NULL on failure; its message is kept per thread
      throw std::runtime_error(std::string("point_to_plane_icp: ") + stocs_b200_last_error(nullptr));
    }
  }
  const int ns = (int)segment_cloud->points.size(), nt = (int)model_cloud->points.size();
  // PCL's align() on an empty source or target does not converge; the reference then resets the
  // caller's matrix (src/pose_clustering.cpp:136-139)
  if (ns == 0 || nt == 0) { offset_transform.setIdentity(); return; }
  std::vector<float> sp((size_t)ns * 3), tp((size_t)nt * 3), tn((size_t)nt * 3), moved((size_t)ns * 3);
  for (int i = 0; i < ns; ++i) {
    const CloudPoint& p = segment_cloud->points[i];
    sp[3 * i] = p.x; sp[3 * i + 1] = p.y; sp[3 * i + 2] = p.z;
  }
  for (int i = 0; i < nt; ++i) {
    const CloudPoint& p = model_cloud->points[i];
    tp[3 * i] = p.x; tp[3 * i + 1] = p.y; tp[3 * i + 2] = p.z;
    tn[3 * i] = p.nx; tn[3 * i + 1] = p.ny; tn[3 * i + 2] = p.nz;
  }
  float T[16];
  int32_t converged = 0;
  if (stocs_b200_icp_point_to_plane(ctx, sp.data(), ns, tp.data(), tn.data(), nt, /*setMaximumIterations*/ 5,
                                    /*setMaxCorrespondenceDistance*/ 0.035f, T, moved.data(), nullptr, nullptr,
                                    &converged) != 0)
    throw std::runtime_error(std::string("point_to_plane_icp: ") + stocs_b200_last_error(ctx));
  for (int i = 0; i < ns; ++i) {  // icp->align(*segment_cloud) leaves the moved source in place
    CloudPoint& p = segment_cloud->points[i];
    p.x = moved[3 * i]; p.y = moved[3 * i + 1]; p.z = moved[3 * i + 2];
    const float nx = p.nx, ny = p.ny, nz = p.nz;
    p.nx = T[0] * nx + T[4] * ny + T[8] * nz;
    p.ny = T[1] * nx + T[5] * ny + T[9] * nz;
    p.nz = T[2] * nx + T[6] * ny + T[10] * nz;
  }
  // src/pose_clustering.cpp:136-139: final transformation when converged, identity otherwise
  if (converged) {
    for (int c = 0; c < 4; ++c)
      for (int r = 0; r < 4; ++r) offset_transform(r, c) = T[c * 4 + r];
  } else {
    offset_transform.setIdentity();
  }
}

}  // namespace clustering
