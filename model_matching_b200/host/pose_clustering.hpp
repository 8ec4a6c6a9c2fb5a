// pose_clustering.hpp -- same declarations as the reference's include/pose_clustering.hpp:9-28.
// greedy_clustering is a faithful host restatement, one candidate at a time against every kept pose.
// That suits the shim's few thousand candidates; for the lists the device produces (10^5..10^6 scored
// hypotheses) the same pass runs on the GPU as stocs_b200_cluster_poses, and the fused pipeline
// clusters its own scored list (stocs_b200_run_pipeline[_instance]_clustered).  Both keep the same
// poses: get_pose_diff is csrc/stocs_pose_math.h, which the kernels call too.
// point_to_plane_icp (pcl::IterativeClosestPointWithNormals in the reference, PCL not being part
// of the reference tree) runs PCL's published point-to-plane loop on the GPU through
// stocs_b200_icp_point_to_plane (csrc/icp.cu, arithmetic in csrc/stocs_icp_math.h).
// trimmed_icp is declared but never defined in the reference either.
#ifndef STOCS_B200_POSE_CLUSTERING_HPP_
#define STOCS_B200_POSE_CLUSTERING_HPP_
#include <vector>

#include "rgbd.hpp"

namespace clustering {

void greedy_clustering(std::vector<PoseCandidate*>& hypotheses_set, float acceptable_fraction, float best_score,
                       int maximum_pose_count, float min_distance, float min_angle, Eigen::Vector3f sym_info,
                       std::vector<PoseCandidate*>& clustered_hypotheses_set);

void point_to_plane_icp(PCLPointCloud::Ptr segment, PCLPointCloud::Ptr model, Eigen::Matrix4f& offset_transform);

// exposed for the tests: max |Euler angle| (degrees, after the symmetry folding) and translation
// distance between two poses (reference src/pose_clustering.cpp:28-72)
void get_pose_diff(const Eigen::Matrix4f& test_pose, const Eigen::Matrix4f& base_pose, const Eigen::Vector3f& sym_info,
                   float& mean_rotation_error, float& translation_error);

}  // namespace clustering
#endif
