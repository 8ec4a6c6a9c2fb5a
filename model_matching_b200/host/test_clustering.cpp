// test_clustering -- reads poses (n, then n x (16 col-major floats + lcp)) and parameters from
// stdin, prints the indices greedy_clustering keeps; used by tests/test_clustering.py.
// `test_clustering icp`: reads ns nt, ns source points (x y z), nt model points (x y z nx ny nz),
// runs clustering::point_to_plane_icp (needs the GPU) and prints the 16 column-major entries of
// the offset and the moved source; used by tests/test_icp_gpu.py.
// `test_clustering bin`: the clustering input in binary on stdin (int64 n; float acceptable_fraction,
// best_score; int32 maximum_pose_count; float min_distance, min_angle, sym_info[3]; n x 16 col-major
// floats; n lcps), prints the kept indices (and the loop's wall clock on stderr); bit-exact inputs
// for tests/test_cluster_gpu.py.
// `test_clustering diff`: int64 n; float sym_info[3]; n test poses, n base poses (16 floats each) on
// stdin; writes get_pose_diff's n rotation errors, then n translation errors (float32) to stdout.
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <vector>

#include "pose_clustering.hpp"

// `icp stale`: offset_transform enters as a non-identity matrix, so a run that does not converge
// must come back as identity (src/pose_clustering.cpp:136-139)
static int icp_main(bool stale) {
  int ns, nt;
  if (scanf("%d %d", &ns, &nt) != 2) return 1;
  auto seg = std::make_shared<PCLPointCloud>(), model = std::make_shared<PCLPointCloud>();
  seg->points.resize(ns);
  model->points.resize(nt);
  for (auto& p : seg->points) { if (scanf("%f %f %f", &p.x, &p.y, &p.z) != 3) return 1; p.nx = 0; p.ny = 0; p.nz = 1; }
  for (auto& p : model->points) if (scanf("%f %f %f %f %f %f", &p.x, &p.y, &p.z, &p.nx, &p.ny, &p.nz) != 6) return 1;
  Eigen::Matrix4f off = Eigen::Matrix4f::Identity();
  if (stale) for (int k = 0; k < 16; ++k) off.data()[k] = 7.0f + (float)k;
  clustering::point_to_plane_icp(seg, model, off);
  for (int k = 0; k < 16; ++k) printf("%.9g ", off.data()[k]);
  printf("\n");
  for (auto& p : seg->points) printf("%.9g %.9g %.9g\n", p.x, p.y, p.z);
  return 0;
}

static bool read_all(void* p, size_t bytes) { return fread(p, 1, bytes, stdin) == bytes; }

static int bin_main() {
  int64_t n;
  float frac, best, min_d, min_a, sym[3];
  int32_t max_count;
  if (!read_all(&n, 8) || !read_all(&frac, 4) || !read_all(&best, 4) || !read_all(&max_count, 4) || !read_all(&min_d, 4) ||
      !read_all(&min_a, 4) || !read_all(sym, 12) || n < 0)
    return 1;
  std::vector<float> T((size_t)n * 16), lcp((size_t)n);
  if (!read_all(T.data(), T.size() * 4) || !read_all(lcp.data(), lcp.size() * 4)) return 1;
  std::vector<PoseCandidate> cand;
  cand.reserve((size_t)n);
  std::vector<PoseCandidate*> all, out;
  for (int64_t i = 0; i < n; ++i) {
    Eigen::Matrix4f M;
    memcpy(M.data(), &T[(size_t)i * 16], 64);
    cand.emplace_back(M, lcp[(size_t)i], (int)i);
    all.push_back(&cand.back());
  }
  const auto t0 = std::chrono::steady_clock::now();
  clustering::greedy_clustering(all, frac, best, max_count, min_d, min_a, Eigen::Vector3f(sym[0], sym[1], sym[2]), out);
  const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  for (auto* p : out) printf("%d\n", p->base_index);
  fprintf(stderr, "greedy_clustering_ms %.4f\n", ms);   // the host loop alone (profiles/cluster_latency.py)
  return 0;
}

static int diff_main() {
  int64_t n;
  float sym[3];
  if (!read_all(&n, 8) || !read_all(sym, 12) || n < 0) return 1;
  std::vector<float> Tt((size_t)n * 16), Tb((size_t)n * 16), out((size_t)n * 2);
  if (!read_all(Tt.data(), Tt.size() * 4) || !read_all(Tb.data(), Tb.size() * 4)) return 1;
  const Eigen::Vector3f s(sym[0], sym[1], sym[2]);
  for (int64_t i = 0; i < n; ++i) {
    Eigen::Matrix4f A, B;
    memcpy(A.data(), &Tt[(size_t)i * 16], 64);
    memcpy(B.data(), &Tb[(size_t)i * 16], 64);
    clustering::get_pose_diff(A, B, s, out[(size_t)i], out[(size_t)n + i]);
  }
  return fwrite(out.data(), 4, out.size(), stdout) == out.size() ? 0 : 1;
}

int main(int argc, char** argv) {
  if (argc > 1 && !strcmp(argv[1], "icp")) return icp_main(argc > 2 && !strcmp(argv[2], "stale"));
  if (argc > 1 && !strcmp(argv[1], "bin")) return bin_main();
  if (argc > 1 && !strcmp(argv[1], "diff")) return diff_main();
  int n, max_count;
  float frac, best, min_d, min_a, sym[3];
  if (scanf("%d %f %f %d %f %f %f %f %f", &n, &frac, &best, &max_count, &min_d, &min_a, &sym[0], &sym[1], &sym[2]) != 9) return 1;
  std::vector<PoseCandidate*> all, out;
  for (int i = 0; i < n; ++i) {
    Eigen::Matrix4f T;
    float lcp;
    for (int k = 0; k < 16; ++k) if (scanf("%f", &T.data()[k]) != 1) return 1;
    if (scanf("%f", &lcp) != 1) return 1;
    all.push_back(new PoseCandidate(T, lcp, (float)i));
  }
  clustering::greedy_clustering(all, frac, best, max_count, min_d, min_a, Eigen::Vector3f(sym[0], sym[1], sym[2]), out);
  for (auto* p : out) printf("%d\n", p->base_index);
  if (n >= 2) {
    float r, t;
    clustering::get_pose_diff(all[0]->transform, all[1]->transform, Eigen::Vector3f(sym[0], sym[1], sym[2]), r, t);
    printf("diff %.6f %.6f\n", r, t);
  }
  return 0;
}
