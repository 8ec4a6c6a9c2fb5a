// stocs_cli.cpp -- the two command lines of the drop-in, built from this one source:
//
//   stocs_single <scene_path> <object_name>      online pose estimation
//   model_preprocess <object_name>               offline model preparation
//
// argv, the files read and written, and the progress lines on stdout are those of the reference's
// src/stocs_match_one_object.cpp and src/model_preprocess.cpp (whose sources, unmodified, also
// compile and link against this directory; tests/test_ref_callers.py pins what they write).
// Everything goes through the public stocs::stocs_estimator / stocs::pre_process_model interface
// of stocs.hpp.
//
// The reference keeps its tunables as compile-time globals ("edit and recompile", README.md:47-69);
// here they live in one Settings record whose defaults are the reference's values and which the
// environment can override (names in Settings::from_env).
#include <libgen.h>
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>

#include "stocs.hpp"

#ifndef STOCS_DEFAULT_REPO_PATH
#define STOCS_DEFAULT_REPO_PATH "."
#endif

namespace {

struct Settings {
  std::string repo_path = STOCS_DEFAULT_REPO_PATH;
  // online: src/stocs_match_one_object.cpp:7-24
  float voxel_size = 0.005f, distance_threshold = 0.005f;
  int ppf_tr = 5, ppf_rot = 5;
  float edge_threshold = 0.f, class_threshold = 0.10f, sample_dispersion = 0.9f;
  int bases = 100, max_sets = 200;
  std::vector<float> intrinsics{1066.778f, 312.986f, 1067.487f, 241.310f};  // {fx, cx, fy, cy}, YCB
  float depth_scale = 1 / 10000.0f;
  int width = 640, height = 480;
  // offline: src/model_preprocess.cpp:6-12
  float model_voxel_size = 0.01f, normal_radius = 0.005f, model_scale = 1.0f;
  // STOCS_REF_SHUFFLE=1: pick the transforms of a base with >= max_sets quads the way the reference
  // does (quirk 5, src/stocs_match_one_object.cpp:134-139); default: deterministic even spread
  bool ref_shuffle = false;
  std::string trace_file;  // STOCS_TRACE_FILE: binary dump of every intermediate (tests/test_shim_gpu.py)

  static void num(const char* name, float& v) { if (const char* e = std::getenv(name)) v = (float)std::atof(e); }
  static void num(const char* name, int& v) { if (const char* e = std::getenv(name)) v = std::atoi(e); }
  void from_env() {
    if (const char* e = std::getenv("STOCS_REPO_PATH")) repo_path = e;
    num("STOCS_VOXEL_SIZE", voxel_size);
    num("STOCS_DISTANCE_THRESHOLD", distance_threshold);
    num("STOCS_PPF_TR", ppf_tr);
    num("STOCS_PPF_ROT", ppf_rot);
    num("STOCS_CLASS_THRESHOLD", class_threshold);
    num("STOCS_SAMPLE_DISPERSION", sample_dispersion);
    num("STOCS_NUM_BASES", bases);
    num("STOCS_MAX_SETS", max_sets);
    num("STOCS_DEPTH_SCALE", depth_scale);
    num("STOCS_IMAGE_WIDTH", width);
    num("STOCS_IMAGE_HEIGHT", height);
    num("STOCS_MODEL_VOXEL_SIZE", model_voxel_size);
    num("STOCS_NORMAL_RADIUS", normal_radius);
    num("STOCS_MODEL_SCALE", model_scale);
    if (const char* e = std::getenv("STOCS_CAM_INTRINSICS")) {
      std::vector<float> k;
      std::stringstream ss(e);
      for (std::string t; std::getline(ss, t, ',');) k.push_back((float)std::atof(t.c_str()));
      if (k.size() == 4) intrinsics = k;
      else std::cerr << "STOCS_CAM_INTRINSICS wants fx,cx,fy,cy -- ignored" << std::endl;
    }
    if (const char* e = std::getenv("STOCS_REF_SHUFFLE")) ref_shuffle = std::atoi(e) != 0;
    if (const char* e = std::getenv("STOCS_TRACE_FILE")) trace_file = e;
  }
};

// the estimator with its protected lists readable (for the trace only)
struct TracedEstimator : stocs::stocs_estimator {
  using stocs::stocs_estimator::stocs_estimator;
  const std::vector<MatrixType>& centred_transforms() { flush_pending(); return all_transforms; }
  int best() const { return best_index; }
};

struct Base {
  std::vector<int> ids;
  float inv1 = 0, inv2 = 0;
  std::vector<Quadrilateral> quads;
  std::vector<int> picked;
};

struct Trace {  // little-endian binary, layout documented in tests/test_shim_gpu.py
  std::ofstream f;
  explicit Trace(const std::string& path) { if (!path.empty()) f.open(path, std::ios::binary); }
  bool on() const { return f.is_open(); }
  template <class T> void put(const T& v) { if (on()) f.write((const char*)&v, sizeof(T)); }
  template <class T> void put(const T* p, size_t n) { if (on()) f.write((const char*)p, (std::streamsize)(sizeof(T) * n)); }
};

// which of a base's n quads become hypotheses (at most `limit`)
std::vector<int> pick_quads(int n, int limit, bool ref_shuffle) {
  std::vector<int> out;
  if (n < limit) {
    for (int i = 0; i < n; ++i) out.push_back(i);
  } else if (ref_shuffle) {
    // the reference builds an index vector of n ZEROS followed by 0..n-1, shuffles it with the
    // unseeded C rand() and takes the first `limit` entries -- so about half of them are quad 0
    std::vector<int> idx((size_t)n);
    for (int i = 0; i < n; ++i) idx.push_back(i);
    std::random_shuffle(idx.begin(), idx.end());
    out.assign(idx.begin(), idx.begin() + limit);
  } else {
    for (int k = 0; k < limit; ++k) out.push_back((int)(((long long)k * n) / limit));
  }
  return out;
}

long long us_since(std::chrono::high_resolution_clock::time_point t0) {
  return std::chrono::duration_cast<micro>(std::chrono::high_resolution_clock::now() - t0).count();
}

int online(const Settings& s, const std::string& scene, const std::string& object) {
  std::cout << "############# LOADING OBJECT MAPS ################" << std::endl;
  PPFMapType model_map;
  rgbd::load_ppf_map(s.repo_path + "/models/" + object + "/ppf_map", model_map);
  std::cout << "############# LOADING OBJECT COMPLETE ################" << std::endl;
  if (std::system(("rm -rf " + scene + "/dbg").c_str()) != 0 || std::system(("mkdir " + scene + "/dbg").c_str()) != 0) return 1;
  std::cout << "############# RUNNING STOCS for Scene: " << scene << ", Object: " << object << " ##############" << std::endl;

  const std::string edge_map = scene + "/probability_maps/edge.png";
  TracedEstimator est(s.repo_path + "/models/" + object + "/model_search.ply", model_map, scene + "/rgb.png",
                      scene + "/depth.png", scene + "/probability_maps/" + object + ".png", edge_map, scene + "/dbg",
                      s.intrinsics, s.width, s.height, s.depth_scale, 1.0f, s.voxel_size, s.distance_threshold, s.ppf_tr,
                      s.ppf_rot, s.edge_threshold, s.class_threshold);
  Trace tr(s.trace_file);
  tr.put("STOCSTR1", 8);

  // 1. bases: instance mode when the scene ships an edge map (src/stocs_match_one_object.cpp:89-93)
  struct stat sb;
  const bool instance_mode = stat(edge_map.c_str(), &sb) == 0;
  std::vector<Base> bases;
  auto t0 = std::chrono::high_resolution_clock::now();
  tr.put<int32_t>(s.bases);
  for (int i = 0; i < s.bases; ++i) {
    Base b;
    b.ids.assign(4, -1);
    std::vector<Point3D> segment;
    const bool ok = instance_mode ? est.sample_instance_base(b.ids, b.inv1, b.inv2, segment, s.sample_dispersion, i + 1)
                                  : est.sample_class_base(b.ids, b.inv1, b.inv2);
    tr.put<uint8_t>(ok ? 1 : 0);
    tr.put(b.ids.data(), 4);
    tr.put(b.inv1); tr.put(b.inv2);
    if (ok) bases.push_back(std::move(b));
  }
  long long total_us = us_since(t0);
  std::cout << "Sampled " << bases.size() << " bases in " << total_us << " microseconds\n";

  // 2. congruent sets, 3. at most max_sets hypotheses per base
  t0 = std::chrono::high_resolution_clock::now();
  for (Base& b : bases) est.find_congruent_sets_on_model(b.ids, b.inv1, b.inv2, &b.quads);
  long long sets = 0;
  int base_number = 0;
  for (Base& b : bases) {
    b.picked = pick_quads((int)b.quads.size(), s.max_sets, s.ref_shuffle);
    for (int k : b.picked) est.get_rigid_transform_from_congruent_pair(b.ids, b.quads[(size_t)k], base_number);
    sets += (long long)b.quads.size();
    ++base_number;
  }
  long long us = us_since(t0);
  std::cout << "found " << sets << " congruent sets in " << us << " microseconds\n";
  total_us += us;

  // 4. score every hypothesis, keep the best
  t0 = std::chrono::high_resolution_clock::now();
  est.compute_best_transform();
  us = us_since(t0);
  std::cout << "evaluated transforms in " << us << " microseconds\n";
  total_us += us;
  std::cout << "total " << total_us << " microseconds\n";

  if (tr.on()) {
    tr.put<int32_t>((int32_t)bases.size());
    for (const Base& b : bases) {
      tr.put<int64_t>((int64_t)b.quads.size());
      for (const Quadrilateral& q : b.quads) tr.put(q.vertices.data(), 4);
      tr.put<int64_t>((int64_t)b.picked.size());
      tr.put(b.picked.data(), b.picked.size());
    }
    const std::vector<MatrixType>& Tc = est.centred_transforms();
    std::vector<PoseCandidate*> poses = est.get_pose_candidates();
    tr.put<int64_t>((int64_t)Tc.size());
    for (size_t i = 0; i < Tc.size(); ++i) {
      tr.put(Tc[i].data(), 16);
      tr.put(poses[i]->transform.data(), 16);
      tr.put(poses[i]->lcp);
      tr.put<int32_t>(poses[i]->base_index);
    }
    tr.put<int32_t>(est.best());
    tr.put<float>(est.get_best_score());
  }

  est.visualize_best_pose();
  PoseCandidate* best = est.get_best_pose();
  if (best == NULL) {
    std::cout << "no pose found" << std::endl;
    return 0;
  }
  // 12 numbers: rows 0..2 of the un-centred pose, row-major, one line (src/stocs_match_one_object.cpp:173-179)
  std::ofstream out(scene + "/best_pose_candidate_" + object + ".txt", std::ofstream::out);
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 4; ++c) out << best->transform(r, c) << ((r == 2 && c == 3) ? "" : " ");
  out << std::endl;
  return 0;
}

int offline(const Settings& s, const std::string& object) {
  const std::string dir = s.repo_path + "/models/" + object;
  std::remove((dir + "/model_search.ply").c_str());  // src/model_preprocess.cpp:25-26
  std::remove((dir + "/ppf_map").c_str());
  stocs::pre_process_model(dir + "/textured_vertices.ply", s.normal_radius, s.model_scale, 1.0f, s.model_voxel_size,
                           (float)s.ppf_tr, (float)s.ppf_rot, dir + "/model_search.ply", dir + "/ppf_map");
  return 0;
}

}  // namespace

int main(int argc, char** argv) {
  Settings s;
  s.from_env();
  std::string self = argc > 0 ? argv[0] : "";
  const size_t slash = self.find_last_of('/');
  if (slash != std::string::npos) self = self.substr(slash + 1);
  if (self.find("model_preprocess") != std::string::npos) {
    if (argc < 2) {
      std::cout << "Enter name of the object model!!" << std::endl;
      return 255;  // the reference calls exit(-1)
    }
    return offline(s, argv[1]);
  }
  if (argc < 3) {
    std::cout << "Enter scene path and object name as arguments!" << std::endl;
    return 255;
  }
  return online(s, argv[1], argv[2]);
}
