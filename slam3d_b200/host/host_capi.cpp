// host_capi.cpp — flat C entry points over the C++ host mirror so the pytest suite can drive it through ctypes.
// (Test/driver glue only; a slam3d application uses the C++ classes directly.)
#include <cstring>
#include <thread>

#include "MiniHost.hpp"

using namespace slam3d_b200;

namespace {
PointCloud::Ptr makeCloud(const float* xyzw, uint64_t n) {
  PointCloud::Ptr c(new PointCloud);
  c->points.resize(n);
  if (n) std::memcpy(&c->points[0].x, xyzw, 16 * n);
  return c;
}
Transform makeTransform(const double* m) { Transform t; if (m) for (int i = 0; i < 16; ++i) t.m[i] = m[i]; return t; }
thread_local std::string g_msg;
// 0 ok, 1 NoMatch, 2 BadMeasurementType, 3 runtime_error
template <typename F> int wrap(F&& f) {
  try { f(); return 0; }
  catch (NoMatch& e) { g_msg = e.what(); return 1; }
  catch (BadMeasurementType& e) { g_msg = e.what(); return 2; }
  catch (std::exception& e) { g_msg = e.what(); return 3; }
}
struct OtherMeasurement : Measurement {
  OtherMeasurement() : Measurement("r", "s", Transform()) {}
  const char* getTypeName() const override { return "other"; }
};
}  // namespace

extern "C" {

const char* s3dhost_last_message() { return g_msg.c_str(); }
void s3dhost_set_cache_capacity(uint64_t n) { setPreparedCacheCapacity((size_t)n); }
uint64_t s3dhost_cache_hits() { return (uint64_t)preparedCacheHits(); }

void* s3dhost_sensor_create(const char* name) { return new PointCloudSensor(name, nullptr); }
void s3dhost_sensor_destroy(void* s) { delete static_cast<PointCloudSensor*>(s); }

void s3dhost_sensor_set_params(void* s, const s3d_registration_parameters* c, int coarse) {
  RegistrationParameters p;
  p.registration_algorithm = static_cast<RegistrationAlgorithm>(c->registration_algorithm);
  p.point_cloud_density = c->point_cloud_density; p.max_fitness_score = c->max_fitness_score; p.max_translation = c->max_translation;
  p.max_rotation = c->max_rotation; p.euclidean_fitness_epsilon = c->euclidean_fitness_epsilon; p.transformation_epsilon = c->transformation_epsilon;
  p.max_correspondence_distance = c->max_correspondence_distance; p.maximum_iterations = c->maximum_iterations; p.rotation_epsilon = c->rotation_epsilon;
  p.correspondence_randomness = c->correspondence_randomness; p.maximum_optimizer_iterations = c->maximum_optimizer_iterations;
  p.resolution = c->resolution; p.step_size = c->step_size; p.outlier_ratio = c->outlier_ratio;
  static_cast<PointCloudSensor*>(s)->setRegistrationParameters(p, coarse != 0);
}
void s3dhost_sensor_set_covariance_scale(void* s, double v) { static_cast<PointCloudSensor*>(s)->setCovarianceScale(v); }

// createConstraint(source, target, odometry, loop): out_T 16 doubles (column-major), out_info 36 doubles.
// bad_type != 0 passes a non-point-cloud measurement as target (BadMeasurementType path, :279-283).
int s3dhost_create_constraint(void* s, const float* src, uint64_t nsrc, const double* src_sensor_pose, const float* tgt, uint64_t ntgt,
                              const double* tgt_sensor_pose, const double* odometry, int loop, int bad_type, double* out_T, double* out_info) {
  return wrap([&] {
    Measurement::Ptr ms(new PointCloudMeasurement(makeCloud(src, nsrc), "robot", "sensor", makeTransform(src_sensor_pose)));
    Measurement::Ptr mt;
    if (bad_type) mt.reset(new OtherMeasurement()); else mt.reset(new PointCloudMeasurement(makeCloud(tgt, ntgt), "robot", "sensor", makeTransform(tgt_sensor_pose)));
    Constraint::Ptr c = static_cast<PointCloudSensor*>(s)->createConstraint(ms, mt, makeTransform(odometry), loop != 0);
    SE3Constraint::Ptr se3 = std::dynamic_pointer_cast<SE3Constraint>(c);
    for (int i = 0; i < 16; ++i) out_T[i] = se3->getRelativePose().m[i];
    for (int i = 0; i < 36; ++i) out_info[i] = se3->getInformation().m[i];
  });
}

// PointCloudSensor::downsample; out must hold n points. Returns the number of output points or -1.
int64_t s3dhost_downsample(const float* in, uint64_t n, double leaf, float* out) {
  int64_t m = -1;
  wrap([&] { PointCloud::Ptr o = PointCloudSensor::downsample(makeCloud(in, n), leaf); m = (int64_t)o->size(); if (m) std::memcpy(out, &o->points[0].x, 16 * m); });
  return m;
}

// PointCloudSensor::buildMap on n posed scans (sensor pose = identity); out must hold the sum of the sizes. Returns the map size or -1.
int64_t s3dhost_build_map(void* s, const float* const* scans, const uint64_t* sizes, int n, const double* poses, double resolution,
                          double outlier_radius, unsigned outlier_neighbors, float* out) {
  int64_t m = -1;
  wrap([&] {
    PointCloudSensor* sensor = static_cast<PointCloudSensor*>(s);
    sensor->setMapResolution(resolution);
    sensor->setMapOutlierRemoval(outlier_radius, outlier_neighbors);
    PointCloudSensor::PosedMeasurements v;
    for (int i = 0; i < n; ++i)
      v.emplace_back(PointCloudMeasurement::Ptr(new PointCloudMeasurement(makeCloud(scans[i], sizes[i]), "robot", sensor->getName(), Transform())),
                     makeTransform(poses + 16 * i));
    PointCloud::Ptr map = sensor->buildMap(v);
    PointCloud::Ptr accu = sensor->getAccumulatedCloud(v);
    PointCloud::Ptr filt = sensor->removeOutliers(accu, outlier_radius, outlier_neighbors);
    PointCloud::Ptr map2 = PointCloudSensor::downsample(filt, resolution);   // the three public steps give the same map
    if (map2->size() != map->size() || (map->size() && std::memcmp(&map->points[0].x, &map2->points[0].x, 16 * map->size()) != 0)) { m = -2; return; }
    m = (int64_t)map->size();
    if (m) std::memcpy(out, &map->points[0].x, 16 * m);
  });
  return m;
}

// Mini-host: n scans fed to addMeasurement(m, odom) in order (link-to-previous), from `threads` host threads when > 1
// (each thread owns a MiniHost but all share the sensor and the process-wide context => concurrent createConstraint).
// out_T: (n-1) x 16 doubles per thread-0 run; returns the number of recorded edges of run 0 or -1.
int s3dhost_run_odometry(void* s, const float* const* scans, const uint64_t* sizes, int n, const double* odoms, int threads, double* out_T, int* n_warnings) {
  PointCloudSensor* sensor = static_cast<PointCloudSensor*>(s);
  std::vector<std::vector<RecordedEdge>> all(threads > 1 ? threads : 1);
  std::vector<int> warn(all.size(), 0);
  auto run = [&](int t) {
    MiniHost host(sensor);
    for (int i = 0; i < n; ++i) {
      Measurement::Ptr m(new PointCloudMeasurement(makeCloud(scans[i], sizes[i]), "robot", sensor->getName(), Transform()));
      host.addMeasurement(m, makeTransform(odoms + 16 * i));
    }
    all[t] = host.edges; warn[t] = (int)host.warnings.size();
  };
  if (all.size() == 1) run(0);
  else { std::vector<std::thread> th; for (size_t t = 0; t < all.size(); ++t) th.emplace_back(run, (int)t); for (auto& x : th) x.join(); }
  for (size_t t = 1; t < all.size(); ++t) {  // concurrent runs must give identical edges
    if (all[t].size() != all[0].size()) return -2;
    for (size_t e = 0; e < all[0].size(); ++e) if (all[t][e].relative.m != all[0][e].relative.m) return -3;
  }
  for (size_t e = 0; e < all[0].size(); ++e) for (int i = 0; i < 16; ++i) out_T[16 * e + i] = all[0][e].relative.m[i];
  if (n_warnings) *n_warnings = warn[0];
  return (int)all[0].size();
}

// BASELINE configs[4] (trajectory): n scans through addMeasurement(m, odom) + linkLastToNeighbors() after every new vertex.
// edges_out: per recorded edge {source, target, loop} as 3 ints followed by nothing; T_out: 16 doubles per edge (relative pose);
// poses_out: n x 16 doubles (corrected poses).  Returns the number of edges (<= max_edges) or -1.
static int run_trajectory(void* s, const float* const* scans, const uint64_t* sizes, int n, const double* odoms, double neighbor_radius,
                          int max_links, int min_loop_length, int patch_range, int batched, int max_edges, int* edges_out, double* T_out,
                          double* poses_out, int* n_warnings) {
  PointCloudSensor* sensor = static_cast<PointCloudSensor*>(s);
  try {
    MiniHost host(sensor);
    host.setNeighborRadius((float)neighbor_radius, max_links);
    host.setMinLoopLength((unsigned)min_loop_length);
    host.setPatchBuildingRange((unsigned)patch_range);
    for (int i = 0; i < n; ++i) {
      Measurement::Ptr m(new PointCloudMeasurement(makeCloud(scans[i], sizes[i]), "robot", sensor->getName(), Transform()));
      if (host.addMeasurement(m, makeTransform(odoms + 16 * i))) host.linkLastToNeighbors(batched != 0);
    }
    const int ne = (int)std::min<size_t>(host.edges.size(), (size_t)max_edges);
    for (int e = 0; e < ne; ++e) {
      edges_out[3 * e] = (int)host.edges[e].source; edges_out[3 * e + 1] = (int)host.edges[e].target; edges_out[3 * e + 2] = host.edges[e].loop ? 1 : 0;
      for (int i = 0; i < 16; ++i) T_out[16 * e + i] = host.edges[e].relative.m[i];
    }
    if (poses_out) for (int v = 0; v < n; ++v) for (int i = 0; i < 16; ++i) poses_out[16 * v + i] = host.correctedPose((unsigned)v).m[i];
    if (n_warnings) *n_warnings = (int)host.warnings.size();
    g_msg = host.warnings.empty() ? "" : host.warnings.back();
    return ne;
  } catch (std::exception& e) {
    g_msg = e.what();
    return -1;
  }
}

int s3dhost_run_trajectory(void* s, const float* const* scans, const uint64_t* sizes, int n, const double* odoms, double neighbor_radius,
                           int max_links, int min_loop_length, int max_edges, int* edges_out, double* T_out, double* poses_out, int* n_warnings) {
  return run_trajectory(s, scans, sizes, n, odoms, neighbor_radius, max_links, min_loop_length, 0, 0, max_edges, edges_out, T_out, poses_out, n_warnings);
}

// the same with Sensor::mPatchBuildingRange = patch_range (loop closures match patches of scans, ScanSensor.cpp:215-270) and,
// when batched != 0, all candidates of a vertex matched in one device batch (PointCloudSensor::createConstraints)
int s3dhost_run_trajectory2(void* s, const float* const* scans, const uint64_t* sizes, int n, const double* odoms, double neighbor_radius,
                            int max_links, int min_loop_length, int patch_range, int batched, int max_edges, int* edges_out, double* T_out,
                            double* poses_out, int* n_warnings) {
  return run_trajectory(s, scans, sizes, n, odoms, neighbor_radius, max_links, min_loop_length, patch_range, batched, max_edges, edges_out, T_out, poses_out, n_warnings);
}

// ScanSensor::addMeasurement(m) without odometry (core/ScanSensor.cpp:49-79): the guess is chained from the previous result and
// a scan becomes a vertex only after min_translation / min_rotation.  T_out: 16 doubles per recorded edge.  Returns the edges or -1.
int s3dhost_run_no_odometry(void* s, const float* const* scans, const uint64_t* sizes, int n, double min_translation, double min_rotation,
                            int* added_out, double* T_out, int* n_warnings) {
  PointCloudSensor* sensor = static_cast<PointCloudSensor*>(s);
  try {
    MiniHost host(sensor);
    host.setMinPoseDistance((float)min_translation, (float)min_rotation);
    for (int i = 0; i < n; ++i) {
      Measurement::Ptr m(new PointCloudMeasurement(makeCloud(scans[i], sizes[i]), "robot", sensor->getName(), Transform()));
      const bool added = host.addMeasurement(m);
      if (added_out) added_out[i] = added ? 1 : 0;
    }
    for (size_t e = 0; e < host.edges.size(); ++e) for (int i = 0; i < 16; ++i) T_out[16 * e + i] = host.edges[e].relative.m[i];
    if (n_warnings) *n_warnings = (int)host.warnings.size();
    g_msg = host.warnings.empty() ? "" : host.warnings.back();
    return (int)host.edges.size();
  } catch (std::exception& e) {
    g_msg = e.what();
    return -1;
  }
}

// createCombinedMeasurement on n posed scans (sensor pose = identity): out must hold the sum of the sizes. Returns the size or -1.
int64_t s3dhost_combined_measurement(void* s, const float* const* scans, const uint64_t* sizes, int n, const double* poses, const double* patch_pose, float* out) {
  int64_t m = -1;
  wrap([&] {
    PointCloudSensor* sensor = static_cast<PointCloudSensor*>(s);
    PointCloudSensor::PosedMeasurements v;
    for (int i = 0; i < n; ++i)
      v.emplace_back(PointCloudMeasurement::Ptr(new PointCloudMeasurement(makeCloud(scans[i], sizes[i]), "robot", sensor->getName(), Transform())),
                     makeTransform(poses + 16 * i));
    Measurement::Ptr c = sensor->createCombinedMeasurement(v, makeTransform(patch_pose));
    PointCloudMeasurement::Ptr pc = std::dynamic_pointer_cast<PointCloudMeasurement>(c);
    m = (int64_t)pc->getPointCloud()->size();
    if (m) std::memcpy(out, &pc->getPointCloud()->points[0].x, 16 * m);
  });
  return m;
}

// fillGroundPlane on a copy of the n input points with map resolution `resolution`: out receives the whole resulting cloud
// (input then fill points) and must hold n + s3d_ground_fill_size(resolution, radius) points.  Returns its size or -1.
int64_t s3dhost_fill_ground_plane(void* s, const float* in, uint64_t n, double resolution, double radius, float* out) {
  int64_t m = -1;
  wrap([&] {
    PointCloudSensor* sensor = static_cast<PointCloudSensor*>(s);
    sensor->setMapResolution(resolution);
    PointCloud::Ptr cloud = makeCloud(in, n);
    sensor->fillGroundPlane(cloud, radius);
    m = (int64_t)cloud->size();
    if (m) std::memcpy(out, &cloud->points[0].x, 16 * m);
  });
  return m;
}

}  // extern "C"
