// PointCloudSensor.cpp — host mirror bodies; all arithmetic goes through the C-ABI (libs3d_b200.so, CUDA sm_100a).
// Reference behaviour cited per function (slam3d/sensor/pcl/PointCloudSensor.cpp).
#include "PointCloudSensor.hpp"

#include <cmath>
#include <list>
#include <stdexcept>

namespace slam3d_b200 {

s3d_context* defaultContext() {
  static std::once_flag once;
  static s3d_context* ctx = nullptr;
  static int status = S3D_OK;
  static std::string err;
  std::call_once(once, [] {
    status = s3d_create_context(nullptr, 0, &ctx);
#ifdef S3D_GICP_USE_BFGS  // built against PCL < 1.14 (shim/CMakeLists.txt): GICP runs that PCL's BFGS inner optimiser
    if (status == S3D_OK) status = s3d_set_gicp_optimizer(ctx, S3D_GICP_BFGS, nullptr);
#endif
#ifdef S3D_NDT_OMP_USE_DIRECT7  // shim/CMakeLists.txt: NDT_OMP runs pclomp's default DIRECT7 neighbour search
    if (status == S3D_OK) status = s3d_set_ndt_omp_search(ctx, S3D_NDT_OMP_DIRECT7, nullptr);
#endif
    if (status != S3D_OK) err = s3d_last_error();
  });
  if (!ctx) throw std::runtime_error("slam3d_b200: cannot create CUDA context: " + err);
  return ctx;
}

namespace {
struct Prepared {
  s3d_prepared_cloud* h = nullptr;
  ~Prepared() { if (h) s3d_release_cloud(defaultContext(), h); }
};
// key: (cloud, density, kind, k | resolution); GICP entries have resolution 0, NDT entries k 0
struct CacheEntry { const PointCloud* key; std::weak_ptr<PointCloud> alive; double density; int k; float resolution; std::shared_ptr<Prepared> prepared; };
std::mutex g_cache_mutex;
std::list<CacheEntry> g_cache;  // front = most recently used
size_t g_cache_capacity = 32;
size_t g_cache_hits = 0;
}  // namespace

void setPreparedCacheCapacity(size_t capacity) {
  std::lock_guard<std::mutex> g(g_cache_mutex);
  g_cache_capacity = capacity;
  while (g_cache.size() > g_cache_capacity) g_cache.pop_back();
}
size_t preparedCacheHits() { std::lock_guard<std::mutex> g(g_cache_mutex); return g_cache_hits; }

static s3d_cloud asCloud(const PointCloud::Ptr& c);

// the prepared form of `cloud` for (density, k) — or, with resolution > 0, its NDT form for (density, resolution): from the
// cache, or built now and remembered
static std::shared_ptr<Prepared> prepared(const PointCloud::Ptr& cloud, double density, int k, float resolution = 0.f) {
  {
    std::lock_guard<std::mutex> g(g_cache_mutex);
    for (auto it = g_cache.begin(); it != g_cache.end();) {
      if (it->alive.expired()) { it = g_cache.erase(it); continue; }  // the measurement is gone; its address may be reused
      if (it->key == cloud.get() && it->density == density && it->k == k && it->resolution == resolution) {
        ++g_cache_hits;
        g_cache.splice(g_cache.begin(), g_cache, it);
        return g_cache.front().prepared;
      }
      ++it;
    }
  }
  std::shared_ptr<Prepared> p(new Prepared());
  const int st = resolution > 0.f ? s3d_prepare_cloud_ndt(defaultContext(), 0, asCloud(cloud), density, resolution, &p->h)
                                  : s3d_prepare_cloud(defaultContext(), 0, asCloud(cloud), density, k, &p->h);
  if (st != S3D_OK) throw std::runtime_error(s3d_last_error());
  std::lock_guard<std::mutex> g(g_cache_mutex);
  g_cache.push_front({cloud.get(), cloud, density, k, resolution, p});
  while (g_cache.size() > g_cache_capacity) g_cache.pop_back();
  return p;
}

static s3d_cloud asCloud(const PointCloud::Ptr& c) {
  s3d_cloud o;
  o.xyzw = c && c->size() ? &c->points[0].x : nullptr;
  o.n = c ? c->size() : 0;
  return o;
}

// :119-174
Transform align(PointCloudMeasurement::Ptr source, PointCloudMeasurement::Ptr target, const Transform& guess,
                const RegistrationParameters& config, s3d_result* result_info) {
  const s3d_registration_parameters c = config.toC();
  s3d_result res;
  int st;
  bool use_cache;
  { std::lock_guard<std::mutex> g(g_cache_mutex); use_cache = g_cache_capacity > 0; }
  const bool ndt = config.registration_algorithm == NDT || config.registration_algorithm == NDT_OMP;
  if (use_cache && (config.registration_algorithm == GICP || config.registration_algorithm == GICP_OMP) && config.correspondence_randomness >= 1 && config.correspondence_randomness <= 4096) {
    std::shared_ptr<Prepared> ps = prepared(source->getPointCloud(), config.point_cloud_density, config.correspondence_randomness);
    std::shared_ptr<Prepared> pt = prepared(target->getPointCloud(), config.point_cloud_density, config.correspondence_randomness);
    st = s3d_gicp_align_prepared(defaultContext(), ps->h, pt->h, guess.data(), &c, &res);
  } else if (use_cache && ndt && config.resolution > 0.f && std::isfinite(config.resolution) && !std::isnan(config.point_cloud_density)) {
    std::shared_ptr<Prepared> ps = prepared(source->getPointCloud(), config.point_cloud_density, 0, config.resolution);
    std::shared_ptr<Prepared> pt = prepared(target->getPointCloud(), config.point_cloud_density, 0, config.resolution);
    st = s3d_gicp_align_prepared(defaultContext(), ps->h, pt->h, guess.data(), &c, &res);
  } else {
    st = s3d_gicp_align(defaultContext(), asCloud(source->getPointCloud()), asCloud(target->getPointCloud()), guess.data(), &c, &res);
  }
  if (result_info) *result_info = res;
  switch (st) {
    case S3D_OK: break;
    case S3D_TOO_FEW_POINTS:        // :134-135
    case S3D_NOT_CONVERGED:         // :74-77
    case S3D_TOO_FAR_FROM_GUESS:    // :167-172
      throw NoMatch(s3d_last_error());
    case S3D_UNKNOWN_ALGORITHM:     // :158-164
    default:
      throw std::runtime_error(s3d_last_error());
  }
  Transform result;
  for (int i = 0; i < 16; ++i) result.m[i] = res.T[i];
  return result;
}

PointCloudSensor::PointCloudSensor(const std::string& n, Logger* l) : mName(n), mLogger(l), mCovarianceScale(1.0) {
  mScanResolution = 0.1;  // :179-182
  mMapResolution = 0.1;
  mMapOutlierRadius = 0.2;
  mMapOutlierNeighbors = 3;
}

PointCloudSensor::~PointCloudSensor() {}

// :190-201
PointCloud::Ptr PointCloudSensor::downsample(PointCloud::Ptr in, double leaf_size) {
  PointCloud::Ptr out(new PointCloud);
  if (in->size() > 0) {
    out->points.resize(in->size());
    uint64_t n_out = 0;
    const int st = s3d_voxel_downsample(defaultContext(), asCloud(in), static_cast<float>(leaf_size), &out->points[0].x, &n_out, nullptr, nullptr);
    if (st != S3D_OK) throw std::runtime_error(s3d_last_error());
    out->points.resize(n_out);
  }
  return out;
}

// :203-209
PointCloud::Ptr PointCloudSensor::downsampleScan(PointCloud::Ptr source) {
  if (mScanResolution > 0) return downsample(source, mScanResolution);
  return source;
}

// :228-233  pcl::transformPointCloud(*source, *out, tf.matrix()) — double matrix, float points
PointCloud::Ptr PointCloudSensor::transform(PointCloud::ConstPtr source, const Transform tf) const {
  PointCloud::Ptr out(new PointCloud);
  out->points.resize(source->size());
  if (source->size()) {
    s3d_cloud in{&source->points[0].x, source->size()};
    if (s3d_transform_cloud(defaultContext(), in, tf.data(), &out->points[0].x) != S3D_OK) throw std::runtime_error(s3d_last_error());
  }
  return out;
}

// :211-226
PointCloud::Ptr PointCloudSensor::removeOutliers(PointCloud::Ptr in, double radius, unsigned min_neighbors) const {
  if (in->size() > 0 && radius > 0 && min_neighbors > 0) {
    PointCloud::Ptr out(new PointCloud);
    out->points.resize(in->size());
    uint64_t n = 0;
    if (s3d_remove_outliers(defaultContext(), asCloud(in), radius, min_neighbors, &out->points[0].x, &n) != S3D_OK) throw std::runtime_error(s3d_last_error());
    out->points.resize(n);
    return out;
  }
  return in;
}

// :362-388  RANSAC ground plane of the cloud, then rings of points every mMapResolution up to `radius` appended to it
void PointCloudSensor::fillGroundPlane(PointCloud::Ptr cloud, ScalarType radius) {
  uint64_t m = 0;
  if (s3d_ground_fill_size(mMapResolution, radius, &m) != S3D_OK) throw std::runtime_error(s3d_last_error());
  std::vector<PointType> fill(m);
  if (s3d_fill_ground_plane(defaultContext(), asCloud(cloud), mMapResolution, radius, m ? &fill[0].x : nullptr, nullptr) != S3D_OK)
    throw std::runtime_error(s3d_last_error());
  cloud->points.insert(cloud->points.end(), fill.begin(), fill.end());
}

// :235-256  (pose = vertex.correctedPose * measurement.sensorPose, accumulated in list order)
PointCloud::Ptr PointCloudSensor::getAccumulatedCloud(const PosedMeasurements& vertices) const {
  PointCloud::Ptr accu(new PointCloud);
  for (size_t i = 0; i < vertices.size(); ++i) {
    PointCloud::Ptr t = transform(vertices[i].first->getPointCloud(), vertices[i].second * vertices[i].first->getSensorPose());
    accu->points.insert(accu->points.end(), t->points.begin(), t->points.end());
  }
  return accu;
}

// :258-266  one device pass: transform(cloud_i, pose_i) appended in list order, then transformPointCloud(pose.inverse())
Measurement::Ptr PointCloudSensor::createCombinedMeasurement(const PosedMeasurements& vertices, Transform pose) const {
  std::vector<s3d_cloud> clouds(vertices.size());
  std::vector<double> poses(16 * vertices.size());
  size_t total = 0;
  for (size_t i = 0; i < vertices.size(); ++i) {
    clouds[i] = asCloud(vertices[i].first->getPointCloud());
    const Transform p = vertices[i].second * vertices[i].first->getSensorPose();  // :248
    for (int j = 0; j < 16; ++j) poses[16 * i + j] = p.m[j];
    total += clouds[i].n;
  }
  PointCloud::Ptr shifted(new PointCloud);
  shifted->points.resize(total);
  uint64_t n = 0;
  if (s3d_create_combined_measurement(defaultContext(), clouds.data(), poses.data(), (int)vertices.size(), pose.data(),
                                      total ? &shifted->points[0].x : nullptr, &n) != S3D_OK)
    throw std::runtime_error(s3d_last_error());
  shifted->points.resize(n);
  if (mLogger) mLogger->message(DEBUG, "Patch pointcloud has " + std::to_string(n) + " points.");
  return Measurement::Ptr(new PointCloudMeasurement(shifted, "AccumulatedPointcloud", mName, Transform::Identity()));
}

// :301-318  one device pass: accumulate -> removeOutliers -> downsample
PointCloud::Ptr PointCloudSensor::buildMap(const PosedMeasurements& vertices) const {
  PointCloud::Ptr map(new PointCloud);
  std::vector<s3d_cloud> clouds(vertices.size());
  std::vector<double> poses(16 * vertices.size());
  size_t total = 0;
  for (size_t i = 0; i < vertices.size(); ++i) {
    clouds[i] = asCloud(vertices[i].first->getPointCloud());
    const Transform p = vertices[i].second * vertices[i].first->getSensorPose();
    for (int j = 0; j < 16; ++j) poses[16 * i + j] = p.m[j];
    total += clouds[i].n;
  }
  map->points.resize(total);
  uint64_t n = 0;
  const int st = s3d_build_map(defaultContext(), clouds.data(), poses.data(), (int)vertices.size(), mMapOutlierRadius, mMapOutlierNeighbors,
                               mMapResolution, total ? &map->points[0].x : nullptr, &n);
  if (st != S3D_OK && mLogger) mLogger->message(ERROR, s3d_last_error());  // :309-312 logs and returns what it has
  map->points.resize(st == S3D_OK ? n : 0);
  return map;
}

// :269-299
Constraint::Ptr PointCloudSensor::createConstraint(const Measurement::Ptr& source, const Measurement::Ptr& target, const Transform& odometry, bool loop) {
  // Transform guess in sensor frame  (:274)
  Transform guess = source->getInverseSensorPose() * odometry * target->getSensorPose();
  PointCloudMeasurement::Ptr sourceCloud = std::dynamic_pointer_cast<PointCloudMeasurement>(source);
  PointCloudMeasurement::Ptr targetCloud = std::dynamic_pointer_cast<PointCloudMeasurement>(target);
  if (!sourceCloud || !targetCloud) {  // :279-283
    if (mLogger) mLogger->message(ERROR, "Measurement given to createConstraint() is not a PointCloud!");
    throw BadMeasurementType();
  }
  if (loop) guess = align(sourceCloud, targetCloud, guess, mCoarseConfiguration);  // :286-289
  Transform icp_result = align(sourceCloud, targetCloud, guess, mFineConfiguration);  // :292
  Transform tf = source->getSensorPose() * icp_result * target->getInverseSensorPose();  // :295
  Covariance<6> covariance = Covariance<6>::Identity() * mCovarianceScale;  // :296
  return Constraint::Ptr(new SE3Constraint(mName, tf, covariance.inverseDiagonal()));
}

// what align() throws for a per-pair status of a batch call (same texts as the single call, PointCloudSensor.cpp:74-77, :134-135, :167-172)
static void failureOf(int st, const s3d_result& r, const RegistrationParameters& cfg, int& kind, std::string& msg) {
  switch (st) {
    case S3D_TOO_FEW_POINTS: kind = 1; msg = "Too few points after filtering, you may have to decrease 'point_cloud_density'."; break;
    case S3D_NOT_CONVERGED:
      kind = 1;
      msg = std::string(cfg.registration_algorithm == NDT || cfg.registration_algorithm == NDT_OMP ? "NDT" : "ICP") + " failed with Fitness-Score " +
            std::to_string(r.fitness) + " > " + std::to_string(cfg.max_fitness_score);
      break;
    case S3D_TOO_FAR_FROM_GUESS: kind = 1; msg = "ICP result is to far away from guess"; break;
    case S3D_UNKNOWN_ALGORITHM: kind = 3; msg = "Unknown registration algorithm specified."; break;
    default: kind = 3; msg = s3d_last_error(); break;
  }
}

std::vector<PointCloudSensor::ConstraintResult> PointCloudSensor::createConstraints(const std::vector<ConstraintRequest>& requests, bool loop) {
  std::vector<ConstraintResult> out(requests.size());
  std::vector<size_t> idx;
  std::vector<s3d_cloud> src, tgt;
  std::vector<double> guesses;
  for (size_t i = 0; i < requests.size(); ++i) {
    PointCloudMeasurement::Ptr sc = std::dynamic_pointer_cast<PointCloudMeasurement>(requests[i].source);
    PointCloudMeasurement::Ptr tc = std::dynamic_pointer_cast<PointCloudMeasurement>(requests[i].target);
    if (!sc || !tc) {  // :279-283
      if (mLogger) mLogger->message(ERROR, "Measurement given to createConstraint() is not a PointCloud!");
      out[i].error = 2; out[i].message = BadMeasurementType().what();
      continue;
    }
    const Transform guess = requests[i].source->getInverseSensorPose() * requests[i].odometry * requests[i].target->getSensorPose();  // :274
    idx.push_back(i); src.push_back(asCloud(sc->getPointCloud())); tgt.push_back(asCloud(tc->getPointCloud()));
    guesses.insert(guesses.end(), guess.m.begin(), guess.m.end());
  }
  const int n = (int)idx.size();
  if (n == 0) return out;
  std::vector<s3d_result> coarse(n), fine(n);
  const s3d_registration_parameters cc = mCoarseConfiguration.toC(), cf = mFineConfiguration.toC();
  const int st = loop ? s3d_gicp_align_loop_batch(defaultContext(), src.data(), tgt.data(), guesses.data(), &cc, &cf, n, coarse.data(), fine.data())  // :286-292
                      : s3d_gicp_align_batch(defaultContext(), src.data(), tgt.data(), guesses.data(), &cf, n, fine.data());                           // :292
  if (st != S3D_OK) throw std::runtime_error(s3d_last_error());
  for (int k = 0; k < n; ++k) {
    ConstraintResult& r = out[idx[k]];
    if (loop && coarse[k].status != S3D_OK) { failureOf(coarse[k].status, coarse[k], mCoarseConfiguration, r.error, r.message); continue; }  // the coarse align threw
    if (fine[k].status != S3D_OK) { failureOf(fine[k].status, fine[k], mFineConfiguration, r.error, r.message); continue; }
    Transform icp_result;
    for (int j = 0; j < 16; ++j) icp_result.m[j] = fine[k].T[j];
    const Transform tf = requests[idx[k]].source->getSensorPose() * icp_result * requests[idx[k]].target->getInverseSensorPose();  // :295
    Covariance<6> covariance = Covariance<6>::Identity() * mCovarianceScale;                                                      // :296
    r.constraint.reset(new SE3Constraint(mName, tf, covariance.inverseDiagonal()));
  }
  return out;
}

// :320-340
void PointCloudSensor::setRegistrationParameters(const RegistrationParameters& conf, bool coarse) {
  if (coarse) mCoarseConfiguration = conf; else mFineConfiguration = conf;
  if (mLogger) mLogger->message(INFO, coarse ? " = RegistrationParameters (Coarse) =" : " = RegistrationParameters (Fine) =");
}

// :342-360
void PointCloudSensor::setScanResolution(double r) { mScanResolution = r; }
void PointCloudSensor::setMapResolution(double r) { mMapResolution = r; }
void PointCloudSensor::setMapOutlierRemoval(double r, unsigned n) { mMapOutlierRadius = r; mMapOutlierNeighbors = n; }

}  // namespace slam3d_b200
