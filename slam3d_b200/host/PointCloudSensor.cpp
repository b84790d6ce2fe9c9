// PointCloudSensor.cpp — host mirror bodies; all arithmetic goes through the C-ABI (libs3d_b200.so, CUDA sm_100a).
// Reference behaviour cited per function (slam3d/sensor/pcl/PointCloudSensor.cpp).
#include "PointCloudSensor.hpp"

#include <cmath>
#include <cstring>
#include <list>
#include <map>
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

static s3d_cloud asCloud(const PointCloud::Ptr& c) {
  s3d_cloud o;
  o.xyzw = c && c->size() ? &c->points[0].x : nullptr;
  o.n = c ? c->size() : 0;
  return o;
}

namespace {
struct Resident {
  s3d_resident_scan* h = nullptr;
  ~Resident() { if (h) s3d_release_scan(defaultContext(), h); }
};
struct StoreEntry { const PointCloud* key; std::weak_ptr<PointCloud> alive; size_t bytes; std::shared_ptr<Resident> scan; };
std::mutex g_store_mutex;
std::list<StoreEntry> g_store;  // front = most recently used
size_t g_store_budget = 0, g_store_bytes = 0;
uint64_t g_store_uploads = 0, g_store_hits = 0;

// under g_store_mutex: entries whose measurement is gone, then least-recently-used ones while the bytes exceed the budget.  A call
// that still holds an evicted scan keeps it until the call ends.
void storeTrim() {
  for (auto it = g_store.begin(); it != g_store.end();) {
    if (it->alive.expired()) { g_store_bytes -= it->bytes; it = g_store.erase(it); } else ++it;
  }
  while (g_store_bytes > g_store_budget) { g_store_bytes -= g_store.back().bytes; g_store.pop_back(); }
}

// The clouds one call reads, as device views of stored scans where the store holds (or now takes) them; host clouds otherwise.
// The misses of the call are uploaded together, once each.  `hold` keeps the scans of the views alive until the call is done.
struct Views {
  std::vector<s3d_cloud> clouds;
  std::vector<std::shared_ptr<Resident>> hold;
};
Views residentViews(const std::vector<PointCloud::Ptr>& clouds) {
  Views v;
  v.hold.resize(clouds.size());
  for (const PointCloud::Ptr& c : clouds) v.clouds.push_back(asCloud(c));
  std::map<const PointCloud*, size_t> miss;  // cloud -> index of its first occurrence in `clouds`
  {
    std::lock_guard<std::mutex> g(g_store_mutex);
    if (g_store_budget == 0) return v;
    storeTrim();
    for (size_t i = 0; i < clouds.size(); ++i) {
      const size_t bytes = 16 * size_t(v.clouds[i].n);
      if (bytes == 0 || bytes > g_store_budget || miss.count(clouds[i].get())) continue;
      auto it = g_store.begin();
      while (it != g_store.end() && it->key != clouds[i].get()) ++it;
      if (it == g_store.end()) { miss.emplace(clouds[i].get(), i); continue; }
      ++g_store_hits;
      g_store.splice(g_store.begin(), g_store, it);
      v.hold[i] = it->scan;
    }
  }
  if (!miss.empty()) {
    std::vector<s3d_cloud> up;
    for (const auto& m : miss) up.push_back(v.clouds[m.second]);
    std::vector<s3d_resident_scan*> h(up.size(), nullptr);
    if (s3d_upload_scans(defaultContext(), 0, up.data(), (int)up.size(), h.data()) != S3D_OK) throw std::runtime_error(s3d_last_error());
    std::lock_guard<std::mutex> g(g_store_mutex);
    size_t k = 0;
    for (const auto& m : miss) {
      std::shared_ptr<Resident> r(new Resident());
      r->h = h[k++];
      v.hold[m.second] = r;
      ++g_store_uploads;
      bool stored = false;  // another thread may have stored the same cloud meanwhile
      for (const StoreEntry& e : g_store) stored = stored || e.key == m.first;
      if (stored) continue;
      g_store.push_front({m.first, clouds[m.second], 16 * size_t(up[k - 1].n), r});
      g_store_bytes += g_store.front().bytes;
    }
    storeTrim();
  }
  for (size_t i = 0; i < clouds.size(); ++i) {
    if (!v.hold[i]) {  // a later occurrence of a cloud uploaded by this call
      auto m = miss.find(clouds[i].get());
      if (m != miss.end()) v.hold[i] = v.hold[m->second];
    }
    if (v.hold[i]) v.clouds[i] = s3d_resident_scan_cloud(v.hold[i]->h);
  }
  return v;
}
}  // namespace

void setResidentScanBudget(size_t bytes) {
  std::lock_guard<std::mutex> g(g_store_mutex);
  g_store_budget = bytes;
  storeTrim();
}

ResidentScanStats residentScanStats() {
  std::lock_guard<std::mutex> g(g_store_mutex);
  storeTrim();
  ResidentScanStats s;
  s.uploads = g_store_uploads; s.hits = g_store_hits; s.bytes_resident = g_store_bytes;
  return s;
}

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
  const Views v = residentViews({cloud});
  const int st = resolution > 0.f ? s3d_prepare_cloud_ndt(defaultContext(), 0, v.clouds[0], density, resolution, &p->h)
                                  : s3d_prepare_cloud(defaultContext(), 0, v.clouds[0], density, k, &p->h);
  if (st != S3D_OK) throw std::runtime_error(s3d_last_error());
  std::lock_guard<std::mutex> g(g_cache_mutex);
  g_cache.push_front({cloud.get(), cloud, density, k, resolution, p});
  while (g_cache.size() > g_cache_capacity) g_cache.pop_back();
  return p;
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
    const Views v = residentViews({source->getPointCloud(), target->getPointCloud()});
    st = s3d_gicp_align(defaultContext(), v.clouds[0], v.clouds[1], guess.data(), &c, &res);
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
  std::vector<PointCloud::Ptr> clouds;
  for (const auto& v : vertices) clouds.push_back(v.first->getPointCloud());
  const Views views = residentViews(clouds);
  PointCloud::Ptr accu(new PointCloud);
  for (size_t i = 0; i < vertices.size(); ++i) {  // transform(cloud_i, pose_i) of every vertex, appended
    const size_t at = accu->size();
    accu->points.resize(at + views.clouds[i].n);
    const Transform tf = vertices[i].second * vertices[i].first->getSensorPose();
    if (views.clouds[i].n && s3d_transform_cloud(defaultContext(), views.clouds[i], tf.data(), &accu->points[at].x) != S3D_OK)
      throw std::runtime_error(s3d_last_error());
  }
  return accu;
}

// :258-266  one device pass: transform(cloud_i, pose_i) appended in list order, then transformPointCloud(pose.inverse())
Measurement::Ptr PointCloudSensor::createCombinedMeasurement(const PosedMeasurements& vertices, Transform pose) const {
  std::vector<PointCloud::Ptr> scans;
  for (const auto& v : vertices) scans.push_back(v.first->getPointCloud());
  const Views views = residentViews(scans);
  const std::vector<s3d_cloud>& clouds = views.clouds;
  std::vector<double> poses(16 * vertices.size());
  size_t total = 0;
  for (size_t i = 0; i < vertices.size(); ++i) {
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
  std::vector<PointCloud::Ptr> scans;
  for (const auto& v : vertices) scans.push_back(v.first->getPointCloud());
  const Views views = residentViews(scans);
  const std::vector<s3d_cloud>& clouds = views.clouds;
  std::vector<double> poses(16 * vertices.size());
  size_t total = 0;
  for (size_t i = 0; i < vertices.size(); ++i) {
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
  std::vector<PointCloud::Ptr> clouds;  // source, target of each request that reaches the batch
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
    idx.push_back(i); clouds.push_back(sc->getPointCloud()); clouds.push_back(tc->getPointCloud());
    guesses.insert(guesses.end(), guess.m.begin(), guess.m.end());
  }
  const int n = (int)idx.size();
  if (n == 0) return out;
  const Views views = residentViews(clouds);
  std::vector<s3d_cloud> src, tgt;
  for (int k = 0; k < n; ++k) { src.push_back(views.clouds[2 * k]); tgt.push_back(views.clouds[2 * k + 1]); }
  std::vector<s3d_result> coarse(n), fine(n);
  const s3d_registration_parameters cc = mCoarseConfiguration.toC(), cf = mFineConfiguration.toC();
  const int st = loop ? s3d_gicp_align_loop_batch(defaultContext(), src.data(), tgt.data(), guesses.data(), &cc, &cf, n, coarse.data(), fine.data())  // :286-292
                      : s3d_gicp_align_batch(defaultContext(), src.data(), tgt.data(), guesses.data(), &cf, n, fine.data());                           // :292
  if (st != S3D_OK) throw std::runtime_error(s3d_last_error());
  for (int k = 0; k < n; ++k)
    out[idx[k]] = resultOf(coarse[k], fine[k], loop, requests[idx[k]].source->getSensorPose(), requests[idx[k]].target->getInverseSensorPose());
  return out;
}

PointCloudSensor::ConstraintResult PointCloudSensor::resultOf(const s3d_result& coarse, const s3d_result& fine, bool loop,
                                                              const Transform& source_sensor_pose, const Transform& target_inverse_sensor_pose) const {
  ConstraintResult r;
  if (loop && coarse.status != S3D_OK) { failureOf(coarse.status, coarse, mCoarseConfiguration, r.error, r.message); return r; }  // the coarse align threw
  if (fine.status != S3D_OK) { failureOf(fine.status, fine, mFineConfiguration, r.error, r.message); return r; }
  Transform icp_result;
  for (int j = 0; j < 16; ++j) icp_result.m[j] = fine.T[j];
  const Transform tf = source_sensor_pose * icp_result * target_inverse_sensor_pose;  // :295
  Covariance<6> covariance = Covariance<6>::Identity() * mCovarianceScale;          // :296
  r.constraint.reset(new SE3Constraint(mName, tf, covariance.inverseDiagonal()));
  return r;
}

// the spec of the prepared handles an align() with `c` runs on (the cases in which align() takes the prepared path)
static bool preparedSpec(const RegistrationParameters& c, s3d_prepare_spec& spec) {
  if (std::isnan(c.point_cloud_density)) return false;
  if ((c.registration_algorithm == GICP || c.registration_algorithm == GICP_OMP) && c.correspondence_randomness >= 1 && c.correspondence_randomness <= 4096) {
    spec = s3d_prepare_spec{c.point_cloud_density, c.correspondence_randomness, 0.f};
    return true;
  }
  if ((c.registration_algorithm == NDT || c.registration_algorithm == NDT_OMP) && c.resolution > 0.f && std::isfinite(c.resolution)) {
    spec = s3d_prepare_spec{c.point_cloud_density, 0, c.resolution};
    return true;
  }
  return false;
}

std::vector<PointCloudSensor::ConstraintResult> PointCloudSensor::createLoopConstraints(const std::vector<LoopRequest>& requests) {
  std::vector<ConstraintResult> out(requests.size());
  if (requests.empty()) return out;
  s3d_prepare_spec coarse_spec, fine_spec;
  if (!preparedSpec(mCoarseConfiguration, coarse_spec) || !preparedSpec(mFineConfiguration, fine_spec)) {
    std::vector<ConstraintRequest> req;
    for (const LoopRequest& r : requests)
      req.push_back({createCombinedMeasurement(r.source.vertices, r.source.pose), createCombinedMeasurement(r.target.vertices, r.target.pose), r.odometry});
    return createConstraints(req, true);
  }
  // distinct scans by cloud object, distinct patches by (member scans, member poses, patch pose) as bit patterns
  std::vector<PointCloud::Ptr> scans;
  std::map<const PointCloud*, int32_t> scan_of;
  std::vector<int32_t> member_scan, first{0};
  std::vector<double> member_poses, patch_poses;
  std::vector<uint64_t> patch_points;
  std::map<std::vector<uint64_t>, int32_t> patch_of;
  auto bits = [](std::vector<uint64_t>& key, const Transform& t) {
    for (double d : t.m) { uint64_t b; std::memcpy(&b, &d, sizeof b); key.push_back(b); }
  };
  auto patchIndex = [&](const Patch& p) {
    std::vector<uint64_t> key;
    std::vector<int32_t> ms;
    std::vector<Transform> mp;
    uint64_t n = 0;
    for (const auto& v : p.vertices) {
      const PointCloud::Ptr& c = v.first->getPointCloud();
      auto it = scan_of.find(c.get());
      if (it == scan_of.end()) { it = scan_of.emplace(c.get(), (int32_t)scans.size()).first; scans.push_back(c); }
      mp.push_back(v.second * v.first->getSensorPose());  // :248
      ms.push_back(it->second);
      key.push_back((uint64_t)it->second);
      bits(key, mp.back());
      n += c ? c->size() : 0;
    }
    bits(key, p.pose);
    const auto ins = patch_of.emplace(key, (int32_t)patch_points.size());
    if (ins.second) {
      member_scan.insert(member_scan.end(), ms.begin(), ms.end());
      for (const Transform& t : mp) member_poses.insert(member_poses.end(), t.m.begin(), t.m.end());
      first.push_back((int32_t)member_scan.size());
      patch_poses.insert(patch_poses.end(), p.pose.m.begin(), p.pose.m.end());
      patch_points.push_back(n);
      if (mLogger) mLogger->message(DEBUG, "Patch pointcloud has " + std::to_string(n) + " points.");  // :258-266
    }
    return ins.first->second;
  };
  std::vector<int32_t> src(requests.size()), tgt(requests.size());
  for (size_t i = 0; i < requests.size(); ++i) { src[i] = patchIndex(requests[i].source); tgt[i] = patchIndex(requests[i].target); }
  const int n_patches = (int)patch_points.size();
  std::vector<s3d_prepare_spec> specs{coarse_spec};
  if (fine_spec.density != coarse_spec.density || fine_spec.k != coarse_spec.k || fine_spec.resolution != coarse_spec.resolution) specs.push_back(fine_spec);
  const int ns = (int)specs.size();
  struct Handles {  // released when the batch is done, whatever happens
    std::vector<s3d_prepared_cloud*> h;
    ~Handles() { for (s3d_prepared_cloud* p : h) s3d_release_cloud(defaultContext(), p); }
  } hh;
  hh.h.assign((size_t)n_patches * ns, nullptr);
  const Views views = residentViews(scans);
  if (s3d_prepare_combined_measurements(defaultContext(), 0, views.clouds.data(), (int)scans.size(), member_scan.data(), member_poses.data(), first.data(),
                                        patch_poses.data(), n_patches, specs.data(), ns, hh.h.data()) != S3D_OK)
    throw std::runtime_error(s3d_last_error());
  // a patch's sensor pose is the identity (createCombinedMeasurement :265); the guess and the edge are formed as createConstraint
  // forms them (:274, :295)
  const Transform identity = Transform::Identity();
  const int n = (int)requests.size();
  std::vector<const s3d_prepared_cloud*> cs(n), ct(n), fs(n), ft(n);
  std::vector<double> guesses;
  for (int i = 0; i < n; ++i) {
    cs[i] = hh.h[(size_t)src[i] * ns]; ct[i] = hh.h[(size_t)tgt[i] * ns];
    fs[i] = hh.h[(size_t)src[i] * ns + ns - 1]; ft[i] = hh.h[(size_t)tgt[i] * ns + ns - 1];
    const Transform guess = identity.inverse() * requests[i].odometry * identity;
    guesses.insert(guesses.end(), guess.m.begin(), guess.m.end());
  }
  std::vector<s3d_result> coarse(n), fine(n);
  const s3d_registration_parameters cc = mCoarseConfiguration.toC(), cf = mFineConfiguration.toC();
  if (s3d_gicp_align_loop_batch_prepared(defaultContext(), cs.data(), ct.data(), fs.data(), ft.data(), guesses.data(), &cc, &cf, n, coarse.data(),
                                         fine.data()) != S3D_OK)
    throw std::runtime_error(s3d_last_error());
  for (int i = 0; i < n; ++i) out[i] = resultOf(coarse[i], fine[i], true, identity, identity.inverse());
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
