// shim/PointCloudSensor.cpp — replacement translation unit for slam3d/sensor/pcl/PointCloudSensor.cpp.
//
// Compiled INSIDE a slam3d source tree (shim/CMakeLists.txt) against the reference's own, unmodified headers
// (slam3d/sensor/pcl/PointCloudSensor.hpp:106-244, RegistrationParameters.hpp, slam3d/core/*), so the class layout, the Boost
// serializers at the end of PointCloudSensor.hpp, ScanSensor, the graph and the g2o back end are untouched and the library keeps
// its name (libslam3d_sensor_pcl, sensor/pcl/CMakeLists.txt:57-59).  Every method of the class is defined here:
//   * the arithmetic ones go to libs3d_b200.so (include/s3d_b200.h): downsample, transform, removeOutliers, getAccumulatedCloud,
//     createCombinedMeasurement, buildMap, fillGroundPlane and the free function align() behind createConstraint;
//   * loadPLY keeps PCL's PLY reader, so the target still links pcl_io — but no longer pcl_registration, pcl_filters or
//     pcl_sample_consensus.
// This file cannot be compiled in this repository's environment (no PCL / Boost / Eigen, SURVEY 8c); the same bodies with
// stand-in types are compiled and tested as slam3d_b200/host/PointCloudSensor.cpp (tests/test_gpu_host.py).
#include <slam3d/sensor/pcl/PointCloudSensor.hpp>

#include <slam3d/core/Mapper.hpp>

#include <pcl/io/ply_io.h>

#include <boost/format.hpp>

#include <cmath>
#include <stdexcept>
#include <vector>

#include <s3d_b200.h>

using namespace slam3d;

namespace {

// One GPU context per process; the C-ABI is re-entrant (ScanSensor.cpp:209-210 enters createConstraint from a second thread).
s3d_context* gpu() {
  static s3d_context* ctx = [] {
    s3d_context* c = nullptr;
    if (s3d_create_context(nullptr, 0, &c) != S3D_OK) throw std::runtime_error(s3d_last_error());
#ifdef S3D_GICP_USE_BFGS  // built against PCL < 1.14 (shim/CMakeLists.txt): GICP runs that PCL's BFGS inner optimiser
    if (s3d_set_gicp_optimizer(c, S3D_GICP_BFGS, nullptr) != S3D_OK) throw std::runtime_error(s3d_last_error());
#endif
#ifdef S3D_NDT_OMP_USE_DIRECT7  // shim/CMakeLists.txt: NDT_OMP runs pclomp's default DIRECT7 neighbour search
    if (s3d_set_ndt_omp_search(c, S3D_NDT_OMP_DIRECT7, nullptr) != S3D_OK) throw std::runtime_error(s3d_last_error());
#endif
    return c;
  }();
  return ctx;
}

static_assert(sizeof(PointType) == 16, "pcl::PointXYZ is x, y, z, padding: the C-ABI's point layout");

s3d_cloud view(const PointCloud& c) { return s3d_cloud{c.empty() ? nullptr : &c.points[0].x, c.size()}; }

void finish(PointCloud& c, size_t n) {  // what pcl's filters leave behind on an unorganised output cloud
  c.points.resize(n);
  c.width = static_cast<uint32_t>(n);
  c.height = 1;
  c.is_dense = true;
}

s3d_registration_parameters toC(const RegistrationParameters& p) {  // RegistrationParameters.hpp:36-97, same order
  s3d_registration_parameters c;
  c.registration_algorithm = static_cast<int32_t>(p.registration_algorithm);
  c.point_cloud_density = p.point_cloud_density;
  c.max_fitness_score = p.max_fitness_score;
  c.max_translation = p.max_translation;
  c.max_rotation = p.max_rotation;
  c.euclidean_fitness_epsilon = p.euclidean_fitness_epsilon;
  c.transformation_epsilon = p.transformation_epsilon;
  c.max_correspondence_distance = p.max_correspondence_distance;
  c.maximum_iterations = p.maximum_iterations;
  c.rotation_epsilon = p.rotation_epsilon;
  c.correspondence_randomness = p.correspondence_randomness;
  c.maximum_optimizer_iterations = p.maximum_optimizer_iterations;
  c.resolution = p.resolution;
  c.step_size = p.step_size;
  c.outlier_ratio = p.outlier_ratio;
  return c;
}

// (cloud, pose) lists of a vertex list, pose = vertex.correctedPose * measurement.sensorPose   (reference :243-248)
struct PosedClouds {
  std::vector<PointCloud::Ptr> keep;
  std::vector<s3d_cloud> clouds;
  std::vector<double> poses;
  size_t total = 0;
};

PosedClouds collect(const VertexObjectList& vertices, Graph* graph, Logger* logger) {
  PosedClouds pc;
  for (const VertexObject& v : vertices) {
    PointCloudMeasurement::Ptr m = boost::dynamic_pointer_cast<PointCloudMeasurement>(graph->getMeasurement(v.measurementUuid));
    if (!m) {
      logger->message(ERROR, "Measurement in getAccumulatedCloud() is not a point cloud!");
      throw BadMeasurementType();
    }
    const Transform pose = v.correctedPose * m->getSensorPose();
    pc.keep.push_back(m->getPointCloud());
    pc.clouds.push_back(view(*m->getPointCloud()));
    pc.poses.insert(pc.poses.end(), pose.matrix().data(), pose.matrix().data() + 16);  // column-major, like the C-ABI
    pc.total += m->getPointCloud()->size();
  }
  return pc;
}

// align(source, target, guess, config) — reference :119-174.  GICP, GICP_OMP, NDT and NDT_OMP all run on the GPU behind this one
// call; the three NoMatch texts and the runtime_error texts are the reference's (s3d_last_error()).
Transform align(PointCloudMeasurement::Ptr source, PointCloudMeasurement::Ptr target, const Transform& guess, const RegistrationParameters& config) {
  const s3d_registration_parameters c = toC(config);
  s3d_result r;
  switch (s3d_gicp_align(gpu(), view(*source->getPointCloud()), view(*target->getPointCloud()), guess.matrix().data(), &c, &r)) {
    case S3D_OK: break;
    case S3D_TOO_FEW_POINTS:
    case S3D_NOT_CONVERGED:
    case S3D_TOO_FAR_FROM_GUESS: throw NoMatch(s3d_last_error());
    default: throw std::runtime_error(s3d_last_error());
  }
  Transform result;
  for (int i = 0; i < 16; ++i) result.matrix().data()[i] = r.T[i];
  return result;
}

}  // namespace

PointCloudSensor::PointCloudSensor(const std::string& n, Logger* l) : ScanSensor(n, l) {
  mScanResolution = 0.1;
  mMapResolution = 0.1;
  mMapOutlierRadius = 0.2;
  mMapOutlierNeighbors = 3;
}

PointCloudSensor::~PointCloudSensor() {}

PointCloud::Ptr PointCloudSensor::downsample(PointCloud::Ptr in, double leaf_size) {
  PointCloud::Ptr out(new PointCloud);
  if (in->size() > 0) {
    out->points.resize(in->size());
    uint64_t n = 0;
    if (s3d_voxel_downsample(gpu(), view(*in), static_cast<float>(leaf_size), &out->points[0].x, &n, nullptr, nullptr) != S3D_OK)
      throw std::runtime_error(s3d_last_error());
    finish(*out, n);
  }
  return out;
}

PointCloud::Ptr PointCloudSensor::downsampleScan(PointCloud::Ptr source) { return mScanResolution > 0 ? downsample(source, mScanResolution) : source; }

PointCloud::Ptr PointCloudSensor::removeOutliers(PointCloud::Ptr in, double radius, unsigned min_neighbors) const {
  if (!(in->size() > 0 && radius > 0 && min_neighbors > 0)) return in;
  PointCloud::Ptr out(new PointCloud);
  out->points.resize(in->size());
  uint64_t n = 0;
  if (s3d_remove_outliers(gpu(), view(*in), radius, min_neighbors, &out->points[0].x, &n) != S3D_OK) throw std::runtime_error(s3d_last_error());
  finish(*out, n);
  return out;
}

PointCloud::Ptr PointCloudSensor::transform(PointCloud::ConstPtr source, const Transform tf) const {
  PointCloud::Ptr out(new PointCloud(*source));  // header, sensor origin and orientation travel with the copy, as in pcl::transformPointCloud
  if (source->size() && s3d_transform_cloud(gpu(), view(*source), tf.matrix().data(), &out->points[0].x) != S3D_OK) throw std::runtime_error(s3d_last_error());
  return out;
}

PointCloud::Ptr PointCloudSensor::getAccumulatedCloud(const VertexObjectList& vertices) const {
  PosedClouds pc = collect(vertices, mMapper->getGraph(), mLogger);
  PointCloud::Ptr accu(new PointCloud);
  accu->points.resize(pc.total);
  uint64_t n = 0;
  if (s3d_create_combined_measurement(gpu(), pc.clouds.data(), pc.poses.data(), static_cast<int>(pc.clouds.size()), nullptr,
                                      pc.total ? &accu->points[0].x : nullptr, &n) != S3D_OK)
    throw std::runtime_error(s3d_last_error());
  finish(*accu, n);
  return accu;
}

Measurement::Ptr PointCloudSensor::createCombinedMeasurement(const VertexObjectList& vertices, Transform pose) const {
  PosedClouds pc = collect(vertices, mMapper->getGraph(), mLogger);
  PointCloud::Ptr shifted(new PointCloud);
  shifted->points.resize(pc.total);
  uint64_t n = 0;
  if (s3d_create_combined_measurement(gpu(), pc.clouds.data(), pc.poses.data(), static_cast<int>(pc.clouds.size()), pose.matrix().data(),
                                      pc.total ? &shifted->points[0].x : nullptr, &n) != S3D_OK)
    throw std::runtime_error(s3d_last_error());
  finish(*shifted, n);
  mLogger->message(DEBUG, (boost::format("Patch pointcloud has %1% points.") % n).str());
  return Measurement::Ptr(new PointCloudMeasurement(shifted, "AccumulatedPointcloud", mName, Transform::Identity()));
}

Constraint::Ptr PointCloudSensor::createConstraint(const Measurement::Ptr& source, const Measurement::Ptr& target, const Transform& odometry, bool loop) {
  Transform guess = source->getInverseSensorPose() * odometry * target->getSensorPose();  // the guess in the sensor frame
  PointCloudMeasurement::Ptr sourceCloud = boost::dynamic_pointer_cast<PointCloudMeasurement>(source);
  PointCloudMeasurement::Ptr targetCloud = boost::dynamic_pointer_cast<PointCloudMeasurement>(target);
  if (!sourceCloud || !targetCloud) {
    mLogger->message(ERROR, "Measurement given to createConstraint() is not a PointCloud!");
    throw BadMeasurementType();
  }
  if (loop) guess = align(sourceCloud, targetCloud, guess, mCoarseConfiguration);  // a loop closure is initialised by the coarse set
  const Transform icp_result = align(sourceCloud, targetCloud, guess, mFineConfiguration);
  const Transform tf = source->getSensorPose() * icp_result * target->getInverseSensorPose();  // back to the robot frame
  const Covariance<6> covariance = Covariance<6>::Identity() * mCovarianceScale;
  return Constraint::Ptr(new SE3Constraint(mName, tf, covariance.inverse()));
}

PointCloud::Ptr PointCloudSensor::buildMap(const VertexObjectList& vertices) const {
  Clock clock;
  const timeval start = clock.now();
  PointCloud::Ptr map(new PointCloud);
  try {
    PosedClouds pc = collect(vertices, mMapper->getGraph(), mLogger);
    map->points.resize(pc.total);
    uint64_t n = 0;
    // accumulate + removeOutliers + downsample in one device pass
    if (s3d_build_map(gpu(), pc.clouds.data(), pc.poses.data(), static_cast<int>(pc.clouds.size()), mMapOutlierRadius, mMapOutlierNeighbors, mMapResolution,
                      pc.total ? &map->points[0].x : nullptr, &n) != S3D_OK)
      throw std::runtime_error(s3d_last_error());
    finish(*map, n);
  } catch (BadMeasurementType&) {
    throw;  // getAccumulatedCloud sits outside the reference's try block
  } catch (std::exception& e) {
    mLogger->message(ERROR, e.what());
  }
  const timeval end = clock.now();
  mLogger->message(INFO, (boost::format("Generated Pointcloud from %1% scans in %2% seconds.") % vertices.size() % (end.tv_sec - start.tv_sec)).str());
  return map;
}

void PointCloudSensor::setRegistrationParameters(const RegistrationParameters& conf, bool coarse) {
  (coarse ? mCoarseConfiguration : mFineConfiguration) = conf;
  mLogger->message(INFO, coarse ? " = RegistrationParameters (Coarse) =" : " = RegistrationParameters (Fine) =");
  auto line = [this](const char* name, double value) { mLogger->message(INFO, (boost::format("%-29s %2%") % (std::string(name) + ":") % value).str()); };
  line("correspondence_randomness", conf.correspondence_randomness);
  line("euclidean_fitness_epsilon", conf.euclidean_fitness_epsilon);
  line("max_correspondence_distance", conf.max_correspondence_distance);
  line("max_fitness_score", conf.max_fitness_score);
  line("maximum_iterations", conf.maximum_iterations);
  line("maximum_optimizer_iterations", conf.maximum_optimizer_iterations);
  line("point_cloud_density", conf.point_cloud_density);
  line("rotation_epsilon", conf.rotation_epsilon);
  line("transformation_epsilon", conf.transformation_epsilon);
}

void PointCloudSensor::setScanResolution(double r) {
  mLogger->message(INFO, (boost::format("scan_resolution:        %1%") % r).str());
  mScanResolution = r;
}

void PointCloudSensor::setMapResolution(double r) {
  mLogger->message(INFO, (boost::format("map_resolution:         %1%") % r).str());
  mMapResolution = r;
}

void PointCloudSensor::setMapOutlierRemoval(double r, unsigned n) {
  mLogger->message(INFO, (boost::format("map_outlier_radius:     %1%") % r).str());
  mLogger->message(INFO, (boost::format("map_outlier_neighbors:  %1%") % n).str());
  mMapOutlierRadius = r;
  mMapOutlierNeighbors = n;
}

// :362-388 on the GPU: PCL's RANSAC plane fit (same seed, same samples, same plane) and the rings of points at map resolution laid
// into the plane around the origin (s3d_fill_ground_plane, DESIGN.md 6f).
void PointCloudSensor::fillGroundPlane(PointCloud::Ptr cloud, ScalarType radius) {
  uint64_t m = 0;
  if (s3d_ground_fill_size(mMapResolution, radius, &m) != S3D_OK) throw std::runtime_error(s3d_last_error());
  std::vector<PointType, Eigen::aligned_allocator<PointType> > fill(m);
  if (s3d_fill_ground_plane(gpu(), view(*cloud), mMapResolution, radius, m ? &fill[0].x : nullptr, nullptr) != S3D_OK)
    throw std::runtime_error(s3d_last_error());
  for (const PointType& p : fill) cloud->push_back(p);
}

// Not on the hot path: the PLY reader stays with PCL; the cloud becomes vertex + pose prior exactly as before.
void PointCloudSensor::loadPLY(const std::string& path, const std::string& robot) {
  PointCloud::Ptr cloud(new PointCloud());
  pcl::PLYReader reader;
  if (reader.read(path, *cloud) != 0) {
    mLogger->message(ERROR, "Could not load initial map.");
    return;
  }
  Transform sensor_pose(cloud->sensor_orientation_.cast<ScalarType>());
  sensor_pose.translation() = cloud->sensor_origin_.block(0, 0, 3, 1).cast<ScalarType>();
  PointCloudMeasurement::Ptr initial_map(new PointCloudMeasurement(cloud, robot, mName, sensor_pose));
  try {
    const IdType id = mMapper->getGraph()->addVertex(initial_map, Transform::Identity());
    Constraint::Ptr prior(new PoseConstraint(mName, Transform::Identity(), Covariance<6>::Identity()));
    mMapper->getGraph()->addConstraint(id, 0, prior);
    mLogger->message(INFO, "Successfully loaded initial map.");
  } catch (std::exception& e) {
    mLogger->message(ERROR, (boost::format("Adding initial point cloud failed: %1%") % e.what()).str());
  }
}
