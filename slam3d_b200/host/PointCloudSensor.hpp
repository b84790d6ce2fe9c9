// PointCloudSensor.hpp — host-side mirror of slam3d::PointCloudSensor's scan-matching interface
// (slam3d/sensor/pcl/PointCloudSensor.hpp:106-244) on top of the C-ABI of include/s3d_b200.h.
//
// Same method names, argument meaning and exception behaviour as the reference for the hot path:
//   createConstraint(source, target, odometry, loop)   PointCloudSensor.cpp:269-299
//   setRegistrationParameters(param, coarse)           :320-340
//   setScanResolution / downsample / downsampleScan    :342-346, :190-209
//   transform                                          :228-233
//   removeOutliers / getAccumulatedCloud / createCombinedMeasurement / buildMap   :211-266, :301-318 (vertex lists passed explicitly)
//   fillGroundPlane                                    :362-388 (RANSAC plane fit and ring fill, s3d_fill_ground_plane)
// plus the free function align() (:119-174) and createConstraints(), a batch form of createConstraint for callers that have
// several candidates at hand (ScanSensor::linkToNeighbors, core/ScanSensor.cpp:179-201).  loadPLY and the serializers do no
// arithmetic on this path and stay with the reference (shim/PointCloudSensor.cpp passes them through).
// In a real slam3d build the same bodies replace PointCloudSensor.cpp's downsample()/align() — see INTEGRATION.md.
#pragma once

#include <mutex>

#include "RegistrationParameters.hpp"
#include "Types.hpp"

namespace slam3d_b200 {

// Process-wide C-ABI context (created on first use; re-entrant, see s3d_b200.h).
s3d_context* defaultContext();

// Per-measurement device cache (SURVEY 8f rank 1).  The reference rebuilds filter, trees and covariances (GICP) or the NDT voxel
// Gaussians in every align(); here a scan that is matched again (target then source in odometry, repeated loop-closure candidate)
// is preprocessed once.  GICP and GICP_OMP use handles of s3d_prepare_cloud, NDT and NDT_OMP handles of s3d_prepare_cloud_ndt.
// Keyed by the cloud object (slam3d measurements are immutable once stored, MeasurementStorage.cpp:13-21), the density, the kind
// of handle and its k (GICP) or resolution (NDT); least-recently-used entries are dropped beyond `capacity`.  capacity 0 disables
// the cache (every align() runs the raw path).  preparedCacheHits() counts the hits of both kinds.
void setPreparedCacheCapacity(size_t capacity);
size_t preparedCacheHits();

// Resident scans (optional, off by default).  With a budget > 0 the cloud of a PointCloudMeasurement is uploaded once, on its first
// use, with s3d_upload_scans, and every later call that reads it (align() on the raw path and on prepared-cache misses,
// createConstraints, createLoopConstraints, getAccumulatedCloud, createCombinedMeasurement, buildMap) passes the device view instead
// of uploading it again.  Results are bit for bit those of the host clouds.  Free-standing clouds (the arguments of downsample,
// downsampleScan, transform, removeOutliers, fillGroundPlane) are never stored.  Keyed by the cloud object like the prepared cache;
// an entry is released when its measurement is gone, and least-recently-used entries are released while the stored bytes exceed
// the budget.  A cloud larger than the budget is not stored.  Budget 0 releases every entry and reads host clouds again.
void setResidentScanBudget(size_t bytes);
struct ResidentScanStats { uint64_t uploads = 0, hits = 0, bytes_resident = 0; };  // scans uploaded, lookups served, 16 B per stored point
ResidentScanStats residentScanStats();

// align(source, target, guess, config) — PointCloudSensor.cpp:119-174.  Throws NoMatch / std::runtime_error exactly
// where the reference does.  `result_info` (optional) receives the C-ABI result (fitness, iterations...).
Transform align(PointCloudMeasurement::Ptr source, PointCloudMeasurement::Ptr target, const Transform& guess,
                const RegistrationParameters& config, s3d_result* result_info = nullptr);

class PointCloudSensor {
 public:
  PointCloudSensor(const std::string& n, Logger* l);
  virtual ~PointCloudSensor();

  const std::string& getName() const { return mName; }
  void setCovarianceScale(ScalarType s) { mCovarianceScale = s; }  // core/Sensor.hpp:138

  virtual Constraint::Ptr createConstraint(const Measurement::Ptr& source, const Measurement::Ptr& target, const Transform& odometry, bool loop);
  void setRegistrationParameters(const RegistrationParameters& param, bool coarse);
  void setScanResolution(double r);
  void setMapResolution(double r);                            // :348-352
  void setMapOutlierRemoval(double r, unsigned n);            // :354-360
  static PointCloud::Ptr downsample(PointCloud::Ptr source, double resolution);
  PointCloud::Ptr downsampleScan(PointCloud::Ptr source);
  PointCloud::Ptr transform(PointCloud::ConstPtr source, const Transform tf) const;
  PointCloud::Ptr removeOutliers(PointCloud::Ptr source, double radius, unsigned min_neighbors) const;   // :211-226
  // getAccumulatedCloud / buildMap take the graph's VertexObjectList in the reference (:235-256, :301-318); without a graph
  // the caller passes the same information explicitly: each measurement with its corrected vertex pose.
  typedef std::vector<std::pair<PointCloudMeasurement::Ptr, Transform> > PosedMeasurements;
  PointCloud::Ptr getAccumulatedCloud(const PosedMeasurements& vertices) const;
  PointCloud::Ptr buildMap(const PosedMeasurements& vertices) const;
  // :258-266 — the patch a loop closure is matched with: accumulated cloud re-expressed in the frame `pose`, sensor pose identity
  Measurement::Ptr createCombinedMeasurement(const PosedMeasurements& vertices, Transform pose) const;
  // :362-388 — appends the rings of the RANSAC ground plane (map resolution spacing, up to `radius`) to `cloud`
  void fillGroundPlane(PointCloud::Ptr cloud, ScalarType radius);

  // Batch form of createConstraint (extension): request i gives the same constraint — or fails with the same exception type and
  // message — as createConstraint(source_i, target_i, odometry_i, loop), but all registrations run as ONE device batch
  // (s3d_gicp_align_batch / s3d_gicp_align_loop_batch), which is what the GPU path is fastest at.
  struct ConstraintRequest { Measurement::Ptr source, target; Transform odometry; };
  struct ConstraintResult {
    Constraint::Ptr constraint;  // null when the request failed
    int error = 0;               // 0 none, 1 NoMatch, 2 BadMeasurementType, 3 std::runtime_error
    std::string message;
  };
  std::vector<ConstraintResult> createConstraints(const std::vector<ConstraintRequest>& requests, bool loop);

  // Loop closures between patches (extension): request i gives the same constraint — or fails with the same exception type and
  // message — as createConstraint(createCombinedMeasurement(source_i), createCombinedMeasurement(target_i), odometry_i, true),
  // but the patches never exist on the host: one s3d_prepare_combined_measurements call builds every distinct patch on the device
  // from the distinct scans (each uploaded once) and prepares it for the coarse and the fine configuration, and one
  // s3d_gicp_align_loop_batch_prepared runs all coarse and fine aligns.  Scans are told apart by cloud object, patches by
  // (members, their poses, patch pose); each distinct patch logs createCombinedMeasurement's DEBUG line.  A configuration that no
  // prepared handle serves (ICP, k or resolution out of range) takes the host patches and createConstraints instead.
  struct Patch { PosedMeasurements vertices; Transform pose; };  // the arguments of createCombinedMeasurement
  struct LoopRequest { Patch source, target; Transform odometry; };
  std::vector<ConstraintResult> createLoopConstraints(const std::vector<LoopRequest>& requests);

 protected:
  std::string mName;
  Logger* mLogger;
  ScalarType mCovarianceScale;
  RegistrationParameters mFineConfiguration;
  RegistrationParameters mCoarseConfiguration;
  double mScanResolution;
  double mMapResolution;
  double mMapOutlierRadius;
  unsigned mMapOutlierNeighbors;

 private:
  // the ConstraintResult of one batched createConstraint from its align results (:286-299)
  ConstraintResult resultOf(const s3d_result& coarse, const s3d_result& fine, bool loop, const Transform& source_sensor_pose,
                            const Transform& target_inverse_sensor_pose) const;
};

}  // namespace slam3d_b200
