// MiniHost.hpp — a dependency-free stand-in for the CALLER of the hot path: the link-to-previous policy of
// slam3d::ScanSensor::addMeasurement(m, odom) (slam3d/core/ScanSensor.cpp:94-135) and the loop-closure call of
// ScanSensor::link (:137-168), with a recording "graph" instead of BoostGraph/g2o (not installed here, SURVEY 8c).
// It exists so tests can drive createConstraint in the reference's call order, with its exception handling
// (NoMatch -> warning, vertex stays unlinked) and from two threads at once (ScanSensor.cpp:209-210).
// linkLastToNeighbors() reproduces ScanSensor::linkToNeighbors (:170-202) on the recorded graph: vertices within
// mNeighborRadius of the new vertex's corrected pose (Graph::getNearbyVertices, core/Graph.cpp:240-261), newest first, no
// existing edge, hop distance (BoostGraph::calculateGraphDistance, unit edge weights) >= mMinLoopLength, at most
// mMaxNeighorLinks links, each through link(index, vertex) with the graph's current relative pose as the guess (:137-142).
// link() matches PATCHES (ScanSensor::buildPatch, :215-270, without a patch solver: mPatchSolver == NULL): the scans within
// mPatchBuildingRange hops of a vertex (BoostGraph::getVerticesInRange, graph/boost/BoostGraph.cpp:274-299, vertex-id order),
// accumulated and re-expressed in the vertex' frame by PointCloudSensor::createCombinedMeasurement.
// linkLastToNeighbors(true) hands all candidates of a vertex to PointCloudSensor::createConstraints — ONE device batch through
// s3d_gicp_align_loop_batch — instead of one createConstraint per candidate; edges and warnings are the same.  With
// setDevicePatches(true) and patches, that batch goes through PointCloudSensor::createLoopConstraints: the patches are built and
// prepared on the device and never copied to the host.
#pragma once

#include <cmath>
#include <map>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "PointCloudSensor.hpp"

namespace slam3d_b200 {

struct RecordedEdge { unsigned source, target; Transform relative; Covariance<6> information; bool loop; };

class MiniHost {
 public:
  explicit MiniHost(PointCloudSensor* s) : mSensor(s), mLastVertex(0), mHasVertex(false), mLinkPrevious(true) {}

  // Sensor::checkMinDistance  core/Sensor.cpp:33-41 (angle of the rotation part like Eigen::AngleAxis: via the trace, in [0, pi])
  bool checkMinDistance(const Transform& t) const {
    const double tr = t(0, 0) + t(1, 1) + t(2, 2);
    const double rot = std::acos(std::fmin(1.0, std::fmax(-1.0, (tr - 1.0) / 2.0)));
    return !(t.translationNorm() < mMinTranslation && std::fabs(rot) < mMinRotation);
  }
  void setMinPoseDistance(float t, float r) { mMinTranslation = t; mMinRotation = r; }  // Sensor::setMinPoseDistance :43-48

  // ScanSensor::addMeasurement(m)  :49-79 — no odometry: the guess is the motion since the last vertex, chained from the
  // previous registration results (mLastTransform), and a scan only becomes a vertex once it has moved far enough
  bool addMeasurement(const Measurement::Ptr& m) {
    if (!mHasVertex) {  // :51-55
      mMeasurements.push_back(m); mLastVertex = 0; mHasVertex = true;
      mCorrected.push_back(Transform::Identity()); mAdjacency.emplace_back();
      return true;
    }
    try {
      Constraint::Ptr c = mSensor->createConstraint(mMeasurements[mLastVertex], m, mLastTransform, false);  // :60
      SE3Constraint::Ptr se3 = std::dynamic_pointer_cast<SE3Constraint>(c);
      if (se3) mLastTransform = se3->getRelativePose();
      if (!se3 || checkMinDistance(mLastTransform)) {  // :62
        const unsigned newVertex = static_cast<unsigned>(mMeasurements.size());
        mMeasurements.push_back(m);
        mCorrected.push_back(mCorrected[mLastVertex]); mAdjacency.emplace_back();
        if (se3) { mCorrected[newVertex] = mCorrected[mLastVertex] * mLastTransform; mLastTransform = Transform::Identity(); }  // :65-69: getCurrentPose()
        record(mLastVertex, newVertex, c, false);  // :70
        mLastVertex = newVertex;
        return true;
      }
    } catch (std::exception& e) {  // :74-77
      std::lock_guard<std::mutex> g(mMutex);
      warnings.push_back(std::string("Could not add Measurement: ") + e.what());
    }
    return false;
  }

  // ScanSensor::addMeasurement(m, odom)  :94-135
  bool addMeasurement(const Measurement::Ptr& m, const Transform& odom) {
    if (!mHasVertex) {  // :96-101
      mMeasurements.push_back(m); mLastVertex = 0; mHasVertex = true; mLastOdometry = odom;
      mCorrected.push_back(Transform::Identity()); mAdjacency.emplace_back();  // Mapper::addMeasurement: vertex at mStartPose
      return true;
    }
    Transform lastTransform = mLastOdometry.inverse() * odom;  // :104
    if (!checkMinDistance(lastTransform)) return false;         // :105, :134
    const unsigned newVertex = static_cast<unsigned>(mMeasurements.size());
    Measurement::Ptr source = mMeasurements[mLastVertex];
    mMeasurements.push_back(m);  // :107
    mCorrected.push_back(mCorrected[mLastVertex]); mAdjacency.emplace_back();  // Mapper.cpp:89: new vertex at the mapper's current pose
    if (mLinkPrevious) {
      try {
        Constraint::Ptr c = mSensor->createConstraint(source, m, lastTransform, false);  // :113
        record(mLastVertex, newVertex, c, false);                                        // :114
        SE3Constraint::Ptr se3 = std::dynamic_pointer_cast<SE3Constraint>(c);            // :117-123
        if (se3) mCorrected[newVertex] = mCorrected[mLastVertex] * se3->getRelativePose();
      } catch (std::exception& e) {  // :124-127
        std::lock_guard<std::mutex> g(mMutex);
        warnings.push_back(std::string("Could not link Measurement to previous: ") + e.what());
      }
    }
    mLastOdometry = odom; mLastVertex = newVertex;  // :129-131
    return true;
  }

  // ScanSensor::buildPatch(source)  :215-270 with mPatchSolver == NULL
  Measurement::Ptr buildPatch(unsigned source) const {
    if (mPatchBuildingRange == 0) return mMeasurements[source];  // :217-220
    const PointCloudSensor::Patch p = patchOf(source);
    return mSensor->createCombinedMeasurement(p.vertices, p.pose);  // :269
  }

  // the arguments buildPatch hands to createCombinedMeasurement (mPatchBuildingRange > 0)
  PointCloudSensor::Patch patchOf(unsigned source) const {
    // Graph::getVerticesInRange: breadth-first search to depth mPatchBuildingRange, result in vertex order (std::map<Vertex, depth>)
    std::map<unsigned, unsigned> depth;
    depth[source] = 0;
    std::vector<unsigned> queue{source};
    for (size_t h = 0; h < queue.size(); ++h) {
      const unsigned v = queue[h];
      if (depth[v] >= mPatchBuildingRange) continue;
      for (unsigned o : mAdjacency[v]) if (!depth.count(o)) { depth[o] = depth[v] + 1; queue.push_back(o); }
    }
    PointCloudSensor::PosedMeasurements v_objects;
    for (const auto& d : depth) v_objects.emplace_back(std::dynamic_pointer_cast<PointCloudMeasurement>(mMeasurements[d.first]), mCorrected[d.first]);
    return PointCloudSensor::Patch{v_objects, mCorrected[source]};
  }

  // ScanSensor::link(source_id, target_id, guess)  :144-168
  void link(unsigned source_id, unsigned target_id, const Transform& guess) {
    Measurement::Ptr source_m = buildPatch(source_id);  // :150-151
    Measurement::Ptr target_m = buildPatch(target_id);
    try {
      Constraint::Ptr se3 = mSensor->createConstraint(source_m, target_m, guess, true);  // :156
      record(source_id, target_id, se3, true);
    } catch (NoMatch& e) {  // :159-166
      std::lock_guard<std::mutex> g(mMutex);
      warnings.push_back(std::string("Failed to link vertex: ") + e.what());
    }
  }

  // ScanSensor::linkLastToNeighbors(false) -> linkToNeighbors(mLastVertex)  :170-213.
  // batched: the candidates are matched in ONE createConstraints() call and the results are then replayed in the reference's
  // order.  The reference inserts each edge before it tests the next candidate, and a new loop edge can only SHORTEN hop
  // distances, so every candidate it attempts also passes the tests on the graph as it is before the first link: the batch
  // takes the first mMaxNeighorLinks of those, the replay repeats the tests on the growing graph, drops a batched result whose
  // candidate no longer qualifies and falls back to a single link() for a candidate the batch did not cover.  Edges and
  // warnings are therefore exactly those of the sequential loop.
  void linkLastToNeighbors(bool batched = false) {
    if (mMaxNeighorLinks < 1 || !mHasVertex) return;
    const unsigned vertex = mLastVertex;
    std::vector<unsigned> neighbors;  // Graph::getNearbyVertices: index order, d < radius
    for (unsigned v = 0; v < mCorrected.size(); ++v) {
      double d2 = 0;
      for (int a = 0; a < 3; ++a) { const double d = mCorrected[v](a, 3) - mCorrected[vertex](a, 3); d2 += d * d; }
      if (std::sqrt(d2) < mNeighborRadius) neighbors.push_back(v);
    }
    auto qualifies = [&](unsigned index) {  // :183-198 on the graph as it is now
      if (index == vertex) return false;
      for (unsigned o : mAdjacency[vertex]) if (o == index) return false;
      const float dist = graphDistance(index, vertex);
      return !(dist <= (float)(mPatchBuildingRange * 2) || dist < (float)mMinLoopLength);
    };
    std::vector<unsigned> batch;
    std::vector<PointCloudSensor::ConstraintResult> res;
    if (batched) {
      for (auto i = neighbors.rbegin(); i != neighbors.rend() && (int)batch.size() < mMaxNeighorLinks; ++i) if (qualifies(*i)) batch.push_back(*i);
      if (batch.empty()) return;
      if (mDevicePatches && mPatchBuildingRange > 0) {  // the patches are built and prepared on the device
        std::vector<PointCloudSensor::LoopRequest> req;
        const PointCloudSensor::Patch target_p = patchOf(vertex);
        for (unsigned index : batch) req.push_back({patchOf(index), target_p, mCorrected[index].inverse() * mCorrected[vertex]});
        res = mSensor->createLoopConstraints(req);
      } else {
        std::vector<PointCloudSensor::ConstraintRequest> req;
        Measurement::Ptr target_m = buildPatch(vertex);
        for (unsigned index : batch) req.push_back({buildPatch(index), target_m, mCorrected[index].inverse() * mCorrected[vertex]});
        res = mSensor->createConstraints(req, true);
      }
    }
    int count = 0;
    for (auto i = neighbors.rbegin(); i != neighbors.rend() && count < mMaxNeighorLinks; ++i) {
      const unsigned index = *i;
      if (!qualifies(index)) continue;
      ++count;
      size_t k = 0;
      while (k < batch.size() && batch[k] != index) ++k;
      if (k == batch.size()) { link(index, vertex, mCorrected[index].inverse() * mCorrected[vertex]); continue; }  // :137-142: guess = Graph::getTransform(source, target)
      if (res[k].constraint) record(index, vertex, res[k].constraint, true);
      else if (res[k].error == 1) { std::lock_guard<std::mutex> g(mMutex); warnings.push_back(std::string("Failed to link vertex: ") + res[k].message); }
      else throw std::runtime_error(res[k].message);  // link() lets everything but NoMatch propagate
    }
  }

  void setNeighborRadius(float r, int max_links) { mNeighborRadius = r; mMaxNeighorLinks = max_links; }  // ScanSensor.hpp setters
  void setMinLoopLength(unsigned l) { mMinLoopLength = l; }
  void setPatchBuildingRange(unsigned r) { mPatchBuildingRange = r; }
  // linkLastToNeighbors(true) with patches: build the patches on the device from their scans (PointCloudSensor::createLoopConstraints)
  // instead of on the host (createCombinedMeasurement + createConstraints).  Same edges and warnings; off by default.
  void setDevicePatches(bool on) { mDevicePatches = on; }
  const Transform& correctedPose(unsigned v) const { return mCorrected[v]; }
  // every vertex with its corrected pose, in vertex order: the list a slam3d application hands to PointCloudSensor::buildMap
  PointCloudSensor::PosedMeasurements vertices() const {
    PointCloudSensor::PosedMeasurements v;
    for (size_t i = 0; i < mMeasurements.size(); ++i) v.emplace_back(std::dynamic_pointer_cast<PointCloudMeasurement>(mMeasurements[i]), mCorrected[i]);
    return v;
  }

  std::vector<RecordedEdge> edges;
  std::vector<std::string> warnings;

 private:
  void record(unsigned s, unsigned t, const Constraint::Ptr& c, bool loop) {
    SE3Constraint::Ptr se3 = std::dynamic_pointer_cast<SE3Constraint>(c);
    std::lock_guard<std::mutex> g(mMutex);
    edges.push_back({s, t, se3->getRelativePose(), se3->getInformation(), loop});
    mAdjacency[s].push_back(t); mAdjacency[t].push_back(s);
  }
  // hop count between two vertices (dijkstra with unit weights == BFS); unreachable = max float like boost's distance map
  float graphDistance(unsigned from, unsigned to) const {
    std::vector<int> dist(mAdjacency.size(), -1);
    std::vector<unsigned> queue{from};
    dist[from] = 0;
    for (size_t h = 0; h < queue.size(); ++h) {
      const unsigned v = queue[h];
      if (v == to) return (float)dist[v];
      for (unsigned o : mAdjacency[v]) if (dist[o] < 0) { dist[o] = dist[v] + 1; queue.push_back(o); }
    }
    return 3.4028235e38f;
  }
  std::vector<Transform> mCorrected;                // VertexObject::correctedPose (no optimiser here: poses are chained edges)
  std::vector<std::vector<unsigned>> mAdjacency;
  float mNeighborRadius = 1.0f;                     // ScanSensor.cpp:37-39 defaults
  int mMaxNeighorLinks = 1;
  unsigned mMinLoopLength = 10;
  unsigned mPatchBuildingRange = 0;                 // ScanSensor.hpp: Sensor::mPatchBuildingRange (core/Sensor.hpp)
  bool mDevicePatches = false;                      // setDevicePatches
  float mMinTranslation = 0.f, mMinRotation = 0.f;  // Sensor::mMinTranslation / mMinRotation (0: every scan qualifies)
  Transform mLastTransform;                         // ScanSensor::mLastTransform
  PointCloudSensor* mSensor;
  std::vector<Measurement::Ptr> mMeasurements;
  unsigned mLastVertex;
  bool mHasVertex, mLinkPrevious;
  Transform mLastOdometry;
  std::mutex mMutex;
};

}  // namespace slam3d_b200
