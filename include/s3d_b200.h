/*
 * s3d_b200.h — C-ABI of the B200-native scan-matching path behind slam3d::PointCloudSensor.
 *
 * This is the drop-in boundary (SURVEY.md §8b): the two call sites in the reference that do all the
 * arithmetic — PointCloudSensor::downsample (slam3d/sensor/pcl/PointCloudSensor.cpp:190-201) and the
 * free function align() (PointCloudSensor.cpp:119-174, which calls doICP<> :52-82) — are replaced by
 * s3d_voxel_downsample() and s3d_gicp_align().  Everything above (createConstraint :269-299,
 * ScanSensor::addMeasurement / link, the graph, the g2o solver) stays host code and is untouched.
 *
 * Conventions
 *   - plain C, no C++/torch types; all pointers are caller-owned and only read/written during the call;
 *   - point clouds are arrays of 16-byte points {x,y,z,w} == pcl::PointXYZ memory
 *     (PointCloudSensor.hpp:43-44); `w` is ignored on input and written as 1.0f on output;
 *   - cloud pointers may be HOST or DEVICE pointers (the library asks cudaPointerGetAttributes);
 *     result structs and 4x4 poses are always host memory.  Host clouds may be pageable (a std::vector, a pcl::PointCloud);
 *     pinned memory (cudaHostRegister on the cloud's buffer, or cudaMallocHost) roughly doubles the upload rate;
 *   - DEVICE inputs are read in place on the library's own (non-blocking) streams: they must be complete before the call.
 *     Either synchronise the producing stream first, or name it once with s3d_set_input_stream() and every call orders its
 *     work after what that stream holds at the time of the call.  Every call is synchronous: outputs are complete on return;
 *   - 4x4 poses are column-major doubles == Eigen::Isometry3d::matrix().data() (core/Types.hpp:53);
 *   - every entry point is re-entrant (ScanSensor.cpp:209-210 enters createConstraint from two threads);
 *   - functions return an s3d_status; they never throw across the boundary.  s3d_last_error() returns a
 *     thread-local message for the last non-OK return on the calling thread.
 */
#ifndef S3D_B200_H
#define S3D_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Status codes.  1..4 map 1:1 on the exceptions thrown by the reference's align()/doICP()
 * (SURVEY.md §8b "Error convention"); the C++ host mirror re-throws the reference's exception types. */
typedef enum s3d_status {
  S3D_OK = 0,
  S3D_TOO_FEW_POINTS = 1,      /* NoMatch  "Too few points after filtering..."   PointCloudSensor.cpp:134-135 */
  S3D_NOT_CONVERGED = 2,       /* NoMatch  "ICP failed with Fitness-Score..."    PointCloudSensor.cpp:74-77   */
  S3D_TOO_FAR_FROM_GUESS = 3,  /* NoMatch  "ICP result is to far away from guess" PointCloudSensor.cpp:167-172 */
  S3D_UNKNOWN_ALGORITHM = 4,   /* std::runtime_error                              PointCloudSensor.cpp:158-164 */
  S3D_INTERNAL_ERROR = 5,      /* CUDA failure, bad argument, workspace problem   (std::runtime_error in the mirror) */
  S3D_INVALID_ARGUMENT = 6
} s3d_status;

/* enum RegistrationAlgorithm {ICP, GICP, GICP_OMP, NDT, NDT_OMP}  — RegistrationParameters.hpp:30 */
enum { S3D_ALG_ICP = 0, S3D_ALG_GICP = 1, S3D_ALG_GICP_OMP = 2, S3D_ALG_NDT = 3, S3D_ALG_NDT_OMP = 4 };

/* Field-for-field mirror of slam3d::RegistrationParameters (RegistrationParameters.hpp:36-97),
 * same order, same defaults (see s3d_default_parameters). */
typedef struct s3d_registration_parameters {
  int32_t registration_algorithm;      /* GICP */
  double  point_cloud_density;         /* 0.2   voxel leaf applied to both clouds before matching; <=0: none */
  double  max_fitness_score;           /* 2.0   */
  double  max_translation;             /* 1.0   */
  double  max_rotation;                /* 1.0   */
  double  euclidean_fitness_epsilon;   /* 1.0   stored, never read by GICP (SURVEY A.4 note) */
  double  transformation_epsilon;      /* 1e-5  */
  double  max_correspondence_distance; /* 2.5   */
  int32_t maximum_iterations;          /* 50    */
  double  rotation_epsilon;            /* 2e-3  */
  int32_t correspondence_randomness;   /* 20    k of the covariance kNN */
  int32_t maximum_optimizer_iterations;/* 20    */
  float   resolution;                  /* 1.0   NDT only */
  double  step_size;                   /* 0.05  NDT only */
  double  outlier_ratio;               /* 0.35  NDT only */
} s3d_registration_parameters;

typedef struct s3d_cloud {
  const float* xyzw; /* n * 4 floats, 16-byte aligned; host or device pointer */
  uint64_t     n;
} s3d_cloud;

/* Output of one align().  T is the pose of the *target* scan in the *source* scan's frame, i.e. what the
 * reference's align() returns (the PCL source/target swap of PointCloudSensor.cpp:68-69 is done inside). */
typedef struct s3d_result {
  double   T[16];            /* column-major 4x4; valid whenever the GICP loop ran (status 0,2,3) */
  double   fitness;          /* pcl getFitnessScore(max_correspondence_distance)  :73 */
  int32_t  status;           /* s3d_status */
  int32_t  converged;        /* pcl hasConverged() */
  int32_t  outer_iterations; /* pcl nr_iterations_ */
  int32_t  inner_iterations; /* total optimiser iterations over all outer iterations */
  uint32_t n_source;         /* points of the (filtered) slam3d source cloud = PCL target */
  uint32_t n_target;         /* points of the (filtered) slam3d target cloud = PCL source (the queries) */
  uint32_t n_correspondences;/* pairs within max_correspondence_distance in the last outer iteration */
  uint32_t reserved;
} s3d_result;

typedef struct s3d_context s3d_context;

/* Library / device bring-up.  `devices` = CUDA ordinals to shard batches over (NULL/0: current device).
 * Scheduling knobs, read from the environment when the context is created (measurement aids; results never depend on them,
 * tests/test_gpu_gicp.py::test_batch_scheduling_is_invisible):
 *   S3D_STREAMS_PER_DEVICE   host threads / streams that push chunks of a batch call through one device (default: 4 for GICP
 *                            on raw scans, 3 for prepared clouds and NDT)
 *   S3D_MAX_PAIRS_PER_LAUNCH upper bound of a chunk (default 32 pairs)
 *   S3D_GATE_UPLOADS=0       lets the chunks of a device upload concurrently instead of one after the other
 *   S3D_BLOCKING_SYNC=0      chunk threads spin on their stream instead of sleeping on a blocking event
 *   S3D_PINNED_BOUNCE=0      pageable clouds go straight to cudaMemcpyAsync instead of through the library's pinned buffer;
 *   S3D_COPY_THREADS=n       helper threads for that staging copy (default: half of the rank's cores, at most 8)
 *   S3D_LOOP_MODE=1|2|3      GICP loop as one persistent kernel / as a graph replay of per-pass kernels / launched from the host
 *                            (default: persistent for single calls, graph replay for the chunks of a batch)
 *   S3D_GRID_FRAC=f          pins the filtered / raw ratio the launch grids are sized with (default: learned per leaf size)
 *   S3D_WATCHDOG_MCYCLES=n   cycles (millions) after which a loop kernel that finds no work reports an internal error */
int s3d_create_context(const int* devices, int n_devices, s3d_context** out);
int s3d_destroy_context(s3d_context* ctx);

void        s3d_default_parameters(s3d_registration_parameters* p); /* RegistrationParameters.hpp defaults */
const char* s3d_last_error(void);
const char* s3d_version(void);

/* PointCloudSensor::downsample(cloud, leaf)  — PointCloudSensor.cpp:190-201 (pcl::VoxelGrid semantics,
 * SURVEY Appendix A.1).  out_xyzw must hold in.n points (host or device).  *n_out receives the number of
 * output points.  If leaf_index (host or device, in.n x uint32, may be NULL) is given it receives the
 * voxel index of every input point (the "leaf assignment"; 0xFFFFFFFF for skipped non-finite points).
 * overflow (may be NULL) is set to 1 when PCL's int32 index guard fires and the input is returned as is. */
int s3d_voxel_downsample(s3d_context* ctx, s3d_cloud in, float leaf, float* out_xyzw, uint64_t* n_out,
                         uint32_t* leaf_index, int32_t* overflow);

/* align(source, target, guess, config) — PointCloudSensor.cpp:119-174.  Always fills *out (status inside
 * is the same value as the return code).  registration_algorithm selects the branch of the reference's switch (:139-165):
 *   GICP  doICP<pcl::GeneralizedIterativeClosestPoint>  (:52-82)
 *   NDT   doNDT<pcl::NormalDistributionsTransform>      (:84-117): resolution, step_size, outlier_ratio, maximum_iterations,
 *         transformation_epsilon are read; out->outer_iterations = nr_iterations_, out->inner_iterations = More-Thuente
 *         line-search iterations, out->n_correspondences = (point, voxel) pairs of the last evaluation
 *   GICP_OMP / NDT_OMP  (:149-157, pclomp's multi-threaded builds of GICP and NDT) run the GICP / NDT branch of this library.
 *         pclomp's GICP is PCL's; pclomp's NDT has PCL's optimiser but by default another neighbour search (DIRECT7: the
 *         query's voxel and its 6 face neighbours, not PCL's kd-tree radius search), which s3d_set_ndt_omp_search selects.
 *         A build with -DS3D_OMP_UNAVAILABLE keeps the error of a reference build without pclomp (:158-161)
 *   anything else -> S3D_UNKNOWN_ALGORITHM with the reference's message (:162-164). */
int s3d_gicp_align(s3d_context* ctx, s3d_cloud source, s3d_cloud target, const double guess[16],
                   const s3d_registration_parameters* params, s3d_result* out);

/* n_pairs independent align() calls (loop-closure candidates, odometry pairs), sharded over the context's
 * devices.  guesses = n_pairs x 16 doubles.  Returns S3D_OK if the batch ran; per-pair status is in out[i]. */
int s3d_gicp_align_batch(s3d_context* ctx, const s3d_cloud* sources, const s3d_cloud* targets,
                         const double* guesses, const s3d_registration_parameters* params, int n_pairs,
                         s3d_result* out);

/* n_pairs loop-closure constraints, i.e. the align sequence of createConstraint(source, target, odometry, loop = true)
 * (PointCloudSensor.cpp:286-292): align with the coarse parameters and `guesses`, then align with the fine parameters and
 * the coarse result as the guess.  Same results as two s3d_gicp_align_batch calls, but every scan is uploaded once and a
 * chunk's fine pass overlaps the other chunks' coarse pass.  out_fine[i] is what the caller turns into the edge; when the
 * coarse align of pair i fails (the reference throws there and never runs the fine align) out_fine[i] = out_coarse[i].
 * out_coarse may be NULL. */
int s3d_gicp_align_loop_batch(s3d_context* ctx, const s3d_cloud* sources, const s3d_cloud* targets, const double* guesses,
                              const s3d_registration_parameters* coarse, const s3d_registration_parameters* fine, int n_pairs,
                              s3d_result* out_coarse, s3d_result* out_fine);

/* Inner optimiser of PCL's GICP (estimateRigidTransformation*), the one step in which PCL versions differ:
 *   S3D_GICP_NEWTON  estimateRigidTransformationNewton, PCL >= 1.14's default (back-tracking Newton; the default here)
 *   S3D_GICP_BFGS    estimateRigidTransformationBFGS, the only optimiser of PCL 1.8.1 ... 1.13 (pcl/registration/bfgs.h, GSL's
 *                    vector_bfgs2 with Fletcher's line search).  About 10x the evaluation passes of Newton (DESIGN.md 4).
 * The setting belongs to the context, not to s3d_registration_parameters (which mirrors slam3d's struct field for field): it is a
 * property of the PCL a build replaces.  It applies to every GICP (and GICP_OMP) entry point — s3d_gicp_align, _batch,
 * _loop_batch (coarse and fine), _prepared, _prepared_batch — and NDT ignores it; prepared clouds serve both.  Calls that start
 * after it returns use the new setting: change it while no call is running on the context.  `previous` (may be NULL) receives the
 * setting it replaces.  Any other value returns S3D_INVALID_ARGUMENT and changes nothing. */
enum { S3D_GICP_NEWTON = 0, S3D_GICP_BFGS = 1 };
int s3d_set_gicp_optimizer(s3d_context* ctx, int optimizer, int* previous);

/* Neighbour search of registration_algorithm = NDT_OMP, the one step in which pclomp's NDT differs from PCL's:
 *   S3D_NDT_OMP_KDTREE   PCL's kd-tree radius search (every centroid within `resolution`): NDT_OMP returns what NDT returns
 *                        (the default here; pclomp's KDTREE mode)
 *   S3D_NDT_OMP_DIRECT7  pclomp's default, DIRECT7 (VoxelGridCovariance::getNeighborhoodAtPoint7, never changed by slam3d's
 *                        doNDT): the query's own voxel and its 6 face neighbours, in the order (0,0,0) (+-1,0,0) (0,+-1,0)
 *                        (0,0,+-1), cell = floor(p / leaf size), leaves with >= 6 points that PCL did not mark invalid.
 * Like s3d_set_gicp_optimizer it belongs to the context: it applies to NDT_OMP in every align entry point — s3d_gicp_align,
 * _batch, _loop_batch (coarse and fine each by their own algorithm), _prepared, _prepared_batch — and NDT, GICP and GICP_OMP
 * ignore it.  Calls that start after it returns use the new setting: change it while no call is running on the context.
 * `previous` (may be NULL) receives the setting it replaces.  Any other value returns S3D_INVALID_ARGUMENT and changes nothing. */
enum { S3D_NDT_OMP_KDTREE = 0, S3D_NDT_OMP_DIRECT7 = 1 };
int s3d_set_ndt_omp_search(s3d_context* ctx, int method, int* previous);

/* ---- stage-level entry points (used by the parity tests and the bench; same kernels as align) ---------- */

/* GICP computeCovariances (SURVEY A.3): exact kNN (k neighbours, self included, ascending (d2, index)),
 * moments, regularised covariance.  Outputs are optional (NULL to skip), host or device:
 *   knn_index  n*k uint32 (original indices), knn_dist2 n*k float, covariances n*9 doubles (column-major 3x3). */
int s3d_knn_covariances(s3d_context* ctx, s3d_cloud cloud, int k, uint32_t* knn_index, float* knn_dist2,
                        double* covariances);

/* Exact 1-NN of T_f32*query[i] in `reference` (SURVEY A.2/A.4): nn_index n uint32, nn_dist2 n float.
 * transform = column-major 4x4 (cast to float and applied as in the GICP loop); NULL = identity. */
int s3d_nearest_neighbors(s3d_context* ctx, s3d_cloud reference, s3d_cloud queries, const double* transform,
                          uint32_t* nn_index, float* nn_dist2);

/* The CUDA stream (cudaStream_t) of the FIRST workspace of device slot `device_slot`: single (non-batch) calls issued by one
 * host thread run on it, so a caller can bracket such calls with events.  Batch calls and concurrent callers use further
 * streams of their own — this handle is a measurement aid, not a way to order work; calls are synchronous anyway.
 * Returns NULL on a bad slot. */
void* s3d_context_stream(s3d_context* ctx, int device_slot);

/* Names the CUDA stream (cudaStream_t; NULL = the legacy default stream) on which the caller produces DEVICE-pointer inputs.
 * While enabled, every call records an event on that stream and lets its own streams wait for it before they touch an input.
 * enabled = 0 switches the ordering off again (inputs must then be complete before a call, see "Conventions"). */
int s3d_set_input_stream(s3d_context* ctx, void* stream, int enabled);

/* Counters since context creation: kernel launches issued by this library, bytes copied H2D / D2H. */
typedef struct s3d_counters { uint64_t kernel_launches, h2d_bytes, d2h_bytes; } s3d_counters;
int s3d_get_counters(s3d_context* ctx, s3d_counters* out);

/* Work done by the GICP loop kernel since context creation (or the last reset): 256-point tiles processed by its search,
 * trial and fitness passes, and control steps (optimiser advances) — the units behind bench.py's algorithmic bytes. */
int s3d_get_loop_stats(s3d_context* ctx, uint64_t* tiles, uint64_t* control_steps, int reset);

/* ---- per-measurement device cache (SURVEY 8f rank 1) ------------------------------------------------------
 * The reference rebuilds the voxel filter, both kd-trees and all covariances inside every align()
 * (PointCloudSensor.cpp:58,125-131 are locals), although each scan is matched several times (once as target and once as
 * source in odometry, many times as a loop-closure candidate).  s3d_prepare_cloud runs the per-cloud stages ONCE
 * (H2D, voxel filter at `density`, NN grid, kNN-k covariances) and keeps the result on the device;
 * s3d_gicp_align_prepared(_batch) then runs only the GICP loop + fitness + gates.  Results are bit-identical to
 * s3d_gicp_align on the raw clouds with point_cloud_density == density and correspondence_randomness == k
 * (status 6 if the handle was prepared with other values).  Handles are immutable and may be shared by threads.
 * s3d_prepare_cloud_ndt does the same for the NDT branch: voxel filter, NN grid and the VoxelGridCovariance at `resolution`
 * that doNDT builds for its target (PointCloudSensor.cpp:84-117); the handle holds no normals. */
typedef struct s3d_prepared_cloud s3d_prepared_cloud;
int s3d_prepare_cloud(s3d_context* ctx, int device_slot, s3d_cloud cloud, double density, int k, s3d_prepared_cloud** out);
/* n clouds in one pass (same result as n calls of s3d_prepare_cloud; out receives n handles, all-or-nothing). */
int s3d_prepare_clouds(s3d_context* ctx, int device_slot, const s3d_cloud* clouds, int n, double density, int k,
                       s3d_prepared_cloud** out);
/* n clouds in one pass: voxel filter at `density`, NN grid, and the NDT VoxelGridCovariance at `resolution`.  All-or-nothing like
 * s3d_prepare_clouds.  resolution <= 0 or not finite, a NaN density or a bad device slot: S3D_INVALID_ARGUMENT and no handle.
 * A cloud whose grid is not searchable (no finite point, PCL's int32 voxel-count guard) still gets a handle; an align on it
 * ends like the raw call ("Voxel grid is not searchable": not converged, identity pose). */
int s3d_prepare_clouds_ndt(s3d_context* ctx, int device_slot, const s3d_cloud* clouds, int n, double density, float resolution,
                           s3d_prepared_cloud** out);
int s3d_prepare_cloud_ndt(s3d_context* ctx, int device_slot, s3d_cloud cloud, double density, float resolution,
                          s3d_prepared_cloud** out);
int s3d_release_cloud(s3d_context* ctx, s3d_prepared_cloud* cloud);
uint64_t s3d_prepared_cloud_size(const s3d_prepared_cloud* cloud); /* points after filtering */
/* Device blocks of prepared clouds since context creation, over all devices: obtained from cudaMalloc, and reused from
 * released handles (s3d_release_cloud hands a block back to its device; a later prepare takes it when it fits). */
int s3d_get_prepared_block_stats(s3d_context* ctx, uint64_t* allocated, uint64_t* reused);
/* Align on prepared clouds; the algorithm comes from params->registration_algorithm as in s3d_gicp_align.
 *   GICP / GICP_OMP  both handles from s3d_prepare_cloud(s) with k == correspondence_randomness (an NDT handle: status 6).
 *   NDT / NDT_OMP    the source (the scan whose grid NDT matches against) from s3d_prepare_cloud(s)_ndt with
 *                    resolution == params->resolution (compared as floats; another value: status 6).  The target is read as
 *                    points only, so a GICP handle of the same density serves too.  A pair whose source is a GICP handle ends
 *                    with S3D_UNKNOWN_ALGORITHM (S3D_TOO_FEW_POINTS under 100 points), as before NDT handles existed.
 * Every handle must match point_cloud_density (status 6 otherwise).  Results are bit-identical to s3d_gicp_align(_batch) on the
 * raw clouds with the same parameters. */
int s3d_gicp_align_prepared(s3d_context* ctx, const s3d_prepared_cloud* source, const s3d_prepared_cloud* target,
                            const double guess[16], const s3d_registration_parameters* params, s3d_result* out);
int s3d_gicp_align_prepared_batch(s3d_context* ctx, const s3d_prepared_cloud* const* sources,
                                  const s3d_prepared_cloud* const* targets, const double* guesses,
                                  const s3d_registration_parameters* params, int n_pairs, s3d_result* out);

/* ---- patch and map building (SURVEY 8f rank 2/3) -------------------------------------------------------------
 * PointCloudSensor::transform (PointCloudSensor.cpp:228-233): pcl::transformPointCloud with a double 4x4.
 * out_xyzw holds in.n points (host or device). */
int s3d_transform_cloud(s3d_context* ctx, s3d_cloud in, const double T[16], float* out_xyzw);
/* PointCloudSensor::removeOutliers (:211-226): pcl::RadiusOutlierRemoval — a point stays iff at least min_neighbors other
 * points lie within `radius`; returns the input unchanged unless in.n > 0, radius > 0 and min_neighbors > 0.
 * Output keeps the input order. */
int s3d_remove_outliers(s3d_context* ctx, s3d_cloud in, double radius, unsigned min_neighbors, float* out_xyzw, uint64_t* n_out);
/* PointCloudSensor::buildMap (:301-318) on explicit lists: accumulate transform(cloud_i, pose_i) in list order
 * (getAccumulatedCloud :235-256, pose_i = vertex.correctedPose * measurement.sensorPose), removeOutliers, downsample.
 * poses = n x 16 doubles; out_xyzw holds sum(clouds[i].n) points. */
int s3d_build_map(s3d_context* ctx, const s3d_cloud* clouds, const double* poses, int n, double outlier_radius,
                  unsigned outlier_neighbors, double resolution, float* out_xyzw, uint64_t* n_out);

/* PointCloudSensor::createCombinedMeasurement (:258-266) on explicit lists — the patch of scans a loop closure is matched
 * with (ScanSensor::buildPatch, core/ScanSensor.cpp:215-270): getAccumulatedCloud (transform(cloud_i, pose_i) appended in list
 * order, pose_i = vertex.correctedPose * measurement.sensorPose), then pcl::transformPointCloud with patch_pose.inverse().
 * Both transforms run on the device in one pass over the points (two float roundings per coordinate, like the two PCL calls).
 * poses = n x 16 doubles, patch_pose = 16 doubles; out_xyzw (host or device) holds sum(clouds[i].n) points.
 * patch_pose == NULL stops after the accumulation: PointCloudSensor::getAccumulatedCloud (:235-256). */
int s3d_create_combined_measurement(s3d_context* ctx, const s3d_cloud* clouds, const double* poses, int n, const double patch_pose[16],
                                    float* out_xyzw, uint64_t* n_out);

/* ---- ground plane (PointCloudSensor::fillGroundPlane, PointCloudSensor.cpp:362-388) ---------------------------------------
 * pcl::RandomSampleConsensus + SampleConsensusModelPlane (DESIGN.md 6f): coefficients[4] = (a, b, c, d), unit normal.
 * iterations = PCL's iterations_, n_inliers = points with |a x + b y + c z + d| < threshold; inliers (may be NULL; host or device,
 * cloud.n entries) receives their indices in ascending order.  N < 3, no non-degenerate sample in 1000 draws, or no plane with
 * an inlier: S3D_INVALID_ARGUMENT.  threshold must be positive and finite, probability in (0, 1), max_iterations >= 1.
 * S3D_RANSAC_BLOCK (environment, read once; measurement aid) sets how many planes are sampled and scored per round (default
 * 256, at most 2048); results never depend on it. */
int s3d_fit_plane_ransac(s3d_context* ctx, s3d_cloud cloud, double threshold, int max_iterations, double probability,
                         float coefficients[4], int32_t* iterations, uint64_t* n_inliers, uint32_t* inliers);
/* Number of points that fillGroundPlane appends for (map_resolution, radius): it depends on these two values only.  Both must be
 * positive and finite; more than 2^31 - 1 points is S3D_INVALID_ARGUMENT. */
int s3d_ground_fill_size(double map_resolution, double radius, uint64_t* n);
/* PointCloudSensor::fillGroundPlane (:362-388): RANSAC plane (threshold 0.01, PCL defaults), then rings of points.  out_xyzw
 * (host or device) receives the s3d_ground_fill_size() new points; the caller appends them.  coefficients may be NULL. */
int s3d_fill_ground_plane(s3d_context* ctx, s3d_cloud cloud, double map_resolution, double radius, float* out_xyzw,
                          float coefficients[4]);

/* Optional per-stage device timing (CUDA events on the launching stream, read back at the call's final
 * synchronisation).  Stage ids: 0 voxel filter, 1 NN grid build, 2 kNN+covariances (NDT: the target's Gaussian voxel
 * grid), 3 the GICP loop kernel — search, trial and fitness passes and the control steps of all outer iterations (NDT:
 * derivative evaluation), 4 GICP loop set-up kernel (NDT: line-search control), 5 NDT fitness (GICP: part of stage 3).
 * ms[i] / launches[i] accumulate since the last reset. */
#define S3D_N_STAGES 6
int s3d_set_profiling(s3d_context* ctx, int enabled);
int s3d_get_stage_times(s3d_context* ctx, double ms[S3D_N_STAGES], uint64_t launches[S3D_N_STAGES], int reset);

#ifdef __cplusplus
}
#endif
#endif /* S3D_B200_H */
