/* limu_cuda.h -- C ABI of liblimu_cuda.so: the B200 (sm_100a) LiDAR odometry hot path.
 *
 * Drop-in boundary for Oreoluwa-Se/Lidar-Imu-Slam's lidar:: classes ("L/" = env_ws/src/limu of the
 * reference). The reference has no FFI layer: its boundary is the C++ class surface called from the
 * single odometry thread (L/src/odom_run.cpp:154-185). Each entry point below names the reference
 * interface it replaces; the header-only C++ classes in include/limu_dropin/ put the reference's own
 * signatures (lidar::VoxelHashMap, lidar::ICP, lidar::KissICP, ...) back on top of these calls, and
 * INTEGRATION.md shows the binding a maintainer adds.
 *
 * Conventions
 *   - plain C: pointers + sizes, no exceptions, no STL, no torch types.
 *   - every call returns LIMU_OK (0) or a negative limu_status; limu_last_error() gives the message of
 *     the calling thread's last failure.
 *   - points : double xyz[3*n] array-of-structs == utils::Vec3dVector storage (L/include/limu/utils/types.hpp:19)
 *   - raw scan points : float xyzt[4*n] = {x, y, z, t}, t in [0,1] = normalised per-point timestamp
 *     (float x,y,z as in pcl::PointXYZINormal, types.hpp:36; t as produced by
 *     utils::normalize_timestamps, L/src/utils/calculation_helpers.cpp:52-66)
 *   - pose   : double[7] = {qx,qy,qz,qw, tx,ty,tz} == Sophus::SE3d::data() order
 *   - voxel  : int32[3] == utils::Voxel (types.hpp:15)
 *   - pointers are HOST memory unless the function name ends in _dev (then: device memory of the
 *     handle's GPU, e.g. torch.Tensor.data_ptr()); host buffers may be pageable or pinned
 *     (limu_host_alloc gives pinned memory; pinned makes the copies asynchronous DMA).
 *   - a handle owns its device buffers and one CUDA stream; calls on one handle are serialised by the
 *     caller (the reference is single-threaded here too); different handles are independent.
 *   - there is NO CPU fallback: every entry point fails with LIMU_ERR_CUDA when no device is usable.
 */
#ifndef LIMU_CUDA_H
#define LIMU_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LIMU_ABI_VERSION 1

typedef enum limu_status {
    LIMU_OK = 0,
    LIMU_ERR_INVALID = -1,   /* bad argument (null pointer, negative size, cap < 1, ...) */
    LIMU_ERR_CUDA = -2,      /* CUDA runtime failure (message carries cudaGetErrorString) */
    LIMU_ERR_KEY_RANGE = -3, /* a voxel index fell outside +-2^20 (the packed 3x21-bit key range) */
    LIMU_ERR_MAP_FULL = -4,  /* hash table could not grow (out of device memory) */
    LIMU_ERR_NOMEM = -5,
    LIMU_ERR_COMM = -6       /* multi-GPU exchange failed */
} limu_status;

const char *limu_last_error(void);
int limu_abi_version(void);
/* First 16 hex digits of the SHA-256 of the sources (csrc + this header) the loaded library was built from: bench.py quotes a committed
 * ncu capture only when it was taken from the same sources. */
const char *limu_source_hash(void);
/* Number of kernel launches issued by this process so far (all handles). bench.py reports the delta. */
uint64_t limu_kernel_launches(void);
int limu_device_count(void);
/* Pinned host memory (cudaHostAlloc); optional, any host pointer is accepted everywhere. */
void *limu_host_alloc(size_t bytes);
void limu_host_free(void *p);

/* ---- context: one GPU, one stream, scratch memory ---------------------------------------------- */
typedef struct limu_ctx limu_ctx;
int limu_ctx_create(int device, limu_ctx **out);
void limu_ctx_destroy(limu_ctx *c);
int limu_ctx_sync(limu_ctx *c);
void *limu_ctx_stream(limu_ctx *c); /* cudaStream_t, for callers that enqueue their own work around ours */
/* Optional per-stage device timing of limu_odom_register_* with CUDA events on the context's stream
 * (what bench.py's roofline reads). Stages: */
enum { LIMU_STAGE_PREPARE = 0, /* deskew / widen */
       LIMU_STAGE_DOWNSAMPLE = 1, LIMU_STAGE_IQR = 2, LIMU_STAGE_ICP = 3, /* the fused registration kernel alone */
       LIMU_STAGE_MAP_UPDATE = 4, LIMU_NUM_STAGES = 5 };
int limu_ctx_set_profiling(limu_ctx *c, int enabled);   /* also resets the accumulators */
int limu_ctx_get_profile(limu_ctx *c, double ms[LIMU_NUM_STAGES], int64_t frames[1]);

/* ---- stateless point operations ------------------------------------------------------------------ */
/* utils::get_vox_index, calculation_helpers.cpp:142-147: keys[3i+a] = (int)(xyz[3i+a] / v). */
int limu_voxel_keys(limu_ctx *c, const double *xyz, int64_t n, double v, int32_t *keys);
/* utils::transform_points, calculation_helpers.cpp:121-133: xyz <- T * xyz in place. */
int limu_transform_points(limu_ctx *c, const double pose[7], double *xyz, int64_t n);
/* lidar::MotionCompensator::deskew_scan, helpers/deskew.cpp:10-28:
 * out[i] = exp((t_i - 0.5) * log(T0^-1 T1)) * (x_i,y_i,z_i). */
int limu_deskew(limu_ctx *c, const float *xyzt, int64_t n, const double T0[7], const double T1[7], double *out_xyz);
/* The same on the reference's own input layout: point records `stride_bytes` apart with float x,y,z at offset 0
 * (pcl::PointXYZINormal = 48 B, types.hpp:36) and FP64 timestamps (std::vector<double>). */
int limu_deskew_cloud(limu_ctx *c, const void *points, int32_t stride_bytes, const double *timestamps, int64_t n, const double T0[7],
                      const double T1[7], double *out_xyz);
/* IMU-propagated backward deskew: the per-point loop of kalman::EKF::motion_compensation_with_imu, L/src/kalman/ekf.cpp:420-468
 * (dead code at runtime in the reference; SURVEY section 8f N1). The host IMU forward pass (:315-410) supplies: `table` = its
 * kalman::Pose6D rows (ekf.hpp:88-105), rot_end (row-major) and pos_lidar_end (:393-418), p_imu_lidar = state POS_IMU_LIDAR.
 * points: records stride_bytes apart with float x,y,z at offset 0 and the float per-point offset time in ms (PCL
 * `curvature`: offset 36 in pcl::PointXYZINormal) at curvature_offset_bytes, sorted by that time (lidar/frame.cpp:28-51).
 * out_xyz (optional, n x 3 doubles) = meas->deskewed (:458-468); write_back != 0 also stores the float x,y,z into the records (:451-453). */
typedef struct limu_imu_pose { double offset_time, acc[3], gyr[3], vel[3], pos[3], rot[9]; } limu_imu_pose;
int limu_deskew_imu(limu_ctx *c, void *points, int32_t stride_bytes, int32_t curvature_offset_bytes, int64_t n, const limu_imu_pose *table,
                    int32_t n_poses, const double rot_end[9], const double pos_lidar_end[3], const double p_imu_lidar[3], double *out_xyz,
                    int32_t write_back);
/* The IMU forward pass of the same function (ekf.cpp:292-418): HOST code inside the library (about 20 IMU samples per scan) that builds
 * what limu_deskew_imu consumes, so a caller does not need the reference's EKF object. samples[0] is the last sample of the previous window
 * (mc_tracker->last_imu, :295), samples[1..k-1] the IMU buffer of this scan. state: the EKF state entries the function reads; in/out members
 * carry what the reference keeps between windows. The quaternion 4-vector is used exactly as the reference does (S acts on it as stored,
 * the rotation matrix reads it as x,y,z,w without normalising). exp(S) is closed-form here, Eigen's Pade approximant there: ~1e-16 apart. */
typedef struct limu_imu_sample { double t, gyr[3], acc[3]; } limu_imu_sample;
typedef struct limu_imu_state {
    double pos[3], vel[3], quat[4];                          /* POS, VEL, ORI at the start of the window (position(), velocity(), orientation()) */
    double bga[3], baa[3], bat[3], grav[3], p_imu_lidar[3];  /* BGA, BAA, BAT, GRAV, POS_IMU_LIDAR */
    double mean_acc_norm, gravity_norm;                      /* meas->get_mean_acc_norm(); the reference's `gravity` constant 9.81 (common.hpp:16) */
    double last_lidar_end_time;                              /* in/out (:413) */
    double acc_s_last[3], ang_vel_last[3];                   /* in/out: the tracker members that fill row 0 of the table (:307, :386-387) */
    double tracker_vel[3], tracker_pos[3], tracker_quat[4];  /* out: mc_tracker->vel / pos and the quaternion after the last IMU pair */
} limu_imu_state;
int limu_imu_forward_pass(limu_imu_state *state, const limu_imu_sample *samples, int32_t k, double lidar_beg_time, double last_point_curvature_ms,
                          limu_imu_pose *table_out, int32_t max_rows, int32_t *n_rows, double rot_end[9], double pos_lidar_end[3]);
/* voxel_downsample (file-local), sensors/lidar/icp.cpp:9-30: first point per voxel of edge s wins;
 * output in first-occurrence order. out_xyz must hold n points; out_idx (optional) the source indices. */
int limu_voxel_downsample(limu_ctx *c, const double *xyz, int64_t n, double s, double *out_xyz, int64_t *out_idx, int64_t *n_out);
/* KissICP::iqr_processing, icp.cpp:88-124 + outlier::IQR, common.hpp:22-63. bounds (optional) = {low, high}. */
int limu_iqr_filter(limu_ctx *c, const double *xyz, int64_t n, double *out_xyz, int64_t *n_out, double bounds[2]);
/* KissICP::voxelize, icp.cpp:126-136: down = ds(frame, 0.5 v); src = IQR(ds(down, 1.5 v)). */
int limu_voxelize(limu_ctx *c, const double *xyz, int64_t n, double v, double *src_xyz, int64_t *n_src, double *down_xyz, int64_t *n_down);
/* lidar::align_clouds, helpers/registration.cpp:43-92. H (6x6 row-major), g, x optional. */
int limu_align(limu_ctx *c, const double *src, const double *tgt, int64_t n, double th, double H[36], double g[6], double x[6], double pose_out[7]);

/* ---- lidar::VoxelHashMap, helpers/voxel_hash_map.hpp:14-48 -------------------------------------- */
typedef struct limu_map limu_map;
/* ctor (:17-19). capacity_voxels: expected number of occupied voxels (the table grows when exceeded). */
int limu_map_create(limu_ctx *c, double vox_size, double max_distance, int max_points_per_voxel, int64_t capacity_voxels, limu_map **out);
void limu_map_destroy(limu_map *m);
int limu_map_clear(limu_map *m);                                   /* clear() :200-204 */
int limu_map_empty(limu_map *m, int *out);                         /* empty() :206-210 */
int limu_map_size(limu_map *m, int64_t *n_voxels, int64_t *n_points);
int limu_map_insert(limu_map *m, const double *xyz, int64_t n);    /* insert_points :12-62 */
int limu_map_insert_dev(limu_map *m, const double *xyz_dev, int64_t n);
int limu_map_update(limu_map *m, const double *xyz, int64_t n, const double pose[7]); /* update(points, pose) :138-144 */
int limu_map_update_origin(limu_map *m, const double *xyz, int64_t n, const double origin[3]); /* update(points, origin) :132-136 */
int limu_map_remove_far(limu_map *m, const double origin[3]);      /* remove_points_from_far :146-171 */
/* get_closest_neighbour :64-102 for n queries. Optional out_key[3n] = voxel of the match (INT32_MIN x3
 * when nothing was found and (0,0,0) is returned), out_rank[n] = position of the match inside its voxel (-1). */
int limu_map_closest(limu_map *m, const double *xyz, int64_t n, double *out_xyz, int32_t *out_key, int32_t *out_rank);
/* get_correspondences :104-130. src/tgt hold up to n points; pairs come out in query order. out_idx optional. */
int limu_map_correspondences(limu_map *m, const double *xyz, int64_t n, double max_correspondance, double *src, double *tgt, int64_t *out_idx, int64_t *n_out);
/* pointcloud() :173-198, in voxel creation order. Pass out_xyz = NULL to query the size. */
int limu_map_pointcloud(limu_map *m, double *out_xyz, int64_t max_points, int64_t *n_out);
/* Structured dump in voxel creation order (replaces reading the public robin_map member, hpp:40). */
int limu_map_dump(limu_map *m, int32_t *keys, int32_t *counts, double *pts, int64_t max_voxels, int64_t max_points, int64_t *n_voxels, int64_t *n_points);

/* ---- lidar::ICP, helpers/registration.cpp:94-130 ------------------------------------------------ */
typedef struct limu_icp_stats {
    int32_t iterations;       /* Gauss-Newton iterations executed */
    int32_t converged;        /* 1 if |log(estimate)| < est_threshold stopped the loop */
    int64_t last_ncorr;       /* correspondences in the last iteration */
    double mean_candidates;   /* k-bar: mean points compared per query (last iteration) */
    double miss_fraction;     /* f_miss: share of queries whose own voxel was absent (last iteration) */
} limu_icp_stats;
/* Whole loop on device (persistent cooperative kernel, no host round trip per iteration).
 * Optional traces: est_trace[7*max_iter], ncorr_trace[max_iter], hg_trace[42*max_iter] (H row-major + g). */
int limu_icp(limu_map *m, const double *xyz, int64_t n, const double init_guess[7], double max_corresp_dist, double kernel,
             int icp_max_iteration, double est_threshold, double pose_out[7], limu_icp_stats *stats,
             double *est_trace, int64_t *ncorr_trace, double *hg_trace);
int limu_icp_dev(limu_map *m, const double *xyz_dev, int64_t n, const double init_guess[7], double max_corresp_dist, double kernel,
                 int icp_max_iteration, double est_threshold, double pose_out[7], limu_icp_stats *stats);

/* Opt-in variants of the registration loop (SURVEY section 8f N2). They have NO counterpart in the reference (whose neighbour rule
 * is own-voxel-only and whose residual is point-to-point, SURVEY section 0 F1); the C oracle's restatement of the same definition is
 * their parity oracle.
 *   LIMU_ICP_NN27: correspondence = the NEAREST stored point over all 27 cells of the query's neighbourhood (what the north star and
 *   upstream KISS-ICP describe), cells visited x-outermost, points in storage order, first minimum wins.
 *   LIMU_ICP_PLANE: point-to-plane residual e = n.(s - t) with n = normal of the matched point's voxel (smallest-eigenvalue
 *   direction of the scatter of its >= 5 stored points, planar when l_min <= 0.04 l_mid; other correspondences are dropped),
 *   weight th^2/(th + e^2)^2, Jacobian row [n ; s x n]; the solve carries a weak prior on the initial guess,
 *   x = LDLT(H + D).solve(-(g + D log(T_icp))) with D = diag(1, 1, 1, 100, 100, 100) (negligible against a populated map; where only a
 *   handful of planar voxels can be matched, e.g. on the first scans of a sequence, the directions they do not observe stay at the
 *   prediction instead of running away). Not available in the point-sharded loop. */
enum { LIMU_ICP_REFERENCE = 0, LIMU_ICP_NN27 = 1, LIMU_ICP_PLANE = 2 };
int limu_icp_ex(limu_map *m, const double *xyz, int64_t n, const double init_guess[7], double max_corresp_dist, double kernel,
                int icp_max_iteration, double est_threshold, int32_t icp_mode, double pose_out[7], limu_icp_stats *stats,
                double *est_trace, int64_t *ncorr_trace, double *hg_trace);
/* get_closest_neighbour under a neighbour rule (icp_mode as above); outputs as limu_map_closest. */
int limu_map_closest_ex(limu_map *m, const double *xyz, int64_t n, int32_t icp_mode, double *out_xyz, int32_t *out_key, int32_t *out_rank);

/* ---- point-sharded ICP over several GPUs (BASELINE configs[4]; no counterpart in the single-process reference) ----
 * One process per GPU. Every rank holds a full replica of the map and a contiguous shard of the query points; per
 * Gauss-Newton iteration the ranks exchange ONE row of 20 doubles (the normal-equation sums). LIMU_SHARD_FUSED does
 * that inside the persistent kernel with stores into peer-mapped mailboxes over NVLink; LIMU_SHARD_NCCL is the un-fused
 * baseline (kernel -> ncclAllReduce -> solve kernel, host in the loop). All ranks return the same pose.
 * Setup: limu_comm_create on every rank -> exchange the 64-byte handles (any transport) -> limu_comm_connect. */
enum { LIMU_SHARD_FUSED = 0, LIMU_SHARD_NCCL = 1 };
int limu_comm_create(limu_ctx *c, int rank, int nranks, unsigned char ipc_handle_out[64]);
int limu_comm_connect(limu_ctx *c, const unsigned char *all_handles /* nranks x 64 bytes, rank order */);
void limu_comm_destroy(limu_ctx *c);
int limu_comm_nccl_unique_id(unsigned char id_out[128]);            /* rank 0, then broadcast */
int limu_comm_nccl_init(limu_ctx *c, const unsigned char id[128]);  /* only needed for LIMU_SHARD_NCCL */
/* stats->mean_candidates / miss_fraction carry GLOBAL candidate / miss COUNTS in a sharded call. */
int limu_icp_sharded_dev(limu_map *m, const double *xyz_dev, int64_t n_local, const double init_guess[7], double max_corresp_dist, double kernel,
                         int icp_max_iteration, double est_threshold, int mode, double pose_out[7], limu_icp_stats *stats);

/* ---- lidar::KissICP, sensors/lidar/icp.hpp:31-68 ------------------------------------------------ */
typedef struct limu_odom_config {   /* frame::Lidar::ProcessingInfo fields the path reads, lidar/frame.hpp:34-58, defaults :64-80 */
    double voxel_size;            /* 1.0 (= max_range / 100) */
    double max_range;             /* 100.0 */
    int32_t max_points_per_voxel; /* 10 */
    int32_t deskew;               /* 0 */
    double min_motion_th;         /* 0.1 */
    int32_t icp_max_iteration;    /* 500 */
    int32_t icp_mode;             /* 0 = the reference's rules (default); LIMU_ICP_* bits opt into the north star's variants */
    double initial_threshold;     /* 2.0 */
    double estimation_threshold;  /* 1e-4 */
    int64_t map_capacity_voxels;  /* 0 = derive from max_range / voxel_size */
    int64_t max_points_per_scan;  /* 0 = grow on demand */
} limu_odom_config;
void limu_odom_default_config(limu_odom_config *cfg);

typedef struct limu_frame_stats {
    int64_t n_points, n_down, n_keypoints;
    double sigma;                 /* adaptive threshold used (icp.cpp:138-144) */
    limu_icp_stats icp;
    int32_t deskewed;             /* 1 if the deskew gate was open (icp.cpp:40-46); 2: IMU-compensated (limu_odom_register_cloud_imu) */
    int32_t reserved0;
} limu_frame_stats;

typedef struct limu_odom limu_odom;
int limu_odom_create(limu_ctx *c, const limu_odom_config *cfg, limu_odom **out);
void limu_odom_destroy(limu_odom *o);
/* register_frame(cloud, timestamps) icp.cpp:49-55. Outputs are optional (NULL = not copied back):
 * down_xyz / keypoints_xyz must hold n points each.
 * Error behaviour of every limu_odom_register_*: LIMU_ERR_KEY_RANGE / LIMU_ERR_MAP_FULL are reported AFTER the frame has been committed
 * (pose appended, threshold state and map updated, outputs filled): the offending points -- voxel index outside +-2^20, e.g. an inf
 * coordinate that frame::Lidar::process_frame would have dropped -- were left out of the downsampled cloud and of the map. */
int limu_odom_register_frame(limu_odom *o, const float *xyzt, int64_t n, double pose_out[7], double *down_xyz, int64_t *n_down,
                             double *keypoints_xyz, int64_t *n_keypoints, limu_frame_stats *stats);
/* Replay / batch use: start uploading the NEXT scan (pinned host memory) on a separate stream while the current one is
 * being registered; the following limu_odom_register_frame call with the same pointer and size skips its own upload.
 * The buffer must stay untouched until that call. Results are identical with or without prefetching. */
int limu_odom_prefetch(limu_odom *o, const float *xyzt, int64_t n);
/* register_frame(cloud, timestamps) on the reference's own layout (PCL point records + FP64 timestamps). */
int limu_odom_register_cloud(limu_odom *o, const void *points, int32_t stride_bytes, const double *timestamps, int64_t n, double pose_out[7],
                             double *down_xyz, int64_t *n_down, double *keypoints_xyz, int64_t *n_keypoints, limu_frame_stats *stats);
/* limu_odom_prefetch for the reference's own layout: start uploading the NEXT cloud (records + FP64 timestamps, ideally pinned) while the
 * current one is being registered; the following limu_odom_register_cloud call with the same pointers, stride and size finds it on the device
 * (and, with LIMU_OPT_SPECULATE, already deskewed and downsampled). Both buffers must stay untouched until that call. */
int limu_odom_prefetch_cloud(limu_odom *o, const void *points, int32_t stride_bytes, const double *timestamps, int64_t n);
int limu_odom_register_frame_dev(limu_odom *o, const float *xyzt_dev, int64_t n, double pose_out[7], limu_frame_stats *stats);
/* Replay hint: the scan that will be registered AFTER the next limu_odom_register_frame_dev call already sits in device memory at
 * xyzt_dev_next (and stays untouched until it has been registered); limu_odom_prefetch gives the host-pointer entry the same treatment.
 * With LIMU_OPT_SPECULATE on (the default) limu_odom_register_frame[_dev] and limu_odom_register_cloud then PIPELINE consecutive scans
 * (csrc/odometry.cu):
 *   - the hinted scan's deskew + downsampling kernel is released the moment the current scan's Gauss-Newton loop has produced its pose
 *     (its deskew twist stays on the device) and runs beside the current scan's map update;
 *   - the hinted scan's IQR + Gauss-Newton loop is launched before the current call returns -- it only reads the map; the hinted scan's
 *     map update is launched only when the caller registers that scan. A hint that is not followed is simply dropped.
 * What the caller sees: a call returns as soon as its pose and clouds are there, while the map update of its scan may still be running --
 * every later call on the handle or its map is ordered behind it; an error of that update (a voxel index out of range after the transform
 * into the world frame) is returned by the NEXT call on the handle, or by limu_odom_flush. Poses do not depend on hints beyond rounding
 * (the twist of a scan prepared ahead is taken by the device's log instead of the host's: ~1e-15). */
int limu_odom_hint_next_dev(limu_odom *o, const float *xyzt_dev_next, int64_t n_next);
/* register_frame on an IMU-deskewed cloud: EKF::motion_compensation_with_imu (ekf.cpp:420-468; float write-back, then widening to double)
 * followed by register_frame(Vec3dVector) (icp.cpp:58-86) -- what limu_deskew_imu + limu_odom_register_points compute, in one call with
 * the deskew fused into the downsampling kernel and without the deskewed cloud travelling to the host and back. Records, curvature offset
 * and the pose table / rot_end / pos_lidar_end / p_imu_lidar are those of limu_deskew_imu (2 <= n_poses <= 96); n >= 0. The records are
 * not written back. cfg.deskew is ignored (that overload has no constant-velocity deskew); prediction, adaptive threshold, pose history and
 * map update are those of limu_odom_register_points. Pose and clouds refer to the scan-end lidar frame of the IMU deskew;
 * stats->deskewed = 2. The table and the three vectors are copied before the call returns. Constant-velocity and IMU scans may be
 * interleaved on one handle. */
int limu_odom_register_cloud_imu(limu_odom *o, const void *points, int32_t stride_bytes, int32_t curvature_offset_bytes, int64_t n,
                                 const limu_imu_pose *table, int32_t n_poses, const double rot_end[9], const double pos_lidar_end[3],
                                 const double p_imu_lidar[3], double pose_out[7], double *down_xyz, int64_t *n_down, double *keypoints_xyz,
                                 int64_t *n_keypoints, limu_frame_stats *stats);
/* limu_odom_prefetch_cloud for limu_odom_register_cloud_imu: start uploading the NEXT cloud and its pose table. The following
 * limu_odom_register_cloud_imu call with the same pointer, stride, curvature offset and size and byte-equal IMU arguments finds it on the
 * device (and, with LIMU_OPT_SPECULATE, already deskewed and downsampled: the IMU deskew does not depend on the previous pose); any other
 * call drops what was prepared. The records must stay untouched until that call; the table and the vectors are copied before this call
 * returns. Results are identical with or without prefetching. */
int limu_odom_prefetch_cloud_imu(limu_odom *o, const void *points, int32_t stride_bytes, int32_t curvature_offset_bytes, int64_t n,
                                 const limu_imu_pose *table, int32_t n_poses, const double rot_end[9], const double pos_lidar_end[3],
                                 const double p_imu_lidar[3]);
/* Handle options. LIMU_OPT_SPECULATE (default 1; the environment variable LIMU_SPECULATE=0 changes the default): see above.
 * LIMU_OPT_CLUSTER_LOOP: retired, accepted and ignored -- the loop shape it selected gave the same results more slowly (DESIGN.md section 9). */
enum { LIMU_OPT_SPECULATE = 1, LIMU_OPT_CLUSTER_LOOP = 2 };
int limu_odom_set_option(limu_odom *o, int32_t option, int64_t value);
/* Wait for everything the handle has in flight (a map update, kernels launched ahead for a hinted scan) and return the status of a map
 * update that no call has reported yet. Not needed for correctness of later calls; useful before timing or tearing down. */
int limu_odom_flush(limu_odom *o);
/* register_frame(Vec3dVector) icp.cpp:58-86 (no deskew). */
int limu_odom_register_points(limu_odom *o, const double *xyz, int64_t n, double pose_out[7], double *down_xyz, int64_t *n_down,
                              double *keypoints_xyz, int64_t *n_keypoints, limu_frame_stats *stats);
int limu_odom_num_poses(limu_odom *o, int64_t *n);                 /* poses_() icp.hpp:57 */
int limu_odom_pose(limu_odom *o, int64_t i, double pose_out[7]);
int limu_odom_adaptive_threshold(limu_odom *o, double *sigma);     /* get_adaptive_threshold() icp.cpp:138-144 (has the reference's side effect) */
int limu_odom_prediction(limu_odom *o, double pose_out[7]);        /* get_prediction_model() icp.cpp:146-154 */
int limu_odom_has_moved(limu_odom *o, int *out);                   /* has_moved() icp.cpp:156-163 */
limu_map *limu_odom_map(limu_odom *o);                             /* the local map (owned by the odometry handle) */

/* ---- frame::Lidar::process_frame, L/src/sensors/lidar/frame.cpp:101-193 (SURVEY section 8f N3) ------------------------------
 * The host preprocessing in front of register_frame: range gate [min_range, max_range] + NaN drop (:143-145), per-point offset
 * time in ms ("curvature", :156; or the constant-rotation model :159-182 when the last point carries no offset time), order by
 * that time (sort_clouds :28-51), drop the first point and cut into frame_split_num segments (split_clouds :53-99), per-point
 * timestamps via utils::get_time_stamps / normalize_timestamps (L/src/utils/calculation_helpers.cpp:3-81).
 * Input: the sensor_msgs::PointCloud2 payload as it arrives (n records of point_step bytes). */
typedef struct limu_cloud_fields {   /* byte offsets inside one record; -1 = the message has no such field (the member stays 0) */
    int32_t point_step;
    int32_t off_x, off_y, off_z;     /* FLOAT32: what pcl::fromROSMsg copies into the reference's LidarPoint (lidar/frame.hpp:12-23) */
    int32_t off_intensity;           /* UINT8 */
    int32_t off_ring;                /* UINT16 */
    int32_t off_timestamp;           /* FLOAT64 LidarPoint::timestamp, absolute seconds */
    int32_t off_time_field;          /* the field utils::get_time_stamps picks: the LAST one named "t", "timestamp" or "time" */
    int32_t time_field_is_f64;       /* 1: that field is "time" (read as double, used as is); 0: "t"/"timestamp" (its first 4 bytes read as
                                      * uint32 whatever the datatype, then divided by the maximum when that is >= 1) */
} limu_cloud_fields;
/* Applies the reference's field selection rules to a PointField list (names: nf NUL-terminated strings back to back; datatypes:
 * sensor_msgs::PointField codes). LIMU_ERR_INVALID with the reference's exception text when no timestamp field exists. */
int limu_cloud_fields_from_pointfields(int32_t nf, const char *names, const int32_t *offsets, const int32_t *datatypes, const int32_t *counts,
                                       int32_t point_step, limu_cloud_fields *out);
typedef struct limu_lidar_config {   /* frame::Lidar::ProcessingInfo, lidar/frame.hpp:39-45, defaults :64-70 */
    double min_range, max_range, min_angle, max_angle, frame_rate;
    int32_t num_scan_lines, frame_split_num;
} limu_lidar_config;
void limu_lidar_default_config(limu_lidar_config *cfg);
/* scan_count: value of the reference's message counter during process_frame (initialize() has incremented it, frame.cpp:13): the
 * 1-based index of this message; below MIN_SCAN_COUNT = 20 the frame is never split (:64).
 * Outputs: segments back to back -- out_points (optional): 48-byte pcl::PointXYZINormal records {x,y,z,1 | 0,0,0,0 | intensity,
 * curvature,0,0}, out_ts (optional): normalised FP64 timestamps, both with room for n entries; seg_sizes / seg_time
 * (accumulated_segment_time, seconds) with room for max_segments. Points of EQUAL offset time keep message order (std::sort leaves
 * their order unspecified in the reference). */
int limu_preprocess_frame(limu_ctx *c, const void *data, int64_t n, const limu_cloud_fields *fields, const limu_lidar_config *cfg, double message_time,
                          int32_t scan_count, void *out_points, double *out_ts, int32_t max_segments, int64_t *seg_sizes, double *seg_time,
                          int32_t *n_segments);
/* lidar_callback -> lidar_process -> estimate_lidar_odometry (L/src/odom_run.cpp:51-106) for one message: preprocess on the device, then
 * register_frame on every segment straight from device memory (no host copy of the processed cloud). poses_out: 7 doubles per
 * segment; stats (optional): one entry per segment. Segments of <= 1 point are skipped like odom_run.cpp:78-83 (their pose slot
 * repeats the previous pose and seg_sizes keeps the size). */
int limu_odom_register_msg(limu_odom *o, const void *data, int64_t n, const limu_cloud_fields *fields, const limu_lidar_config *cfg, double message_time,
                           int32_t scan_count, int32_t max_segments, double *poses_out, int64_t *seg_sizes, double *seg_time, int32_t *n_segments,
                           limu_frame_stats *stats);

/* ---- kalman::EKF predict / update, L/src/kalman/ekf.cpp (SURVEY section 8f N4) -------------------------------------------------
 * HOST code inside the library (the north star keeps the small state solve on the host): the reference's error-state-free quaternion EKF --
 * 30 inner states + a trail of `lidar_pose_trail` poses of 7 -- restated without Eigen. The reference constructs this filter and never
 * steps it at runtime; parity is pinned against the compiled original (oracle/ref_ekf_driver.cpp). State layout, ekf.hpp:32-44: POS 0,
 * VEL 3, ORI 6 (w x y z), BGA 10, BAA 13, BAT 16, GRAV 19, POS_IMU_LIDAR 22, ROT_IMU_LIDAR 25 (x y z w as Eigen stores it), SFT 29,
 * trail poses from 30. Matrices are row-major, dim = 30 + 7 * lidar_pose_trail. */
typedef struct limu_ekf_params {   /* kalman::EKF_PARAMETERS, ekf.hpp:62-86 */
    int32_t lidar_pose_trail, reserved0;
    double noise_scale, init_pos_noise, init_vel_noise, init_ori_noise, init_bga_noise, init_baa_noise, init_bat_noise;
    double acc_process_noise, gyro_process_noise, acc_process_noise_rev, gyro_process_noise_rev;
    double init_lidar_imu_time_noise, init_pos_trail_noise, init_ori_trail_noise, visualZuptR;
} limu_ekf_params;
typedef struct limu_ekf limu_ekf;
void limu_ekf_default_params(limu_ekf_params *p);
int limu_ekf_create(const limu_ekf_params *p, limu_ekf **out);       /* EKF::EKF :63-190 */
void limu_ekf_destroy(limu_ekf *e);
int limu_ekf_state_dim(limu_ekf *e, int32_t *dim);
int limu_ekf_get_state(limu_ekf *e, double *m /* dim */, double *P /* dim x dim */, double *current_time); /* any pointer may be NULL */
int limu_ekf_set_state(limu_ekf *e, const double *m, const double *P);
/* initialize_imu_global_orientation :194-211 as evidently intended (the original has undefined behaviour: four coefficients into a Vector3d) */
int limu_ekf_initialize_orientation(limu_ekf *e, const double xa[3], const double calc_grav[3]);
/* predict :214-290: state propagation with gyro xg / accelerometer xa at time t, Jacobians, covariance */
int limu_ekf_predict(limu_ekf *e, double t, const double xg[3], const double xa[3], const double calc_grav[3], const double trans_lidar_imu[3],
                     const double rot_lidar_imu[9]);
int limu_ekf_normalize_quaternions(limu_ekf *e, int only_current);   /* :619-636 */
int limu_ekf_zero_velocity_update(limu_ekf *e, double r);            /* zero_vel_update :657-678 */
int limu_ekf_augment_pose_trail(limu_ekf *e);                        /* update_visual_pose_aug :700-734 */
int limu_ekf_undo_augmentation(limu_ekf *e);                         /* update_undo_augmentation :736-756 */
int limu_ekf_update_and_propagate(limu_ekf *e);                      /* :680-698 */
/* The registration result as a measurement of the filter -- what the reference's design promised and its code never wired (SURVEY F2):
 * pose {qx,qy,qz,qw, tx,ty,tz} (limu_odom_register_*) observes POS and ORI directly, R = diag(pos_sigma^2 x3, ori_sigma^2 x4) * noise_scale.
 * No counterpart in the reference (parity unpinned). */
int limu_ekf_update_lidar_pose(limu_ekf *e, const double pose[7], double pos_sigma, double ori_sigma);

/* ---- host-side SE(3) helpers (the same restatement of Sophus 1.22.10 the device code uses) ------ */
void limu_se3_exp(const double x[6], double pose_out[7]);
void limu_se3_log(const double pose[7], double x_out[6]);
void limu_se3_mul(const double a[7], const double b[7], double out[7]);
void limu_se3_inverse(const double a[7], double out[7]);

#ifdef __cplusplus
}
#endif
#endif /* LIMU_CUDA_H */
