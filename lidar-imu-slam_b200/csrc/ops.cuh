// ops.cuh -- device-pointer entry points of the per-scan stages (shared by the C ABI wrappers in
// ops.cu and the fused pipeline in odometry.cu). All counts may live in device memory (n_dev) so
// stages chain without a host round trip; n_max is the launch bound.
#pragma once
#include "common.cuh"

namespace limu {

// Scratch owned by whoever runs a downsample / IQR stage.
struct StageScratch {
    DevBuf table;     // [keys u64 x Cs | minidx u32 x Cs]
    DevBuf pslot;     // u32 per point
    DevBuf flags;     // u8 per point
    DevBuf blockcnt;  // int per 1024 points
    DevBuf idx;       // int per point (survivor indices)
    DevBuf d2;        // double per point (IQR)
    void release() { table.release(); pslot.release(); flags.release(); blockcnt.release(); idx.release(); d2.release(); }
};

// Scratch of the fused deskew + two-stage downsample kernel (voxelize.cu).
struct VoxelizeScratch {
    DevBuf table, pslot, tiles;
    int64_t cap_slots = 0, pslot_n = 0;   // allocated slots per table / entries per pslot array
    int parity = 0;                       // which of the two stage-2 tables the NEXT launch uses
    int st_word = 0;                      // which of the owner's three status words the NEXT launch reports into
    unsigned int epoch = 0;               // launch counter: validates the per-tile count words
    void release() { table.release(); pslot.release(); tiles.release(); cap_slots = pslot_n = 0; parity = 0; st_word = 0; }
};
// The IMU deskew of a cloud of point records (limu_deskew_imu's arguments): `table` = M pose rows of 22 doubles in DEVICE memory, the float
// curvature (ms) of each record at byte offset toff, the scan-end rotation (row-major) and lidar position, the IMU->lidar lever arm.
struct ImuDeskew {
    const double *table;
    int M, toff;
    double rot_end[9], pos_lidar_end[3], p_il[3];
};
struct ImuCall;   // the arguments of one IMU-deskewing call (imu_compensate.cuh)
// One scan in device memory as k_voxelize reads it.
enum ScanLayout {
    SCAN_XYZT = 0,      // float4 {x,y,z,t}
    SCAN_RECORDS = 1,   // records `stride` bytes apart (float x,y,z first) + FP64 timestamps `ts`
    SCAN_XYZ = 2,       // double xyz (register_frame(Vec3dVector)): already a frame, never deskewed
    SCAN_IMU = 3,       // records `stride` bytes apart, IMU-deskewed as limu_deskew_imu does with `imu` and the pose table at `imu_table`
};
struct Scan {
    int layout = SCAN_XYZT;
    const void *ptr = nullptr;
    int stride = 0;
    const double *ts = nullptr;
    const ImuCall *imu = nullptr;
    const double *imu_table = nullptr;
    int64_t n = 0;
};
// KissICP::deskew_scan + the two voxel_downsample stages of KissICP::voxelize in one cooperative launch. deskew (layouts 0 and 1): with the
// twist at twist_host, or at twist_dev (device memory: speculative launches, odometry.cu).
// own_status: THREE status words private to the pipeline that owns `sc` (zero at first use): consecutive launches rotate through them and each
// launch zeroes the next one late, so a word is clean when its launch starts without a memset per scan; *status_used = which word this launch
// reports into. nullptr = the context's shared word.
// stream: where to enqueue (nullptr = the context's); beside: the lean kernel on all but GATE_SLACK_SMS SMs, so that the launch runs next to the
// map update of the pipelined path.
int voxelize_device(limu_ctx *c, VoxelizeScratch &sc, const Scan &scan, int deskew, const double *twist_host, double v, double *frame_dev, double *down_dev,
                    double *src0_dev, int *counts_dev, const double *twist_dev = nullptr, DevStatus *own_status = nullptr, int *status_used = nullptr,
                    cudaStream_t stream = nullptr, bool beside = false);
// One-thread kernel on stream s that returns once *flag has reached seq (voxelize.cu).
int gate_device(cudaStream_t s, const unsigned int *flag, unsigned int seq);

// deskew.cpp:10-28. twist_dev: 6 doubles (device). out: n x 3 doubles.
int deskew_device(limu_ctx *c, const float *xyzt_dev, int64_t n, const double *twist_dev, double *out_dev);
// the same for strided point records + FP64 timestamps (the reference's PCL cloud + std::vector<double>)
int deskew_records_device(limu_ctx *c, const void *rec_dev, int stride, const double *ts_dev, int64_t n, const double *twist_dev, double *out_dev);
int widen_records_device(limu_ctx *c, const void *rec_dev, int stride, int64_t n, double *out_dev);
// pointcloud2eigen, calculation_helpers.cpp:83-97: widen float xyz to double.
int widen_device(limu_ctx *c, const float *xyzt_dev, int64_t n, double *out_dev);
// icp.cpp:9-30 first-point-wins downsample. out_idx_dev: survivor indices (int, n_max), out_count_dev: int.
int downsample_device(limu_ctx *c, StageScratch &sc, const double *xyz_dev, int64_t n_max, const int *n_dev, double s,
                      double *out_xyz_dev, int *out_count_dev);
// icp.cpp:88-124 + common.hpp:22-63. bounds_dev: 2 doubles (optional).
int iqr_device(limu_ctx *c, StageScratch &sc, const double *xyz_dev, int64_t n_max, const int *n_dev, double *out_xyz_dev,
               int *out_count_dev, double *bounds_dev);


// ---- frame::Lidar::process_frame on the device (preprocess.cu; SURVEY section 8f N3) ----
constexpr int PRE_MAX_SEG = 64;
struct SegTable {                      // device + pinned host mirror
    int nseg, m, pad0, pad1;
    int begin[PRE_MAX_SEG], end[PRE_MAX_SEG];   // sorted positions (begin, end] -> output rows begin .. end-1
    double adj[PRE_MAX_SEG];           // message_time_ms - last_frame_end_time of the segment (frame.cpp:74)
    double time[PRE_MAX_SEG];          // accumulated_segment_time (:89)
    double tmax[PRE_MAX_SEG];          // maximum of the segment's timestamps (normalize_timestamps :87)
};
struct PreScratch {
    DevBuf raw, curv, ext, flags, blockcnt, sidx, keys[2], vals[2], hist, small, rec, ts;
    SegTable *h_seg = nullptr;   // pinned
    void release() {
        DevBuf *b[] = {&raw, &curv, &ext, &flags, &blockcnt, &sidx, &keys[0], &keys[1], &vals[0], &vals[1], &hist, &small, &rec, &ts};
        for (auto *x : b) x->release();
        if (h_seg) { cudaFreeHost(h_seg); h_seg = nullptr; }
    }
};
// Everything up to the processed records in device memory. data_dev: the message payload on the device. On return
// sc.rec / sc.ts hold the concatenated segments (48-byte pcl::PointXYZINormal records + FP64 timestamps) and *sc.h_seg the
// segment table (host; the call synchronises once to read it).
int preprocess_device(limu_ctx *c, PreScratch &sc, const unsigned char *data_dev, int64_t n, const limu_cloud_fields &f, const limu_lidar_config &cfg,
                      double message_time, int scan_count);
int preprocess_validate(const limu_cloud_fields *f, const limu_lidar_config *cfg, int max_segments);

}  // namespace limu
