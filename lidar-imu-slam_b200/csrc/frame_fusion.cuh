// frame_fusion.cuh -- what the odometry pipeline asks the persistent registration kernel to do around the ICP loop.
#pragma once
#include "common.cuh"
namespace limu {
struct FrameFusion {
    const double *iqr_in;      // src0 after the two downsampling stages (nullptr: no IQR prologue)
    const int *iqr_n;
    double *iqr_d2, *iqr_out;
    int *iqr_count;
    const double *upd_down;    // downsampled scan, sensor frame (nullptr: no map-update epilogue)
    const int *upd_n;
    double *upd_world;
    unsigned int *upd_pslot;
    unsigned long long upd_birth_base;
    double *twist_out;         // non-null: leave log(last_pose^-1 * new_pose) here for the NEXT scan's deskew (delta_pose, deskew.cpp:14)
    double last_pose[7];       // poses.back() before this scan
    unsigned int *loop_flag;   // non-null: the kernel stores loop_seq here once its pose is in memory and its reads of the map are over (what k_gate waits for)
    unsigned int loop_seq;
    double *host_res;          // non-null (launches without the map update only): pinned host copy of res_block[0 .. res_doubles), word 31 <- loop_seq when it is complete
    const double *res_block;
    int res_doubles;
    DevStatus *status;         // the frame kernel's status word (per odometry handle); nullptr = the context's
    cudaStream_t stream;       // where to launch (nullptr: the context's stream)
    unsigned int *barrier;     // 8 zero-at-rest words private to the caller for the grid barriers (nullptr: the context's; launches on different streams need their own)
};
}  // namespace limu
struct limu_map;
namespace limu {
// The map-update half of a frame as a launch of its own: pose_dev = the 7 doubles the loop kernel left (registration.cu).
int frame_update_device(limu_map *m, const FrameFusion &fuse, const double *pose_dev);
}  // namespace limu
