// icp_args.cuh -- the parameter block of the persistent registration kernel and of the map-update kernel (registration.cu). The odometry
// pipeline (odometry.cu) fills the fields of the frame around the ICP loop; icp_device / frame_update_device fill what they derive themselves.
#pragma once
#include "voxel_map.cuh"

namespace limu {

constexpr int NS_MAX = 32;   // doubles of the widest per-CTA partial row (the point-to-plane variant)
constexpr int MBOX_MAX_RANKS = 8, MBOX_ROW = 24, MBOX_RING = 4;   // mailbox row: NS doubles + stamp + pad; ring of 4 exchange slots

struct IcpArgs {
    MapView map;
    const unsigned long long *map_counters;   // [0] = live voxels (empty map -> return init_guess, registration.cpp:99-100)
    const double *points;       // n x 3, sensor frame (read only)
    double *work;               // n x 3, running source cloud
    int64_t n_max;
    const int *n_dev;
    double init_pose[7];        // init_guess, by value (no staging copy per call)
    double tau_sq;              // max_corresp_dist^2 (voxel_hash_map.cpp:112)
    double th;                  // kernel (registration.cpp:57-58)
    int max_iter;
    double eps;
    double *partials;           // [2][icp_blocks][NSX] (value, stamp) word pairs: the per-CTA rows of an iteration, self-validating (see ll_* below)
    unsigned int ll_stamp_base; // stamps of this launch are 0x80000000 | ((ll_stamp_base + iteration) & 0x7FFFFFFF): never 0, never reused soon
    unsigned int *barrier;      // zeroed before launch; nullptr when filled by the caller: the context's words (launches on different streams need their own)
    double *out;                // [0..6] pose, [7] iterations, [8] converged, [9] ncorr, [10] ncand, [11] nmiss, [12] n
    int grouped;                // 1: eight lanes per query (latency shape: a few thousand keypoints)
    int stage_doubles;          // > 0: the launch carries dynamic shared memory for the staged pass of the bandwidth shape
    int iqr_cap;                // latency shape: candidates the grid-wide IQR ranking can hold per CTA: IQR_GRID_MAX (static shared memory), or 8192 / 16384
                                // (the launch then carries iqr_cap * 10 bytes of dynamic shared memory: squared ranges + index list)
    int coop_scan;              // 1: sub-warp cooperative candidate scan (bandwidth shape); 0: one lane per query (latency shape)
    // point-sharded multi-GPU (SURVEY section 8e): every rank owns a contiguous shard of the queries and a full replica of
    // the map; per iteration the ranks exchange their NS-double row through peer-mapped mailboxes (NVLink stores).
    int nranks, rank;
    double *mbox_local;         // [MBOX_RING][MAX_RANKS][MBOX_ROW] in this rank's memory
    double *mbox_peer[MBOX_MAX_RANKS];   // the same buffer of every rank (peer mappings; [rank] == mbox_local)
    unsigned long long stamp_base;   // exchanges completed by earlier calls: iteration j of this call is exchange number stamp_base + j, its
                                     // stamp is that number + 1 and its ring slot that number mod MBOX_RING (contiguous ACROSS calls, so a rank
                                     // that is already in the next call can never overwrite a slot a slower peer is still reading)
    int *comm_error;            // set to 1 if a peer did not show up in time
    // ---- fused frame mode (odometry.cu): optional IQR prologue and local_map.update epilogue in the same launch ----
    const double *iqr_in;       // src0 (after the two downsampling stages); nullptr = no prologue
    const int *iqr_n;           // its count (device)
    double *iqr_d2;             // scratch, one double per point
    double *iqr_out;            // filtered keypoints (== points); count written to iqr_count
    int *iqr_count;
    const double *upd_down;     // downsampled scan (sensor frame); nullptr = no epilogue
    const int *upd_n;           // its count (device)
    double *upd_world;          // transformed copy
    unsigned int *upd_pslot;
    unsigned long long *upd_counters;   // map counters (writable)
    unsigned long long upd_birth_base;
    long long upd_capacity;     // C
    double upd_max_distance;
    DevStatus *status;          // nullptr when filled by the caller: the context's status word
    unsigned int *exit_count;   // last CTA out resets the barrier words (no memset per launch)
    unsigned int *barrier_icp;  // barrier of the leading `icp_blocks` CTAs that run the Gauss-Newton loop
    int icp_blocks;
    double *twist_out;          // non-null: leave log(last_pose^-1 * new_pose) here for the NEXT scan's deskew (delta_pose, deskew.cpp:14)
    double last_pose[7];        // poses.back() before this scan
    unsigned int *loop_flag;    // non-null: set to loop_seq (release, GPU scope) once the pose of this launch is in memory and its reads of the map are over (what k_gate waits for)
    unsigned int loop_seq;
    double *host_res;           // non-null: pinned host memory; CTA 0 copies the handle's result block (res_block, res_doubles) there when the
    const double *res_block;    // launch is over and then stores loop_seq into word 31 (system scope): the host reads its pose without a copy
    int res_doubles;            // engine round trip in the stream, and the next kernel of the stream starts right behind this one
    double *est_trace;          // optional [max_iter][7]
    long long *ncorr_trace;     // optional [max_iter]
    double *hg_trace;           // optional [max_iter][42]
};

// Enqueue the persistent ICP kernel on `stream` (nullptr: the context's). A: zeroed, then the caller's fields (points .. out, the fused-frame
// fields, the traces); n_hint: query count the launch shape is chosen for; sharded: the point-sharded loop of the context's communicator.
int icp_device(limu_map *m, IcpArgs A, int64_t n_hint, int icp_mode, bool sharded, cudaStream_t stream);
// The map-update half of a frame as a launch of its own on the context's stream: A holds the upd_* fields, status, barrier and out = the
// 7 pose doubles the loop kernel left.
int frame_update_device(limu_map *m, IcpArgs A);
// Reserve the per-CTA partial rows of the loop in `rows`; a fresh allocation is zero-filled, so that nothing in it looks like a stamp.
int icp_partials_reserve(limu_ctx *c, DevBuf &rows, cudaStream_t s);

}  // namespace limu
