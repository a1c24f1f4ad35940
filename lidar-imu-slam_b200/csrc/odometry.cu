// odometry.cu -- lidar::KissICP (L/include/limu/sensors/lidar/icp.hpp:31-68, L/src/sensors/lidar/icp.cpp)
// as a device pipeline: one H2D of the raw scan, every stage enqueued on the handle's stream with
// device-side counts, ONE host synchronisation per scan (to read the pose the scalar host glue needs:
// adaptive threshold, constant-velocity prediction -- L/src/sensors/lidar/helpers/threshold.cpp, icp.cpp:138-163).
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "icp_args.cuh"
#include "imu_compensate.cuh"
#include "ops.cuh"

namespace limu {

// theta = Eigen::AngleAxisd(model_dev.rotationMatrix()).angle() (threshold.cpp:7): quaternion -> matrix
// (Eigen Quaternion::toRotationMatrix) -> quaternion (Eigen RotationBase assign, Quaternion.h) -> 2 atan2(|v|, |w|).
static double rotation_angle(const Pose &T) {
    const double x = T.qx, y = T.qy, z = T.qz, w = T.qw;
    const double tx = 2 * x, ty = 2 * y, tz = 2 * z;
    const double twx = tx * w, twy = ty * w, twz = tz * w, txx = tx * x, txy = ty * x, txz = tz * x, tyy = ty * y, tyz = tz * y, tzz = tz * z;
    double m[3][3];
    m[0][0] = 1 - (tyy + tzz); m[0][1] = txy - twz; m[0][2] = txz + twy;
    m[1][0] = txy + twz; m[1][1] = 1 - (txx + tzz); m[1][2] = tyz - twx;
    m[2][0] = txz - twy; m[2][1] = tyz + twx; m[2][2] = 1 - (txx + tyy);
    double c[4];
    double t = (m[0][0] + m[1][1]) + m[2][2];
    if (t > 0) {
        t = sqrt(t + 1.0);
        c[3] = 0.5 * t; t = 0.5 / t;
        c[0] = (m[2][1] - m[1][2]) * t; c[1] = (m[0][2] - m[2][0]) * t; c[2] = (m[1][0] - m[0][1]) * t;
    } else {
        int i = 0;
        if (m[1][1] > m[0][0]) i = 1;
        if (m[2][2] > m[i][i]) i = 2;
        const int j = (i + 1) % 3, k = (j + 1) % 3;
        t = sqrt(m[i][i] - m[j][j] - m[k][k] + 1.0);
        c[i] = 0.5 * t; t = 0.5 / t;
        c[3] = (m[k][j] - m[j][k]) * t; c[j] = (m[j][i] + m[i][j]) * t; c[k] = (m[k][i] + m[i][k]) * t;
    }
    const double n = sqrt(sqnorm3(c[0], c[1], c[2]));
    return n != 0.0 ? 2.0 * atan2(n, fabs(c[3])) : 0.0;
}

static void imu_call_copy(ImuCall &dst, const ImuCall &src) {   // (the rows past M are not part of the call)
    dst.M = src.M; dst.toff = src.toff;
    memcpy(dst.rot_end, src.rot_end, sizeof dst.rot_end); memcpy(dst.pos_lidar_end, src.pos_lidar_end, sizeof dst.pos_lidar_end); memcpy(dst.p_il, src.p_il, sizeof dst.p_il);
    memcpy(dst.table, src.table, (size_t)src.M * 22 * sizeof(double));
}
static bool imu_call_same(const ImuCall &a, const ImuCall &b) {
    return a.M == b.M && a.toff == b.toff && !memcmp(a.rot_end, b.rot_end, sizeof a.rot_end) && !memcmp(a.pos_lidar_end, b.pos_lidar_end, sizeof a.pos_lidar_end) &&
           !memcmp(a.p_il, b.p_il, sizeof a.p_il) && !memcmp(a.table, b.table, (size_t)a.M * 22 * sizeof(double));
}

// Is `call` the scan `prepared` describes? The same layout, buffer, count and stride, and for an IMU-deskewed scan the same IMU arguments.
// One test for every place that reuses prepared work: a prefetch slot against a call (host pointers), the scan whose k_voxelize ran ahead
// against a slot or a call (device pointers). FP64 timestamps are not compared: a prefetch slot is known by its points pointer (the caller keeps
// both buffers untouched until the call), and on the device a record buffer and its timestamp buffer are uploaded and handed over together.
static bool scan_is(const Scan &prepared, const Scan &call) {
    if (!(prepared.layout == call.layout && prepared.ptr == call.ptr && prepared.n == call.n && prepared.stride == call.stride)) return false;
    return prepared.layout != SCAN_IMU || prepared.imu == call.imu || imu_call_same(*prepared.imu, *call.imu);
}
}  // namespace limu

// Device result block of one handle (per HANDLE: two handles of one context may interleave their scans). 28 ints, then 13 doubles:
//   [0] n_down, [1] n_src0 of the scans with parity 0     [20] [21] the same for parity 1 (consecutive scans alternate: in the pipelined
//   [2] n_keypoints (written by the loop kernel)                    path the next scan's k_voxelize runs while this scan's update reads its count)
//   [3] the loop flag: sequence number of the last Gauss-Newton loop that is over and has its pose in memory (k_gate waits for it)
//   [4..7] / [24..27] status word of the map update of a parity-0 / parity-1 scan
//   [8..19] three status words k_voxelize rotates through
//   doubles 14..26: pose + loop statistics (out13).     ONE copy of RES_DOUBLES per scan.
namespace {
constexpr int RES_CNT1 = 20, RES_FLAG = 3, RES_BARRIER = 64 /* 8 words, zero at rest: grid barriers of the pipelined kernels */, RES_UPD_ST0 = 4, RES_UPD_ST1 = 24, RES_VOX_ST = 8, RES_OUT = 14, RES_DOUBLES = 27;
inline int *res_counts(int *cnt, int par) { return cnt + (par ? RES_CNT1 : 0); }
inline limu::DevStatus *res_update_status(int *cnt, int par) { return reinterpret_cast<limu::DevStatus *>(cnt + (par ? RES_UPD_ST1 : RES_UPD_ST0)); }
}  // namespace

struct limu_odom {
    limu_ctx *ctx = nullptr;
    limu_odom_config cfg;
    limu_map *map = nullptr;
    std::vector<limu::Pose> poses;
    // AdaptiveThreshold (helpers/threshold.hpp:9-33)
    double model_error_sq = 0.0;
    int num_samples = 0;
    limu::Pose model_deviation = limu::pose_identity();
    // device buffers. down / src0 / src exist twice: consecutive scans alternate (`par`), so that the next scan's kernels and this scan's
    // cloud copies never touch the same buffer.
    limu::DevBuf raw, ts, frame, down[2], src0[2], src[2], work, world, partials, d2, res;
    int par = 0;                            // parity of the scan registered last
    limu::VoxelizeScratch vx;
    limu::PreScratch pre;                   // limu_odom_register_msg: frame::Lidar::process_frame on the device
    int64_t nk_hint = 2048, nd_hint = 16384;   // keypoints / downsampled points of the previous scan (launch shapes; the kernels take any count)
    // limu_odom_prefetch*: the next scan is uploaded on its own stream while the current one is being registered. Two slots: the scan about
    // to be registered and the one after it.
    struct Prefetch {
        limu::Scan call;                    // the prefetch call: host pointers, imu = the pinned copy below; call.ptr == nullptr: nothing a call can claim
        limu::DevBuf buf, ts, imu_tab;      // the device copy: points, FP64 timestamps (records), pose table (IMU records)
        limu::ImuCall *imu = nullptr;       // pinned: the IMU arguments of the call (its table upload's source)
        cudaEvent_t done = nullptr;         // behind the upload on copy_stream
        uint64_t seq = 0;                   // order in which the pending uploads were requested
    } pf[2];
    uint64_t pf_counter = 0;
    limu::DevBuf imu_tab;                   // pose table of the IMU scan being registered when it was not prefetched (swaps with pf[].imu_tab like raw / pf[].buf)
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t clouds_done = nullptr;
    // ---- pipelined path (LIMU_OPT_SPECULATE, on by default; packed float4 scans) -------------------------------------------------------
    // When the library knows which scan comes next (a device-pointer hint from limu_odom_hint_next_dev, or the scan limu_odom_prefetch is
    // uploading) the work of consecutive scans overlaps on the device and with the host:
    //   pipe stream     [loop X] [vox X+1] [loop X+1] [vox X+2] ...     loop   = IQR + Gauss-Newton loop (reads the map, writes a pose)
    //   context stream     [gate|update X]    [gate|update X+1]         update = local_map.update: insert + eviction
    //   * the critical chain -- loop X, deskew + downsampling of scan X+1 (its deskew twist is log(pose X-1^-1 pose X), left on the device
    //     by loop X), loop X+1 -- is one in-order stream without events or host round trips in it;
    //   * the map update of scan X runs BESIDE vox X+1 on the context's stream: a one-thread gate kernel releases it the moment loop X
    //     is over (loop X+1 waits for its event, normally long complete);
    //   * loop X+1 is launched at the END of call X -- before the caller has asked for scan X+1 -- because it only reads the map: if the
    //     caller then registers something else its result is dropped. The map update of a scan is launched only once that scan has been
    //     registered by the caller. So a call finds its pose computed (or in flight), and the GPU never waits for the host round trip;
    //   * the loop kernel leaves its result block in pinned host memory itself (no copy engine in the chain); the host polls for it.
    // Consequences for the caller: a call returns while the map update of its scan may still run (everything else on the handle or its map
    // goes to the context's stream behind it); an error of that update (voxel index out of range AFTER the transform into the world) is
    // reported by the next call on the handle or by limu_odom_flush.
    bool speculate = true;
    const void *hint_ptr = nullptr;         // next scan (device float4 rows), set by the caller before registering the current one
    int64_t hint_n = 0;
    cudaStream_t pipe_stream = nullptr;
    cudaEvent_t loop_done[2] = {nullptr, nullptr}, upd_done[2] = {nullptr, nullptr}, pipe_tail = nullptr, input_ready = nullptr;
    bool upd_recorded[2] = {false, false};
    cudaEvent_t pev_vox[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}}, pev_upd[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   // profiling: device time of launches collected one call later
    bool pev_vox_used[2] = {false, false}, pev_upd_used[2] = {false, false};
    double *h_res[2] = {nullptr, nullptr};  // pinned: the result block of a scan of either parity (256 bytes; word 30 checksum, word 31 sequence number)
    unsigned int loop_seq = 0;              // sequence number of the last loop launch of this handle
    unsigned int loop_seq_of[2] = {0, 0};   // ... and of the last launch for either parity (what the host waits for in h_res[par][31])
    limu::DevBuf twist_next;                // 6 doubles written by the loop kernel
    int pending_update_par = -1;            // parity of a map update whose status word has not been read yet
    struct Ahead {                          // what is in flight for the scan the caller said comes next
        limu::Scan scan;                    // that scan (device pointers): a hint, or the device copy of prefetch slot `slot`
        int deskewed = 0, slot = -1, par = 0, vox_word = 0;
        bool vox = false, loop = false;
        double sigma = 0.0;                 // what the loop was launched with
        limu::Pose init = limu::pose_identity();
        uint64_t map_mutations = 0;         // the map's mutation count when the loop was launched (the caller may touch the map between calls)
        double stash_model_error_sq = 0.0;  // AdaptiveThreshold state before the glue of that launch: restored if the launch is not used
        int stash_num_samples = 0;
    } ahead;
};

using namespace limu;

// The device copy of the scan in a prefetch slot.
static Scan prefetched(const limu_odom::Prefetch &p) {
    Scan s = p.call;
    s.ptr = p.buf.p;
    s.ts = s.layout == SCAN_RECORDS ? p.ts.as<double>() : nullptr;
    s.imu_table = s.layout == SCAN_IMU ? p.imu_tab.as<double>() : nullptr;
    return s;
}

static bool odom_has_moved(const limu_odom *o) {   // icp.cpp:156-163
    if (o->poses.empty()) return false;
    const Pose d = mul(inverse(o->poses.front()), o->poses.back());
    return sqrt(sqnorm3(d.tx, d.ty, d.tz)) > 5.0 * o->cfg.min_motion_th;
}
static double odom_compute_threshold(limu_odom *o) {   // threshold.cpp:16-28 (+ :5-12)
    const double theta = rotation_angle(o->model_deviation);
    const double delta_rot = 2.0 * o->cfg.max_range * sin(theta / 2.0);
    const double delta_trans = sqrt(sqnorm3(o->model_deviation.tx, o->model_deviation.ty, o->model_deviation.tz));
    const double model_error = delta_rot + delta_trans;
    if (model_error > o->cfg.min_motion_th) { o->model_error_sq += model_error * model_error; o->num_samples++; }
    if (o->num_samples < 1) return o->cfg.initial_threshold;
    return sqrt(o->model_error_sq / o->num_samples);
}
static double odom_adaptive_threshold(limu_odom *o) {   // icp.cpp:138-144
    if (!odom_has_moved(o)) return o->cfg.initial_threshold;
    return odom_compute_threshold(o);
}
static Pose odom_prediction(const limu_odom *o) {   // icp.cpp:146-154
    const size_t N = o->poses.size();
    if (N < 2) return pose_identity();
    return mul(inverse(o->poses[N - 2]), o->poses[N - 1]);
}

static int odom_side_stream(limu_odom *o) {
    if (!o->copy_stream) {
        LIMU_CUDA_TRY(cudaStreamCreateWithFlags(&o->copy_stream, cudaStreamNonBlocking));
        for (int sl = 0; sl < 2; ++sl) LIMU_CUDA_TRY(cudaEventCreateWithFlags(&o->pf[sl].done, cudaEventDisableTiming));
    }
    if (!o->clouds_done) LIMU_CUDA_TRY(cudaEventCreateWithFlags(&o->clouds_done, cudaEventDisableTiming));
    return LIMU_OK;
}

static int odom_res_block(limu_odom *o) {
    if (!o->res.p) {
        LIMU_TRY(o->res.reserve(48 * sizeof(double)));
        LIMU_CUDA_TRY(cudaMemsetAsync(o->res.p, 0, o->res.bytes, o->ctx->stream));
    }
    return LIMU_OK;
}

// Forget what is in flight for a scan that will not be registered (or not as it was prepared). The kernels themselves are harmless -- they
// write buffers of the other parity and scratch -- but the threshold model must not keep a sample that was added for a registration that
// did not happen (get_adaptive_threshold accumulates on every call, threshold.cpp:16-28). to_context_stream: what follows goes to the
// context's stream (plain path), which therefore waits for whatever the pipe stream still has to do.
static int odom_drop_ahead(limu_odom *o, bool keep_voxelize, bool to_context_stream = false) {
    limu_odom::Ahead &ah = o->ahead;
    if (ah.loop) { o->model_error_sq = ah.stash_model_error_sq; o->num_samples = ah.stash_num_samples; ah.loop = false; }
    if (!keep_voxelize && ah.vox) { ah.vox = false; ah.slot = -1; }
    if (to_context_stream && o->pipe_stream) {
        LIMU_CUDA_TRY(cudaEventRecord(o->pipe_tail, o->pipe_stream));
        LIMU_CUDA_TRY(cudaStreamWaitEvent(o->ctx->stream, o->pipe_tail, 0));
    }
    return LIMU_OK;
}

// Status word of a map update that was launched by an earlier call and is complete by now (stream order): report and clear it.
static int odom_deferred_status(limu_odom *o, const int *host_res) {
    if (o->pending_update_par < 0) return LIMU_OK;
    const int p = o->pending_update_par;
    o->pending_update_par = -1;
    DevStatus st;
    memcpy(&st, host_res + (p ? RES_UPD_ST1 : RES_UPD_ST0), sizeof st);
    if (!(st.key_range | st.table_full)) return LIMU_OK;
    LIMU_CUDA_TRY(cudaMemsetAsync(res_update_status(o->res.as<int>(), p), 0, sizeof(DevStatus), o->ctx->stream));
    if (st.key_range) { set_error("map update of the PREVIOUS frame: voxel index outside the packed key range (|index| >= 2^20); the frame was inserted without those points"); return LIMU_ERR_KEY_RANGE; }
    set_error("map update of the previous frame: voxel hash table full");
    return LIMU_ERR_MAP_FULL;
}

static int odom_report(limu_odom *o, const int *hc, int vox_word, int upd_par, bool spec_hit, int64_t n, int deskewed, double sigma, limu_frame_stats *stats) {
    const double *ho = reinterpret_cast<const double *>(hc) + RES_OUT;
    const int64_t nk = hc[2];
    if (stats) {
        stats->n_points = n; stats->n_down = res_counts(const_cast<int *>(hc), o->par)[0]; stats->n_keypoints = nk; stats->sigma = sigma; stats->deskewed = deskewed;
        stats->reserved0 = spec_hit ? 1 : 0;
        stats->icp.iterations = (int)ho[7]; stats->icp.converged = (int)ho[8]; stats->icp.last_ncorr = (int64_t)ho[9];
        stats->icp.mean_candidates = nk > 0 ? ho[10] / (double)nk : 0.0;
        stats->icp.miss_fraction = nk > 0 ? ho[11] / (double)nk : 0.0;
    }
    // device status of this scan: its own k_voxelize word and (plain path) the frame kernel's word
    DevStatus st = {0, 0, {0, 0}}, sv;
    if (upd_par >= 0) memcpy(&st, hc + (upd_par ? RES_UPD_ST1 : RES_UPD_ST0), sizeof st);
    memcpy(&sv, hc + RES_VOX_ST + 4 * vox_word, sizeof sv);
    if (st.key_range | st.table_full | st.pad[0]) LIMU_CUDA_TRY(cudaMemsetAsync(res_update_status(o->res.as<int>(), upd_par), 0, sizeof(DevStatus), o->ctx->stream));   // (the next frame kernel is launched after this)
    st.key_range |= sv.key_range; st.table_full |= sv.table_full;
    if (st.key_range) { set_error("voxel index outside the packed key range (|index| >= 2^20) or NaN coordinate: the frame was registered without those points"); return LIMU_ERR_KEY_RANGE; }
    if (st.table_full) { set_error("voxel hash table full"); return LIMU_ERR_MAP_FULL; }
    return LIMU_OK;
}

// Copy this scan's clouds to the caller. `side`: the main stream is busy with later work, use the copy stream (what the copies read is complete).
static int odom_copy_clouds(limu_odom *o, bool side, int par, const int *hc, double *down_xyz, double *keypoints_xyz) {
    limu_ctx *c = o->ctx;
    const int64_t nd = res_counts(const_cast<int *>(hc), par)[0], nk = hc[2];
    if (!((down_xyz && nd > 0) || (keypoints_xyz && nk > 0))) return LIMU_OK;
    cudaStream_t s = c->stream;
    if (side) { LIMU_TRY(odom_side_stream(o)); s = o->copy_stream; }
    if (down_xyz && nd > 0) LIMU_CUDA_TRY(cudaMemcpyAsync(down_xyz, o->down[par].p, (size_t)nd * 24, cudaMemcpyDeviceToHost, s));
    if (keypoints_xyz && nk > 0) LIMU_CUDA_TRY(cudaMemcpyAsync(keypoints_xyz, o->src[par].p, (size_t)nk * 24, cudaMemcpyDeviceToHost, s));
    if (side) {
        LIMU_CUDA_TRY(cudaEventRecord(o->clouds_done, s));
        LIMU_CUDA_TRY(cudaEventSynchronize(o->clouds_done));
    } else {
        LIMU_CUDA_TRY(cudaStreamSynchronize(s));
    }
    return LIMU_OK;
}

// ---- the steps of one scan that the plain and the pipelined path share ----------------------------------------------------------------
// Deskew gate (icp.cpp:40-46) of a scan registered with n_poses poses in the history: 1 = constant-velocity deskew (config.deskew &&
// poses.size() > 2), 2 = IMU-compensated, 0 = none.
static int odom_deskew_gate(const limu_odom *o, int layout, size_t n_poses) {
    if (layout == SCAN_IMU) return 2;
    return (layout != SCAN_XYZ && o->cfg.deskew && n_poses > 2) ? 1 : 0;
}
static void odom_deskew_twist(const limu_odom *o, double twist[6]) {   // twist = delta_pose(poses[N-2], poses[N-1]) (deskew.cpp:14)
    const size_t N = o->poses.size();
    se3_log(mul(inverse(o->poses[N - 2]), o->poses[N - 1]), twist);
}
// What k_voxelize writes for a scan of n points and parity par.
static int odom_reserve_voxelize(limu_odom *o, int par, int64_t n, cudaStream_t s) {
    const size_t nb = (size_t)std::max<int64_t>(n, 1) * 24;
    LIMU_TRY(o->frame.reserve(nb, s));
    LIMU_TRY(o->down[par].reserve(nb, s));
    LIMU_TRY(o->src0[par].reserve(nb, s));
    return LIMU_OK;
}
// The loop half of a frame of parity par: iqr_processing of src0[par] into src[par] (icp.cpp:133), then ICP (icp.cpp:74-76) from init with
// the adaptive threshold sigma; the pose and loop statistics go to the result block.
static void odom_loop_args(limu_odom *o, IcpArgs &A, int par, int64_t n, const Pose &init, const Pose &last, double sigma) {
    int *cnt = o->res.as<int>();
    A.points = o->src[par].as<double>(); A.work = o->work.as<double>(); A.n_max = n; A.n_dev = cnt + 2;
    pose_store(init, A.init_pose);
    const double tau = 3.0 * sigma;
    A.tau_sq = tau * tau; A.th = sigma / 3.0; A.max_iter = o->cfg.icp_max_iteration; A.eps = o->cfg.estimation_threshold;
    A.partials = o->partials.as<double>(); A.out = o->res.as<double>() + RES_OUT;
    A.iqr_in = o->src0[par].as<double>(); A.iqr_n = res_counts(cnt, par) + 1; A.iqr_d2 = o->d2.as<double>(); A.iqr_out = o->src[par].as<double>(); A.iqr_count = cnt + 2;
    pose_store(last, A.last_pose);
}
// The map-update half of a frame of parity par: local_map.update(down_sampled, new_pose) (icp.cpp:81; voxel_hash_map.cpp:138-144).
static int odom_update_args(limu_odom *o, IcpArgs &A, int par, int64_t n) {
    limu_ctx *c = o->ctx;
    LIMU_TRY(map_maybe_grow(o->map, n));
    LIMU_TRY(o->map->pslot.reserve((size_t)std::max<int64_t>(n, 1) * 4, c->stream));
    LIMU_TRY(o->world.reserve((size_t)std::max<int64_t>(n, 1) * 24, c->stream));
    int *cnt = o->res.as<int>();
    A.upd_down = o->down[par].as<double>(); A.upd_n = res_counts(cnt, par); A.upd_world = o->world.as<double>(); A.upd_pslot = o->map->pslot.as<unsigned int>();
    A.upd_birth_base = o->map->birth_base;
    A.status = res_update_status(cnt, par);
    return LIMU_OK;
}
// The map bookkeeping of an update that has been launched; returns used_upper from before it.
static int64_t odom_map_claim(limu_odom *o, int64_t n) {
    const int64_t upper_before = o->map->used_upper;
    o->map->birth_base += (uint64_t)n;
    o->map->used_upper = upper_before + std::max<int64_t>(n, 0);   // safe bound until the exact count arrives (at most one new voxel per point)
    return upper_before;
}
// Commit the whole frame of parity par from its result block hc -- map bookkeeping, pose history, threshold state, outputs -- BEFORE anyone
// looks at the device status: the map update inserts this scan (points with out-of-range voxel indices were left out by both downsampling
// and the insert), so an error return must not leave a map that holds a scan without a pose.
static Pose odom_commit(limu_odom *o, const int *hc, int par, const Pose &init, int64_t upper_before, double pose_out[7], int64_t *n_down,
                        int64_t *n_keypoints) {
    const int64_t nd = res_counts(const_cast<int *>(hc), par)[0], nk = hc[2];
    const Pose new_pose = pose_load(reinterpret_cast<const double *>(hc) + RES_OUT);
    o->map->used_upper = upper_before + nd;   // exact: at most one new voxel per inserted point
    o->nk_hint = std::max<int64_t>(nk, 256);
    o->nd_hint = std::max<int64_t>(nd, 256);
    o->model_deviation = mul(inverse(init), new_pose);   // icp.cpp:78-79
    o->poses.push_back(new_pose);                        // :82
    o->par = par;
    if (pose_out) pose_store(new_pose, pose_out);
    if (n_down) *n_down = nd;
    if (n_keypoints) *n_keypoints = nk;
    return new_pose;
}

// Plain path: everything of one scan enqueued on the context's stream, one synchronisation, nothing left in flight. The scan is in device
// memory (an IMU scan: register_frame(Vec3dVector) on the compensated cloud, no constant-velocity deskew).
static int odom_register_device(limu_odom *o, const Scan &scan, double pose_out[7], double *down_xyz, int64_t *n_down, double *keypoints_xyz,
                                int64_t *n_keypoints, limu_frame_stats *stats) {
    limu_ctx *c = o->ctx;
    LIMU_TRY(odom_drop_ahead(o, false, true));
    o->hint_ptr = nullptr; o->hint_n = 0;
    const int64_t n = scan.n;
    const int deskewed = odom_deskew_gate(o, scan.layout, o->poses.size());
    double twist[6] = {0, 0, 0, 0, 0, 0};
    if (deskewed == 1) odom_deskew_twist(o, twist);
    const int par = o->par ^ 1;
    const size_t nb = (size_t)std::max<int64_t>(n, 1) * 24;
    LIMU_TRY(odom_reserve_voxelize(o, par, n, c->stream));
    LIMU_TRY(o->src[par].reserve(nb, c->stream));
    LIMU_TRY(o->work.reserve(nb, c->stream));
    LIMU_TRY(o->world.reserve(nb, c->stream));
    LIMU_TRY(icp_partials_reserve(c, o->partials, c->stream));
    LIMU_TRY(odom_res_block(o));
    int *cnt = o->res.as<int>();
    DevStatus *vox_status = reinterpret_cast<DevStatus *>(cnt + RES_VOX_ST);

    // deskew_scan + voxelize's two downsampling stages (icp.cpp:36-47, :126-131): one cooperative launch
    int vox_word = 0;
    LIMU_TRY(prof_begin(c, LIMU_STAGE_DOWNSAMPLE));
    LIMU_TRY(voxelize_device(c, o->vx, scan, deskewed == 1, twist, o->cfg.voxel_size, o->frame.as<double>(), o->down[par].as<double>(),
                             o->src0[par].as<double>(), res_counts(cnt, par), nullptr, vox_status, &vox_word));
    LIMU_TRY(prof_end(c, LIMU_STAGE_DOWNSAMPLE));
    // host scalar glue (icp.cpp:66-71)
    const double sigma = odom_adaptive_threshold(o);
    const Pose last = o->poses.empty() ? pose_identity() : o->poses.back();
    const Pose init = mul(last, odom_prediction(o));

    // the IQR, the Gauss-Newton loop and the map update: ONE persistent cooperative launch (registration.cu)
    IcpArgs A;
    memset(&A, 0, sizeof A);
    LIMU_TRY(odom_update_args(o, A, par, n));
    LIMU_TRY(o->d2.reserve((size_t)std::max<int64_t>(n, 1) * 8, c->stream));
    odom_loop_args(o, A, par, n, init, last, sigma);
    LIMU_TRY(icp_device(o->map, A, o->nk_hint, o->cfg.icp_mode, false, nullptr));
    const int64_t upper_before = odom_map_claim(o, n);

    // the one synchronisation of the scan (nothing is left in flight: a later call on the pipelined path need not wait for anything)
    double *h = static_cast<double *>(c->h_pinned) + 32;
    LIMU_CUDA_TRY(cudaMemcpyAsync(h, o->res.p, RES_DOUBLES * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
    o->upd_recorded[0] = o->upd_recorded[1] = false;
    LIMU_TRY(prof_collect(c));
    const int *hc = reinterpret_cast<const int *>(h);
    odom_commit(o, hc, par, init, upper_before, pose_out, n_down, n_keypoints);
    LIMU_TRY(odom_copy_clouds(o, false, par, hc, down_xyz, keypoints_xyz));
    const int deferred = odom_deferred_status(o, hc);   // (an update of the pipelined path that nobody has asked about yet)
    LIMU_TRY(odom_report(o, hc, vox_word, par, false, n, deskewed, sigma, stats));
    return deferred;
}

static int odom_pipe_init(limu_odom *o) {
    if (o->pipe_stream) return LIMU_OK;
    LIMU_TRY(odom_res_block(o));
    LIMU_CUDA_TRY(cudaStreamSynchronize(o->ctx->stream));   // (the result block is zeroed before the pipe stream sees it)
    LIMU_CUDA_TRY(cudaStreamCreateWithFlags(&o->pipe_stream, cudaStreamNonBlocking));
    LIMU_CUDA_TRY(cudaEventCreateWithFlags(&o->pipe_tail, cudaEventDisableTiming));
    LIMU_CUDA_TRY(cudaEventCreateWithFlags(&o->input_ready, cudaEventDisableTiming));
    for (int k = 0; k < 2; ++k) {
        LIMU_CUDA_TRY(cudaEventCreateWithFlags(&o->loop_done[k], cudaEventDisableTiming));
        LIMU_CUDA_TRY(cudaEventCreateWithFlags(&o->upd_done[k], cudaEventDisableTiming));
        LIMU_CUDA_TRY(cudaEventCreate(&o->pev_vox[k][0]));
        LIMU_CUDA_TRY(cudaEventCreate(&o->pev_vox[k][1]));
        LIMU_CUDA_TRY(cudaEventCreate(&o->pev_upd[k][0]));
        LIMU_CUDA_TRY(cudaEventCreate(&o->pev_upd[k][1]));
        LIMU_CUDA_TRY(cudaMallocHost(&o->h_res[k], 32 * sizeof(double)));
        memset(o->h_res[k], 0, 32 * sizeof(double));
    }
    return odom_side_stream(o);
}

// The IQR + Gauss-Newton half of a frame as a launch of its own on the pipe stream (no map update). It waits for the map update of the
// previous scan (context stream); its result block goes to h_res[par] (pinned), loop_done[par] is recorded behind it.
static int odom_launch_loop(limu_odom *o, int par, int64_t n, const Pose &init, const Pose &last, double sigma) {
    limu_ctx *c = o->ctx;
    cudaStream_t ps = o->pipe_stream;
    const size_t nb = (size_t)std::max<int64_t>(n, 1) * 24;
    LIMU_TRY(o->src[par].reserve(nb, ps));
    LIMU_TRY(o->work.reserve(nb, ps));
    LIMU_TRY(o->d2.reserve((size_t)std::max<int64_t>(n, 1) * 8, ps));
    LIMU_TRY(o->twist_next.reserve(6 * sizeof(double), ps));
    LIMU_TRY(icp_partials_reserve(c, o->partials, ps));
    int *cnt = o->res.as<int>();
    IcpArgs A;
    memset(&A, 0, sizeof A);
    odom_loop_args(o, A, par, n, init, last, sigma);
    A.twist_out = o->twist_next.as<double>();
    A.loop_flag = reinterpret_cast<unsigned int *>(cnt + RES_FLAG);
    A.loop_seq = ++o->loop_seq;
    A.host_res = o->h_res[par]; A.res_block = o->res.as<double>(); A.res_doubles = RES_DOUBLES;
    A.barrier = reinterpret_cast<unsigned int *>(cnt + RES_BARRIER);
    if (o->upd_recorded[par ^ 1]) LIMU_CUDA_TRY(cudaStreamWaitEvent(ps, o->upd_done[par ^ 1], 0));
    LIMU_TRY(icp_device(o->map, A, o->nk_hint, o->cfg.icp_mode, false, ps));
    LIMU_CUDA_TRY(cudaEventRecord(o->loop_done[par], ps));
    o->map->readers_done = o->loop_done[par];   // (entry points that change the map from the context's stream wait for this reader)
    o->loop_seq_of[par] = o->loop_seq;
    return LIMU_OK;
}

// Wait until the loop launched for parity `par` has left its result block in h_res[par]: word 31 carries its sequence number, word 30 the
// XOR of the other words (the kernel stores the block without a system-scope fence, so a torn read is possible -- and read again).
static int odom_wait_loop(limu_odom *o, int par, unsigned long long out[32]) {
    const volatile unsigned long long *src = reinterpret_cast<const volatile unsigned long long *>(o->h_res[par]);
    const unsigned long long want = o->loop_seq_of[par];
    for (unsigned int spins = 1;; ++spins) {
        if (src[31] == want) {
            unsigned long long x = 0ull;
            for (int k = 0; k < 32; ++k) { out[k] = src[k]; if (k != 30) x ^= out[k]; }
            if (out[31] == want && x == out[30]) return LIMU_OK;
        }
        if ((spins & 0x3FFFu) == 0u) {   // now and then: is the kernel still alive?
            const cudaError_t e = cudaEventQuery(o->loop_done[par]);
            if (e == cudaSuccess) {
                unsigned long long x = 0ull;
                for (int k = 0; k < 32; ++k) { out[k] = src[k]; if (k != 30) x ^= out[k]; }
                if (out[31] == want && x == out[30]) return LIMU_OK;
                set_error("registration kernel finished without publishing its result");
                return LIMU_ERR_CUDA;
            }
            if (e != cudaErrorNotReady) { set_error("registration kernel failed: %s", cudaGetErrorString(e)); return LIMU_ERR_CUDA; }
        }
    }
}

// Pipelined path (see limu_odom): scan in device memory (float4 rows, point records with FP64 timestamps, or IMU-deskewed records).
// input_ready: event behind the scan's upload (nullptr: it is there).
static int odom_register_pipelined(limu_odom *o, const Scan &scan, cudaEvent_t input_ready, double pose_out[7], double *down_xyz, int64_t *n_down,
                                   double *keypoints_xyz, int64_t *n_keypoints, limu_frame_stats *stats) {
    limu_ctx *c = o->ctx;
    LIMU_TRY(odom_pipe_init(o));
    cudaStream_t ps = o->pipe_stream;
    limu_odom::Ahead &ah = o->ahead;
    const int64_t n = scan.n;
    const size_t NP = o->poses.size();
    const int deskewed = odom_deskew_gate(o, scan.layout, NP);
    const int par = o->par ^ 1, npar = par ^ 1;
    const bool hit_vox = ah.vox && n > 0 && scan_is(ah.scan, scan) && ah.deskewed == deskewed && ah.par == par;
    const bool hit_loop = hit_vox && ah.loop && ah.map_mutations == o->map->mutations;
    if (ah.vox && !hit_vox && ah.slot >= 0 && scan_is(prefetched(o->pf[ah.slot]), ah.scan)) {
        // the caller registered something else than the scan it had prefetched: that upload is stale, do not prepare it again
        o->pf[ah.slot].call.ptr = nullptr;
    }
    // the scan after this one, if the caller told us where it is: a device-pointer hint, or the OLDEST upload limu_odom_prefetch has pending
    Scan next;
    int next_slot = -1;
    if (o->hint_ptr) { next.ptr = o->hint_ptr; next.n = o->hint_n; }
    else {
        for (int sl = 0; sl < 2; ++sl)
            if (o->pf[sl].call.ptr && o->pf[sl].buf.p != scan.ptr && (next_slot < 0 || o->pf[sl].seq < o->pf[next_slot].seq)) next_slot = sl;
        if (next_slot >= 0) next = prefetched(o->pf[next_slot]);
    }
    o->hint_ptr = nullptr; o->hint_n = 0;   // a hint is good for one call only
    int *cnt = o->res.as<int>();
    DevStatus *vox_status = reinterpret_cast<DevStatus *>(cnt + RES_VOX_ST);
    const double v = o->cfg.voxel_size;
    const Pose last = o->poses.empty() ? pose_identity() : o->poses.back();

    // 1. this scan's k_voxelize, unless it ran ahead (pipe stream: behind whatever was prepared for a scan that did not come)
    int vox_word = ah.vox_word;
    if (!hit_vox) {
        LIMU_TRY(odom_drop_ahead(o, false));
        double twist[6] = {0, 0, 0, 0, 0, 0};
        if (deskewed == 1) odom_deskew_twist(o, twist);
        LIMU_TRY(odom_reserve_voxelize(o, par, n, ps));
        if (input_ready) LIMU_CUDA_TRY(cudaStreamWaitEvent(ps, input_ready, 0));
        if (c->profiling) LIMU_CUDA_TRY(cudaEventRecord(o->pev_vox[par][0], ps));
        LIMU_TRY(voxelize_device(c, o->vx, scan, deskewed == 1, twist, v, o->frame.as<double>(), o->down[par].as<double>(), o->src0[par].as<double>(),
                                 res_counts(cnt, par), nullptr, vox_status, &vox_word, ps, false));
        if (c->profiling) { LIMU_CUDA_TRY(cudaEventRecord(o->pev_vox[par][1], ps)); o->pev_vox_used[par] = true; }
    }
    // 2. its loop, unless that ran ahead too (with exactly the glue this call would compute)
    double sigma;
    Pose init;
    if (hit_loop) {
        sigma = ah.sigma; init = ah.init;
        ah.loop = false;   // consumed: the threshold sample it added stays
    } else {
        LIMU_TRY(odom_drop_ahead(o, true));
        sigma = odom_adaptive_threshold(o);              // host scalar glue (icp.cpp:66-71)
        init = mul(last, odom_prediction(o));
        LIMU_TRY(odom_launch_loop(o, par, n, init, last, sigma));
    }
    const unsigned int my_seq = o->loop_seq_of[par];
    ah.vox = false; ah.slot = -1;
    // 3. its map update on the context's stream: the caller has registered this scan (local_map.update, icp.cpp:81). A gate kernel holds it
    //    until the loop is over.
    {
        IcpArgs A;
        memset(&A, 0, sizeof A);
        LIMU_TRY(odom_update_args(o, A, par, n));
        A.barrier = reinterpret_cast<unsigned int *>(cnt + RES_BARRIER) + 4;   // (its own words: the next scan's loop may be running on the pipe stream)
        A.out = o->res.as<double>() + RES_OUT;                                  // the pose the loop left
        LIMU_TRY(gate_device(c->stream, reinterpret_cast<unsigned int *>(cnt + RES_FLAG), my_seq));
        if (c->profiling) LIMU_CUDA_TRY(cudaEventRecord(o->pev_upd[par][0], c->stream));
        LIMU_TRY(frame_update_device(o->map, A));
        if (c->profiling) { LIMU_CUDA_TRY(cudaEventRecord(o->pev_upd[par][1], c->stream)); o->pev_upd_used[par] = true; }
        LIMU_CUDA_TRY(cudaEventRecord(o->upd_done[par], c->stream));
        o->upd_recorded[par] = true;
    }
    const int64_t upper_before = odom_map_claim(o, n);
    // 4. the next scan's k_voxelize right behind this scan's loop in the pipe stream (its deskew twist, log(last^-1 * new) (deskew.cpp:14),
    //    is left on the device by that loop; an IMU-deskewed scan needs only its own slot's arguments); lean CTAs: it runs beside the map update
    if (next.ptr && next.n > 0) {
        const int next_deskewed = odom_deskew_gate(o, next.layout, NP + 1);   // the gate as the next scan will see it
        LIMU_TRY(odom_reserve_voxelize(o, npar, next.n, ps));
        if (next_slot >= 0) LIMU_CUDA_TRY(cudaStreamWaitEvent(ps, o->pf[next_slot].done, 0));
        int w = 0;
        if (c->profiling) LIMU_CUDA_TRY(cudaEventRecord(o->pev_vox[npar][0], ps));
        LIMU_TRY(voxelize_device(c, o->vx, next, next_deskewed == 1, nullptr, v, o->frame.as<double>(), o->down[npar].as<double>(), o->src0[npar].as<double>(),
                                 res_counts(cnt, npar), next_deskewed == 1 ? o->twist_next.as<double>() : nullptr, vox_status, &w, ps, true));
        if (c->profiling) { LIMU_CUDA_TRY(cudaEventRecord(o->pev_vox[npar][1], ps)); o->pev_vox_used[npar] = true; }
        ah.vox = true; ah.scan = next; ah.slot = next_slot; ah.deskewed = next_deskewed; ah.par = npar; ah.vox_word = w;
    }
    // 5. the one wait of the call: this scan's pose
    unsigned long long hw[32];
    LIMU_TRY(odom_wait_loop(o, par, hw));
    if (c->profiling) {
        LIMU_CUDA_TRY(cudaEventSynchronize(o->loop_done[par]));   // (the stage events sit behind the kernel in the stream)
        LIMU_TRY(prof_collect(c));
        float ms = 0.f;
        if (o->pev_vox_used[par]) {   // this scan's k_voxelize
            if (cudaEventElapsedTime(&ms, o->pev_vox[par][0], o->pev_vox[par][1]) == cudaSuccess) c->stage_ms[LIMU_STAGE_DOWNSAMPLE] += (double)ms; else (void)cudaGetLastError();
            o->pev_vox_used[par] = false;
        }
        if (o->pev_upd_used[npar]) {   // the previous scan's map update (this scan's loop waited for it)
            if (cudaEventElapsedTime(&ms, o->pev_upd[npar][0], o->pev_upd[npar][1]) == cudaSuccess) c->stage_ms[LIMU_STAGE_MAP_UPDATE] += (double)ms; else (void)cudaGetLastError();
            o->pev_upd_used[npar] = false;
        }
    }
    const int *hc = reinterpret_cast<const int *>(hw);
    const Pose new_pose = odom_commit(o, hc, par, init, upper_before, pose_out, n_down, n_keypoints);
    const int deferred = odom_deferred_status(o, hc);   // the previous scan's map update ran in front of this scan's loop
    o->pending_update_par = par;
    // 6. the next scan's loop, ahead of the caller asking for it: it only reads the map (it waits for this scan's update)
    if (ah.vox) {
        ah.stash_model_error_sq = o->model_error_sq; ah.stash_num_samples = o->num_samples;
        ah.sigma = odom_adaptive_threshold(o);
        ah.init = mul(new_pose, odom_prediction(o));
        ah.map_mutations = o->map->mutations;
        ah.loop = true;
        const int st = odom_launch_loop(o, npar, ah.scan.n, ah.init, new_pose, ah.sigma);
        if (st != LIMU_OK) { (void)odom_drop_ahead(o, true); return st; }
    }
    // 7. this scan's clouds (both streams are busy with later work). The keypoint cloud is the last thing the loop kernel writes -- after the
    //    result block this call woke up on -- so a caller who wants it waits for the kernel itself.
    if (keypoints_xyz && hc[2] > 0) LIMU_CUDA_TRY(cudaEventSynchronize(o->loop_done[par]));
    LIMU_TRY(odom_copy_clouds(o, true, par, hc, down_xyz, keypoints_xyz));
    LIMU_TRY(odom_report(o, hc, vox_word, -1, hit_vox, n, deskewed, sigma, stats));
    return deferred;
}

// Wait for everything the handle has in flight and report what a deferred map update had to say.
static int odom_flush(limu_odom *o) {
    limu_ctx *c = o->ctx;
    LIMU_TRY(odom_drop_ahead(o, false, true));
    LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (o->pending_update_par < 0 || !o->res.p) return LIMU_OK;
    double *h = static_cast<double *>(c->h_pinned) + 32;
    LIMU_CUDA_TRY(cudaMemcpyAsync(h, o->res.p, RES_DOUBLES * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
    return odom_deferred_status(o, reinterpret_cast<const int *>(h));
}

extern "C" {

void limu_odom_default_config(limu_odom_config *cfg) {   // lidar/frame.hpp:64-80
    if (!cfg) return;
    memset(cfg, 0, sizeof *cfg);
    cfg->max_range = 100.0;
    cfg->voxel_size = cfg->max_range / 100.0;
    cfg->max_points_per_voxel = 10;
    cfg->deskew = 0;
    cfg->min_motion_th = 0.1;
    cfg->icp_max_iteration = 500;
    cfg->initial_threshold = 2.0;
    cfg->estimation_threshold = 0.0001;
}

int limu_odom_create(limu_ctx *c, const limu_odom_config *cfg, limu_odom **out) {
    LIMU_TRY(bind(c));
    LIMU_REQUIRE(cfg && out, "limu_odom_create: null argument");
    LIMU_REQUIRE(cfg->voxel_size > 0 && cfg->max_points_per_voxel >= 1, "limu_odom_create: voxel_size must be > 0 and max_points_per_voxel >= 1");
    LIMU_REQUIRE((cfg->icp_mode & ~(LIMU_ICP_NN27 | LIMU_ICP_PLANE)) == 0, "limu_odom_create: unknown icp_mode bits");
    limu_odom *o = new limu_odom;
    o->ctx = c;
    o->cfg = *cfg;
    if (const char *e = getenv("LIMU_SPECULATE")) o->speculate = atoi(e) != 0;        // default of LIMU_OPT_SPECULATE (on)
    int64_t capv = cfg->map_capacity_voxels;
    if (capv <= 0) {   // a sensor sees a shell, not a ball: ~ (2 r / v)^2 * 8 voxels is generous for one neighbourhood
        const double side = 2.0 * cfg->max_range / cfg->voxel_size;
        capv = (int64_t)std::min(4.0e6, std::max(65536.0, side * side * 8.0));
    }
    int st = limu_map_create(c, cfg->voxel_size, cfg->max_range, cfg->max_points_per_voxel, capv, &o->map);   // icp.hpp:35-37
    if (st != LIMU_OK) { delete o; return st; }
    *out = o;
    return LIMU_OK;
}

void limu_odom_destroy(limu_odom *o) {
    if (!o) return;
    cudaSetDevice(o->ctx->device);
    if (o->pipe_stream) cudaStreamSynchronize(o->pipe_stream);
    cudaStreamSynchronize(o->ctx->stream);
    o->map->readers_done = nullptr;
    limu_map_destroy(o->map);
    if (o->copy_stream) { cudaStreamSynchronize(o->copy_stream); cudaStreamDestroy(o->copy_stream); cudaEventDestroy(o->pf[0].done); cudaEventDestroy(o->pf[1].done); }
    DevBuf *bufs[] = {&o->res, &o->pf[0].buf, &o->pf[1].buf, &o->pf[0].ts, &o->pf[1].ts, &o->pf[0].imu_tab, &o->pf[1].imu_tab, &o->imu_tab, &o->d2, &o->raw, &o->ts, &o->frame, &o->down[0], &o->down[1], &o->src0[0], &o->src0[1], &o->src[0], &o->src[1],
                      &o->work, &o->world, &o->partials, &o->twist_next};
    for (auto *b : bufs) b->release();
    o->vx.release();
    o->pre.release();
    if (o->pipe_stream) {
        cudaStreamDestroy(o->pipe_stream);
        cudaEventDestroy(o->pipe_tail); cudaEventDestroy(o->input_ready);
        for (int k = 0; k < 2; ++k) {
            cudaEventDestroy(o->loop_done[k]); cudaEventDestroy(o->upd_done[k]);
            cudaEventDestroy(o->pev_vox[k][0]); cudaEventDestroy(o->pev_vox[k][1]); cudaEventDestroy(o->pev_upd[k][0]); cudaEventDestroy(o->pev_upd[k][1]);
            cudaFreeHost(o->h_res[k]);
        }
    }
    if (o->clouds_done) cudaEventDestroy(o->clouds_done);
    if (o->pf[0].imu) cudaFreeHost(o->pf[0].imu);
    delete o;
}

// A scan in host memory -> device memory, on the way noting whether limu_odom_prefetch* has uploaded it (and whether its k_voxelize has
// even run ahead). call: the scan as the caller gave it (host pointers). Returns the scan in device memory and the event to wait for.
static int odom_host_scan(limu_odom *o, const Scan &call, Scan *dev, cudaEvent_t *ready) {
    limu_ctx *c = o->ctx;
    const int64_t n = call.n;
    const size_t bytes = (size_t)n * (call.stride ? call.stride : 16);
    const bool with_ts = call.layout == SCAN_RECORDS, with_imu = call.layout == SCAN_IMU;
    int hit = -1;
    for (int s = 0; s < 2; ++s) if (n > 0 && scan_is(o->pf[s].call, call)) hit = s;
    *ready = nullptr;
    if (hit >= 0 && o->speculate && o->ahead.vox && scan_is(o->ahead.scan, prefetched(o->pf[hit]))) {
        // uploaded ahead of time AND already through k_voxelize (behind the previous scan's loop): register it where it lies
        o->pf[hit].call.ptr = nullptr;
        *dev = prefetched(o->pf[hit]);
        return LIMU_OK;
    }
    if (o->speculate) LIMU_TRY(odom_pipe_init(o));
    if (o->pipe_stream) LIMU_CUDA_TRY(cudaStreamSynchronize(o->pipe_stream));   // (o->raw may still be read by a kernel prepared for another scan)
    if (hit >= 0) {   // uploaded ahead of time: the buffers change hands
        LIMU_CUDA_TRY(cudaStreamWaitEvent(c->stream, o->pf[hit].done, 0));
        std::swap(o->raw, o->pf[hit].buf);
        if (with_ts) std::swap(o->ts, o->pf[hit].ts);
        if (with_imu) std::swap(o->imu_tab, o->pf[hit].imu_tab);
        o->pf[hit].call.ptr = nullptr;
        *ready = o->pf[hit].done;
    } else {
        LIMU_TRY(stage_in(c, o->raw, call.ptr, bytes));
        if (with_ts) LIMU_TRY(stage_in(c, o->ts, call.ts, (size_t)n * 8));
        if (with_imu) LIMU_TRY(stage_in(c, o->imu_tab, call.imu->table, (size_t)call.imu->M * 22 * sizeof(double)));
        if (o->speculate) { LIMU_CUDA_TRY(cudaEventRecord(o->input_ready, c->stream)); *ready = o->input_ready; }
    }
    *dev = call;
    dev->ptr = o->raw.p;
    dev->ts = with_ts ? o->ts.as<double>() : nullptr;
    dev->imu_table = with_imu ? o->imu_tab.as<double>() : nullptr;
    return LIMU_OK;
}

// Start the upload of a scan that will be registered later (two slots; the OLDEST pending upload gives way). call: the scan as the caller
// gave it (host pointers); an IMU scan's arguments are copied (pinned) and its pose table uploaded with the records.
static int odom_prefetch_scan(limu_odom *o, const Scan &call) {
    const int64_t n = call.n;
    if (n == 0) return LIMU_OK;
    LIMU_TRY(odom_side_stream(o));
    for (int s = 0; s < 2; ++s) if (scan_is(o->pf[s].call, call)) return LIMU_OK;   // already in flight
    const bool with_ts = call.layout == SCAN_RECORDS;
    const int s = o->pf[0].call.ptr == nullptr ? 0 : (o->pf[1].call.ptr == nullptr ? 1 : (o->pf[0].seq < o->pf[1].seq ? 0 : 1));
    limu_odom::Prefetch &p = o->pf[s];
    if (o->ahead.vox && scan_is(o->ahead.scan, prefetched(p))) {
        // the k_voxelize that ran ahead on the scan in this slot may still be reading it: let it finish, and forget what was prepared (the
        // slot is about to hold a different scan, possibly of the same size)
        LIMU_CUDA_TRY(cudaStreamSynchronize(o->pipe_stream));
        LIMU_TRY(odom_drop_ahead(o, false));
    }
    p.call.ptr = nullptr;
    const size_t bytes = (size_t)n * (call.stride ? call.stride : 16);
    if (p.buf.bytes < bytes || (with_ts && p.ts.bytes < (size_t)n * 8)) {   // growing may free a buffer the copy stream still writes: drain it first
        LIMU_CUDA_TRY(cudaStreamSynchronize(o->copy_stream));
        LIMU_TRY(p.buf.reserve(bytes, o->copy_stream));
        if (with_ts) LIMU_TRY(p.ts.reserve((size_t)n * 8, o->copy_stream));
    }
    if (call.layout == SCAN_IMU) {
        if (!p.imu) {   // (one pinned allocation for both slots)
            ImuCall *both = nullptr;
            LIMU_CUDA_TRY(cudaMallocHost(&both, 2 * sizeof(ImuCall)));
            o->pf[0].imu = both; o->pf[1].imu = both + 1;
        }
        LIMU_CUDA_TRY(cudaEventSynchronize(p.done));   // (the slot's previous table upload has read the host copy)
        imu_call_copy(*p.imu, *call.imu);
        LIMU_TRY(p.imu_tab.reserve(sizeof p.imu->table, o->copy_stream));
        LIMU_CUDA_TRY(cudaMemcpyAsync(p.imu_tab.p, p.imu->table, (size_t)p.imu->M * 22 * sizeof(double), cudaMemcpyHostToDevice, o->copy_stream));
    }
    LIMU_CUDA_TRY(cudaMemcpyAsync(p.buf.p, call.ptr, bytes, cudaMemcpyHostToDevice, o->copy_stream));
    if (with_ts) LIMU_CUDA_TRY(cudaMemcpyAsync(p.ts.p, call.ts, (size_t)n * 8, cudaMemcpyHostToDevice, o->copy_stream));
    LIMU_CUDA_TRY(cudaEventRecord(p.done, o->copy_stream));
    p.call = call;
    if (call.layout == SCAN_IMU) p.call.imu = p.imu;
    p.seq = ++o->pf_counter;
    return LIMU_OK;
}

// The scan of a register / prefetch call as the caller gave it: float4 rows (stride 0), records + FP64 timestamps, or with imu IMU-deskewed records.
static Scan odom_call(const void *pts, int stride, const double *ts, int64_t n, const ImuCall *imu = nullptr) {
    Scan s;
    s.layout = imu ? SCAN_IMU : stride ? SCAN_RECORDS : SCAN_XYZT;
    s.ptr = pts; s.stride = stride; s.ts = ts; s.imu = imu; s.n = n;
    return s;
}

// Register a scan given in host memory: on the pipelined path with LIMU_OPT_SPECULATE, else on the plain path.
static int odom_register_host(limu_odom *o, const Scan &call, double pose_out[7], double *down_xyz, int64_t *n_down, double *keypoints_xyz,
                              int64_t *n_keypoints, limu_frame_stats *stats) {
    Scan dev;
    cudaEvent_t ready = nullptr;   // what the scan's first kernel has to wait for when it is not launched on the context's stream
    LIMU_TRY(odom_host_scan(o, call, &dev, &ready));
    if (o->speculate) return odom_register_pipelined(o, dev, ready, pose_out, down_xyz, n_down, keypoints_xyz, n_keypoints, stats);
    return odom_register_device(o, dev, pose_out, down_xyz, n_down, keypoints_xyz, n_keypoints, stats);
}

int limu_odom_register_frame(limu_odom *o, const float *xyzt, int64_t n, double pose_out[7], double *down_xyz, int64_t *n_down,
                             double *keypoints_xyz, int64_t *n_keypoints, limu_frame_stats *stats) {
    LIMU_REQUIRE(o && n >= 0 && (n == 0 || xyzt), "limu_odom_register_frame: bad arguments");
    LIMU_TRY(bind(o->ctx));
    return odom_register_host(o, odom_call(xyzt, 0, nullptr, n), pose_out, down_xyz, n_down, keypoints_xyz, n_keypoints, stats);
}

int limu_odom_prefetch(limu_odom *o, const float *xyzt, int64_t n) {
    LIMU_REQUIRE(o && n >= 0 && (n == 0 || xyzt), "limu_odom_prefetch: bad arguments");
    LIMU_TRY(bind(o->ctx));
    return odom_prefetch_scan(o, odom_call(xyzt, 0, nullptr, n));
}

int limu_odom_register_cloud(limu_odom *o, const void *points, int32_t stride_bytes, const double *timestamps, int64_t n, double pose_out[7],
                             double *down_xyz, int64_t *n_down, double *keypoints_xyz, int64_t *n_keypoints, limu_frame_stats *stats) {
    LIMU_REQUIRE(o && n >= 0 && stride_bytes >= 12 && stride_bytes % 4 == 0 && (n == 0 || (points && timestamps)), "limu_odom_register_cloud: bad arguments");
    LIMU_TRY(bind(o->ctx));
    return odom_register_host(o, odom_call(points, stride_bytes, timestamps, n), pose_out, down_xyz, n_down, keypoints_xyz, n_keypoints, stats);
}

int limu_odom_prefetch_cloud(limu_odom *o, const void *points, int32_t stride_bytes, const double *timestamps, int64_t n) {
    LIMU_REQUIRE(o && n >= 0 && stride_bytes >= 12 && stride_bytes % 4 == 0 && (n == 0 || (points && timestamps)), "limu_odom_prefetch_cloud: bad arguments");
    LIMU_TRY(bind(o->ctx));
    return odom_prefetch_scan(o, odom_call(points, stride_bytes, timestamps, n));
}

// Arguments of the IMU entry points: where limu_deskew_imu accepts them (n >= 0 as for limu_odom_register_cloud). Copied into *a.
static int odom_imu_args(ImuCall *a, const char *fn, limu_odom *o, const void *points, int32_t stride, int32_t toff, int64_t n, const limu_imu_pose *table,
                         int32_t n_poses, const double *rot_end, const double *pos_lidar_end, const double *p_imu_lidar) {
    if (!(o && n >= 0 && (n == 0 || points) && table && rot_end && pos_lidar_end && p_imu_lidar && n_poses >= 2 && n_poses <= IMU_MAX_ROWS && stride >= 16 &&
          stride % 4 == 0 && toff >= 12 && toff + 4 <= stride && toff % 4 == 0)) {
        set_error("%s: bad arguments (need n >= 0, 2 <= n_poses <= 96, float x,y,z at offset 0 and a float time field inside each record)", fn);
        return LIMU_ERR_INVALID;
    }
    static_assert(sizeof(limu_imu_pose) == 22 * sizeof(double), "limu_imu_pose layout");
    a->M = n_poses; a->toff = toff;
    memcpy(a->rot_end, rot_end, sizeof a->rot_end); memcpy(a->pos_lidar_end, pos_lidar_end, sizeof a->pos_lidar_end); memcpy(a->p_il, p_imu_lidar, sizeof a->p_il);
    memcpy(a->table, table, (size_t)n_poses * sizeof(limu_imu_pose));
    return LIMU_OK;
}

int limu_odom_register_cloud_imu(limu_odom *o, const void *points, int32_t stride_bytes, int32_t curvature_offset_bytes, int64_t n, const limu_imu_pose *table,
                                 int32_t n_poses, const double rot_end[9], const double pos_lidar_end[3], const double p_imu_lidar[3], double pose_out[7],
                                 double *down_xyz, int64_t *n_down, double *keypoints_xyz, int64_t *n_keypoints, limu_frame_stats *stats) {
    ImuCall a;
    LIMU_TRY(odom_imu_args(&a, "limu_odom_register_cloud_imu", o, points, stride_bytes, curvature_offset_bytes, n, table, n_poses, rot_end, pos_lidar_end, p_imu_lidar));
    LIMU_TRY(bind(o->ctx));
    return odom_register_host(o, odom_call(points, stride_bytes, nullptr, n, &a), pose_out, down_xyz, n_down, keypoints_xyz, n_keypoints, stats);
}

int limu_odom_prefetch_cloud_imu(limu_odom *o, const void *points, int32_t stride_bytes, int32_t curvature_offset_bytes, int64_t n, const limu_imu_pose *table,
                                 int32_t n_poses, const double rot_end[9], const double pos_lidar_end[3], const double p_imu_lidar[3]) {
    ImuCall a;
    LIMU_TRY(odom_imu_args(&a, "limu_odom_prefetch_cloud_imu", o, points, stride_bytes, curvature_offset_bytes, n, table, n_poses, rot_end, pos_lidar_end, p_imu_lidar));
    LIMU_TRY(bind(o->ctx));
    return odom_prefetch_scan(o, odom_call(points, stride_bytes, nullptr, n, &a));
}

int limu_odom_register_frame_dev(limu_odom *o, const float *xyzt_dev, int64_t n, double pose_out[7], limu_frame_stats *stats) {
    LIMU_REQUIRE(o && n >= 0 && (n == 0 || xyzt_dev), "limu_odom_register_frame_dev: bad arguments");
    LIMU_TRY(bind(o->ctx));
    const Scan scan = odom_call(xyzt_dev, 0, nullptr, n);
    if (o->speculate) return odom_register_pipelined(o, scan, nullptr, pose_out, nullptr, nullptr, nullptr, nullptr, stats);
    return odom_register_device(o, scan, pose_out, nullptr, nullptr, nullptr, nullptr, stats);
}

int limu_odom_hint_next_dev(limu_odom *o, const float *xyzt_dev_next, int64_t n_next) {
    LIMU_REQUIRE(o && n_next >= 0, "limu_odom_hint_next_dev: bad arguments");
    o->hint_ptr = (o->speculate && n_next > 0) ? xyzt_dev_next : nullptr;   // with LIMU_OPT_SPECULATE off a hint is ignored
    o->hint_n = (o->speculate && n_next > 0) ? n_next : 0;
    return LIMU_OK;
}

int limu_odom_register_points(limu_odom *o, const double *xyz, int64_t n, double pose_out[7], double *down_xyz, int64_t *n_down,
                              double *keypoints_xyz, int64_t *n_keypoints, limu_frame_stats *stats) {
    LIMU_REQUIRE(o && n >= 0 && (n == 0 || xyz), "limu_odom_register_points: bad arguments");
    LIMU_TRY(bind(o->ctx));
    LIMU_TRY(stage_in(o->ctx, o->raw, xyz, (size_t)n * 24));
    Scan scan;
    scan.layout = SCAN_XYZ; scan.ptr = o->raw.p; scan.n = n;
    return odom_register_device(o, scan, pose_out, down_xyz, n_down, keypoints_xyz, n_keypoints, stats);
}

int limu_odom_register_msg(limu_odom *o, const void *data, int64_t n, const limu_cloud_fields *fields, const limu_lidar_config *cfg, double message_time,
                           int32_t scan_count, int32_t max_segments, double *poses_out, int64_t *seg_sizes, double *seg_time, int32_t *n_segments,
                           limu_frame_stats *stats) {
    LIMU_REQUIRE(o && n >= 0 && (n == 0 || data) && n_segments && max_segments >= 0 && (max_segments == 0 || (poses_out && seg_sizes && seg_time)) &&
                     n < (int64_t(1) << 31), "limu_odom_register_msg: bad arguments");
    LIMU_TRY(bind(o->ctx));
    LIMU_TRY(preprocess_validate(fields, cfg, max_segments));
    *n_segments = 0;
    if (n == 0) return LIMU_OK;
    limu_ctx *c = o->ctx;
    LIMU_TRY(stage_in(c, o->pre.raw, data, (size_t)n * fields->point_step));
    LIMU_TRY(preprocess_device(c, o->pre, o->pre.raw.as<unsigned char>(), n, *fields, *cfg, message_time, scan_count));   // lidar_callback, odom_run.cpp:51-67
    const SegTable &T = *o->pre.h_seg;
    const int ns = std::min<int>(T.nseg, max_segments);
    for (int k = 0; k < ns; ++k) {
        const int64_t off = T.begin[k], nk = T.end[k] - T.begin[k];
        seg_sizes[k] = nk; seg_time[k] = T.time[k];
        if (stats) memset(&stats[k], 0, sizeof(limu_frame_stats));
        if (nk <= 1) {   // "Too few input point cloud!" (odom_run.cpp:78-83): the segment is popped without being registered
            pose_store(o->poses.empty() ? pose_identity() : o->poses.back(), poses_out + 7 * k);
            continue;
        }
        // estimate_lidar_odometry -> register_frame(*processed_frame, time_buffer) (odom_run.cpp:103-106) on the device-resident segment
        const Scan seg = odom_call(o->pre.rec.as<unsigned char>() + (size_t)off * 48, 48, o->pre.ts.as<double>() + off, nk);
        LIMU_TRY(odom_register_device(o, seg, poses_out + 7 * k, nullptr, nullptr, nullptr, nullptr, stats ? &stats[k] : nullptr));
    }
    *n_segments = ns;
    return LIMU_OK;
}

int limu_odom_num_poses(limu_odom *o, int64_t *n) {
    LIMU_REQUIRE(o && n, "limu_odom_num_poses: null argument");
    *n = (int64_t)o->poses.size();
    return LIMU_OK;
}
int limu_odom_pose(limu_odom *o, int64_t i, double pose_out[7]) {
    LIMU_REQUIRE(o && pose_out && i >= 0 && i < (int64_t)o->poses.size(), "limu_odom_pose: index out of range");
    pose_store(o->poses[(size_t)i], pose_out);
    return LIMU_OK;
}
int limu_odom_adaptive_threshold(limu_odom *o, double *sigma) {
    LIMU_REQUIRE(o && sigma, "limu_odom_adaptive_threshold: null argument");
    // get_adaptive_threshold() adds a sample on every call (threshold.cpp:16-28): a loop that ran ahead did so with a threshold that does
    // not contain this one, and is dropped
    if (o->ahead.loop) { LIMU_TRY(bind(o->ctx)); LIMU_TRY(odom_drop_ahead(o, true)); }
    *sigma = odom_adaptive_threshold(o);
    return LIMU_OK;
}
int limu_odom_prediction(limu_odom *o, double pose_out[7]) {
    LIMU_REQUIRE(o && pose_out, "limu_odom_prediction: null argument");
    pose_store(odom_prediction(o), pose_out);
    return LIMU_OK;
}
int limu_odom_has_moved(limu_odom *o, int *out) {
    LIMU_REQUIRE(o && out, "limu_odom_has_moved: null argument");
    *out = odom_has_moved(o) ? 1 : 0;
    return LIMU_OK;
}
limu_map *limu_odom_map(limu_odom *o) { return o ? o->map : nullptr; }

int limu_odom_set_option(limu_odom *o, int32_t option, int64_t value) {
    LIMU_REQUIRE(o, "limu_odom_set_option: null handle");
    if (option == LIMU_OPT_SPECULATE) {
        LIMU_TRY(bind(o->ctx));
        int st = LIMU_OK;
        if (!value && o->speculate) st = odom_flush(o);   // nothing stays in flight on the plain path
        o->speculate = value != 0;
        if (!o->speculate) { o->hint_ptr = nullptr; o->hint_n = 0; }
        return st;
    }
    if (option == LIMU_OPT_CLUSTER_LOOP) return LIMU_OK;   // retired: accepted and ignored (limu_cuda.h)
    set_error("limu_odom_set_option: unknown option %d", (int)option);
    return LIMU_ERR_INVALID;
}

int limu_odom_flush(limu_odom *o) {
    LIMU_REQUIRE(o, "limu_odom_flush: null handle");
    LIMU_TRY(bind(o->ctx));
    return odom_flush(o);
}

}  // extern "C"
