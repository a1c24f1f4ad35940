// ops.cu -- per-scan stages before registration: voxel keys, rigid transform, constant-velocity deskew,
// first-point-wins voxel downsampling, IQR keypoint filter. Replaces (L/ = env_ws/src/limu):
//   utils::get_vox_index / transform_points      L/src/utils/calculation_helpers.cpp:142-147, :121-133
//   MotionCompensator::deskew_scan               L/src/sensors/lidar/helpers/deskew.cpp:10-28
//   voxel_downsample / voxelize / iqr_processing L/src/sensors/lidar/icp.cpp:9-30, :126-136, :88-124
//   outlier::IQR / median                        L/include/common.hpp:22-63
#include <algorithm>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "compact.cuh"
#include "iqr.cuh"
#include "ops.cuh"
#include "voxel_map.cuh"

namespace limu {

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
static __global__ void k_voxel_keys(const double *__restrict__ xyz, int64_t n3, double v, int *__restrict__ keys) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n3; i += (int64_t)gridDim.x * blockDim.x)
        keys[i] = vox_index(xyz[i], v);
}

// One thread per raw point: one coalesced 16-byte load {x,y,z,t}; motion = exp((t - 0.5) * twist)
// (deskew.cpp:24, mid_pose_timestamp deskew.hpp:12); out = motion * point (:25) in FP64.
static __global__ void __launch_bounds__(256) k_deskew(const float4 *__restrict__ xyzt, int64_t n, const double *__restrict__ twist, double *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 q = __ldg(xyzt + i);
    const double s = (double)q.w - 0.5;
    double st[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) st[k] = s * twist[k];
    const Pose M = se3_exp(st);
    const V3 o = apply(M, V3{(double)q.x, (double)q.y, (double)q.z});
    out[3 * i] = o.x; out[3 * i + 1] = o.y; out[3 * i + 2] = o.z;
}

// The same two stages for the reference's own input layout: an array of point records `stride` bytes apart with
// float x,y,z at offset 0 (pcl::PointXYZINormal: 48 B, types.hpp:36) and a separate double timestamp per point
// (std::vector<double>, icp.cpp:49-50). Timestamps stay FP64, so results match the reference bit for bit up to libm.
static __global__ void __launch_bounds__(256) k_deskew_rec(const unsigned char *__restrict__ rec, int stride, const double *__restrict__ ts, int64_t n,
                                                          const double *__restrict__ twist, double *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float *q = reinterpret_cast<const float *>(rec + (size_t)i * stride);
    const double s = ts[i] - 0.5;
    double st[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) st[k] = s * twist[k];
    const Pose M = se3_exp(st);
    const V3 o = apply(M, V3{(double)q[0], (double)q[1], (double)q[2]});
    out[3 * i] = o.x; out[3 * i + 1] = o.y; out[3 * i + 2] = o.z;
}
static __global__ void __launch_bounds__(256) k_widen_rec(const unsigned char *__restrict__ rec, int stride, int64_t n, double *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float *q = reinterpret_cast<const float *>(rec + (size_t)i * stride);
    out[3 * i] = (double)q[0]; out[3 * i + 1] = (double)q[1]; out[3 * i + 2] = (double)q[2];
}

static __global__ void __launch_bounds__(256) k_widen(const float4 *__restrict__ xyzt, int64_t n, double *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 q = __ldg(xyzt + i);
    out[3 * i] = (double)q.x; out[3 * i + 1] = (double)q.y; out[3 * i + 2] = (double)q.z;
}

// voxel_downsample pass 1 (icp.cpp:13-19): claim-or-find the voxel in a scan-local table and keep the
// smallest input index per voxel ("first point wins" of the serial loop).
static __global__ void __launch_bounds__(256) k_ds_claim(const double *__restrict__ xyz, int64_t n_max, const int *n_dev, double vs,
                                                        unsigned long long *keys, unsigned int *minidx, unsigned int mask, int shift,
                                                        unsigned int *__restrict__ pslot, DevStatus *st) {
    const int64_t n = n_dev ? (int64_t)*n_dev : n_max;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int kx = vox_index(xyz[3 * i], vs), ky = vox_index(xyz[3 * i + 1], vs), kz = vox_index(xyz[3 * i + 2], vs);
    unsigned int slot = PEND_NONE;
    if (!key_in_range(kx, ky, kz)) {
        st->key_range = 1;
    } else {
        const unsigned long long key = pack_key(kx, ky, kz);
        unsigned int s = slot_of(key, shift);
        for (unsigned int probes = 0; probes <= mask; ++probes) {
            unsigned long long cur = __ldcg(&keys[s]);
            if (cur == KEY_EMPTY) {
                cur = atomicCAS(&keys[s], KEY_EMPTY, key);
                if (cur == KEY_EMPTY) cur = key;
            }
            if (cur == key) { slot = s; break; }
            s = (s + 1) & mask;
        }
        if (slot != PEND_NONE) atomicMin(&minidx[slot], (unsigned int)i);
        else st->table_full = 1;
    }
    pslot[i] = slot;
}
// pass 2: a point survives iff it holds its voxel's smallest index.
static __global__ void __launch_bounds__(256) k_ds_flag(int64_t n_max, const int *n_dev, const unsigned int *__restrict__ minidx,
                                                       const unsigned int *__restrict__ pslot, unsigned char *__restrict__ flags) {
    const int64_t n = n_dev ? (int64_t)*n_dev : n_max;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned int s = pslot[i];
    flags[i] = (s != PEND_NONE && minidx[s] == (unsigned int)i) ? 1 : 0;
}

static __global__ void __launch_bounds__(1024) k_iqr(const double *__restrict__ xyz, int64_t n_max, const int *n_dev, double *__restrict__ d2,
                                                   double *__restrict__ out, int *out_count, double *bounds) {
    __shared__ IqrSmem sm;
    iqr_block<1024>(sm, xyz, (int)(n_dev ? (int64_t)*n_dev : n_max), d2, out, out_count, bounds);
}

// ------------------------------------------------------------------------------------------------
// device-pointer stage entry points
// ------------------------------------------------------------------------------------------------
int deskew_device(limu_ctx *c, const float *xyzt_dev, int64_t n, const double *twist_dev, double *out_dev) {
    if (n <= 0) return LIMU_OK;
    k_deskew<<<div_up(n, 256), 256, 0, c->stream>>>(reinterpret_cast<const float4 *>(xyzt_dev), n, twist_dev, out_dev);
    LIMU_LAUNCHED();
    return LIMU_OK;
}
int widen_device(limu_ctx *c, const float *xyzt_dev, int64_t n, double *out_dev) {
    if (n <= 0) return LIMU_OK;
    k_widen<<<div_up(n, 256), 256, 0, c->stream>>>(reinterpret_cast<const float4 *>(xyzt_dev), n, out_dev);
    LIMU_LAUNCHED();
    return LIMU_OK;
}

int deskew_records_device(limu_ctx *c, const void *rec_dev, int stride, const double *ts_dev, int64_t n, const double *twist_dev, double *out_dev) {
    if (n <= 0) return LIMU_OK;
    k_deskew_rec<<<div_up(n, 256), 256, 0, c->stream>>>(static_cast<const unsigned char *>(rec_dev), stride, ts_dev, n, twist_dev, out_dev);
    LIMU_LAUNCHED();
    return LIMU_OK;
}
int widen_records_device(limu_ctx *c, const void *rec_dev, int stride, int64_t n, double *out_dev) {
    if (n <= 0) return LIMU_OK;
    k_widen_rec<<<div_up(n, 256), 256, 0, c->stream>>>(static_cast<const unsigned char *>(rec_dev), stride, n, out_dev);
    LIMU_LAUNCHED();
    return LIMU_OK;
}

static int64_t table_slots(int64_t n) { int64_t p = 1024; while (p < 2 * n) p <<= 1; return p; }

int downsample_device(limu_ctx *c, StageScratch &sc, const double *xyz_dev, int64_t n_max, const int *n_dev, double s, double *out_xyz_dev,
                      int *out_count_dev) {
    if (n_max <= 0) { LIMU_CUDA_TRY(cudaMemsetAsync(out_count_dev, 0, sizeof(int), c->stream)); return LIMU_OK; }
    const int64_t Cs = table_slots(n_max);
    int lg = 0;
    while ((int64_t(1) << lg) < Cs) ++lg;
    LIMU_TRY(sc.table.reserve((size_t)Cs * 12, c->stream));
    LIMU_TRY(sc.pslot.reserve((size_t)n_max * 4, c->stream));
    LIMU_TRY(sc.flags.reserve((size_t)n_max, c->stream));
    LIMU_TRY(sc.blockcnt.reserve((size_t)div_up(n_max, COMPACT_BLOCK) * 4 + 16, c->stream));
    LIMU_TRY(sc.idx.reserve((size_t)n_max * 4 + 16, c->stream));
    unsigned long long *keys = sc.table.as<unsigned long long>();
    unsigned int *minidx = reinterpret_cast<unsigned int *>(keys + Cs);
    LIMU_CUDA_TRY(cudaMemsetAsync(sc.table.p, 0xFF, (size_t)Cs * 12, c->stream));   // KEY_EMPTY and "no index" are all-ones
    const int blocks = div_up(n_max, 256);
    k_ds_claim<<<blocks, 256, 0, c->stream>>>(xyz_dev, n_max, n_dev, s, keys, minidx, (unsigned int)(Cs - 1), 64 - lg, sc.pslot.as<unsigned int>(), c->d_status);
    LIMU_LAUNCHED();
    k_ds_flag<<<blocks, 256, 0, c->stream>>>(n_max, n_dev, minidx, sc.pslot.as<unsigned int>(), sc.flags.as<unsigned char>());
    LIMU_LAUNCHED();
    LIMU_TRY(compact_flags(c, sc.flags.as<unsigned char>(), n_max, n_dev, sc.blockcnt.as<int>(), sc.idx.as<int>(), out_count_dev));
    const int gb = std::min<int64_t>(div_up(n_max, 256), (int64_t)c->sm_count * 8);
    k_gather_points<<<gb, 256, 0, c->stream>>>(xyz_dev, sc.idx.as<int>(), out_count_dev, out_xyz_dev, nullptr);
    LIMU_LAUNCHED();
    return LIMU_OK;
}

int iqr_device(limu_ctx *c, StageScratch &sc, const double *xyz_dev, int64_t n_max, const int *n_dev, double *out_xyz_dev, int *out_count_dev,
               double *bounds_dev) {
    if (n_max <= 0) { LIMU_CUDA_TRY(cudaMemsetAsync(out_count_dev, 0, sizeof(int), c->stream)); return LIMU_OK; }
    LIMU_TRY(sc.d2.reserve((size_t)n_max * 8, c->stream));
    k_iqr<<<1, 1024, 0, c->stream>>>(xyz_dev, n_max, n_dev, sc.d2.as<double>(), out_xyz_dev, out_count_dev, bounds_dev);
    LIMU_LAUNCHED();
    return LIMU_OK;
}

// Stage scratch of the stateless C entry points, one pair per context (the voxelize chain uses both).
struct CtxScratch { StageScratch a, b; VoxelizeScratch vx; };
static std::mutex g_sc_mu;
static std::unordered_map<limu_ctx *, CtxScratch *> g_sc;
static StageScratch *scratch_of(limu_ctx *c, int which) {
    std::lock_guard<std::mutex> lk(g_sc_mu);
    auto it = g_sc.find(c);
    if (it == g_sc.end()) it = g_sc.emplace(c, new CtxScratch).first;
    return which == 0 ? &it->second->a : &it->second->b;
}
static VoxelizeScratch *vx_scratch_of(limu_ctx *c) {
    scratch_of(c, 0);
    std::lock_guard<std::mutex> lk(g_sc_mu);
    return &g_sc.find(c)->second->vx;
}
void release_ctx_scratch(limu_ctx *c) {
    std::lock_guard<std::mutex> lk(g_sc_mu);
    auto it = g_sc.find(c);
    if (it == g_sc.end()) return;
    it->second->a.release(); it->second->b.release(); it->second->vx.release();
    delete it->second;
    g_sc.erase(it);
}

}  // namespace limu

using namespace limu;

extern "C" {

int limu_voxel_keys(limu_ctx *c, const double *xyz, int64_t n, double v, int32_t *keys) {
    LIMU_TRY(bind(c));
    LIMU_REQUIRE(n >= 0 && (n == 0 || (xyz && keys)) && v > 0, "limu_voxel_keys: bad arguments");
    if (n == 0) return LIMU_OK;
    LIMU_TRY(stage_in(c, c->in0, xyz, (size_t)n * 24));
    LIMU_TRY(c->out0.reserve((size_t)n * 12, c->stream));
    const int blocks = std::min<int64_t>(div_up(3 * n, 256), (int64_t)c->sm_count * 16);
    k_voxel_keys<<<blocks, 256, 0, c->stream>>>(c->in0.as<double>(), 3 * n, v, c->out0.as<int>());
    LIMU_LAUNCHED();
    LIMU_CUDA_TRY(cudaMemcpyAsync(keys, c->out0.p, (size_t)n * 12, cudaMemcpyDeviceToHost, c->stream));
    return check_status(c);
}

int limu_transform_points(limu_ctx *c, const double pose[7], double *xyz, int64_t n) {
    LIMU_TRY(bind(c));
    LIMU_REQUIRE(pose && n >= 0 && (n == 0 || xyz), "limu_transform_points: bad arguments");
    if (n == 0) { printf("[INFO] utils::transform_points the points vector is empty\n"); return LIMU_OK; }   // calculation_helpers.cpp:123-127
    double *dpose;
    LIMU_TRY(stage_small(c, pose, 7, 0, &dpose));
    LIMU_TRY(stage_in(c, c->in0, xyz, (size_t)n * 24));
    LIMU_TRY(transform_device(c, dpose, c->in0.as<double>(), c->in0.as<double>(), n, nullptr));
    LIMU_CUDA_TRY(cudaMemcpyAsync(xyz, c->in0.p, (size_t)n * 24, cudaMemcpyDeviceToHost, c->stream));
    return check_status(c);
}

int limu_deskew(limu_ctx *c, const float *xyzt, int64_t n, const double T0[7], const double T1[7], double *out_xyz) {
    LIMU_TRY(bind(c));
    LIMU_REQUIRE(T0 && T1 && n >= 0 && (n == 0 || (xyzt && out_xyz)), "limu_deskew: bad arguments");
    if (n == 0) return LIMU_OK;
    double twist[6];
    se3_log(mul(inverse(pose_load(T0)), pose_load(T1)), twist);   // utils::delta_pose, calculation_helpers.cpp:99-102
    double *dtw;
    LIMU_TRY(stage_small(c, twist, 6, 0, &dtw));
    LIMU_TRY(stage_in(c, c->in1, xyzt, (size_t)n * 16));
    LIMU_TRY(c->out0.reserve((size_t)n * 24, c->stream));
    LIMU_TRY(deskew_device(c, c->in1.as<float>(), n, dtw, c->out0.as<double>()));
    LIMU_CUDA_TRY(cudaMemcpyAsync(out_xyz, c->out0.p, (size_t)n * 24, cudaMemcpyDeviceToHost, c->stream));
    return check_status(c);
}

}  // extern "C"

extern "C" {

int limu_deskew_cloud(limu_ctx *c, const void *points, int32_t stride_bytes, const double *timestamps, int64_t n, const double T0[7],
                      const double T1[7], double *out_xyz) {
    LIMU_TRY(bind(c));
    LIMU_REQUIRE(T0 && T1 && n >= 0 && stride_bytes >= 12 && stride_bytes % 4 == 0 && (n == 0 || (points && timestamps && out_xyz)), "limu_deskew_cloud: bad arguments");
    if (n == 0) return LIMU_OK;
    double twist[6];
    se3_log(mul(inverse(pose_load(T0)), pose_load(T1)), twist);   // utils::delta_pose, calculation_helpers.cpp:99-102
    double *dtw;
    LIMU_TRY(stage_small(c, twist, 6, 0, &dtw));
    LIMU_TRY(stage_in(c, c->in1, points, (size_t)n * stride_bytes));
    LIMU_TRY(stage_in(c, c->in0, timestamps, (size_t)n * 8));
    LIMU_TRY(c->out0.reserve((size_t)n * 24, c->stream));
    LIMU_TRY(deskew_records_device(c, c->in1.p, stride_bytes, c->in0.as<double>(), n, dtw, c->out0.as<double>()));
    LIMU_CUDA_TRY(cudaMemcpyAsync(out_xyz, c->out0.p, (size_t)n * 24, cudaMemcpyDeviceToHost, c->stream));
    return check_status(c);
}

int limu_voxel_downsample(limu_ctx *c, const double *xyz, int64_t n, double s, double *out_xyz, int64_t *out_idx, int64_t *n_out) {
    LIMU_TRY(bind(c));
    LIMU_REQUIRE(n >= 0 && n_out && s > 0 && (n == 0 || xyz), "limu_voxel_downsample: bad arguments");
    *n_out = 0;
    if (n == 0) return LIMU_OK;
    StageScratch &sc = *scratch_of(c, 0);
    LIMU_TRY(stage_in(c, c->in0, xyz, (size_t)n * 24));
    LIMU_TRY(c->out0.reserve((size_t)n * 24, c->stream));
    int *count_dev = reinterpret_cast<int *>(c->d_small.as<double>());
    LIMU_TRY(downsample_device(c, sc, c->in0.as<double>(), n, nullptr, s, c->out0.as<double>(), count_dev));
    int *h = static_cast<int *>(c->h_pinned);
    LIMU_CUDA_TRY(cudaMemcpyAsync(h, count_dev, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
    const int64_t k = h[0];
    *n_out = k;
    if (k > 0 && out_xyz) LIMU_CUDA_TRY(cudaMemcpyAsync(out_xyz, c->out0.p, (size_t)k * 24, cudaMemcpyDeviceToHost, c->stream));
    if (k > 0 && out_idx) {
        std::vector<int> tmp((size_t)k);
        LIMU_CUDA_TRY(cudaMemcpyAsync(tmp.data(), sc.idx.p, (size_t)k * 4, cudaMemcpyDeviceToHost, c->stream));
        LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
        for (int64_t j = 0; j < k; ++j) out_idx[j] = tmp[(size_t)j];
    }
    return check_status(c);
}

int limu_iqr_filter(limu_ctx *c, const double *xyz, int64_t n, double *out_xyz, int64_t *n_out, double bounds[2]) {
    LIMU_TRY(bind(c));
    LIMU_REQUIRE(n >= 0 && n_out && (n == 0 || xyz), "limu_iqr_filter: bad arguments");
    *n_out = 0;
    if (n == 0) return LIMU_OK;
    StageScratch &sc = *scratch_of(c, 0);
    LIMU_TRY(stage_in(c, c->in0, xyz, (size_t)n * 24));
    LIMU_TRY(c->out0.reserve((size_t)n * 24, c->stream));
    int *count_dev = reinterpret_cast<int *>(c->d_small.as<double>());
    double *bounds_dev = c->d_small.as<double>() + 8;
    LIMU_TRY(iqr_device(c, sc, c->in0.as<double>(), n, nullptr, c->out0.as<double>(), count_dev, bounds_dev));
    double *h = static_cast<double *>(c->h_pinned);
    LIMU_CUDA_TRY(cudaMemcpyAsync(h, c->d_small.p, 10 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
    const int64_t k = *reinterpret_cast<int *>(h);
    *n_out = k;
    if (bounds) { bounds[0] = h[8]; bounds[1] = h[9]; }
    if (k > 0 && out_xyz) LIMU_CUDA_TRY(cudaMemcpyAsync(out_xyz, c->out0.p, (size_t)k * 24, cudaMemcpyDeviceToHost, c->stream));
    return check_status(c);
}

int limu_voxelize(limu_ctx *c, const double *xyz, int64_t n, double v, double *src_xyz, int64_t *n_src, double *down_xyz, int64_t *n_down) {
    LIMU_TRY(bind(c));
    LIMU_REQUIRE(n >= 0 && n_src && n_down && v > 0 && (n == 0 || xyz), "limu_voxelize: bad arguments");
    *n_src = *n_down = 0;
    if (n == 0) return LIMU_OK;
    StageScratch &sb = *scratch_of(c, 1);
    LIMU_TRY(stage_in(c, c->in0, xyz, (size_t)n * 24));
    LIMU_TRY(c->in1.reserve((size_t)n * 24, c->stream));    // frame copy written by the fused kernel
    LIMU_TRY(c->out0.reserve((size_t)n * 24, c->stream));   // down
    LIMU_TRY(c->out1.reserve((size_t)n * 24, c->stream));   // ds(down, 1.5v)
    LIMU_TRY(c->out2.reserve((size_t)n * 24, c->stream));   // after IQR
    int *cnt = reinterpret_cast<int *>(c->d_small.as<double>());   // [0]=n_down [1]=n_src0 [2]=n_src
    Scan scan;
    scan.layout = SCAN_XYZ; scan.ptr = c->in0.p; scan.n = n;
    LIMU_TRY(voxelize_device(c, *vx_scratch_of(c), scan, 0, nullptr, v, c->in1.as<double>(), c->out0.as<double>(), c->out1.as<double>(), cnt + 0));   // icp.cpp:129-130
    LIMU_TRY(iqr_device(c, sb, c->out1.as<double>(), n, cnt + 1, c->out2.as<double>(), cnt + 2, nullptr));             // :133
    int *h = static_cast<int *>(c->h_pinned);
    LIMU_CUDA_TRY(cudaMemcpyAsync(h, cnt, 3 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
    *n_down = h[0];
    *n_src = h[2];
    if (h[0] > 0 && down_xyz) LIMU_CUDA_TRY(cudaMemcpyAsync(down_xyz, c->out0.p, (size_t)h[0] * 24, cudaMemcpyDeviceToHost, c->stream));
    if (h[2] > 0 && src_xyz) LIMU_CUDA_TRY(cudaMemcpyAsync(src_xyz, c->out2.p, (size_t)h[2] * 24, cudaMemcpyDeviceToHost, c->stream));
    return check_status(c);
}

}  // extern "C"
