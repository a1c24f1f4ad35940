// imu_deskew.cu -- IMU-propagated backward deskew: the per-point loop of kalman::EKF::motion_compensation_with_imu
// (L/src/kalman/ekf.cpp:420-468; SURVEY section 8f N1). The host IMU forward pass (:315-410) stays where it is (it walks
// ~20 IMU samples through the EKF state) and hands over its pose table (kalman::Pose6D rows, ekf.hpp:88-105), the
// scan-end rotation / lidar position (:393-418) and the IMU->lidar lever arm; every point is then independent. The math
// (head rule, compensation, the first point's re-visits) is in imu_compensate.cuh, shared with the fused voxelize kernel.
#include <algorithm>

#include "imu_compensate.cuh"

namespace limu {

struct ImuDeskewArgs {
    unsigned char *rec;      // point records, `stride` bytes apart: float x,y,z at offset 0, float curvature (ms) at `toff`
    int stride, toff;
    int64_t n;
    const double *table;     // M x 22
    int M;
    double rot_end[9], pos_lidar_end[3], p_il[3];
    double *out;             // n x 3 (optional)
};

static __global__ void __launch_bounds__(256) k_deskew_imu(const ImuDeskewArgs A) {
    __shared__ double tab[IMU_MAX_ROWS * 22];
    for (int k = threadIdx.x; k < A.M * 22; k += blockDim.x) tab[k] = A.table[k];
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.n) return;
    float *q = reinterpret_cast<float *>(A.rec + (size_t)i * A.stride);
    float xyz[3] = {q[0], q[1], q[2]};
    const double t = imu_point_time(A.rec + (size_t)i * A.stride, A.toff);
    if (imu_deskew_point(tab, A.M, i, t, A.rot_end, A.pos_lidar_end, A.p_il, xyz)) { q[0] = xyz[0]; q[1] = xyz[1]; q[2] = xyz[2]; }
    if (A.out) { A.out[3 * i] = (double)xyz[0]; A.out[3 * i + 1] = (double)xyz[1]; A.out[3 * i + 2] = (double)xyz[2]; }
}

}  // namespace limu

using namespace limu;

extern "C" int limu_deskew_imu(limu_ctx *c, void *points, int32_t stride_bytes, int32_t curvature_offset_bytes, int64_t n, const limu_imu_pose *table,
                               int32_t n_poses, const double rot_end[9], const double pos_lidar_end[3], const double p_imu_lidar[3], double *out_xyz,
                               int32_t write_back) {
    LIMU_TRY(bind(c));
    LIMU_REQUIRE(points && table && rot_end && pos_lidar_end && p_imu_lidar && n >= 1 && n_poses >= 2 && n_poses <= IMU_MAX_ROWS && stride_bytes >= 16 &&
                     stride_bytes % 4 == 0 && curvature_offset_bytes >= 12 && curvature_offset_bytes + 4 <= stride_bytes && curvature_offset_bytes % 4 == 0,
                 "limu_deskew_imu: bad arguments (need n >= 1, 2 <= n_poses <= 96, float x,y,z at offset 0 and a float time field inside each record)");
    static_assert(sizeof(limu_imu_pose) == 22 * sizeof(double), "limu_imu_pose layout");
    LIMU_TRY(stage_in(c, c->in1, points, (size_t)n * stride_bytes));
    LIMU_TRY(stage_in(c, c->tmp0, table, (size_t)n_poses * sizeof(limu_imu_pose)));
    if (out_xyz) LIMU_TRY(c->out0.reserve((size_t)n * 24, c->stream));
    ImuDeskewArgs A;
    A.rec = c->in1.as<unsigned char>(); A.stride = stride_bytes; A.toff = curvature_offset_bytes; A.n = n;
    A.table = c->tmp0.as<double>(); A.M = n_poses;
    for (int k = 0; k < 9; ++k) A.rot_end[k] = rot_end[k];
    for (int k = 0; k < 3; ++k) { A.pos_lidar_end[k] = pos_lidar_end[k]; A.p_il[k] = p_imu_lidar[k]; }
    A.out = out_xyz ? c->out0.as<double>() : nullptr;
    k_deskew_imu<<<div_up(n, 256), 256, 0, c->stream>>>(A);
    LIMU_LAUNCHED();
    if (out_xyz) LIMU_CUDA_TRY(cudaMemcpyAsync(out_xyz, c->out0.p, (size_t)n * 24, cudaMemcpyDeviceToHost, c->stream));
    if (write_back)   // only the 12 bytes of x,y,z of every record travel back
        LIMU_CUDA_TRY(cudaMemcpy2DAsync(points, (size_t)stride_bytes, c->in1.p, (size_t)stride_bytes, 12, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    return check_status(c);
}
