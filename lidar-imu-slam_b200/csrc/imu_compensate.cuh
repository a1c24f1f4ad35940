// imu_compensate.cuh -- the per-point math of kalman::EKF::motion_compensation_with_imu (L/src/kalman/ekf.cpp:420-468; SURVEY section 8f
// N1), shared by the stand-alone deskew (k_deskew_imu, imu_deskew.cu) and the IMU variant of the fused voxelize kernel (voxelize.cu), so
// that both write the same floats:
//   head   = the latest table row (excluding the last) whose offset_time is below the point's time (:422-433)
//   R_i    = R_head * AngleAxis(dt |w|, w/|w|)                                   (:444, helper.hpp:35-40)
//   T_ei   = p + v dt + 0.5 a dt^2 + R_i p_IL - p_lidar_end                      (:445)
//   P_comp = R_end^T (R_i P_i + T_ei), stored back as FLOAT and widened          (:448-468)
// The reference's serial loop never consumes the first point of the scan (:455-456), so that point is compensated again by every older
// head below its time.
#pragma once
#include "common.cuh"

namespace limu {

constexpr int IMU_MAX_ROWS = 96;   // table rows (kalman::Pose6D, 22 doubles each) a call accepts

// The IMU deskew arguments of one limu_odom_register_cloud_imu / limu_odom_prefetch_cloud_imu call, copied from the caller (host): a prepared
// scan is only used by a call whose arguments are byte for byte the same.
struct ImuCall {
    int32_t M, toff;
    double rot_end[9], pos_lidar_end[3], p_il[3];
    double table[IMU_MAX_ROWS * 22];
};

// Eigen::AngleAxisd(dt*|w|, w.normalized()).toRotationMatrix() (Eigen/src/Geometry/AngleAxis.h)
__device__ __forceinline__ void ang_vel_to_rmat(const double *w, double dt, double *R) {
    const double z = sqnorm3(w[0], w[1], w[2]);
    const double nrm = sqrt(z);
    double ax = w[0], ay = w[1], az = w[2];
    if (z > 0.0) { ax = w[0] / nrm; ay = w[1] / nrm; az = w[2] / nrm; }
    const double angle = dt * nrm;
    const double s = sin(angle), c = cos(angle);
    const double sx = s * ax, sy = s * ay, sz = s * az;
    const double cx = (1.0 - c) * ax, cy = (1.0 - c) * ay, cz = (1.0 - c) * az;
    double tmp;
    tmp = cx * ay; R[1] = tmp - sz; R[3] = tmp + sz;
    tmp = cx * az; R[2] = tmp + sy; R[6] = tmp - sy;
    tmp = cy * az; R[5] = tmp - sx; R[7] = tmp + sx;
    R[0] = cx * ax + c; R[4] = cy * ay + c; R[8] = cz * az + c;
}

// One compensation of xyz (in place, float) under table row T, for a point of time t (seconds after the scan start).
__device__ __forceinline__ void compensate(const double *T, double t, const double *rot_end, const double *pos_lidar_end, const double *p_il, float *xyz) {
    const double dt = t - T[0];
    double Rw[9], Ri[9], t1[3], t2[3];
    ang_vel_to_rmat(T + 4, dt, Rw);
    mat3mul(T + 13, Rw, Ri);
    mat3vec(Ri, p_il, t1);
    const double P[3] = {(double)xyz[0], (double)xyz[1], (double)xyz[2]};
    mat3vec(Ri, P, t2);
    double v[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double Tei = (((T[10 + a] + T[7 + a] * dt) + (0.5 * T[1 + a]) * (dt * dt)) + t1[a]) - pos_lidar_end[a];
        v[a] = t2[a] + Tei;
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) xyz[a] = (float)((rot_end[a] * v[0] + rot_end[3 + a] * v[1]) + rot_end[6 + a] * v[2]);
}

// The point's time from its record: the float `curvature` (ms) at byte offset toff, / double(1000) (ekf.cpp:426).
__device__ __forceinline__ double imu_point_time(const unsigned char *record, int toff) {
    return (double)*reinterpret_cast<const float *>(record + toff) / 1000.0;
}

// Point i of the scan through the serial loop: compensated under its head row and, for i == 0, again under every older row below its time.
// tab: M rows of 22 doubles. Returns false (xyz untouched) when no row below the last lies before t.
__device__ __forceinline__ bool imu_deskew_point(const double *tab, int M, int64_t i, double t, const double *rot_end, const double *pos_lidar_end,
                                                 const double *p_il, float *xyz) {
    int h = M - 2;
    while (h >= 0 && !(t > tab[22 * h])) --h;
    if (h < 0) return false;
    compensate(tab + 22 * h, t, rot_end, pos_lidar_end, p_il, xyz);
    if (i == 0)   // the serial loop re-visits the first point under every older head (:455-456)
        for (int g = h - 1; g >= 0; --g) if (t > tab[22 * g]) compensate(tab + 22 * g, t, rot_end, pos_lidar_end, p_il, xyz);
    return true;
}

}  // namespace limu
