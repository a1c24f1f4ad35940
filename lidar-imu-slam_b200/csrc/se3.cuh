// se3.cuh -- SE(3) / small dense algebra shared by host glue and device kernels.
//
// Restates the parts of Sophus 1.22.10 and Eigen 3.4.0 the reference path calls, with the SAME
// floating-point operation order wherever a result feeds a voxel key, a distance comparison or a
// transformed point (those must be bit-identical to the x86-64 reference build, which has no FMA
// contraction: L/CMakeLists.txt:5 -> this library is compiled with -fmad=false and
// -Xcompiler -ffp-contract=off). Citations are to sophus/{so3,se3}.hpp and Eigen/src/...
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define LIMU_HD __host__ __device__ __forceinline__
#else
#define LIMU_HD inline
#endif

namespace limu {

struct V3 { double x, y, z; };
// Pose = Sophus::SE3d parameters: unit quaternion (x,y,z,w) + translation.
struct Pose { double qx, qy, qz, qw, tx, ty, tz; };

LIMU_HD Pose pose_identity() { return Pose{0, 0, 0, 1, 0, 0, 0}; }
LIMU_HD Pose pose_load(const double *p) { return Pose{p[0], p[1], p[2], p[3], p[4], p[5], p[6]}; }
LIMU_HD void pose_store(const Pose &T, double *p) { p[0] = T.qx; p[1] = T.qy; p[2] = T.qz; p[3] = T.qw; p[4] = T.tx; p[5] = T.ty; p[6] = T.tz; }

// Eigen squaredNorm of a fixed 3-vector under SSE2: (a^2 + b^2) + c^2.
LIMU_HD double sqnorm3(double a, double b, double c) { return (a * a + b * b) + c * c; }

LIMU_HD V3 cross(const V3 &a, const V3 &b) {  // Eigen/src/Geometry/OrthoMethods.h cross3
    return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}

// SO3::operator*(point), so3.hpp:388-399: uv = qv x p; uv += uv; p + w*uv + qv x uv.
LIMU_HD V3 rotate(const Pose &T, const V3 &p) {
    const V3 qv{T.qx, T.qy, T.qz};
    V3 uv = cross(qv, p);
    uv.x += uv.x; uv.y += uv.y; uv.z += uv.z;
    const V3 c = cross(qv, uv);
    return V3{(p.x + T.qw * uv.x) + c.x, (p.y + T.qw * uv.y) + c.y, (p.z + T.qw * uv.z) + c.z};
}
// SE3::operator*(point), se3.hpp:319-322.
LIMU_HD V3 apply(const Pose &T, const V3 &p) {
    const V3 r = rotate(T, p);
    return V3{r.x + T.tx, r.y + T.ty, r.z + T.tz};
}

// SO3(quaternion) constructor -> normalize(), so3.hpp:318-325; 4-vector squaredNorm under SSE2
// reduces two packets: (x^2 + z^2) + (y^2 + w^2).
LIMU_HD void quat_normalize(double &x, double &y, double &z, double &w) {
    const double len = sqrt((x * x + z * z) + (y * y + w * w));
    x /= len; y /= len; z /= len; w /= len;
}

// SE3 product, se3.hpp:302-307 with SO3 product so3.hpp:344-369 (renormalises).
LIMU_HD Pose mul(const Pose &a, const Pose &b) {
    Pose o;
    o.qw = a.qw * b.qw - a.qx * b.qx - a.qy * b.qy - a.qz * b.qz;
    o.qx = a.qw * b.qx + a.qx * b.qw + a.qy * b.qz - a.qz * b.qy;
    o.qy = a.qw * b.qy + a.qy * b.qw + a.qz * b.qx - a.qx * b.qz;
    o.qz = a.qw * b.qz + a.qz * b.qw + a.qx * b.qy - a.qy * b.qx;
    quat_normalize(o.qx, o.qy, o.qz, o.qw);
    const V3 r = rotate(a, V3{b.tx, b.ty, b.tz});
    o.tx = a.tx + r.x; o.ty = a.ty + r.y; o.tz = a.tz + r.z;
    return o;
}
// SE3::inverse, se3.hpp:222-225; SO3::inverse so3.hpp:246-248 (conjugate, renormalised).
LIMU_HD Pose inverse(const Pose &a) {
    Pose o;
    o.qx = -a.qx; o.qy = -a.qy; o.qz = -a.qz; o.qw = a.qw;
    quat_normalize(o.qx, o.qy, o.qz, o.qw);
    o.tx = o.ty = o.tz = 0.0;
    const V3 r = rotate(o, V3{a.tx * -1.0, a.ty * -1.0, a.tz * -1.0});
    o.tx = r.x; o.ty = r.y; o.tz = r.z;
    return o;
}

#define LIMU_SOPHUS_EPS 1e-10  // sophus/common.hpp:157

// Row-major 3x3 helpers. Eigen's fixed 3x3 lazy products (column-major, SSE2): rows 0-1 accumulate
// ((k0 + k1) + k2) through the packet path, row 2 through the scalar unroller k0 + (k1 + k2).
LIMU_HD void hat(const double *w, double *O) {  // so3.hpp:783-792
    O[0] = 0; O[1] = -w[2]; O[2] = w[1];
    O[3] = w[2]; O[4] = 0; O[5] = -w[0];
    O[6] = -w[1]; O[7] = w[0]; O[8] = 0;
}
LIMU_HD void mat3mul(const double *A, const double *B, double *C) {
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        C[j] = (A[0] * B[j] + A[1] * B[3 + j]) + A[2] * B[6 + j];
        C[3 + j] = (A[3] * B[j] + A[4] * B[3 + j]) + A[5] * B[6 + j];
        C[6 + j] = A[6] * B[j] + (A[7] * B[3 + j] + A[8] * B[6 + j]);
    }
}
LIMU_HD void mat3vec(const double *A, const double *v, double *o) {
    o[0] = (A[0] * v[0] + A[1] * v[1]) + A[2] * v[2];
    o[1] = (A[3] * v[0] + A[4] * v[1]) + A[5] * v[2];
    o[2] = A[6] * v[0] + (A[7] * v[1] + A[8] * v[2]);
}

// Correctly rounded 1 / v (on the device without the FP64 division subroutine).
LIMU_HD double rcp(double v) {
#ifdef __CUDA_ARCH__
    return __drcp_rn(v);
#else
    return 1.0 / v;
#endif
}

// SE3::exp, se3.hpp:852-861; SO3::expAndTheta so3.hpp:694-732; SO3::leftJacobian so3.hpp:550-571.
// se3_exp() is the composition of the two halves below and is bit-identical to Sophus on x86-64.
LIMU_HD void se3_exp_rotation(const double *a, double *q /* x y z w */, double *theta_out) {
    const double *om = a + 3;
    const double theta_sq = sqnorm3(om[0], om[1], om[2]);
    double theta, imag, real;
    if (theta_sq < LIMU_SOPHUS_EPS * LIMU_SOPHUS_EPS) {
        theta = 0.0;
        const double theta_po4 = theta_sq * theta_sq;
        imag = 0.5 - (1.0 / 48.0) * theta_sq + (1.0 / 3840.0) * theta_po4;
        real = 1.0 - (1.0 / 8.0) * theta_sq + (1.0 / 384.0) * theta_po4;
    } else {
        theta = sqrt(theta_sq);
        const double half = 0.5 * theta;
#ifdef __CUDA_ARCH__
        double sh, ch;   // one argument reduction for both
        sincos(half, &sh, &ch);
        imag = sh / theta;
        real = ch;
#else
        imag = sin(half) / theta;
        real = cos(half);
#endif
    }
    q[3] = real; q[0] = imag * om[0]; q[1] = imag * om[1]; q[2] = imag * om[2];
    *theta_out = theta;
}
LIMU_HD void se3_exp_translation(const double *a, double *t) {
    const double *ups = a, *om = a + 3;
    const double theta_sq = sqnorm3(om[0], om[1], om[2]);
    const double theta = theta_sq < LIMU_SOPHUS_EPS * LIMU_SOPHUS_EPS ? 0.0 : sqrt(theta_sq);
    const double tsq = theta * theta;  // leftJacobian(omega, theta) recomputes theta^2 (so3.hpp:556)
    double Om[9], Om2[9], V[9];
    hat(om, Om);
    mat3mul(Om, Om, Om2);
    if (tsq < LIMU_SOPHUS_EPS * LIMU_SOPHUS_EPS) {
#pragma unroll
        for (int i = 0; i < 9; ++i) V[i] = ((i % 4 == 0) ? 1.0 : 0.0) + 0.5 * Om[i];
    } else {
#ifdef __CUDA_ARCH__
        double st, ct;
        sincos(theta, &st, &ct);
#else
        const double st = sin(theta), ct = cos(theta);
#endif
        const double c1 = (1.0 - ct) / tsq, c2 = (theta - st) / (tsq * theta);
#pragma unroll
        for (int i = 0; i < 9; ++i) V[i] = (((i % 4 == 0) ? 1.0 : 0.0) + c1 * Om[i]) + c2 * Om2[i];
    }
    mat3vec(V, ups, t);
}
LIMU_HD Pose se3_exp(const double *a) {
    double q[4], t[3], theta;
    se3_exp_rotation(a, q, &theta);
    se3_exp_translation(a, t);
    return Pose{q[0], q[1], q[2], q[3], t[0], t[1], t[2]};
}

// SE3::exp for the Gauss-Newton loop, where it runs on one thread while the grid waits: the same formulas as se3_exp() from one sqrt
// and one sincos(theta/2) -- sin(theta) = 2 sh ch, 1 - cos(theta) = 2 sh^2 -- and one reciprocal of theta, and V v as
// v + c1 (w x v) + c2 (w x (w x v)). Not bit-identical to Sophus: the quaternion differs by rounding, and the translation is the more
// accurate one where Sophus's 1 - cos(theta) cancels (theta between ~1e-10 and ~1e-5). Nothing keyed or compared bit for bit uses it.
LIMU_HD Pose se3_exp_gn(const double *a) {
    const V3 ups{a[0], a[1], a[2]}, om{a[3], a[4], a[5]};
    const double theta_sq = sqnorm3(om.x, om.y, om.z);
    const V3 wu = cross(om, ups), wwu = cross(om, wu);
    double imag, real, c1, c2;
    if (theta_sq < LIMU_SOPHUS_EPS * LIMU_SOPHUS_EPS) {   // Sophus's small-angle branches: V = I + Omega / 2
        const double theta_po4 = theta_sq * theta_sq;
        imag = 0.5 - (1.0 / 48.0) * theta_sq + (1.0 / 3840.0) * theta_po4;
        real = 1.0 - (1.0 / 8.0) * theta_sq + (1.0 / 384.0) * theta_po4;
        c1 = 0.5;
        c2 = 0.0;
    } else {
        const double theta = sqrt(theta_sq), it = rcp(theta), half = 0.5 * theta;
        double sh, ch;
#ifdef __CUDA_ARCH__
        sincos(half, &sh, &ch);
#else
        sh = sin(half); ch = cos(half);
#endif
        imag = sh * it;
        real = ch;
        c1 = 2.0 * (imag * imag);                          // (1 - cos theta) / theta^2
        c2 = (theta - 2.0 * (sh * ch)) * (it * (it * it)); // (theta - sin theta) / theta^3
    }
    return Pose{imag * om.x, imag * om.y, imag * om.z, real,
                (ups.x + c1 * wu.x) + c2 * wwu.x, (ups.y + c1 * wu.y) + c2 * wwu.y, (ups.z + c1 * wu.z) + c2 * wwu.z};
}

// SE3::log, se3.hpp:237-253; SO3::logAndTheta so3.hpp:264-310; leftJacobianInverse so3.hpp:573-597.
LIMU_HD void se3_log(const Pose &T, double *x) {
    const double sqn = sqnorm3(T.qx, T.qy, T.qz), w = T.qw;
    double two_atan, theta;
    if (sqn < LIMU_SOPHUS_EPS * LIMU_SOPHUS_EPS) {
        const double sw = w * w;
        two_atan = 2.0 / w - (2.0 / 3.0) * sqn / (w * sw);
        theta = 2.0 * sqn / w;
    } else {
        const double n = sqrt(sqn);
        const double at = (w < 0.0) ? atan2(-n, -w) : atan2(n, w);
        two_atan = 2.0 * at / n;
        theta = two_atan * n;
    }
    const double om[3] = {two_atan * T.qx, two_atan * T.qy, two_atan * T.qz};
    const double tsq = theta * theta;
    double Om[9], Om2[9], Vi[9];
    hat(om, Om);
    mat3mul(Om, Om, Om2);
    if (tsq < LIMU_SOPHUS_EPS * LIMU_SOPHUS_EPS) {
#pragma unroll
        for (int i = 0; i < 9; ++i) Vi[i] = (((i % 4 == 0) ? 1.0 : 0.0) - 0.5 * Om[i]) + (1. / 12.) * Om2[i];
    } else {
        const double half = 0.5 * theta;
        const double c = (1.0 - 0.5 * theta * cos(half) / sin(half)) / (theta * theta);
#pragma unroll
        for (int i = 0; i < 9; ++i) Vi[i] = (((i % 4 == 0) ? 1.0 : 0.0) - 0.5 * Om[i]) + c * Om2[i];
    }
    const double t[3] = {T.tx, T.ty, T.tz};
    mat3vec(Vi, t, x);
    x[3] = om[0]; x[4] = om[1]; x[5] = om[2];
}

// |v| of a 6-vector as Eigen reduces it (three SSE2 packets, then the horizontal add).
LIMU_HD double norm6(const double *x) {
    const double a = (x[0] * x[0] + x[2] * x[2]) + x[4] * x[4];
    const double b = (x[1] * x[1] + x[3] * x[3]) + x[5] * x[5];
    return sqrt(a + b);
}

// Convergence of a Gauss-Newton iteration, |log(exp(x))| < eps (icp.cpp:124), from the twist itself: log(exp(x)) is x up to rounding
// while the rotation is below pi, so the verdict is 1 (converged) when |x| < eps (1 - 1e-6) and 0 when |x| > eps (1 + 1e-6). Inside
// that band, or for |w| >= 3 (or NaN), it is 2: too close to call, and the caller takes the logarithm as the reference does.
// Compares squares (the band is far wider than their rounding): no sqrt.
LIMU_HD int gn_verdict(const double *x, double eps) {
    const double n2 = ((x[0] * x[0] + x[2] * x[2]) + x[4] * x[4]) + ((x[1] * x[1] + x[3] * x[3]) + x[5] * x[5]);   // norm6(x)^2
    const double lo = eps * (1.0 - 1e-6), hi = eps * (1.0 + 1e-6);
    if (!(sqnorm3(x[3], x[4], x[5]) < 9.0)) return 2;
    return n2 < lo * lo ? 1 : (n2 > hi * hi ? 0 : 2);
}

// Eigen 3.4.0 LDLT<Matrix6d>: diagonal-pivoted in-place factorisation of the lower triangle
// (Cholesky/LDLT.h:300-395) and the solve with pseudo-inverse of D (:569-607). A is row-major 6x6.
// Every loop has compile-time bounds and the runtime pivot index only selects among statically indexed
// swaps, so on the device the whole factorisation lives in registers (the Gauss-Newton solve runs on ONE
// thread while the grid waits: its latency is on the critical path of every iteration).
LIMU_HD void swapd(double &a, double &b) { const double t = a; a = b; b = t; }
// Conditional swap written as two selects on statically indexed operands (keeps the matrix in registers:
// an `if (pivot == i) swap(...)` chain gets re-rolled by the compiler into a dynamically indexed local array).
LIMU_HD void cswapd(bool sw, double &a, double &b) { const double ta = a, tb = b; a = sw ? tb : ta; b = sw ? ta : tb; }
LIMU_HD void ldlt6_solve(const double *Ain, const double *b, double *x) {
    double a[6][6];
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = 0; j < 6; ++j) a[i][j] = Ain[6 * i + j];
    int tr[6];
    double inv[6];       // 1 / D_k: FP64 division is a ~200-cycle subroutine on the device and this solve sits on the critical
                         // path of every Gauss-Newton iteration, so each pivot is inverted once (one division per column instead of
                         // up to six; entries of L and the solution then differ from Eigen's by <= 1 ulp per operation)
    bool zero = false;   // "entire diagonal is zero" exit of LDLT.h:364-375
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        int big = k;
        double bigv = fabs(a[k][k]);
#pragma unroll
        for (int i = k + 1; i < 6; ++i) { const double v = fabs(a[i][i]); if (v > bigv) { bigv = v; big = i; } }
        if (zero) big = k;
        tr[k] = big;
#pragma unroll
        for (int i = k + 1; i < 6; ++i) {
            const bool sw = (big == i);
#pragma unroll
            for (int c = 0; c < k; ++c) cswapd(sw, a[k][c], a[i][c]);
#pragma unroll
            for (int r = i + 1; r < 6; ++r) cswapd(sw, a[r][k], a[r][i]);
            cswapd(sw, a[k][k], a[i][i]);
#pragma unroll
            for (int m = k + 1; m < i; ++m) cswapd(sw, a[m][k], a[i][m]);
        }
        if (!zero) {
            if (k > 0) {
                double temp[6];
#pragma unroll
                for (int c = 0; c < k; ++c) temp[c] = a[c][c] * a[k][c];
                double acc = 0.0;
#pragma unroll
                for (int c = 0; c < k; ++c) acc += a[k][c] * temp[c];
                a[k][k] -= acc;
#pragma unroll
                for (int r = k + 1; r < 6; ++r) {
                    double a2 = 0.0;
#pragma unroll
                    for (int c = 0; c < k; ++c) a2 += a[r][c] * temp[c];
                    a[r][k] -= a2;
                }
            }
            const double akk = a[k][k];
            const bool valid = fabs(akk) > 0.0;
            if (k == 0 && !valid) zero = true;
#ifdef __CUDA_ARCH__
            inv[k] = fabs(akk) > 2.2250738585072014e-308 ? __drcp_rn(akk) : 0.0;   // correctly rounded reciprocal == 1.0 / akk, without the division subroutine
#else
            inv[k] = fabs(akk) > 2.2250738585072014e-308 ? 1.0 / akk : 0.0;   // pseudo-inverse of D (LDLT.h:590-596)
#endif
            if (valid) {
#pragma unroll
                for (int r = k + 1; r < 6; ++r) a[r][k] *= inv[k];
            }
        } else {
            inv[k] = 0.0;
        }
    }
    double d[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) d[i] = b[i];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
#pragma unroll
        for (int i = k + 1; i < 6; ++i) cswapd(tr[k] == i, d[k], d[i]);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int c = 0; c < i; ++c) d[i] -= a[i][c] * d[c];
#pragma unroll
    for (int i = 0; i < 6; ++i) d[i] *= inv[i];
#pragma unroll
    for (int i = 5; i >= 0; --i)
#pragma unroll
        for (int c = i + 1; c < 6; ++c) d[i] -= a[c][i] * d[c];
#pragma unroll
    for (int k = 5; k >= 0; --k) {
#pragma unroll
        for (int i = k + 1; i < 6; ++i) cswapd(tr[k] == i, d[k], d[i]);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) x[i] = d[i];
}

// The 17 sums that determine H = sum w J^T J and g = sum w J^T r for J = [I | -hat(s)]
// (registration.cpp:46-54,75-76): w, w*s (3), w*s*s^T (6, upper), w*r (3), w*(s x r) (3), count.
struct NormalSums {
    double w, ws[3], wss[6] /* xx xy xz yy yz zz */, wr[3], wsxr[3];
};
enum { LIMU_NSUMS = 16 };

// Expand the sums into H (row-major 6x6) and g (6). With A = -hat(s): H = [[wI, wA],[wA^T, wA^T A]],
// A^T A = (s.s) I - s s^T, g = [w r; w (s x r)].
LIMU_HD void expand_normal_equations(const double *S, double *H, double *g) {
    const double w = S[0], sx = S[1], sy = S[2], sz = S[3];
    const double xx = S[4], xy = S[5], xz = S[6], yy = S[7], yz = S[8], zz = S[9];
#pragma unroll
    for (int i = 0; i < 36; ++i) H[i] = 0.0;
    H[0] = H[7] = H[14] = w;
    // A = [[0, sz, -sy], [-sz, 0, sx], [sy, -sx, 0]]
    H[0 * 6 + 4] = sz;  H[0 * 6 + 5] = -sy;
    H[1 * 6 + 3] = -sz; H[1 * 6 + 5] = sx;
    H[2 * 6 + 3] = sy;  H[2 * 6 + 4] = -sx;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) H[(3 + c) * 6 + r] = H[r * 6 + 3 + c];
    H[3 * 6 + 3] = yy + zz; H[3 * 6 + 4] = -xy;     H[3 * 6 + 5] = -xz;
    H[4 * 6 + 3] = -xy;     H[4 * 6 + 4] = xx + zz; H[4 * 6 + 5] = -yz;
    H[5 * 6 + 3] = -xz;     H[5 * 6 + 4] = -yz;     H[5 * 6 + 5] = xx + yy;
    g[0] = S[10]; g[1] = S[11]; g[2] = S[12]; g[3] = S[13]; g[4] = S[14]; g[5] = S[15];
}

// x = H^-1 (-g) straight from the 16 sums, for the point-to-point H above: its top-left block is w I, so eliminating it leaves the 3x3
// Schur complement Sm = D - A^T A / w = D - (|c|^2 I - c c^T) / w (c = sum w s, D the bottom-right block), solved by its adjugate:
//   Sm x2 = -g2 + (c x g1) / w,   x1 = (c x x2 - g1) / w.
// One reciprocal of w, one of det(Sm), no pivot search. Agrees with ldlt6_solve to rounding (the sums are ours, not Eigen's, in any
// case). When w is not positive and finite, when det(Sm) is not clear of the cancellation in D - A^T A / w (det(Sm) <= 1e-9 tr(D)^3:
// fewer than three points, collinear points), or when a sum is not finite, it returns exactly what expand_normal_equations +
// ldlt6_solve return. The choice depends on
// S alone, so every CTA and rank that folds the same sums takes the same branch.
LIMU_HD void solve_point_to_point(const double *S, double *x) {
    const double w = S[0], cx = S[1], cy = S[2], cz = S[3];
    const double xx = S[4], xy = S[5], xz = S[6], yy = S[7], yz = S[8], zz = S[9];
    const double iw = rcp(w), mx = cx * iw, my = cy * iw, mz = cz * iw;   // m = c / w
    const double dxx = yy + zz, dyy = xx + zz, dzz = xx + yy;
    const double s00 = dxx - (cy * my + cz * mz), s11 = dyy - (cx * mx + cz * mz), s22 = dzz - (cx * mx + cy * my);
    const double s01 = cx * my - xy, s02 = cx * mz - xz, s12 = cy * mz - yz;
    const double a00 = s11 * s22 - s12 * s12, a01 = s02 * s12 - s01 * s22, a02 = s01 * s12 - s02 * s11;   // adj(Sm), symmetric
    const double a11 = s00 * s22 - s02 * s02, a12 = s01 * s02 - s00 * s12, a22 = s00 * s11 - s01 * s01;
    const double det = (s00 * a00 + s01 * a01) + s02 * a02;
    const double trd = (dxx + dyy) + dzz, gsum = ((S[10] + S[11]) + (S[12] + S[13])) + (S[14] + S[15]);
    if (!(w > 0.0 && isfinite(w) && det > 1e-9 * (trd * (trd * trd)) && isfinite(gsum))) {
        double H[36], g[6];
        expand_normal_equations(S, H, g);
#pragma unroll
        for (int k = 0; k < 6; ++k) g[k] = -g[k];
        ldlt6_solve(H, g, x);
        return;
    }
    const double g1x = S[10], g1y = S[11], g1z = S[12];
    const double rx = (my * g1z - mz * g1y) - S[13], ry = (mz * g1x - mx * g1z) - S[14], rz = (mx * g1y - my * g1x) - S[15];
    const double id = rcp(det);
    const double x2x = ((a00 * rx + a01 * ry) + a02 * rz) * id;
    const double x2y = ((a01 * rx + a11 * ry) + a12 * rz) * id;
    const double x2z = ((a02 * rx + a12 * ry) + a22 * rz) * id;
    x[0] = (my * x2z - mz * x2y) - g1x * iw;
    x[1] = (mz * x2x - mx * x2z) - g1y * iw;
    x[2] = (mx * x2y - my * x2x) - g1z * iw;
    x[3] = x2x; x[4] = x2y; x[5] = x2z;
}

}  // namespace limu
