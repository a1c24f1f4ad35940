"""The Gauss-Newton step of the ICP loop on the host: solve_point_to_point (Schur complement of the w I block of the point-to-point
normal equations) against expand_normal_equations + ldlt6_solve, se3_exp_gn against se3_exp and an extended-precision exp, and
gn_verdict against |x| < eps. csrc/se3.cuh is compiled with g++ -ffp-contract=off, as the library compiles it (-fmad=false)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lidar-imu-slam_b200", "csrc")

HARNESS = r"""
#include "se3.cuh"
#include <math.h>
using namespace limu;
extern "C" {
void gn_solve(const double *S, double *x) { solve_point_to_point(S, x); }
void ldlt_solve(const double *S, double *x) {
    double H[36], g[6];
    expand_normal_equations(S, H, g);
    for (int k = 0; k < 6; ++k) g[k] = -g[k];
    ldlt6_solve(H, g, x);
}
void exp_gn(const double *a, double *p) { pose_store(se3_exp_gn(a), p); }
void exp_sophus(const double *a, double *p) { pose_store(se3_exp(a), p); }
// SE3::exp in long double: 1 - cos = 2 sin^2(theta/2), so nothing cancels that double rounding would not hide
void exp_exact(const double *a, double *p) {
    const long double ux = a[0], uy = a[1], uz = a[2], wx = a[3], wy = a[4], wz = a[5];
    const long double th = sqrtl(wx * wx + wy * wy + wz * wz);
    long double imag = 0.5L, c1 = 0.5L, c2 = 1.0L / 6.0L;
    if (th > 0) {
        const long double sh = sinl(th / 2), ch = cosl(th / 2);
        imag = sh / th; c1 = 2 * sh * sh / (th * th);
        c2 = th > 1e-3L ? (th - 2 * sh * ch) / (th * th * th) : 1.0L / 6 - th * th / 120 + th * th * th * th / 5040;
    }
    const long double vx = wy * uz - wz * uy, vy = wz * ux - wx * uz, vz = wx * uy - wy * ux;
    const long double ox = wy * vz - wz * vy, oy = wz * vx - wx * vz, oz = wx * vy - wy * vx;
    p[0] = (double)(imag * wx); p[1] = (double)(imag * wy); p[2] = (double)(imag * wz); p[3] = (double)(th > 0 ? cosl(th / 2) : 1.0L);
    p[4] = (double)(ux + c1 * vx + c2 * ox); p[5] = (double)(uy + c1 * vy + c2 * oy); p[6] = (double)(uz + c1 * vz + c2 * oz);
}
int verdict(const double *x, double eps) { return gn_verdict(x, eps); }
}
"""

D6 = ctypes.POINTER(ctypes.c_double)


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("gn_solve")
    src, so = d / "harness.cpp", d / "harness.so"
    src.write_text(HARNESS)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(so)])
    h = ctypes.CDLL(str(so))
    for f in ("gn_solve", "ldlt_solve", "exp_gn", "exp_sophus", "exp_exact"):
        getattr(h, f).argtypes = [D6, D6]
        getattr(h, f).restype = None
    h.verdict.argtypes = [D6, ctypes.c_double]
    h.verdict.restype = ctypes.c_int
    return h


def _p(a):
    return a.ctypes.data_as(D6)


def call(h, f, a, n):
    a = np.ascontiguousarray(a, dtype=np.float64)
    out = np.zeros(n)
    getattr(h, f)(_p(a), _p(out))
    return out


def sums(s, r, w):
    """The 16 sums of NormalSums for sources s, residuals r, weights w."""
    ws = w[:, None] * s
    sxr = np.cross(s, r)
    return np.concatenate([[w.sum()], ws.sum(0),
                           [(ws[:, 0] * s[:, 0]).sum(), (ws[:, 0] * s[:, 1]).sum(), (ws[:, 0] * s[:, 2]).sum(),
                            (ws[:, 1] * s[:, 1]).sum(), (ws[:, 1] * s[:, 2]).sum(), (ws[:, 2] * s[:, 2]).sum()],
                           (w[:, None] * r).sum(0), (w[:, None] * sxr).sum(0)])


def cloud(rng, n, scale, flat, offset):
    s = rng.uniform(-scale, scale, size=(n, 3))
    s[:, 2] *= flat
    s += offset
    r = rng.normal(scale=0.05, size=(n, 3)) + 0.01 * np.cross(rng.normal(size=3), s)
    w = 1.0 / (1.0 + (r * r).sum(1) / 0.1) ** 2    # Geman-McClure-like weights
    return s, r, w


def hessian(S):
    w, cx, cy, cz, xx, xy, xz, yy, yz, zz = S[:10]
    A = np.array([[0, cz, -cy], [-cz, 0, cx], [cy, -cx, 0]])
    D = np.array([[yy + zz, -xy, -xz], [-xy, xx + zz, -yz], [-xz, -yz, xx + yy]])
    return np.block([[w * np.eye(3), A], [A.T, D]])


@pytest.mark.parametrize("scale", [5.0, 40.0])
@pytest.mark.parametrize("flat", [1.0, 0.05, 1e-4, 0.0])
@pytest.mark.parametrize("n", [3, 7, 200, 3200])
def test_structured_solve_matches_ldlt(lib, scale, flat, n):
    """Both solves are backward stable, so they may differ by what the conditioning of H makes of rounding: about eps cond(H) relative
    (a 50-digit solve of the worst sets here finds both within that of the exact step, neither consistently closer)."""
    rng = np.random.default_rng(int(scale) * 1000 + n + int(flat * 1e4))
    for t in range(40):
        offset = rng.normal(size=3) * scale * (2.0 if t % 4 == 3 else 0.2)   # every fourth cloud sits away from the origin
        S = sums(*cloud(rng, n, scale, flat, offset))
        x, ref = call(lib, "gn_solve", S, 6), call(lib, "ldlt_solve", S, 6)
        cond = np.linalg.cond(hessian(S))
        assert np.all(np.isfinite(ref))
        assert np.abs(x - ref).max() <= max(1e-15 * cond, 1e-14) * np.abs(ref).max(), (t, cond, x, ref)
        if cond < 1e3:
            assert np.abs(x - ref).max() <= 1e-13 * np.abs(ref).max(), (t, cond, x, ref)


def test_degenerate_sets_take_the_ldlt_path(lib):
    """No point, one point, two points and collinear points: Sm is singular up to rounding, and the result is ldlt6_solve's, bit for bit."""
    rng = np.random.default_rng(7)
    cases = [np.zeros(16)]
    for t in range(200):
        scale = [0.5, 5.0, 40.0, 300.0][t % 4]
        n = [1, 2, 2, 50][t % 4] if t % 8 < 4 else [1, 2, 3, 500][t % 4]
        s, r, w = cloud(rng, n, scale, 1.0, rng.normal(size=3) * scale)
        if n > 2:   # on a line
            s = s[:1] + rng.uniform(-scale, scale, size=(n, 1)) * rng.normal(size=3)
        cases.append(sums(s, r, w))
    for S in cases:
        x, ref = call(lib, "gn_solve", S, 6), call(lib, "ldlt_solve", S, 6)
        assert np.array_equal(x, ref, equal_nan=True), (S, x, ref)


def test_nonfinite_sums_take_the_ldlt_path(lib):
    rng = np.random.default_rng(9)
    S0 = sums(*cloud(rng, 100, 5.0, 1.0, np.zeros(3)))
    for k in range(16):
        for v in (np.nan, np.inf, -np.inf):
            S = S0.copy()
            S[k] = v
            assert np.array_equal(call(lib, "gn_solve", S, 6), call(lib, "ldlt_solve", S, 6), equal_nan=True), (k, v)


def test_exp_matches_sophus_and_extended_precision(lib):
    """Quaternion within 1e-15 of se3_exp; translation within 2e-15 |v| of the long-double exp. Where se3_exp's 1 - cos(theta)
    cancels (theta ~ 1e-10 .. 1e-5), the two may differ by se3_exp's own error, which the bound below adds back."""
    rng = np.random.default_rng(3)
    eps = 1e-10
    thetas = [0.0, 1e-14, 1e-11, eps * (1 - 1e-12), eps, eps * (1 + 1e-12), 2e-10, 1e-9, 1e-8, 3e-8, 1e-7, 1e-6, 1e-5, 1e-4, 1e-3, 1e-2,
              0.1, 0.5, 1.0, 2.0, 3.0, np.pi - 1e-3, np.pi - 1e-6]
    for th in thetas:
        for t in range(20):
            axis = rng.normal(size=3)
            axis /= np.linalg.norm(axis)
            ups = rng.normal(size=3) * 10.0 ** rng.uniform(-4, 1)
            a = np.concatenate([ups, th * axis])
            p, q, e = call(lib, "exp_gn", a, 7), call(lib, "exp_sophus", a, 7), call(lib, "exp_exact", a, 7)
            nu = np.linalg.norm(ups)
            assert np.abs(p[:4] - q[:4]).max() <= 1e-15, (th, p, q)
            assert np.abs(p[:4] - e[:4]).max() <= 1e-15, (th, p, e)
            err_gn, err_sophus = np.abs(p[4:] - e[4:]).max(), np.abs(q[4:] - e[4:]).max()
            assert err_gn <= 2e-15 * nu, (th, p, e)
            assert np.abs(p[4:] - q[4:]).max() <= 2e-15 * nu + err_sophus, (th, p, q)


def test_verdict_matches_the_norm_of_the_twist(lib):
    rng = np.random.default_rng(5)
    for eps in (1e-4, 1e-6, 0.01):
        for t in range(2000):
            d = rng.normal(size=6)
            ratio = rng.uniform(0.01, 3.0)
            x = d / np.linalg.norm(d) * ratio * eps
            v = lib.verdict(_p(x), eps)
            if abs(ratio - 1.0) > 2e-6:
                assert v == (1 if ratio < 1.0 else 0), (eps, ratio, v)
            else:
                assert v in (2, 1 if ratio < 1.0 else 0)
            assert v != 2 or abs(ratio - 1.0) < 2e-6
        # inside the band: too close to call
        for r in (1.0 - 5e-7, 1.0, 1.0 + 5e-7):
            x = np.array([r * eps, 0, 0, 0, 0, 0])
            assert lib.verdict(_p(x), eps) == 2
    # a rotation of 3 rad or more, and NaN: always left to the logarithm
    for x in ([0, 0, 0, 3.0, 0, 0], [0, 0, 0, 0, 2.0, 2.3], [np.nan, 0, 0, 0, 0, 0], [0, 0, 0, np.nan, 0, 0], [0, 0, 0, np.inf, 0, 0]):
        assert lib.verdict(_p(np.array(x, dtype=np.float64)), 1e-4) == 2, x
