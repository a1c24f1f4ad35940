"""limu_odom_register_cloud_imu / limu_odom_prefetch_cloud_imu: the IMU backward deskew (kalman::EKF::motion_compensation_with_imu, ekf.cpp:420-468)
fused into the downsampling kernel of the odometry handle, followed by register_frame(Vec3dVector) (icp.cpp:58-86).

Two references. The composition: limu_deskew_imu -> its double output -> limu_odom_register_points on a second handle (plain path); the fused
call must give the same clouds, counts, iterations and poses bit for bit. The C port: lo_kiss_register_points on the same device-deskewed cloud
(not the port's own deskew: CUDA sin/cos may move a float by one ulp, which can flip a voxel key; the deskew itself is pinned to <= 1 ulp by
test_imu_forward.py), to the north-star tolerance of 1e-5 m / 1e-6.

Scenes are synth.cast_scan sweeps as 48-byte pcl::PointXYZINormal records with curvature = 100 t ms; the IMU windows follow the synthetic
trajectory (yaw rate, centripetal acceleration, gravity) with the noise of test_imu_forward.window, chained from scan to scan through
limu_imu_forward_pass."""
import os
import re
import time

import numpy as np
import pytest

from conftest import ROOT

REC, CURV = 48, 36                       # record size and curvature offset of pcl::PointXYZINormal
KEY_RANGE, INVALID = -3, -1


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    return g.load_package()


@pytest.fixture(scope="module")
def ctx(pkg):
    c = pkg.Context(0)
    yield c
    c.close()


def synth_mod():
    from importlib import import_module
    return import_module("limu_b200.synth")


def records_of(scan):
    """float32 [n,4] (x, y, z, t in [0,1]) -> [n,12] float32 records {x,y,z,1 | 0,0,0,0 | intensity, curvature = 100 t ms, 0, 0}."""
    r = np.zeros((len(scan), 12), np.float32)
    r[:, :3] = scan[:, :3]
    r[:, 3] = 1.0
    r[:, 9] = (scan[:, 3].astype(np.float64) * 100.0).astype(np.float32)
    return r


# scene shapes of bench.py's workloads: c2 (ground + boxes + cylinders, -25..+2 degrees) and c3 (urban canyon, -25..+15 degrees)
SHAPES = {"c2": dict(scene=dict(), elev=(-25.0, 2.0), beams=64, az=2000), "c3": dict(scene=dict(street=True, n_boxes=60, n_cyl=30), elev=(-25.0, 15.0), beams=128, az=4000)}


def make_sequence(traj, sizes, seed, shape="c2", device="cuda:0"):
    """One sweep per trajectory step, resized to sizes[i] points by synth.pad_scan (time order kept)."""
    synth = synth_mod()
    w = SHAPES[shape]
    scene = synth.Scene(seed=seed % 1000, **w["scene"])
    seq = []
    for i, n in enumerate(sizes):
        s = synth.cast_scan(scene, traj[i], traj[i + 1], beams=w["beams"], azimuth_steps=w["az"], elev=w["elev"], seed=seed + i, device=device)
        seq.append(synth.pad_scan(s, n, seed=seed + i))
    return seq


def imu_windows(pkg, traj, recs, rng, dt=0.005, first_offset=-0.004, gyr_extra=(0.0, 0.0, 0.0), acc_extra=(0.0, 0.0, 0.0), pil=(0.1, -0.05, 0.2),
                bg=(0.001, 0.002, -0.001), scan_dt=0.1, t_begin=50.0):
    """IMU samples along the trajectory (z rate = the sweep's yaw rate, centripetal acceleration, gravity; noise 0.002 rad/s and 0.03 m/s^2),
    cut into one window per scan (row 0 = the last sample of the previous window) and run through limu_imu_forward_pass with the state
    carried from scan to scan. Returns [(table, rot_end, pos_lidar_end, p_imu_lidar)] per scan."""
    from test_imu_forward import make_state
    n = len(recs)
    span = scan_dt * n + 0.05 - first_offset
    T = t_begin + first_offset + np.arange(int(span / dt) + 2) * dt
    k = np.clip(((T - t_begin) / scan_dt).astype(int), 0, n - 1)
    yaw_rate = np.diff(traj[: n + 1, 2]) / scan_dt
    speed = np.linalg.norm(np.diff(traj[: n + 1, :2], axis=0), axis=1) / scan_dt
    gyr = np.stack([np.zeros(len(T)), np.zeros(len(T)), yaw_rate[k]], 1) + np.asarray(gyr_extra) + rng.normal(size=(len(T), 3)) * 0.002
    acc = np.stack([np.zeros(len(T)), speed[k] * yaw_rate[k], np.full(len(T), 9.81)], 1) + np.asarray(acc_extra) + rng.normal(size=(len(T), 3)) * 0.03
    imu = np.concatenate([T[:, None], gyr, acc], 1)
    mean_acc = acc.mean(0)
    st = make_state(pkg, mean_acc, pil, bg, 0.0, np.concatenate([[0.0], acc[0], gyr[0]]))
    out, start = [], 0
    for i, r in enumerate(recs):
        beg = t_begin + i * scan_dt
        last_ms = float(r[-1, CURV // 4]) if len(r) else 0.0
        end = int(np.searchsorted(T, beg + last_ms / 1000.0, side="left"))
        end = max(end, start + 1)
        table, rot_end, ple = pkg.imu_forward_pass(st, imu[start:end + 1], beg, last_ms)
        st.pos[:], st.vel[:], st.quat[:] = st.tracker_pos[:], st.tracker_vel[:], st.tracker_quat[:]
        out.append((table, rot_end, ple, np.array(pil, float)))
        start = end
    return out


def composition(ctx, recs, imus, speculate=False, **cfg):
    """limu_deskew_imu -> out_xyz -> register_points on a fresh handle. Per scan (deskewed cloud, down, keypoints, pose, iterations, status)."""
    k = ctx.KissICP(speculate=speculate, **cfg)
    res = []
    for r, (table, re_, pe, pil) in zip(recs, imus):
        xyzc = np.ascontiguousarray(r[:, [0, 1, 2, 9]]) if len(r) else np.zeros((0, 4), np.float32)
        out = ctx.deskew_imu(xyzc, table, re_, pe, pil)[0] if len(r) else np.zeros((0, 3))
        st = 0
        try:
            d, s, p = k.register_points(out)
        except Exception as e:
            st, d, s, p = e.status, None, None, k.poses()[-1]
        res.append((out, d, s, p.copy(), k.stats.icp.iterations, st))
    dump = k.local_map().dump()
    k.close()
    return res, dump


def fused(ctx, recs, imus, speculate, prefetch=None, **cfg):
    """register_cloud_imu on one handle. prefetch(i) -> (records, imu args) to prefetch before registering scan i, or None."""
    k = ctx.KissICP(speculate=speculate, **cfg)
    res, hits = [], 0
    for i, (r, a) in enumerate(zip(recs, imus)):
        if prefetch is not None:
            pf = prefetch(i)
            if pf is not None:
                k.prefetch_cloud_imu(pf[0], REC, CURV, *pf[1])
        st = 0
        try:
            d, s, p = k.register_cloud_imu(r, REC, CURV, *a)
        except Exception as e:
            st, d, s, p = e.status, None, None, k.poses()[-1]
        assert k.stats.deskewed == 2 or st != 0
        hits += k.stats.reserved0
        res.append((None, d, s, p.copy(), k.stats.icp.iterations, st))
    dump = k.local_map().dump()
    k.close()
    return res, dump, hits


def assert_same(got, ref, pose_tol=0.0, what=""):
    assert len(got) == len(ref)
    for i, (g, r) in enumerate(zip(got, ref)):
        assert g[5] == r[5], (what, i, g[5], r[5])
        if g[1] is not None:
            assert g[1].shape == r[1].shape and g[2].shape == r[2].shape and g[4] == r[4], (what, i, g[1].shape, r[1].shape, g[2].shape, r[2].shape, g[4], r[4])
            assert np.array_equal(g[1], r[1]) and np.array_equal(g[2], r[2]), (what, i)
        if pose_tol == 0.0:
            assert np.array_equal(g[3], r[3]), (what, i, g[3], r[3])
        else:
            np.testing.assert_allclose(g[3], r[3], rtol=0, atol=pose_tol, err_msg=f"{what} scan {i}")


def assert_same_map(a, b, tol=0.0):
    """Map dumps: voxel keys and counts equal, stored points bit-identical (tol = 0) or within tol."""
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    np.testing.assert_allclose(a[2], b[2], rtol=0, atol=tol)


def pinned_records(pkg, recs):
    out = []
    for r in recs:
        p = pkg.PinnedArray((max(len(r), 1), 12), np.float32)
        p.array[: len(r)] = r
        out.append(p)
    return out


def next_prefetch(pins, recs, imus):
    return lambda i: (pins[i + 1].array[: len(recs[i + 1])], imus[i + 1]) if i + 1 < len(recs) else None


# ---- the c2-shaped sequence: 20 scans of 128 k points, voxel 1.0, cap 10 ---------------------------------------------------------------------
C2 = dict(voxel_size=1.0, cap=10, icp_max_iteration=60)


@pytest.fixture(scope="module")
def c2(pkg, ctx):
    synth = synth_mod()
    traj = synth.loop_trajectory(21, radius=30.0, step=0.7)
    seq = make_sequence(traj, [128000] * 20, seed=1000)
    recs = [records_of(s) for s in seq]
    imus = imu_windows(pkg, traj, recs, np.random.default_rng(77))
    comp, comp_dump = composition(ctx, recs, imus, **C2)
    plain, plain_dump, _ = fused(ctx, recs, imus, False, deskew=True, **C2)   # (cfg.deskew is ignored by the IMU call)
    pins = pinned_records(pkg, recs)
    pipe, pipe_dump, hits = fused(ctx, [p.array for p in pins], imus, True, prefetch=next_prefetch(pins, recs, imus), **C2)
    yield dict(seq=seq, recs=recs, imus=imus, comp=comp, comp_dump=comp_dump, plain=plain, plain_dump=plain_dump, pipe=pipe, pipe_dump=pipe_dump, hits=hits)
    for p in pins:
        p.free()


@pytest.mark.gpu
def test_plain_path_equals_the_composition(c2):
    assert_same(c2["plain"], c2["comp"], what="plain vs composition")
    assert_same_map(c2["plain_dump"], c2["comp_dump"])
    assert max(r[2].shape[0] for r in c2["plain"]) > 500


@pytest.mark.gpu
def test_pipelined_prefetched_path_equals_the_plain_path(c2):
    assert c2["hits"] == len(c2["recs"]) - 1                  # every scan but the first was deskewed and downsampled ahead
    assert_same(c2["pipe"], c2["plain"], pose_tol=1e-9, what="pipelined vs plain")
    bitwise = sum(np.array_equal(a[3], b[3]) for a, b in zip(c2["pipe"], c2["plain"]))
    print(f"\npipelined vs plain: {bitwise} of {len(c2['pipe'])} poses bit-identical")
    assert np.array_equal(c2["pipe_dump"][0], c2["plain_dump"][0]) and np.array_equal(c2["pipe_dump"][1], c2["plain_dump"][1])
    np.testing.assert_allclose(c2["pipe_dump"][2], c2["plain_dump"][2], rtol=0, atol=1e-8)


@pytest.mark.gpu
def test_plain_path_matches_the_port(c2):
    import oracle
    kc = oracle.load_port().Kiss(max_range=100.0, **C2)
    for i, (comp, got) in enumerate(zip(c2["comp"], c2["plain"])):
        dc, sc, pc = kc.register_points(comp[0])
        assert (len(dc), len(sc), kc.last_iterations()) == (got[1].shape[0], got[2].shape[0], got[4]), i
        assert np.abs(got[3][4:] - pc[4:]).max() < 1e-5 and np.abs(got[3][:4] - pc[:4]).max() < 1e-6, i


# ---- small sequences for the semantics --------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def small(pkg):
    synth = synth_mod()
    traj = synth.loop_trajectory(11, radius=30.0, step=0.7)
    seq = make_sequence(traj, [30000] * 10, seed=2000)
    recs = [records_of(s) for s in seq]
    imus = imu_windows(pkg, traj, recs, np.random.default_rng(78))
    return dict(traj=traj, seq=seq, recs=recs, imus=imus)


SMALL = dict(voxel_size=1.0, cap=10, icp_max_iteration=60)


@pytest.mark.gpu
def test_stationary_imu_equals_register_cloud_without_deskew(ctx, pkg, small):
    """Identity rotations, zero velocity, acceleration and lever arm: the IMU deskew returns every point unchanged, so the result is
    register_cloud with deskew = 0 on the same records, bit for bit, on both paths."""
    recs, seq = small["recs"][:6], small["seq"][:6]
    table = np.zeros((22, 22))
    table[:, 0] = -0.004 + np.arange(22) * 0.005
    table[:, 13:22] = np.eye(3).reshape(9)
    still = (table, np.eye(3).reshape(9), np.zeros(3), np.zeros(3))
    for spec in (False, True):
        k = ctx.KissICP(speculate=spec, deskew=False, **SMALL)
        ref = []
        for r, s in zip(recs, seq):
            d, sr, p = k.register_cloud(r, REC, s[:, 3].astype(np.float64))
            ref.append((None, d, sr, p.copy(), k.stats.icp.iterations, 0))
        k.close()
        pins = pinned_records(pkg, recs)
        got, _, _ = fused(ctx, [p.array for p in pins], [still] * len(recs), spec, prefetch=lambda i: (pins[i + 1].array, still) if i + 1 < len(recs) else None,
                          deskew=True, **SMALL)
        assert_same(got, ref, what=f"stationary speculate={spec}")
        for p in pins:
            p.free()


@pytest.mark.gpu
def test_rows_before_the_scan_start_repeat_the_first_point(ctx, pkg, small):
    """first_offset = -0.03: several table rows lie below point 0, which the reference's loop compensates again under each of them. down[0] is
    point 0 (first point per voxel wins, first-occurrence order): it must be deskew_imu's point 0 bit for bit, on both paths."""
    recs = small["recs"][:4]
    imus = imu_windows(pkg, small["traj"], recs, np.random.default_rng(5), first_offset=-0.03)
    assert (imus[0][0][:, 0] < 0).sum() >= 4
    comp, _ = composition(ctx, recs, imus, **SMALL)
    for spec in (False, True):
        pins = pinned_records(pkg, recs)
        got, _, _ = fused(ctx, [p.array for p in pins], imus, spec, prefetch=next_prefetch(pins, recs, imus), **SMALL)
        for g, c in zip(got, comp):
            assert np.array_equal(g[1][0], c[0][0])
        assert_same(got, comp, pose_tol=0.0 if not spec else 1e-9, what=f"first_offset speculate={spec}")
        for p in pins:
            p.free()


@pytest.mark.gpu
def test_prefetch_semantics(ctx, pkg, small):
    """A prepared scan is only used by a register call of the same kind with the same records and byte-equal IMU arguments; anything else is
    dropped, and results never depend on prefetching."""
    recs, imus, seq = small["recs"], small["imus"], small["seq"]
    n = len(recs)
    ref, ref_dump = composition(ctx, recs, imus, **SMALL)
    pins = pinned_records(pkg, recs)
    arr = [p.array for p in pins]

    def wrong(a):   # the same window with one row of the table moved by one ulp
        t = a[0].copy()
        t[1, 10] = np.nextafter(t[1, 10], 1.0)
        return (t,) + tuple(a[1:])

    # a prefetch with table A followed by a register with table B == an un-prefetched register with B
    got, dump, hits = fused(ctx, arr, imus, True, prefetch=lambda i: (arr[i + 1], wrong(imus[i + 1])) if i + 1 < n else None, **SMALL)
    assert hits == 0
    assert_same(got, ref, pose_tol=1e-9, what="table A then B")
    assert_same_map(dump, ref_dump, 1e-8)

    # a constant-velocity prefetch_cloud of the same records followed by the IMU register
    ts = [np.ascontiguousarray(s[:, 3].astype(np.float64)) for s in seq]
    k = ctx.KissICP(speculate=True, deskew=True, **SMALL)
    got = []
    for i in range(n):
        if i + 1 < n:
            k.prefetch_cloud(arr[i + 1], REC, ts[i + 1])
        d, s, p = k.register_cloud_imu(arr[i], REC, CURV, *imus[i])
        assert k.stats.reserved0 == 0
        got.append((None, d, s, p.copy(), k.stats.icp.iterations, 0))
    k.close()
    assert_same(got, ref, pose_tol=1e-9, what="cv prefetch then imu register")

    # constant-velocity and IMU scans interleaved on one handle, prefetches of either kind before either kind: against the plain path
    kinds = ["imu", "cv", "cv", "imu", "imu", "cv", "imu", "cv", "cv", "imu"]

    def interleaved(spec, cross):
        k = ctx.KissICP(speculate=spec, deskew=True, **SMALL)
        out = []
        for i in range(n):
            if spec and i + 1 < n:
                kind = kinds[i + 1] if not (cross and i % 3 == 0) else ("cv" if kinds[i + 1] == "imu" else "imu")
                if kind == "imu":
                    k.prefetch_cloud_imu(arr[i + 1], REC, CURV, *imus[i + 1])
                else:
                    k.prefetch_cloud(arr[i + 1], REC, ts[i + 1])
            if kinds[i] == "imu":
                d, s, p = k.register_cloud_imu(arr[i], REC, CURV, *imus[i])
                assert k.stats.deskewed == 2
            else:
                d, s, p = k.register_cloud(arr[i], REC, ts[i])
                assert k.stats.deskewed == (1 if i > 2 else 0)
            out.append((None, d, s, p.copy(), k.stats.icp.iterations, 0))
        dump = k.local_map().dump()
        k.close()
        return out, dump

    plain, plain_dump = interleaved(False, False)
    for cross in (False, True):
        got, dump = interleaved(True, cross)
        for i, (g, r) in enumerate(zip(got, plain)):
            assert g[1].shape == r[1].shape and g[2].shape == r[2].shape and g[4] == r[4], (cross, i)
            np.testing.assert_allclose(g[1], r[1], rtol=0, atol=1e-9)
            np.testing.assert_allclose(g[2], r[2], rtol=0, atol=1e-9)
            np.testing.assert_allclose(g[3], r[3], rtol=0, atol=1e-9)
        assert_same_map(dump, plain_dump, 1e-8)

    # an abandoned IMU prefetch (of a scan that is never registered, and of one registered two calls later) does no harm
    def abandoned(i):
        if i == 2:
            return (arr[9], imus[9])               # never registered in this run
        if i == 4:
            return (arr[6], imus[6])               # registered at i = 6, after scan 5 has used the pipeline
        return None
    got, dump, _ = fused(ctx, arr[:9], imus[:9], True, prefetch=abandoned, **SMALL)
    assert_same(got, ref[:9], pose_tol=1e-9, what="abandoned prefetch")
    for p in pins:
        p.free()


@pytest.mark.gpu
def test_ragged_sizes(ctx, pkg):
    """n = 1, 2, 1023, 1025 and 128 k points, then three scans of 512 000 points at voxel 0.5, cap 20 (the loop kernel then needs every SM):
    pipelined with prefetches, plain and composition; no call may take a second (a gate and a full-GPU cooperative launch waiting for each
    other would take five)."""
    synth = synth_mod()
    for sizes, cfg, seed, shape in (([128000, 1, 2, 1023, 1025, 128000, 2, 1025], dict(voxel_size=1.0, cap=10, icp_max_iteration=60), 3000, "c2"),
                                    ([512000] * 3, dict(voxel_size=0.5, cap=20, max_range=1000.0, icp_max_iteration=60), 3007, "c3")):
        traj = synth.loop_trajectory(len(sizes) + 1, radius=30.0, step=0.5)
        seq = make_sequence(traj, sizes, seed=seed, shape=shape)
        recs = [records_of(s) for s in seq]
        imus = imu_windows(pkg, traj, recs, np.random.default_rng(seed))
        comp, comp_dump = composition(ctx, recs, imus, **cfg)
        plain, plain_dump, _ = fused(ctx, recs, imus, False, **cfg)
        assert_same(plain, comp, what=f"ragged plain {sizes}")
        assert_same_map(plain_dump, comp_dump)
        if sizes[0] == 512000:
            assert min(r[2].shape[0] for r in plain) >= 7000
        pins = pinned_records(pkg, recs)
        k = ctx.KissICP(speculate=True, **cfg)
        worst = 0.0
        for i in range(len(recs)):
            if i + 1 < len(recs):
                k.prefetch_cloud_imu(pins[i + 1].array[: len(recs[i + 1])], REC, CURV, *imus[i + 1])
            t0 = time.perf_counter()
            d, s, p = k.register_cloud_imu(pins[i].array[: len(recs[i])], REC, CURV, *imus[i])
            worst = max(worst, time.perf_counter() - t0) if i > 0 else worst
            assert d.shape == plain[i][1].shape and s.shape == plain[i][2].shape and k.stats.icp.iterations == plain[i][4], (sizes[i], i)
            assert np.array_equal(d, plain[i][1]) and np.array_equal(s, plain[i][2]), (sizes[i], i)
            np.testing.assert_allclose(p, plain[i][3], rtol=0, atol=1e-9)
        k.close()
        for x in pins:
            x.free()
        assert worst < 1.0, f"a call took {worst:.2f} s"


@pytest.mark.gpu
def test_errors(ctx, pkg, small):
    """A NaN coordinate: LIMU_ERR_KEY_RANGE with the frame committed, as the composition reports it. Bad arguments: LIMU_ERR_INVALID, the
    handle untouched (pose count unchanged, the next scan's result unaffected)."""
    import ctypes as C
    recs, imus = [r.copy() for r in small["recs"][:5]], small["imus"][:5]
    recs[2][100, 1] = np.nan
    comp, comp_dump = composition(ctx, recs, imus, **SMALL)
    assert comp[2][5] == KEY_RANGE and all(c[5] == 0 for i, c in enumerate(comp) if i != 2)
    for spec in (False, True):
        pins = pinned_records(pkg, recs)
        got, dump, _ = fused(ctx, [p.array for p in pins], imus, spec, prefetch=next_prefetch(pins, recs, imus), **SMALL)
        assert_same(got, comp, pose_tol=0.0 if not spec else 1e-9, what=f"nan speculate={spec}")
        assert_same_map(dump, comp_dump, 1e-8)
        for p in pins:
            p.free()

    clean = small["recs"][:3]
    ref, _ = composition(ctx, clean, imus[:3], **SMALL)
    L = pkg.lib()
    for spec in (False, True):
        k = ctx.KissICP(speculate=spec, **SMALL)
        k.register_cloud_imu(clean[0], REC, CURV, *imus[0])
        k.register_cloud_imu(clean[1], REC, CURV, *imus[1])
        table, re_, pe, pil = imus[2]
        bad = [(clean[2], REC, CURV, table[:1]), (clean[2], REC, CURV, np.concatenate([table] * 5)[:97]), (clean[2], 12, CURV, table),
               (clean[2], REC, REC, table), (clean[2], REC, 46, table)]
        for r, stride, toff, t in bad:
            with pytest.raises(pkg.LimuError) as e:
                k.register_cloud_imu(r, stride, toff, t, re_, pe, pil)
            assert e.value.status == INVALID, (stride, toff, len(t))
            with pytest.raises(pkg.LimuError) as e:
                k.prefetch_cloud_imu(r, stride, toff, t, re_, pe, pil)
            assert e.value.status == INVALID
            assert len(k.poses()) == 2
        pose = np.empty(7)
        assert L.limu_odom_register_cloud_imu(k.h, clean[2].ctypes.data_as(C.c_void_p), REC, CURV, len(clean[2]), None, 22, pkg._d(re_), pkg._d(pe), pkg._d(pil),
                                              pkg._d(pose), None, None, None, None, None) == INVALID
        assert L.limu_odom_prefetch_cloud_imu(k.h, clean[2].ctypes.data_as(C.c_void_p), REC, CURV, len(clean[2]), None, 22, pkg._d(re_), pkg._d(pe),
                                              pkg._d(pil)) == INVALID
        assert len(k.poses()) == 2
        d, s, p = k.register_cloud_imu(clean[2], REC, CURV, *imus[2])
        assert np.array_equal(d, ref[2][1]) and np.array_equal(s, ref[2][2]) and k.stats.icp.iterations == ref[2][4]
        np.testing.assert_allclose(p, ref[2][3], rtol=0, atol=0.0 if not spec else 1e-9)
        k.close()


def _random_seeds_i():
    """4 seeds in the suite; LIMU_RANDOM_SEEDS_I="lo-hi" widens the campaign."""
    spec = os.environ.get("LIMU_RANDOM_SEEDS_I", "")
    if "-" in spec:
        lo, hi = spec.split("-")
        return range(int(lo), int(hi))
    return range(8000, 8004)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", _random_seeds_i())
def test_random_family(ctx, pkg, seed):
    """Seeded random windows (the ranges of test_cuda_deskew_on_random_windows: 100 / 200 / 400 Hz, rates up to ~3 rad/s, accelerations up to
    ~2 g, windows starting up to 30 ms before the scan), voxel size, cap, scan sizes and prefetch pattern (next scan, a wrong table, a skipped
    or an abandoned prefetch): pipelined, plain and composition with the bars above."""
    r_ = np.random.default_rng(seed)
    synth = synth_mod()
    n_scans = 7
    traj = synth.loop_trajectory(n_scans + 1, radius=30.0, step=float(r_.uniform(0.2, 1.0)))
    sizes = [int(r_.integers(1000, 150000)) for _ in range(n_scans)]
    cfg = dict(voxel_size=float(r_.choice([0.5, 0.75, 1.0, 1.5])), cap=int(r_.choice([3, 10, 20])), icp_max_iteration=60)
    seq = make_sequence(traj, sizes, seed=40 * seed)
    recs = [records_of(s) for s in seq]
    imus = imu_windows(pkg, traj, recs, r_, dt=float(r_.choice([0.0025, 0.005, 0.01])), first_offset=-float(r_.uniform(1e-4, 0.03)),
                       gyr_extra=tuple(r_.normal(size=3) * r_.choice([0.05, 0.5, 1.5])), acc_extra=tuple(r_.normal(size=3) * r_.choice([0.3, 3.0])))
    comp, comp_dump = composition(ctx, recs, imus, **cfg)
    plain, plain_dump, _ = fused(ctx, recs, imus, False, **cfg)
    assert_same(plain, comp, what=f"seed {seed} plain")
    assert_same_map(plain_dump, comp_dump)
    pins = pinned_records(pkg, recs)
    arr = [p.array[: len(r)] for p, r in zip(pins, recs)]
    pattern = r_.integers(0, 4, size=n_scans)

    def prefetch(i):
        if i + 1 >= n_scans or pattern[i] == 3:
            return None
        if pattern[i] == 1:                                        # a wrong table: must be dropped
            t = imus[i + 1][0].copy()
            t[-1, 1] += 1e-3
            return arr[i + 1], (t,) + tuple(imus[i + 1][1:])
        if pattern[i] == 2 and i + 2 < n_scans:                    # the scan after next
            return arr[i + 2], imus[i + 2]
        return arr[i + 1], imus[i + 1]
    pipe, pipe_dump, _ = fused(ctx, arr, imus, True, prefetch=prefetch, **cfg)
    assert_same(pipe, plain, pose_tol=1e-9, what=f"seed {seed} pipelined, pattern {pattern.tolist()}")
    assert_same_map(pipe_dump, plain_dump, 1e-8)
    for p in pins:
        p.free()


def test_imu_voxelize_beside_the_map_update_fits_one_register_file():
    """Pipelined path: the next scan's k_voxelize_imu_lean (1024 threads) runs BESIDE the map update k_frame_update (256 threads), as
    k_voxelize_lean does: both CTAs must fit into the 65 536 registers of an SM. Read from the ptxas logs the build leaves behind."""
    regs = {}
    for log in ("registration.ptxas.log", "voxelize.ptxas.log"):
        path = os.path.join(ROOT, "lidar-imu-slam_b200", "build", log)
        if not os.path.exists(path):
            pytest.skip("no ptxas log (library not built here)")
        for m in re.finditer(r"Compiling entry function '(\w+)'.*?Used (\d+) registers", open(path).read(), re.S):
            regs[m.group(1)] = int(m.group(2))
    upd = [v for k, v in regs.items() if "k_frame_update" in k]
    vox = [v for k, v in regs.items() if "k_voxelize_imu_lean" in k]
    assert upd and vox, sorted(regs)
    alloc = lambda r, threads: ((r + 7) // 8 * 8) * threads
    assert alloc(upd[0], 256) + alloc(vox[0], 1024) <= 65536, (upd, vox)
