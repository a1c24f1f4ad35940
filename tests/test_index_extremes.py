"""Voxel indices at their extremes: the edge of the packed key range (+-(2^20 - 1) per axis), eviction distances whose square leaves
int32, and coordinates that are NaN, infinite or too large for any voxel index.

Pinned semantics (DESIGN section 2/3, INTEGRATION section 5):
* a voxel index is what the reference's x86-64 build computes, (int)(p / v) = cvttsd2si: NaN, or a truncation outside int32, gives
  INT_MIN;
* indices within +-(2^20 - 1) are bit-exact with the C port everywhere;
* eviction tests a voxel with Vector3i::squaredNorm(), int arithmetic that wraps modulo 2^32, and the device reproduces that;
* entries that turn points into map or grid keys drop a point whose index is NaN or outside the key range and return
  LIMU_ERR_KEY_RANGE (-3); everything else equals the port on the cloud without those points;
* queries never fail: their results equal the port's on the same input, NaN and infinite queries included.

The CPU part pins the port and the numpy restatement of the eviction (tests/np_restatement.py) against each other; the GPU part checks the
CUDA path against both.
"""
import ctypes as C

import numpy as np
import pytest

from np_restatement import np_remove_far, np_vox_index_x86

INT_MIN = -2147483648
B = (1 << 20) - 1                                   # largest |index| the packed key holds
KEY_RANGE = -3

# index distances from the origin's voxel to voxel 0: 46340^2 fits int32, 46341^2 wraps negative, 65536^2 wraps to 0, 26754 / 26755 on all
# three axes straddle 2^31 (3 * 26755^2 = 2 147 488 075)
EVICTION_ORIGINS = [(30000, 0, 0), (46340, 0, 0), (46341, 0, 0), (50000, 0, 0), (65535, 0, 0), (65536, 0, 0), (65537, 0, 0),
                    (27000, 27000, 27000), (26754, 26754, 26754), (26755, 26755, 26755), (-46341, 0, 0), (0, -65536, 0), (0, 0, 46341),
                    (3.0e9, 0, 0), (-3.0e9, 5.0, 0)]


def _eviction_map(api, vox=1.0, maxd=100.0):
    """Voxels at index 0 and 1 (and, off the x axis, (0,2,0) and (0,0,-3)) of a map with voxel `vox` and max distance `maxd`."""
    m = api.Map(vox, maxd, 4)
    m.insert(np.array([[0.5, 0.5, 0.5], [1.5, 0.5, 0.5], [0.25, 0.75, 0.5], [0.5, 2.5, 0.5], [0.5, 0.5, -3.5]]) * vox)
    return m


def _origin(o, vox=1.0):
    """An origin whose voxel index is `o` (components given in index units; those beyond int32 stand as they are)."""
    return np.array([(c + 0.5) * vox if abs(c) < 2 ** 31 else c * vox for c in o], np.float64)


# ------------------------------------------------------------------------------------------------------------------------------------
# CPU: the port and the numpy restatement agree, and the port shows the behaviour the device has to reproduce
# ------------------------------------------------------------------------------------------------------------------------------------
def test_port_vox_index_gives_int_min_for_nan_inf_and_int32_overflow(port):
    for v in (1.0, 0.5, 0.3, 1e-3):
        bad = np.array([[np.nan, 0.0, 0.0], [0.0, np.inf, 0.0], [0.0, 0.0, -np.inf], [2.0 ** 31 * v, -(2.0 ** 31) * v * 1.5, 1e300],
                        [-1e300, 2.0 ** 32 * v, np.nan]])
        k = port.vox_index(bad, v)
        assert k[0, 0] == INT_MIN and k[1, 1] == INT_MIN and k[2, 2] == INT_MIN
        assert (k[3] == INT_MIN).all() and (k[4] == INT_MIN).all()
        assert k[0, 1] == 0 and k[1, 0] == 0
        assert np.array_equal(k, np_vox_index_x86(bad, v))
    # the last representable indices on both sides: -2^31 itself is representable, 2^31 is not
    v = 1.0
    edge = np.array([[2.0 ** 31 - 1, 2.0 ** 31 - 0.5, 2.0 ** 31], [-(2.0 ** 31), -(2.0 ** 31) - 0.5, -(2.0 ** 31) - 1]])
    assert np.array_equal(port.vox_index(edge, v), [[2 ** 31 - 1, 2 ** 31 - 1, INT_MIN], [INT_MIN, INT_MIN, INT_MIN]])
    assert np.array_equal(port.vox_index(edge, v), np_vox_index_x86(edge, v))


def test_port_eviction_wraps_like_int32(port):
    """The examples of the eviction test in int32: at 46341 one of the two voxels survives, at 50000 and 65536 both do."""
    expect = {(30000, 0, 0): 0, (46341, 0, 0): 1, (50000, 0, 0): 2, (65536, 0, 0): 2, (27000, 27000, 27000): 2}
    for o, survivors in expect.items():
        m = port.Map(1.0, 100.0, 4)
        m.insert(np.array([[0.5, 0.5, 0.5], [1.5, 0.5, 0.5]]))
        m.remove_far(_origin(o))
        assert m.num_voxels() == survivors, o


def test_numpy_eviction_matches_port_at_crafted_origins(port):
    for vox, maxd in ((1.0, 100.0), (0.5, 100.0), (1.0, 3.0)):
        for o in EVICTION_ORIGINS:
            m = _eviction_map(port, vox, maxd)
            before = m.dump()
            origin = _origin(o, vox)
            m.remove_far(origin)
            got = m.dump()
            want = np_remove_far(*before, origin, vox, maxd)
            assert all(np.array_equal(a, b) for a, b in zip(got, want)), (vox, maxd, o)


@pytest.mark.parametrize("seed", range(6))
def test_numpy_eviction_matches_port_random(port, seed):
    """Voxels all over the key range, origins up to twice as far out (some beyond int32) and max distances from 1 to 1e5."""
    rng = np.random.default_rng(700 + seed)
    vox = float(rng.choice([1.0, 0.5, 0.3]))
    maxd = float(np.exp(rng.uniform(0.0, np.log(1e5))))
    n = 4000
    k = rng.integers(-B, B + 1, size=(n, 3))
    k[: n // 4] = rng.integers(-70000, 70000, size=(n // 4, 3))                     # squares that wrap around 2^31 and 2^32
    k[n // 4: n // 2] = rng.integers(-30, 30, size=(n // 4, 3))                     # a dense cluster near the origin
    pts = (k + rng.uniform(0.05, 0.95, size=(n, 3))) * vox
    pts = np.where(k < 0, (k - rng.uniform(0.05, 0.95, size=(n, 3)) + 1) * vox, pts)
    m = port.Map(vox, maxd, 3)
    m.insert(np.concatenate([pts, pts + 0.01 * vox]))
    for j in range(8):
        if j < 5:
            origin = rng.uniform(-2.0, 2.0, size=3) * B * vox
        elif j < 7:
            origin = (rng.integers(-70000, 70000, size=3) + 0.5) * vox
        else:
            origin = rng.choice([-1.0, 1.0], size=3) * 4.0e9 * vox
        before = m.dump()
        m.remove_far(origin)
        got = m.dump()
        want = np_remove_far(*before, origin, vox, maxd)
        assert all(np.array_equal(a, b) for a, b in zip(got, want)), (seed, j)
    assert 0 < m.num_voxels()


# ------------------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    return g.load_package()


@pytest.fixture(scope="module")
def ctx(pkg):
    c = pkg.Context(0)
    yield c
    c.close()


_dp, _lp = C.POINTER(C.c_double), C.POINTER(C.c_int64)


def _raw_downsample(pkg, ctx, xyz, s):
    """limu_voxel_downsample called directly: the binding raises before it returns the outputs the call did write."""
    xyz = np.ascontiguousarray(xyz, np.float64).reshape(-1, 3)
    out = np.zeros((max(len(xyz), 1), 3))
    idx = np.zeros(max(len(xyz), 1), np.int64)
    n = C.c_int64(-1)
    st = pkg.lib().limu_voxel_downsample(ctx.h, xyz.ctypes.data_as(_dp), len(xyz), float(s), out.ctypes.data_as(_dp), idx.ctypes.data_as(_lp), C.byref(n))
    return st, out[: n.value].copy(), idx[: n.value].copy()


def _raw_voxelize(pkg, ctx, xyz, v):
    xyz = np.ascontiguousarray(xyz, np.float64).reshape(-1, 3)
    src, down = np.zeros((max(len(xyz), 1), 3)), np.zeros((max(len(xyz), 1), 3))
    ns, nd = C.c_int64(-1), C.c_int64(-1)
    st = pkg.lib().limu_voxelize(ctx.h, xyz.ctypes.data_as(_dp), len(xyz), float(v), src.ctypes.data_as(_dp), C.byref(ns), down.ctypes.data_as(_dp), C.byref(nd))
    return st, src[: ns.value].copy(), down[: nd.value].copy()


def _in_range(port, xyz, v):
    k = port.vox_index(xyz, v)
    return (np.abs(k.astype(np.int64)) <= B).all(axis=1)


def _insert_expect_key_range(pkg, gm, xyz):
    with pytest.raises(pkg.LimuError) as e:
        gm.insert_points(xyz)
    assert e.value.status == KEY_RANGE


def _dumps_equal(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


def _boundary_values(v):
    """Coordinates at the edge of the key range for voxel v: index exactly +-(2^20 - 1) (with fractional offsets), -(2^20 - 0.5) v
    (truncates toward zero into range), exactly +-2^20, and one ulp either side of the boundary multiples."""
    vals = []
    for s in (1.0, -1.0):
        for f in (0.0, 0.25, 0.5, 0.999):
            vals.append(s * (B + f) * v)
        for m in (B, B + 1):
            x = s * m * v
            vals += [x, np.nextafter(x, np.inf), np.nextafter(x, -np.inf)]
        vals.append(s * (B + 1.5) * v)
    return np.array(vals)


def _boundary_cloud(v, rng):
    """Background points near the origin, then every boundary value on each axis in turn (the other two coordinates small), each
    boundary point once as the first point of its voxel and once again later, with a neighbour just inside the boundary."""
    vals = _boundary_values(v)
    bg = rng.normal(size=(3000, 3)) * 20 * v
    rows = []
    for ax in range(3):
        p = rng.normal(size=(len(vals), 3)) * 3 * v
        p[:, ax] = vals
        rows.append(p)
        inner = p.copy()
        inner[:, ax] = np.sign(vals) * (B - 0.5) * v             # the in-range neighbour voxel of the boundary one
        rows.append(inner)
    edge = np.concatenate(rows)
    corners = np.array([[sx * (B + 0.5) * v, sy * (B + 0.5) * v, sz * (B + 0.5) * v] for sx in (1, -1) for sy in (1, -1) for sz in (1, -1)])
    return np.concatenate([edge, bg[:1500], edge[::-1], corners, bg[1500:]])


VOXELS = [1.0, 0.5, 0.25, 0.3, 0.1, 1e-3]   # powers of two: the multiply path of the map; the others: the division path


@pytest.mark.gpu
@pytest.mark.parametrize("v", VOXELS)
def test_key_boundary_matches_port(pkg, ctx, port, v):
    rng = np.random.default_rng(int(v * 1000) + 11)
    pts = _boundary_cloud(v, rng)
    ok = _in_range(port, pts, v)
    assert 0 < (~ok).sum() < len(pts)
    clean = pts[ok]
    assert np.array_equal(ctx.voxel_keys(pts, v), port.vox_index(pts, v))

    st, out, _ = _raw_downsample(pkg, ctx, pts, v)
    assert st == KEY_RANGE
    assert np.array_equal(out, port.voxel_downsample(clean, v))

    # voxelize downsamples at half its voxel size first: pass 2v so that the first grid is the one at v
    st, gs, gd = _raw_voxelize(pkg, ctx, pts, 2 * v)
    os_, od = port.voxelize(clean, 2 * v)
    assert st == KEY_RANGE and np.array_equal(gd, od) and np.array_equal(gs, os_)

    for cap in (1, 4):
        gm = ctx.VoxelHashMap(v, 100.0, cap)
        om = port.Map(v, 100.0, cap)
        _insert_expect_key_range(pkg, gm, pts)
        om.insert(clean)
        assert _dumps_equal(gm.dump(), om.dump())
        # queries: every point of the cloud (out-of-range ones included) and small offsets of them, both neighbour rules
        q = np.concatenate([pts, pts + rng.normal(size=pts.shape) * 0.4 * v, [[(B + 1.2) * v, 0.2 * v, 0.1 * v], [-(B + 1.2) * v, 0, 0]]])
        for mode in (0, pkg.ICP_NN27):
            om.set_mode(mode)
            gout, gkey, grank = gm.get_closest_neighbour(q, with_index=True, icp_mode=mode)
            oout, okey, orank = om.closest(q, with_index=True)
            assert np.array_equal(gkey, okey) and np.array_equal(grank, orank) and np.array_equal(gout, oout), mode
        om.set_mode(0)
        outside = np.abs(port.vox_index(q, v).astype(np.int64)).max(axis=1) == B + 1
        assert (outside & (grank >= 0)).any()                # a query just outside found its in-range neighbour
        for tau in (0.5 * v, 3.0 * v):
            gs_, gt_, gi = gm.get_correspondences(q, tau, with_index=True)
            os_, ot_, oi = om.correspondences(q, tau, with_index=True)
            assert np.array_equal(gs_, os_) and np.array_equal(gt_, ot_) and np.array_equal(gi, oi)
        # eviction from origins at the edge: index distances up to 2(2^20 - 1), whose squares wrap
        for origin in ([(B + 0.5) * v, 0.0, 0.0], [-(B + 0.5) * v, 0.0, 0.0], [0.0, (B + 0.5) * v, -(B + 0.5) * v], [5 * v, 5 * v, 5 * v]):
            origin = np.array(origin)
            want = np_remove_far(*om.dump(), origin, v, 100.0)
            gm.remove_points_from_far(origin)
            om.remove_far(origin)
            assert _dumps_equal(gm.dump(), om.dump()) and _dumps_equal(om.dump(), want), origin
        gm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("vox", [1.0, 0.3])
def test_eviction_overflow_matches_port(ctx, port, vox):
    for maxd in (100.0, 3.0):
        for o in EVICTION_ORIGINS:
            origin = _origin(o, vox)
            gm = ctx.VoxelHashMap(vox, maxd, 4)
            om = _eviction_map(port, vox, maxd)
            gm.insert_points(om.dump()[2])
            assert _dumps_equal(gm.dump(), om.dump())
            want = np_remove_far(*om.dump(), origin, vox, maxd)
            gm.remove_points_from_far(origin)
            om.remove_far(origin)
            assert _dumps_equal(gm.dump(), om.dump()) and _dumps_equal(om.dump(), want), (maxd, o)
            # update(points, pose): insert the points moved by the pose, then evict around the pose's translation
            pose = np.array([0.0, 0.0, 0.0, 1.0, *origin]) if np.abs(origin).max() < 2.0e6 * vox else None
            if pose is not None:
                more = np.array([[0.3, 0.2, 0.1], [-0.4, 0.1, 0.2]]) * vox
                gm.update(more, pose)
                om.update(more, pose)
                assert _dumps_equal(gm.dump(), om.dump()), ("update", maxd, o)
            gm.close()


def _cluster_scans(rng, n_scans):
    """A static 3-D scene near the sensor plus, in every scan, a few new points of a cluster 600 m away (60 000 indices at voxel 0.01 m:
    its squared index distance wraps to a negative int, so the reference keeps it) and of one 300 m away (evicted everywhere)."""
    near = rng.uniform(-15, 15, size=(4000, 3))
    near[:, 2] *= 0.2
    scans = []
    for i in range(n_scans):
        far = np.array([600.0, 3.0, 1.0]) + rng.normal(size=(40, 3)) * 0.5
        mid = np.array([0.0, -300.0, 2.0]) + rng.normal(size=(40, 3)) * 0.5
        xyz = np.concatenate([near, far, mid]).astype(np.float32)
        t = rng.random((len(xyz), 1)).astype(np.float32)
        scans.append(np.ascontiguousarray(np.concatenate([xyz, t], 1)))
    return scans


@pytest.mark.gpu
@pytest.mark.parametrize("speculate", [False, True])
def test_odometry_keeps_wrapped_far_cluster_like_port(pkg, ctx, port, speculate):
    rng = np.random.default_rng(21)
    scans = _cluster_scans(rng, 4)
    cfg = dict(voxel_size=0.01, max_range=100.0, cap=10, deskew=False, icp_max_iteration=30)
    gk = ctx.KissICP(speculate=speculate, **cfg)
    ok = port.Kiss(**cfg)
    pins = [pkg.PinnedArray(s.shape, np.float32) for s in scans]
    for p, s in zip(pins, scans):
        p.array[...] = s
    for i, p in enumerate(pins):
        if speculate and i + 1 < len(pins):
            gk.prefetch(pins[i + 1].array)
        gd, gs, gp = gk.register_frame(p.array)
        od, os_, op = ok.register_cloud(scans[i][:, :3], scans[i][:, 3].astype(np.float64))
        assert np.array_equal(gd, od) and np.array_equal(gs, os_), i
        np.testing.assert_allclose(gp, op, rtol=0, atol=1e-9)
        gmap, omap = gk.local_map().dump(), ok.map().dump()
        assert np.array_equal(gmap[0], omap[0]) and np.array_equal(gmap[1], omap[1]), i
        np.testing.assert_allclose(gmap[2], omap[2], rtol=0, atol=1e-9)
        assert (omap[2][:, 0] > 500).any() and not (omap[2][:, 1] < -250).any()
    gk.close()
    for p in pins:
        p.free()


# ---- non-finite coordinates ---------------------------------------------------------------------------------------------------------
def _nonfinite_cloud(v, rng):
    """A finite cloud with NaN in x only, y only and in all axes, +-inf and +-1e300 mixed in: first in the cloud, first in the voxel
    their finite coordinates name, and mid-cloud. Returns (cloud, mask of the finite rows)."""
    base = rng.normal(size=(6000, 3)) * 10 * v
    bad_vals = []
    for b in (np.nan, np.inf, -np.inf, 1e300, -1e300):
        for ax in (0, 1, 2):
            bad_vals.append((ax, b))
    rows = []
    for j, (ax, b) in enumerate(bad_vals):
        p = base[(37 * j) % len(base)].copy()
        p[ax] = b
        rows.append(p)
    allnan = np.array([np.nan, np.nan, np.nan])
    bad = np.array(rows + [allnan])
    pts = np.concatenate([bad[:4], base[:3000], bad, base[3000:], bad[::-1]])
    fin = np.isfinite(pts).all(axis=1) & (np.abs(pts) < 1e200).all(axis=1)
    return pts, fin


@pytest.mark.gpu
@pytest.mark.parametrize("v", [1.0, 0.3])
def test_nonfinite_points_are_dropped_with_key_range(pkg, ctx, port, v):
    rng = np.random.default_rng(31)
    pts, fin = _nonfinite_cloud(v, rng)
    clean = pts[fin]
    k = ctx.voxel_keys(pts, v)
    assert np.array_equal(k, port.vox_index(pts, v)) and np.array_equal(k, np_vox_index_x86(pts, v))
    st, out, idx = _raw_downsample(pkg, ctx, pts, v)
    assert st == KEY_RANGE and np.array_equal(out, port.voxel_downsample(clean, v))
    assert fin[idx].all()
    st, gs, gd = _raw_voxelize(pkg, ctx, pts, v)
    os_, od = port.voxelize(clean, v)
    assert st == KEY_RANGE and np.array_equal(gd, od) and np.array_equal(gs, os_)
    gm, om = ctx.VoxelHashMap(v, 100.0, 5), port.Map(v, 100.0, 5)
    _insert_expect_key_range(pkg, gm, pts)
    om.insert(clean)
    assert _dumps_equal(gm.dump(), om.dump())
    with pytest.raises(pkg.LimuError) as e:
        gm.update(pts, np.array([0.0, 0.0, 0.0, 1.0, 0.5, -0.25, 0.0]))
    assert e.value.status == KEY_RANGE
    om.update(clean, np.array([0.0, 0.0, 0.0, 1.0, 0.5, -0.25, 0.0]))
    assert _dumps_equal(gm.dump(), om.dump())
    gm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("v", [1.0, 0.3])
def test_nonfinite_queries_match_port(pkg, ctx, port, v):
    """The aliasing case: voxels (0,0,0) and (0,ky,kz) are occupied, and a query with NaN x names (INT_MIN, ky, kz)."""
    rng = np.random.default_rng(41)
    ky, kz = 3, -2
    world = np.concatenate([rng.uniform(0.05, 0.95, size=(6, 3)) * v,
                            (np.array([0.0, ky, kz]) + np.array([0.5, 0.5, -0.5]) + rng.uniform(-0.45, 0.45, size=(6, 3))) * v,
                            rng.normal(size=(500, 3)) * 5 * v])
    gm, om = ctx.VoxelHashMap(v, 100.0, 10), port.Map(v, 100.0, 10)
    gm.insert_points(world)
    om.insert(world)
    assert _dumps_equal(gm.dump(), om.dump())
    good = np.array([[0.3, (ky + 0.5) * v, (kz - 0.5) * v], [0.4 * v, 0.4 * v, 0.4 * v], [0.2 * v, (ky + 0.3) * v, (kz - 0.1) * v]])
    q = []
    for g in good:
        for ax in (0, 1, 2):
            for b in (np.nan, np.inf, -np.inf, 1e300, 2.0 ** 31 * v):
                p = g.copy()
                p[ax] = b
                q.append(p)
        q.append(np.full(3, np.nan))
        q.append(g)
    q = np.array(q)
    for mode in (0, pkg.ICP_NN27):
        om.set_mode(mode)
        gout, gkey, grank = gm.get_closest_neighbour(q, with_index=True, icp_mode=mode)
        oout, okey, orank = om.closest(q, with_index=True)
        assert np.array_equal(gkey, okey) and np.array_equal(grank, orank) and np.array_equal(gout, oout), mode
        assert (okey[:, 0] == INT_MIN).sum() >= 3 * 3 * 5
    om.set_mode(0)
    for tau in (0.5 * v, 1e6):
        gs, gt, gi = gm.get_correspondences(q, tau, with_index=True)
        os_, ot, oi = om.correspondences(q, tau, with_index=True)
        assert np.array_equal(gs, os_, equal_nan=True) and np.array_equal(gt, ot) and np.array_equal(gi, oi)
    gm.close()


def _dense_scene(rng, n):
    a = rng.random((n // 3, 3)) * 40 - 20
    a[:, 2] = rng.normal(size=len(a)) * 0.02
    b = rng.random((n // 3, 3)) * 40 - 20
    b[:, 0] = 20 + rng.normal(size=len(b)) * 0.02
    c = rng.random((n // 3, 3)) * 40 - 20
    c[:, 1] = -20 + rng.normal(size=len(c)) * 0.02
    return np.concatenate([a, b, c])


@pytest.mark.gpu
@pytest.mark.parametrize("nq", [300, 40000])
def test_icp_with_nan_sources_matches_port(ctx, port, nq):
    """A few NaN sources in both launch shapes of the Gauss-Newton loop (one lane per query below 32 768 queries, the cooperative
    candidate scan above): they never correspond, in the port as on the device."""
    rng = np.random.default_rng(51)
    world = _dense_scene(rng, 90000)
    gm, om = ctx.VoxelHashMap(1.0, 100.0, 20), port.Map(1.0, 100.0, 20)
    gm.insert_points(world)
    om.insert(world)
    true = port.se3_exp(np.array([0.3, -0.2, 0.05, 0.004, -0.003, 0.02]))
    src = port.transform(port.se3_inv(true), world[rng.choice(len(world), nq, replace=False)])
    src[0, 0] = np.nan
    src[nq // 2, 1] = np.nan
    src[nq // 3] = np.nan
    src[-1, 2] = np.nan
    init = np.array([0, 0, 0, 1.0, 0, 0, 0])
    g = gm.icp(src, init, 6.0, 2.0 / 3.0, 60, 1e-4, trace=True)
    r = port.icp(om, src, init, 6.0, 2.0 / 3.0, 60, 1e-4, trace=True)
    assert g["iters"] == r["iters"]
    assert np.array_equal(g["ncorr"], r["ncorr"]) and r["ncorr"].max() <= nq - 4
    np.testing.assert_allclose(g["est"], r["est"], rtol=0, atol=1e-10)
    np.testing.assert_allclose(g["pose"], r["pose"], rtol=0, atol=1e-9)
    gm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("speculate", [False, True])
def test_register_frame_with_nan_points_commits_the_clean_frame(pkg, ctx, port, speculate):
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    scene = synth.Scene(seed=5)
    traj = synth.loop_trajectory(6, radius=30.0, step=0.6)
    scans = [synth.cast_scan(scene, traj[i], traj[i + 1], beams=16, azimuth_steps=600, seed=90 + i) for i in range(5)]
    bad, clean = list(scans), list(scans)
    for i, rows in ((1, [0, 1, 700]), (3, [5, 2000, len(scans[3]) - 1])):
        b = scans[i].copy()
        b[rows[0], 0] = np.nan            # first in the cloud / in its voxel
        b[rows[1], 1] = np.nan            # mid-cloud
        b[rows[2], :3] = np.nan
        bad[i] = b
        clean[i] = np.delete(scans[i], rows, axis=0)
    gk = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=speculate)
    ok = port.Kiss(deskew=True, icp_max_iteration=60)
    pins = [pkg.PinnedArray(s.shape, np.float32) for s in bad]
    for p, s in zip(pins, bad):
        p.array[...] = s
    for i, p in enumerate(pins):
        if speculate and i + 1 < len(pins):
            gk.prefetch(pins[i + 1].array)
        if i in (1, 3):
            with pytest.raises(pkg.LimuError) as e:
                gk.register_frame(p.array)
            assert e.value.status == KEY_RANGE
        else:
            gk.register_frame(p.array)
        od, os_, op = ok.register_cloud(clean[i][:, :3], clean[i][:, 3].astype(np.float64))
        gp = gk.poses()
        assert len(gp) == i + 1
        assert np.abs(gp[-1][4:] - op[4:]).max() < 1e-5 and np.abs(gp[-1][:4] - op[:4]).max() < 1e-6
        gmap, omap = gk.local_map().dump(), ok.map().dump()
        assert np.array_equal(gmap[0], omap[0]) and np.array_equal(gmap[1], omap[1]), i
        np.testing.assert_allclose(gmap[2], omap[2], rtol=0, atol=1e-6)
        assert np.isfinite(gmap[2]).all()
    gk.close()
    for p in pins:
        p.free()
