"""max_points_per_voxel at every path the device code chooses by it, not only at caps 1-20.

The cap is a user setting of the reference (frame.hpp reads it from the YAML config, default 10; the reference's hash_map_test.hpp uses
50 ... 1000; limu_map_create accepts 1 ... 4096), but the device code dispatches on it (registration.cu / voxel_map.cuh, n = query count):

    queries    cap                 lookup
    <= 16384   1-8 / 9-16 / 17-24  latency shape, group8_closest_at<ROUNDS = 1 / 2 / 3>
    <= 16384   25-64               ROUNDS = 3 plus the tail loop over ranks 24 ..., also on the memo ("known") path
    >  16384   1-20                staged pass (cp.async), block stride 16 / 32 / 48 / 64 doubles for caps 1-4 / 5-8 / 9-12 / 13-20
    >  16384   21-24 / >= 25       icp_query_pass_coop<3> / ... plus the tail
    any        >= 65               the bandwidth build even at 300 queries (in odometry: the frame kernel's SHAPE 1 with the one-CTA IQR select)
    opt-in point-to-plane, bandwidth build: block_closest below 32768 queries, coop_scan<1 / 2 / 3 / 0> from 32768 on (0: cap > 24)

The worlds are dense on purpose: a cap only matters where voxels really hold that many points, and every GPU test asserts that its map has
voxels filled to the cap, counts that are no multiple of 4 or 8 and (cap >= 25) voxels past 24 points, and that its queries include misses
of their own voxel and queries that find nothing. The CPU part pins the C port at these caps against tests/np_restatement.py (a brute-force
restatement independent of the port) and the iteration-0 normal equations against exact (math.fsum) sums.
"""
import math
import os

import numpy as np
import pytest

from np_restatement import np_closest, np_keys, np_map_insert

NN27, PLANE = 1, 2
IDENT = np.array([0, 0, 0, 1.0, 0, 0, 0])
TRUE_TWIST = np.array([0.06, -0.04, 0.02, 0.004, -0.003, 0.01])


def slab_world(rng, cap, vox=1.0):
    """A slab of voxels (8 x 8 x 2 up to cap 100, a 4 x 4 x 1 blob above), each holding points on a small random plane through it (noise
    1 % of the voxel: planar for the point-to-plane variant). About a third of the voxels is offered more than `cap` points (so they fill
    to the cap), about an eighth none (holes: queries there miss their own voxel), the rest a count below the cap drawn uniformly.
    Returned shuffled, so storage order is not creation order of the points."""
    side, layers = (8, 2) if cap <= 100 else (4, 1)
    out = []
    for ix in range(1, side + 1):
        for iy in range(1, side + 1):
            for iz in range(1, layers + 1):
                u = rng.random()
                if u < 0.12:
                    continue
                m = int(cap * rng.uniform(1.0, 1.3)) + 1 if u < 0.45 or cap == 1 else int(rng.integers(1, cap))
                c = (np.array([ix, iy, iz]) + 0.5) * vox
                nrm = rng.normal(size=3)
                nrm /= np.linalg.norm(nrm)
                p = c + (rng.random((m, 3)) - 0.5) * 0.9 * vox
                p -= ((p - c) @ nrm)[:, None] * nrm
                out.append(p + rng.normal(size=(m, 1)) * 0.01 * vox * nrm)
    return rng.permutation(np.concatenate(out))


def make_queries(rng, world, nq, vox=1.0):
    """World points moved by 0.25 voxel (many leave their voxel, some into holes), points anywhere in the slab's box, and a few far away
    (nothing within the 27 cells), seen from a pose off the identity by TRUE_TWIST."""
    lo, hi = world.min(0), world.max(0)
    n_far = max(3, nq // 100)
    n_box = nq // 8
    n_near = nq - n_far - n_box
    near = world[rng.integers(0, len(world), n_near)] + rng.normal(size=(n_near, 3)) * 0.25 * vox
    box = lo + rng.random((n_box, 3)) * (hi - lo)
    far = hi + 5.0 * vox + rng.random((n_far, 3)) * 3.0 * vox
    return rng.permutation(np.concatenate([near, box, far]))


def assert_map_coverage(counts, cap):
    assert counts.max() <= cap
    assert (counts == cap).any(), "no voxel filled to the cap"
    assert (counts % 4 != 0).any() and (counts % 8 != 0).any(), "every count a multiple of 4 / 8"
    if cap >= 25:
        assert (counts > 24).any(), "no voxel past the 24 register-resident ranks"


def assert_query_coverage(q, key, rank, vox):
    found_elsewhere = (rank >= 0) & (key != np_keys(q, vox)).any(axis=1)
    assert found_elsewhere.any(), "no query missed its own voxel"
    assert (rank < 0).any(), "no query found nothing"


def exact_normal_equations(src, tgt, th):
    """H = sum w J^T J, g = sum w J^T (s - t) with J = [I | -hat(s)], w = th^2 / (th + d^2)^2, each of the 42 entries summed exactly
    (math.fsum over the per-point terms). -> (hg [42], sum |terms| [42])."""
    r = src - tgt
    d2 = (r[:, 0] * r[:, 0] + r[:, 1] * r[:, 1]) + r[:, 2] * r[:, 2]
    w = (th * th) / ((th + d2) * (th + d2))
    n = len(src)
    J = np.zeros((n, 3, 6))
    J[:, 0, 0] = J[:, 1, 1] = J[:, 2, 2] = 1.0
    J[:, 0, 4], J[:, 0, 5] = src[:, 2], -src[:, 1]
    J[:, 1, 3], J[:, 1, 5] = -src[:, 2], src[:, 0]
    J[:, 2, 3], J[:, 2, 4] = src[:, 1], -src[:, 0]
    terms = np.concatenate([(w[:, None, None] * np.einsum("nka,nkb->nab", J, J)).reshape(n, 36), w[:, None] * np.einsum("nka,nk->na", J, r)], 1)
    return np.array([math.fsum(terms[:, k]) for k in range(42)]), np.abs(terms).sum(axis=0)


def iteration0_reference(keys, counts, pts, src, vox, tau, th):
    t, _, _ = np_closest(keys, counts, pts, src, vox)
    d = src - t
    gate = ((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]) < tau * tau
    hg, mag = exact_normal_equations(src[gate], t[gate], th)
    return hg, mag, int(gate.sum())


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("cap", [21, 24, 25, 33, 64, 65, 100, 1000, 4096])
def test_port_map_and_closest_match_brute_force(port, cap):
    rng = np.random.default_rng(7000 + cap)
    world = slab_world(rng, cap)
    m = port.Map(1.0, 100.0, cap)
    cuts = (0, len(world) // 3, len(world))
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        m.insert(world[lo:hi])
    ok, oc, op = m.dump()
    nk, nc, npt = np_map_insert(world, 1.0, cap)
    assert np.array_equal(ok, nk) and np.array_equal(oc, nc) and np.array_equal(op, npt)
    assert_map_coverage(oc, cap)
    q = make_queries(rng, world, 3000)
    got = m.closest(q, with_index=True)
    want = np_closest(ok, oc, op, q, 1.0)
    assert all(np.array_equal(a, b) for a, b in zip(got, want))
    assert_query_coverage(q, want[1], want[2], 1.0)


@pytest.mark.parametrize("cap", [25, 100, 1000])
def test_port_iteration0_normal_equations_against_exact_sums(port, cap):
    rng = np.random.default_rng(7100 + cap)
    world = slab_world(rng, cap)
    m = port.Map(1.0, 100.0, cap)
    m.insert(world)
    src = make_queries(rng, world, 2500)
    tau, th = 0.6, 0.2 / 3
    hg, mag, ngate = iteration0_reference(*m.dump(), src, 1.0, tau, th)
    assert 0 < ngate < len(src)                                        # tau rejects some correspondences
    r = port.icp(m, src, IDENT, tau, th, 1, 1e-4, trace=True)
    assert r["ncorr"][0] == ngate
    assert (np.abs(r["hg"][0] - hg) <= 1e-13 * mag).all()


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    return g.load_package()


@pytest.fixture(scope="module")
def ctx(pkg):
    c = pkg.Context(0)
    yield c
    c.close()


def check_loop(ctx, port, cap, nq, seed, vox=1.0, max_iter=30):
    """The comparisons of the grid and the random family: map, stand-alone lookups and the whole Gauss-Newton loop against the C port and
    the brute-force restatement, iteration 0 against exact sums."""
    rng = np.random.default_rng(seed)
    world = slab_world(rng, cap, vox)
    q = make_queries(rng, world, nq, vox)
    src = port.transform(port.se3_inv(port.se3_exp(TRUE_TWIST)), q)
    what = f"cap {cap}, {nq} queries, voxel {vox}, seed {seed}"
    gm, om = ctx.VoxelHashMap(vox, 100.0 * vox, cap), port.Map(vox, 100.0 * vox, cap)
    try:
        half = len(world) // 2
        for b in (world[:half], world[half:]):
            gm.insert_points(b)
            om.insert(b)
        gk, gc, gp = gm.dump()
        ok, oc, op = om.dump()
        assert np.array_equal(gk, ok) and np.array_equal(gc, oc) and np.array_equal(gp, op), what
        assert_map_coverage(gc, cap)
        want = np_closest(gk, gc, gp, src, vox)
        assert_query_coverage(src, want[1], want[2], vox)
        got = gm.get_closest_neighbour(src, with_index=True)
        assert all(np.array_equal(a, b) for a, b in zip(got, want)), what
        assert all(np.array_equal(a, b) for a, b in zip(got, om.closest(src, with_index=True))), what
        sigma = 0.2 * vox
        tau, th = 3 * sigma, sigma / 3
        gs, gt, gi = gm.get_correspondences(src, tau, with_index=True)
        os_, ot, oi = om.correspondences(src, tau, with_index=True)
        assert np.array_equal(gs, os_) and np.array_equal(gt, ot) and np.array_equal(gi, oi), what
        hg0, mag, ngate = iteration0_reference(gk, gc, gp, src, vox, tau, th)
        assert len(gi) == ngate and 0 < ngate < nq, what
        g = gm.icp(src, IDENT, tau, th, max_iter, 1e-4, trace=True)
        r = port.icp(om, src, IDENT, tau, th, max_iter, 1e-4, trace=True)
        assert g["iters"] == r["iters"], what
        assert np.array_equal(g["ncorr"], r["ncorr"]), what                   # the same correspondence sets in every iteration
        assert g["ncorr"][0] == ngate, what
        np.testing.assert_allclose(g["est"], r["est"], rtol=0, atol=1e-10, err_msg=what)
        np.testing.assert_allclose(g["hg"], r["hg"], rtol=0, atol=1e-12 * np.abs(r["hg"]).max(), err_msg=what)
        assert (np.abs(g["hg"][0] - hg0) <= 1e-13 * mag).all(), what
        np.testing.assert_allclose(g["pose"][4:], r["pose"][4:], rtol=0, atol=1e-9, err_msg=what)
        np.testing.assert_allclose(g["pose"][:4], r["pose"][:4], rtol=0, atol=1e-10, err_msg=what)
    finally:
        gm.close()


LOOP_CASES = [
    # latency shape (<= 16384 queries, cap <= 64): ROUNDS = 1 / 2 / 3, then 3 plus the tail over ranks 24 ...
    (1, 300), (4, 16384), (5, 300), (8, 16384), (9, 300), (12, 300), (13, 16384), (16, 300), (17, 16384), (20, 300), (21, 300),
    (24, 16384), (25, 300), (33, 16384), (64, 300), (64, 16384),
    # bandwidth shape, blocks staged through shared memory: strides of 16 / 32 / 48 / 64 doubles
    (1, 16385), (4, 32767), (5, 32768), (8, 16385), (9, 32767), (12, 16385), (13, 40000), (16, 16385), (17, 32768), (20, 16385),
    # bandwidth shape, blocks too large to stage: icp_query_pass_coop<3>, plus the tail from cap 25 on
    (21, 16385), (24, 40000), (25, 16385), (33, 32768), (64, 16385), (65, 40000), (100, 32767), (1000, 16385),
    # cap > 64: the bandwidth build at any query count
    (65, 300), (65, 16384), (100, 300), (1000, 300), (4096, 300), (4096, 16385),
]


@pytest.mark.gpu
@pytest.mark.parametrize("cap,nq", LOOP_CASES)
def test_loop_at_every_lookup_path(ctx, port, cap, nq):
    check_loop(ctx, port, cap, nq, seed=100 * cap + nq % 97)


VARIANT_CASES = [
    # latency shape: eight lanes per query, the plane of voxels of up to 64 points
    (NN27, 25, 2500), (PLANE, 9, 2500), (PLANE, 25, 2500), (PLANE, 64, 2500), (NN27 | PLANE, 16, 2500), (NN27 | PLANE, 100, 2500),
    # bandwidth shape below 32768 queries: one lane per query (block_closest, map_closest27)
    (PLANE, 25, 20000), (PLANE, 100, 20000), (NN27, 64, 20000), (NN27 | PLANE, 9, 20000),
    # from 32768 queries: coop_scan<1 / 2 / 3 / 0>
    (PLANE, 8, 40000), (PLANE, 16, 40000), (PLANE, 17, 40000), (PLANE, 25, 40000), (PLANE, 64, 40000), (PLANE, 100, 40000),
    (NN27, 100, 40000), (NN27 | PLANE, 25, 40000),
]


def check_variant(ctx, port, mode, cap, nq, seed, vox=1.0):
    rng = np.random.default_rng(seed)
    world = slab_world(rng, cap, vox)
    src = port.transform(port.se3_inv(port.se3_exp(TRUE_TWIST)), make_queries(rng, world, nq, vox))
    what = f"mode {mode}, cap {cap}, {nq} queries, voxel {vox}, seed {seed}"
    gm, om = ctx.VoxelHashMap(vox, 100.0 * vox, cap), port.Map(vox, 100.0 * vox, cap)
    try:
        gm.insert_points(world)
        om.insert(world)
        assert_map_coverage(gm.dump()[1], cap)
        om.set_mode(mode)
        if mode & NN27:
            got = gm.get_closest_neighbour(src, with_index=True, icp_mode=NN27)
            assert all(np.array_equal(a, b) for a, b in zip(got, om.closest(src, with_index=True))), what
            assert (got[2] < 0).any(), what
        max_iter = 60 if nq <= 16384 else (10 if nq < 32768 else 4)
        g = gm.icp(src, IDENT, 0.6 * vox, 0.2 * vox / 3, max_iter, 1e-4, trace=True, icp_mode=mode)
        r = port.icp(om, src, IDENT, 0.6 * vox, 0.2 * vox / 3, max_iter, 1e-4, trace=True)
        assert g["iters"] == r["iters"], what
        assert np.array_equal(g["ncorr"], r["ncorr"]) and 0 < r["ncorr"][0] < nq, what   # same correspondences (and planar voxels) every iteration
        np.testing.assert_allclose(g["hg"], r["hg"], rtol=0, atol=1e-11 * np.abs(r["hg"]).max(), err_msg=what)
        np.testing.assert_allclose(g["est"], r["est"], rtol=0, atol=1e-9, err_msg=what)
        np.testing.assert_allclose(g["pose"][4:], r["pose"][4:], rtol=0, atol=1e-8, err_msg=what)
        np.testing.assert_allclose(g["pose"][:4], r["pose"][:4], rtol=0, atol=1e-9, err_msg=what)
    finally:
        gm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode,cap,nq", VARIANT_CASES)
def test_variants_at_large_caps(ctx, port, mode, cap, nq):
    check_variant(ctx, port, mode, cap, nq, seed=200 * cap + 10 * mode + nq % 89)


def _sequence(voxel):
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    scene = synth.Scene(seed=11)
    traj = synth.loop_trajectory(9, radius=30.0, step=0.5)
    dense = voxel < 0.5
    return [synth.cast_scan(scene, traj[i], traj[i + 1], beams=64 if dense else 32, azimuth_steps=1800 if dense else 900, seed=60 + i)
            for i in range(8)]


@pytest.mark.gpu
@pytest.mark.parametrize("cap,voxel", [(21, 1.0), (25, 1.0), (64, 1.0), (65, 1.0), (100, 1.0), (25, 0.2)])
def test_odometry_at_large_caps(ctx, pkg, port, cap, voxel):
    """KissICP with the map update at large caps, plain and pipelined, against the C port scan by scan. A 4096-voxel initial table makes
    the map grow (rehash) with blocks of up to 2.4 kB. Cap 65 and 100 run the frame kernel's bandwidth build at a few thousand keypoints;
    voxel 0.2 m gives more than 16384 keypoints (icp_query_pass_coop<3> and the tail beside the map update)."""
    import torch
    seq = _sequence(voxel)
    cfg = dict(voxel_size=voxel, cap=cap, deskew=True, icp_max_iteration=80)
    k = ctx.KissICP(speculate=False, map_capacity_voxels=4096, **cfg)
    ref = []
    for s_ in seq:
        d, sr, p = k.register_frame(s_)
        ref.append((len(d), len(sr), p.copy(), k.stats.icp.iterations))
        assert (k.stats.n_down, k.stats.n_keypoints) == (len(d), len(sr))
    ref_dump = k.local_map().dump()
    k.close()
    if voxel < 0.5:
        assert max(r[1] for r in ref) > 16384
    if cap >= 25 and voxel >= 0.5:
        assert (ref_dump[1] > 24).any()
    kc = port.Kiss(max_range=100.0, **cfg)
    for i, s_ in enumerate(seq):
        dc, sc, pc = kc.register_cloud(np.ascontiguousarray(s_[:, :3]), s_[:, 3].astype(np.float64))
        assert (len(dc), len(sc), kc.last_iterations()) == ref[i][:2] + (ref[i][3],), i
        assert np.abs(ref[i][2][4:] - pc[4:]).max() < 1e-5 and np.abs(ref[i][2][:4] - pc[:4]).max() < 1e-6, i
    ok, oc, op = kc.map().dump()
    assert np.array_equal(ref_dump[0], ok) and np.array_equal(ref_dump[1], oc)
    np.testing.assert_allclose(ref_dump[2], op, rtol=0, atol=1e-6)
    staged = [torch.from_numpy(s_).cuda() for s_ in seq]
    torch.cuda.synchronize()
    k = ctx.KissICP(speculate=True, map_capacity_voxels=4096, **cfg)
    for i, t in enumerate(staged):
        if i + 1 < len(staged):
            k.hint_next_dev(staged[i + 1].data_ptr(), len(seq[i + 1]))
        p = k.register_frame_dev(t.data_ptr(), len(seq[i]))
        np.testing.assert_allclose(p, ref[i][2], rtol=0, atol=1e-9)
        assert (k.stats.n_down, k.stats.n_keypoints, k.stats.icp.iterations) == ref[i][:2] + (ref[i][3],), i
    dump = k.local_map().dump()
    assert np.array_equal(dump[0], ref_dump[0]) and np.array_equal(dump[1], ref_dump[1])
    np.testing.assert_allclose(dump[2], ref_dump[2], rtol=0, atol=1e-8)   # (deskewed with the device's twist: ~1e-15 from the host's)
    k.close()


@pytest.mark.gpu
def test_cap_4096_keeps_4096_of_5000(ctx, port):
    """META_COUNT_BITS = 13: a voxel offered 5000 points keeps its first 4096, and one ICP through such voxels equals the port."""
    rng = np.random.default_rng(4096)
    cells = np.array([[1, 1, 1], [2, 1, 1], [1, 2, 1], [3, 3, 1]])
    offered = [5000, 4097, 4096, 1234]
    world = rng.permutation(np.concatenate([c + rng.random((m, 3)) for c, m in zip(cells, offered)]))
    gm, om = ctx.VoxelHashMap(1.0, 100.0, 4096), port.Map(1.0, 100.0, 4096)
    gm.insert_points(world)
    om.insert(world)
    gk, gc, gp = gm.dump()
    nk, nc, npt = np_map_insert(world, 1.0, 4096)
    assert np.array_equal(gk, nk) and np.array_equal(gc, nc) and np.array_equal(gp, npt)
    assert sorted(gc.tolist()) == [1234, 4096, 4096, 4096]
    src = world[rng.integers(0, len(world), 2000)] + rng.normal(size=(2000, 3)) * 0.1
    g = gm.icp(src, IDENT, 0.3, 0.1 / 3, 10, 1e-4, trace=True)
    r = port.icp(om, src, IDENT, 0.3, 0.1 / 3, 10, 1e-4, trace=True)
    assert g["iters"] == r["iters"] and np.array_equal(g["ncorr"], r["ncorr"])
    np.testing.assert_allclose(g["hg"], r["hg"], rtol=0, atol=1e-12 * np.abs(r["hg"]).max())
    np.testing.assert_allclose(g["pose"], r["pose"], rtol=0, atol=1e-10)
    gm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [0, 4097])
def test_caps_outside_1_to_4096_are_rejected(ctx, pkg, cap):
    """limu_map_create checks 1 <= cap <= 4096; limu_odom_create checks only cap >= 1 and relies on limu_map_create for the upper bound."""
    with pytest.raises(pkg.LimuError) as e:
        ctx.VoxelHashMap(1.0, 100.0, cap)
    assert e.value.status == -1
    with pytest.raises(pkg.LimuError) as e:
        ctx.KissICP(cap=cap)
    assert e.value.status == -1


def _random_seeds_v():
    """4 seeds in the suite; LIMU_RANDOM_SEEDS_V="lo-hi" widens the campaign (profiles/r2_random_campaign.json)."""
    spec = os.environ.get("LIMU_RANDOM_SEEDS_V", "")
    if "-" in spec:
        lo, hi = spec.split("-")
        return range(int(lo), int(hi))
    return range(5000, 5004)


BOUNDARY_CAPS = [1, 4, 5, 8, 9, 12, 13, 16, 17, 20, 21, 24, 25, 64, 65, 4096]


@pytest.mark.gpu
@pytest.mark.parametrize("seed", _random_seeds_v())
def test_random_caps_query_counts_and_modes(ctx, port, seed):
    """Seeded random configurations: a cap log-uniform over 1 ... 4096 (half the draws a dispatch boundary or its neighbour), a query count
    class on either side of 16384 and 32768, a mode (mostly the reference's rules) and a voxel size; then the comparisons of the grid above."""
    rng = np.random.default_rng(seed)
    if rng.random() < 0.5:
        cap = int(rng.choice(BOUNDARY_CAPS))
    else:
        cap = int(np.exp(rng.uniform(0.0, np.log(4096.0))))
    nq = int(rng.choice([300, int(rng.integers(1000, 16385)), 16385, 32767, 32768, int(rng.integers(32768, 45000))]))
    if cap > 1000:
        nq = min(nq, 2000)
    mode = int(rng.choice([0, 0, 0, NN27, PLANE, NN27 | PLANE]))
    vox = float(rng.choice([0.5, 1.0, 2.0]))
    if mode == 0:
        check_loop(ctx, port, cap, nq, seed=seed, vox=vox)
    else:
        check_variant(ctx, port, mode, min(max(cap, 5) if mode & PLANE else cap, 200), nq, seed=seed, vox=vox)   # (a plane needs 5 points)
