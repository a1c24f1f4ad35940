"""LIMU_OPT_SPECULATE (the pipelined path: the next scan's deskew + downsampling behind the current scan's Gauss-Newton loop in one stream,
the map update beside it, the next scan's loop launched ahead of the caller) and the error behaviour of limu_odom_register_*: results must
not depend on hints / prefetches beyond rounding (the twist of a scan prepared ahead is taken by the device's log: bar 1e-9, far inside the
north-star tolerance of 1e-5 m / 1e-6 rad), whatever the caller does with the slots, the handle or the map between calls."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    return g.load_package()


@pytest.fixture(scope="module")
def ctx(pkg):
    c = pkg.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def scans(pkg):
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    scene = synth.Scene(seed=21)
    traj = synth.loop_trajectory(11, radius=30.0, step=0.7)
    return [synth.cast_scan(scene, traj[i], traj[i + 1], beams=16, azimuth_steps=700, seed=300 + i) for i in range(10)]


def plain_run(ctx, seq, **kw):
    k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=False, **kw)
    out = []
    for s in seq:
        d, sr, p = k.register_frame(s)
        out.append((d, sr, p.copy(), k.stats.icp.iterations))
    dump = k.local_map().dump()
    k.close()
    return out, dump


def close_enough(got, ref):
    assert len(got) == len(ref)
    for (gd, gs, gp, gi), (rd, rs, rp, ri) in zip(got, ref):
        assert gd.shape == rd.shape and gs.shape == rs.shape and gi == ri
        np.testing.assert_allclose(gd, rd, rtol=0, atol=1e-9)
        np.testing.assert_allclose(gs, rs, rtol=0, atol=1e-9)
        np.testing.assert_allclose(gp, rp, rtol=0, atol=1e-9)


def test_hinted_device_replay_matches_plain(ctx, pkg, scans):
    import torch
    ref, ref_dump = plain_run(ctx, scans)
    staged = [torch.from_numpy(s).cuda() for s in scans]
    torch.cuda.synchronize()
    k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=True)
    hits = 0
    for i, t in enumerate(staged):
        if i + 1 < len(staged):
            k.hint_next_dev(staged[i + 1].data_ptr(), len(scans[i + 1]))
        p = k.register_frame_dev(t.data_ptr(), len(scans[i]))
        hits += k.stats.reserved0
        np.testing.assert_allclose(p, ref[i][2], rtol=0, atol=1e-9)
        assert k.stats.icp.iterations == ref[i][3] and k.stats.n_down == len(ref[i][0]) and k.stats.n_keypoints == len(ref[i][1])
    assert hits == len(scans) - 1                       # every scan after the first was voxelized ahead of time
    dump = k.local_map().dump()
    assert np.array_equal(dump[0], ref_dump[0]) and np.array_equal(dump[1], ref_dump[1])
    np.testing.assert_allclose(dump[2], ref_dump[2], rtol=0, atol=1e-9)
    k.close()


def test_prefetched_host_replay_matches_plain(ctx, pkg, scans):
    ref, _ = plain_run(ctx, scans)
    pinned = [pkg.PinnedArray(s.shape, np.float32) for s in scans]
    for p, s in zip(pinned, scans):
        p.array[...] = s
    k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=True)
    got, hits = [], 0
    for i in range(len(scans)):
        if i + 1 < len(scans):
            k.prefetch(pinned[i + 1].array)
        d, sr, p = k.register_frame(pinned[i].array)
        hits += k.stats.reserved0
        got.append((d, sr, p.copy(), k.stats.icp.iterations))
    assert hits == len(scans) - 1
    close_enough(got, ref)
    k.close()
    for p in pinned:
        p.free()


def test_slot_reuse_and_abandoned_prefetches(ctx, pkg, scans):
    """ADVICE round 1: prefetch(B), register(A) speculates on B, prefetch(C), prefetch(D) -- D takes B's slot while the speculative launch
    may still read it, and has B's size. Registering D must give D's result, not B's."""
    eq = [s[: min(len(x) for x in scans)].copy() for s in scans]          # equal sizes: the dangerous case
    order = [0, 3, 4, 5, 2]                                               # A, D, then a few more
    ref, _ = plain_run(ctx, [eq[i] for i in order])
    pinned = [pkg.PinnedArray(s.shape, np.float32) for s in eq]
    for p, s in zip(pinned, eq):
        p.array[...] = s
    k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=True)
    got = []
    k.prefetch(pinned[1].array)                                           # B
    d, sr, p = k.register_frame(pinned[0].array)                          # A (speculates on B)
    got.append((d, sr, p.copy(), k.stats.icp.iterations))
    k.prefetch(pinned[2].array)                                           # C
    k.prefetch(pinned[3].array)                                           # D: evicts the oldest pending upload (B)
    for j in (3, 4, 5, 2):                                                # none of them is what was speculated on last
        d, sr, p = k.register_frame(pinned[j].array)
        got.append((d, sr, p.copy(), k.stats.icp.iterations))
    close_enough(got, ref)
    k.close()
    # a hint that is not followed (device-pointer entry)
    import torch
    staged = [torch.from_numpy(s).cuda() for s in eq[:4]]
    torch.cuda.synchronize()
    ref2, _ = plain_run(ctx, [eq[0], eq[2], eq[3]])
    k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=True)
    k.hint_next_dev(staged[1].data_ptr(), len(eq[1]))
    p0 = k.register_frame_dev(staged[0].data_ptr(), len(eq[0]))
    p2 = k.register_frame_dev(staged[2].data_ptr(), len(eq[2]))           # not the hinted scan: the speculation is discarded
    assert k.stats.reserved0 == 0
    k.set_speculate(False)
    k.hint_next_dev(staged[1].data_ptr(), len(eq[1]))                     # ignored now
    p3 = k.register_frame_dev(staged[3].data_ptr(), len(eq[3]))
    for g_, r_ in zip((p0, p2, p3), ref2):
        np.testing.assert_allclose(g_, r_[2], rtol=0, atol=1e-9)
    k.close()
    for p in pinned:
        p.free()


def test_out_of_range_point_commits_the_frame(ctx, pkg, scans):
    """ADVICE round 1: a device status error (a point whose voxel index leaves the packed key range, e.g. inf) used to return before the
    pose was pushed while the map already held the scan. Now the frame is committed and the error tells the caller points were left out."""
    bad = scans[1].copy()
    bad[100, 0] = np.inf
    clean = np.delete(scans[1], 100, axis=0)
    ref, ref_dump = plain_run(ctx, [scans[0], clean, scans[2], scans[3]])
    for spec in (False, True):
        k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=spec)
        pins = [pkg.PinnedArray(s.shape, np.float32) for s in (scans[0], bad, scans[2], scans[3])]
        for p, s in zip(pins, (scans[0], bad, scans[2], scans[3])):
            p.array[...] = s
        poses = []
        for i, p in enumerate(pins):
            if spec and i + 1 < len(pins):
                k.prefetch(pins[i + 1].array)
            if i == 1:
                with pytest.raises(pkg.LimuError) as e:
                    k.register_frame(p.array)
                assert e.value.status == -3
            else:
                poses.append(k.register_frame(p.array)[2].copy())
        allp = k.poses()
        assert len(allp) == 4                                             # the bad scan has a pose
        for i, r in enumerate(ref):
            np.testing.assert_allclose(allp[i], r[2], rtol=0, atol=1e-9)
        dump = k.local_map().dump()
        assert np.array_equal(dump[0], ref_dump[0]) and np.array_equal(dump[1], ref_dump[1])
        k.close()
        for p in pins:
            p.free()


def test_caller_touches_handle_and_map_between_pipelined_calls(ctx, pkg, scans):
    """The pipelined path launches the NEXT scan's Gauss-Newton loop before the caller asks for that scan. Whatever the caller does in between
    that the loop's inputs depend on -- get_adaptive_threshold (adds a sample to the threshold model, threshold.cpp:16-28), inserting into or
    pruning the local map -- must give what the plain path gives for the same sequence of calls: the loop that ran ahead is dropped."""
    import torch
    rng = np.random.default_rng(5)
    extra = [rng.uniform(-20, 20, size=(500, 3)) for _ in scans]

    def run(spec):
        staged = [torch.from_numpy(s).cuda() for s in scans]
        torch.cuda.synchronize()
        k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=spec)
        out = []
        for i, t in enumerate(staged):
            if spec and i + 1 < len(staged):
                k.hint_next_dev(staged[i + 1].data_ptr(), len(scans[i + 1]))
            p = k.register_frame_dev(t.data_ptr(), len(scans[i]))
            row = [p.copy(), k.stats.icp.iterations, k.stats.n_keypoints]
            if i in (3, 6):
                row.append(k.get_adaptive_threshold())            # (a) the getter with its side effect
            if i == 4:
                k.local_map().insert_points(extra[i])             # (b) the caller adds points to the map
            if i == 7:
                k.local_map().remove_points_from_far(p[4:7] + np.array([60.0, 0.0, 0.0]))   # (c) ... and prunes it around another origin
            if i == 5:
                assert k.local_map().size()[0] > 0                # (d) a read of the map is ordered behind the update in flight
            out.append(row)
        k.flush()
        dump = k.local_map().dump()
        k.close()
        return out, dump

    (a, da), (b, db) = run(False), run(True)
    for ra, rb in zip(a, b):
        assert ra[1] == rb[1] and ra[2] == rb[2]
        np.testing.assert_allclose(ra[0], rb[0], rtol=0, atol=1e-9)
        if len(ra) > 3:
            assert abs(ra[3] - rb[3]) < 1e-9
    assert np.array_equal(da[0], db[0]) and np.array_equal(da[1], db[1])
    np.testing.assert_allclose(da[2], db[2], rtol=0, atol=1e-9)


def test_flush_and_plain_calls_between_pipelined_calls(ctx, pkg, scans):
    """register_cloud / register_points go down the plain path: switching back and forth drops what was prepared and keeps the order of map updates."""
    import torch
    seq = scans[:8]

    def run(spec):
        staged = [torch.from_numpy(s).cuda() for s in seq]
        torch.cuda.synchronize()
        k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=spec)
        poses = []
        for i, t in enumerate(staged):
            if i in (2, 5):     # the same scan through the reference's own layout (float32 xyz records + float64 timestamps), plain path
                rec = np.ascontiguousarray(seq[i][:, :3])
                _, _, p = k.register_cloud(rec, 12, seq[i][:, 3].astype(np.float64))
            else:
                if spec and i + 1 < len(staged):
                    k.hint_next_dev(staged[i + 1].data_ptr(), len(seq[i + 1]))   # (before i = 1 and 4: a hint that the plain call then ignores)
                p = k.register_frame_dev(t.data_ptr(), len(seq[i]))
            poses.append(p.copy())
            if i == 3:
                k.flush()
        dump = k.local_map().dump()
        k.close()
        return poses, dump

    (a, da), (b, db) = run(False), run(True)
    for pa, pb in zip(a, b):
        np.testing.assert_allclose(pa, pb, rtol=0, atol=1e-9)
    assert np.array_equal(da[0], db[0]) and np.array_equal(da[1], db[1])


def test_prefetched_clouds_match_plain(ctx, pkg, scans):
    """limu_odom_prefetch_cloud + limu_odom_register_cloud (point records + FP64 timestamps, the reference's own layout) through the pipelined
    path against the plain path; one prefetch is not followed (the caller registers another cloud instead)."""
    seq = scans[:8]
    recs, tss = [], []
    for s_ in seq:
        r = pkg.PinnedArray((len(s_), 12), np.float32); r.array[...] = 0; r.array[:, :3] = s_[:, :3]
        t = pkg.PinnedArray((len(s_),), np.float64); t.array[...] = s_[:, 3]
        recs.append(r); tss.append(t)
    order = [0, 1, 2, 3, 5, 6, 7]          # cloud 4 is prefetched and then skipped

    def run(spec):
        k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=spec)
        out, hits = [], 0
        for j, i in enumerate(order):
            if spec and i + 1 < len(seq):
                k.prefetch_cloud(recs[i + 1].array, 48, tss[i + 1].array)
            d, sr, p = k.register_cloud(recs[i].array, 48, tss[i].array)
            hits += k.stats.reserved0
            out.append((d, sr, p.copy(), k.stats.icp.iterations))
        dump = k.local_map().dump()
        k.close()
        return out, dump, hits

    (a, da, _), (b, db, hits) = run(False), run(True)
    assert hits == len(order) - 2                      # every cloud but the first and the one after the skipped prefetch ran ahead
    close_enough(b, a)
    assert np.array_equal(da[0], db[0]) and np.array_equal(da[1], db[1])
    for x in recs + tss:
        x.free()


def test_two_pipelined_handles_on_one_context(ctx, pkg, scans):
    """Two odometry handles of one context, calls interleaved: each has its own pipe stream, result block and barrier words, so their loop
    kernels may overlap each other and the other handle's map update; results must be those of the handles run alone."""
    import torch
    seq_a, seq_b = scans[:9], [np.ascontiguousarray(s[::2]) for s in scans[1:10]]   # (different scans, different sizes)
    dev_a = [torch.from_numpy(s).cuda() for s in seq_a]
    dev_b = [torch.from_numpy(s).cuda() for s in seq_b]
    torch.cuda.synchronize()

    def alone(devs, seq):
        k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=False)
        out = [(k.register_frame_dev(t.data_ptr(), len(s)).copy(), k.stats.icp.iterations) for t, s in zip(devs, seq)]
        dump = k.local_map().dump()
        k.close()
        return out, dump

    ref_a, ref_b = alone(dev_a, seq_a), alone(dev_b, seq_b)
    ka = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=True)
    kb = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=True)
    got_a, got_b = [], []
    for i in range(len(seq_a)):
        if i + 1 < len(seq_a):
            ka.hint_next_dev(dev_a[i + 1].data_ptr(), len(seq_a[i + 1]))
            kb.hint_next_dev(dev_b[i + 1].data_ptr(), len(seq_b[i + 1]))
        got_a.append((ka.register_frame_dev(dev_a[i].data_ptr(), len(seq_a[i])).copy(), ka.stats.icp.iterations))
        got_b.append((kb.register_frame_dev(dev_b[i].data_ptr(), len(seq_b[i])).copy(), kb.stats.icp.iterations))
    for (got, k), (ref, ref_dump) in (((got_a, ka), ref_a), ((got_b, kb), ref_b)):
        for (gp, gi), (rp, ri) in zip(got, ref):
            assert gi == ri
            np.testing.assert_allclose(gp, rp, rtol=0, atol=1e-9)
        dump = k.local_map().dump()
        assert np.array_equal(dump[0], ref_dump[0]) and np.array_equal(dump[1], ref_dump[1])
        k.close()


@pytest.mark.parametrize("cap,voxel", [(10, 1.0), (20, 1.0), (3, 1.0), (10, 0.35)])
def test_plain_path_matches_port_across_caps_and_keypoint_counts(ctx, pkg, cap, voxel):
    """The plain path at caps 3, 10 and 20 against the C port scan by scan (cloud sizes and iteration counts equal, the clouds bit-exact
    while the deskew gate is closed, poses to the north-star tolerance of 1e-5 m / 1e-6 rad), and the pipelined path on the same sequence
    against the plain path (poses 1e-9, the same map). Voxel 0.35 m makes > 3840 keypoints per scan, and with the decimated first scan
    the launch hint is small: more than 4096 IQR candidates then go through the one-CTA select behind a whole-grid barrier."""
    import torch
    import oracle
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    scene = synth.Scene(seed=5)
    traj = synth.loop_trajectory(8, radius=30.0, step=0.5)
    dense = voxel < 1.0
    seq = [synth.cast_scan(scene, traj[i], traj[i + 1], beams=64 if dense else 32, azimuth_steps=2000 if dense else 900, seed=40 + i) for i in range(7)]
    if dense:
        seq[0] = np.ascontiguousarray(seq[0][::16])
    cfg = dict(voxel_size=voxel, cap=cap, deskew=True, icp_max_iteration=80)
    k = ctx.KissICP(speculate=False, **cfg)
    ref = []
    for s_ in seq:
        d, sr, p = k.register_frame(s_)
        ref.append((d, sr, p.copy(), k.stats.icp.iterations))
    ref_dump = k.local_map().dump()
    k.close()
    if dense:
        assert max(len(r[1]) for r in ref) > 3840
    kc = oracle.load_port().Kiss(max_range=100.0, **cfg)
    for i, s_ in enumerate(seq):
        dc, sc, pc = kc.register_cloud(np.ascontiguousarray(s_[:, :3]), s_[:, 3].astype(np.float64))
        assert (len(dc), len(sc), kc.last_iterations()) == (len(ref[i][0]), len(ref[i][1]), ref[i][3]), i
        if i < 3:   # deskew gate closed: identical inputs
            assert np.array_equal(dc, ref[i][0]) and np.array_equal(sc, ref[i][1]), i
        assert np.abs(ref[i][2][4:] - pc[4:]).max() < 1e-5 and np.abs(ref[i][2][:4] - pc[:4]).max() < 1e-6, i
    staged = [torch.from_numpy(s_).cuda() for s_ in seq]
    torch.cuda.synchronize()
    k = ctx.KissICP(speculate=True, **cfg)
    for i, t in enumerate(staged):
        if i + 1 < len(staged):
            k.hint_next_dev(staged[i + 1].data_ptr(), len(seq[i + 1]))
        p = k.register_frame_dev(t.data_ptr(), len(seq[i]))
        np.testing.assert_allclose(p, ref[i][2], rtol=0, atol=1e-9)
        assert k.stats.icp.iterations == ref[i][3] and k.stats.n_down == len(ref[i][0]) and k.stats.n_keypoints == len(ref[i][1]), i
    dump = k.local_map().dump()
    assert np.array_equal(dump[0], ref_dump[0]) and np.array_equal(dump[1], ref_dump[1])
    np.testing.assert_allclose(dump[2], ref_dump[2], rtol=0, atol=1e-8)
    k.close()


def test_plain_path_degenerate_inputs(ctx, pkg):
    """Empty map on the first scan (ICP returns init_guess, registration.cpp:99-100), one-point and empty keypoint clouds. The retired
    option LIMU_OPT_CLUSTER_LOOP (2) is still accepted and changes nothing."""
    runs = []
    for retired_option in (False, True):
        k = ctx.KissICP(voxel_size=1.0, cap=10, deskew=False, icp_max_iteration=20, speculate=False)
        if retired_option:
            assert pkg.lib().limu_odom_set_option(k.h, 2, 1) == 0   # LIMU_OK
        one = np.array([[10.0, 2.0, 1.0, 0.5]], np.float32)
        d, sr, p = k.register_frame(one)
        assert len(d) == 1 and len(sr) == 1 and np.array_equal(p, [0, 0, 0, 1, 0, 0, 0])
        rows = [(d, sr, p.copy())]
        d, sr, p = k.register_frame(one)                       # map now holds that point
        assert len(d) == 1 and len(sr) == 1 and np.abs(p[4:]).max() < 1e-9
        rows.append((d, sr, p.copy()))
        two = np.array([[10.0, 2.0, 1.0, 0.5], [30.0, -4.0, 2.0, 0.7]], np.float32)
        d, sr, p = k.register_frame(two)
        assert len(d) == 2 and 1 <= len(sr) <= 2
        assert k.local_map().size()[0] == 2
        rows.append((d, sr, p.copy()))
        runs.append(rows)
        k.close()
    for a, b in zip(*runs):
        assert all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("voxel,beams,az", [(0.3, 64, 2000), (0.1, 64, 2000)])
def test_pipelined_matches_plain_when_the_loop_needs_every_sm(ctx, pkg, voxel, beams, az):
    """Small voxels = many keypoints: at ~5 k keypoints the latency shape of the loop kernel asks for one CTA on EVERY SM, above 16 384 the
    bandwidth shape for several per SM, and the scan's k_voxelize for one 1024-thread CTA per SM. A cooperative grid that needs the whole GPU
    must not wait for the SM a k_gate thread of the same pipeline sits on (that was a 5-second stall with a wrong map state behind it at
    configs[2]'s size): the pipelined path leaves GATE_SLACK_SMS SMs free. Hinted replay against the plain path, timing checked."""
    import time
    import torch
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    scene = synth.Scene(seed=5, n_boxes=60, n_cyl=30)
    traj = synth.loop_trajectory(9, radius=30.0, step=0.5)
    seq = [synth.cast_scan(scene, traj[i], traj[i + 1], beams=beams, azimuth_steps=az, seed=900 + i, device="cuda:0") for i in range(8)]
    ref, _ = plain_run(ctx, seq, voxel_size=voxel, cap=20)
    nk = max(len(r[1]) for r in ref)
    assert nk > (16384 if voxel < 0.2 else 4200), nk          # the regime this test is about
    # ... which is also where the grid-wide IQR ranking keeps its candidate lists in dynamic shared memory (more than 4096 of them; 16384 at
    # most, beyond that one CTA selects): the C port pins the filter's output and the poses
    import oracle
    kc = oracle.load_port().Kiss(voxel_size=voxel, max_range=100.0, cap=20, deskew=True, icp_max_iteration=60)
    for i, s in enumerate(seq):
        dc, sc, pc = kc.register_cloud(np.ascontiguousarray(s[:, :3]), s[:, 3].astype(np.float64))
        assert (len(dc), len(sc), kc.last_iterations()) == (len(ref[i][0]), len(ref[i][1]), ref[i][3]), i
        assert np.array_equal(sc, ref[i][1]) or i >= 3          # keypoint cloud bit-exact while the deskew gate is closed (identical inputs)
        assert np.abs(ref[i][2][4:] - pc[4:]).max() < 1e-5 and np.abs(ref[i][2][:4] - pc[:4]).max() < 1e-6, i
    staged = [torch.from_numpy(s).cuda() for s in seq]
    torch.cuda.synchronize()
    k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=True, voxel_size=voxel, cap=20)
    worst = 0.0
    for i, t in enumerate(staged):
        if i + 1 < len(staged):
            k.hint_next_dev(staged[i + 1].data_ptr(), len(seq[i + 1]))
        t0 = time.perf_counter()
        p = k.register_frame_dev(t.data_ptr(), len(seq[i]))
        worst = max(worst, time.perf_counter() - t0) if i > 0 else worst
        np.testing.assert_allclose(p, ref[i][2], rtol=0, atol=1e-9)
        assert k.stats.icp.iterations == ref[i][3] and k.stats.n_down == len(ref[i][0]) and k.stats.n_keypoints == len(ref[i][1])
    k.close()
    assert worst < 1.0, f"a call took {worst:.2f} s: the gate and a full-GPU cooperative launch waited for each other"


def test_ragged_sequence_through_the_pipelined_path(ctx, pkg):
    """Scan sizes that change from call to call -- 1 point to 4 M points, so every per-scan buffer is re-allocated while earlier launches are
    in flight and the launch shapes change between scans (one tile, many tiles per CTA, latency and bandwidth shape of the loop) -- hinted
    replay on the pipelined path against the plain path (counts and iterations equal, poses 1e-9) and the C port (north-star tolerance)."""
    import torch
    import oracle
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    scene = synth.Scene(seed=9, n_boxes=40, n_cyl=20)
    sizes = [30000, 120000, 300000, 8000, 4194304, 1000, 1048576, 1, 57, 2, 40000]
    n_pinned = 7   # a one-point scan makes the normal equations singular: there the compiled reference and its C port already disagree with each
                   # other (LDLT of a rank-3 matrix), so from that scan on only the pipelined path against the plain path is checked
    traj = synth.loop_trajectory(len(sizes) + 1, radius=30.0, step=0.4)
    rng = np.random.default_rng(4)
    seq = []
    for i, n in enumerate(sizes):
        beams, az = (512, 11059) if n > 2_000_000 else (256, 5530) if n > 100_000 else (64, 2000)   # (rays that hit nothing are dropped: cast more than needed)
        s = synth.cast_scan(scene, traj[i], traj[i + 1], beams=beams, azimuth_steps=az, seed=700 + i, device="cuda:0")
        assert len(s) >= n, (len(s), n)
        keep = np.sort(rng.choice(len(s), size=n, replace=False)) if n < len(s) else np.arange(n)
        seq.append(np.ascontiguousarray(s[keep]))
    ref, ref_dump = plain_run(ctx, seq, cap=10)
    port = oracle.load_port()
    kc = port.Kiss(voxel_size=1.0, max_range=100.0, cap=10, deskew=True, icp_max_iteration=60)
    staged = [torch.from_numpy(s).cuda() for s in seq]
    torch.cuda.synchronize()
    k = ctx.KissICP(deskew=True, icp_max_iteration=60, speculate=True, cap=10)
    for i, t in enumerate(staged):
        if i + 1 < len(staged):
            k.hint_next_dev(staged[i + 1].data_ptr(), len(seq[i + 1]))
        p = k.register_frame_dev(t.data_ptr(), len(seq[i]))
        np.testing.assert_allclose(p, ref[i][2], rtol=0, atol=1e-9, err_msg=f"scan {i} ({sizes[i]} points)")
        assert k.stats.icp.iterations == ref[i][3] and k.stats.n_down == len(ref[i][0]) and k.stats.n_keypoints == len(ref[i][1]), (i, sizes[i])
        if i >= n_pinned:
            continue
        dc, sc, pc = kc.register_cloud(np.ascontiguousarray(seq[i][:, :3]), seq[i][:, 3].astype(np.float64))
        assert (len(dc), len(sc), kc.last_iterations()) == (k.stats.n_down, k.stats.n_keypoints, k.stats.icp.iterations), (i, sizes[i])
        assert np.abs(p[4:] - pc[4:]).max() < 1e-5 and np.abs(p[:4] - pc[:4]).max() < 1e-6, (i, sizes[i])
    dump = k.local_map().dump()
    assert np.array_equal(dump[0], ref_dump[0]) and np.array_equal(dump[1], ref_dump[1])
    np.testing.assert_allclose(dump[2], ref_dump[2], rtol=0, atol=1e-9)
    k.close()


def _random_seeds():
    """16 seeds in the suite; LIMU_RANDOM_SEEDS="lo-hi" widens the campaign (profiles/r2_random_campaign.json: seeds 16..255 on one B200)."""
    import os
    spec = os.environ.get("LIMU_RANDOM_SEEDS", "")
    if "-" in spec:
        lo, hi = spec.split("-")
        return range(int(lo), int(hi))
    return range(16)


@pytest.mark.parametrize("seed", _random_seeds())
def test_random_configurations_pipelined_vs_plain_vs_port(ctx, pkg, seed):
    """Seeded random configurations (voxel size, cap, deskew gate, scan shape, iteration cap, registration variant): hinted replay on the
    pipelined path against the plain path (1e-9) and against the C port (counts and iterations equal, north-star pose tolerance)."""
    import torch
    import oracle
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    rng = np.random.default_rng(1000 + seed)
    voxel = float(rng.choice([0.25, 0.5, 1.0, 2.0]))
    cap = int(rng.choice([1, 3, 10, 20]))
    deskew = bool(rng.integers(0, 2))
    mode = int(rng.choice([0, 0, 0, 3]))
    beams = int(rng.choice([8, 16, 32, 64]))
    az = int(rng.integers(300, 2500))
    max_iter = int(rng.choice([5, 60, 500]))
    step = float(rng.choice([0.1, 0.5, 1.0]))
    scene = synth.Scene(seed=50 + seed, n_boxes=int(rng.integers(10, 80)), n_cyl=int(rng.integers(5, 40)))
    traj = synth.loop_trajectory(8, radius=30.0, step=step)
    seq = [synth.cast_scan(scene, traj[i], traj[i + 1], beams=beams, azimuth_steps=az, seed=40 * seed + i, device="cuda:0") for i in range(7)]
    cfg = dict(voxel_size=voxel, cap=cap, deskew=deskew, icp_max_iteration=max_iter, icp_mode=mode)
    what = f"seed {seed}: {cfg}, {beams} x {az}, {step} m/scan"
    k = ctx.KissICP(speculate=False, **cfg)
    ref = []
    for s in seq:
        d, sr, p = k.register_frame(s)
        ref.append((d, sr, p.copy(), k.stats.icp.iterations))
    k.close()
    kc = oracle.load_port().Kiss(voxel_size=voxel, max_range=100.0, cap=cap, deskew=deskew, icp_max_iteration=max_iter)
    if mode:
        kc.set_mode(mode)
    staged = [torch.from_numpy(s).cuda() for s in seq]
    torch.cuda.synchronize()
    k = ctx.KissICP(speculate=True, **cfg)
    for i, t in enumerate(staged):
        if i + 1 < len(staged):
            k.hint_next_dev(staged[i + 1].data_ptr(), len(seq[i + 1]))
        p = k.register_frame_dev(t.data_ptr(), len(seq[i]))
        np.testing.assert_allclose(p, ref[i][2], rtol=0, atol=1e-9, err_msg=f"{what}, scan {i}")
        assert (k.stats.icp.iterations, k.stats.n_down, k.stats.n_keypoints) == (ref[i][3], len(ref[i][0]), len(ref[i][1])), (what, i)
        dc, sc, pc = kc.register_cloud(np.ascontiguousarray(seq[i][:, :3]), seq[i][:, 3].astype(np.float64))
        assert (len(dc), len(sc), kc.last_iterations()) == (k.stats.n_down, k.stats.n_keypoints, k.stats.icp.iterations), (what, i)
        assert np.abs(p[4:] - pc[4:]).max() < 1e-5 and np.abs(p[:4] - pc[:4]).max() < 1e-6, (what, i, p, pc)
    k.close()


def _random_seeds_b():
    """4 seeds in the suite; LIMU_RANDOM_SEEDS_B="lo-hi" widens the campaign (profiles/r2_random_campaign.json)."""
    import os
    spec = os.environ.get("LIMU_RANDOM_SEEDS_B", "")
    if "-" in spec:
        lo, hi = spec.split("-")
        return range(int(lo), int(hi))
    return range(1000, 1004)


@pytest.mark.parametrize("seed", _random_seeds_b())
def test_random_configurations_with_eviction_and_map_growth(ctx, pkg, seed):
    """Second family of seeded random configurations: a short max_range (the eviction sweep removes voxels on every scan), long steps between
    scans, and a voxel table that starts small (map_capacity_voxels: the table is re-hashed while the sequence runs). Pipelined path with hints
    against the plain path (poses 1e-9, final map: same voxels in the same creation order) and against the C port (counts, iterations, poses)."""
    import torch
    import oracle
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    rng = np.random.default_rng(seed)
    voxel = float(rng.choice([0.25, 0.5, 1.0]))
    cap = int(rng.choice([3, 10, 20]))
    deskew = bool(rng.integers(0, 2))
    mode = int(rng.choice([0, 0, 0, 3]))
    beams = int(rng.choice([16, 32]))
    az = int(rng.integers(500, 2000))
    max_iter = int(rng.choice([30, 100]))
    step = float(rng.choice([1.0, 2.0, 4.0]))
    max_range = float(rng.choice([15.0, 30.0, 60.0]))
    capacity = int(rng.choice([0, 512, 4096]))
    scene = synth.Scene(seed=seed, n_boxes=int(rng.integers(10, 80)), n_cyl=int(rng.integers(5, 40)))
    n = 10
    traj = synth.loop_trajectory(n + 1, radius=30.0, step=step)
    seq = [synth.cast_scan(scene, traj[i], traj[i + 1], beams=beams, azimuth_steps=az, seed=40 * seed + i, device="cuda:0") for i in range(n)]
    cfg = dict(voxel_size=voxel, max_range=max_range, cap=cap, deskew=deskew, icp_max_iteration=max_iter, icp_mode=mode, map_capacity_voxels=capacity)
    what = f"seed {seed}: {cfg}, {beams} x {az}, {step} m/scan"
    k = ctx.KissICP(speculate=False, **cfg)
    ref = []
    for s in seq:
        d, sr, p = k.register_frame(s)
        ref.append((d, sr, p.copy(), k.stats.icp.iterations))
    ref_dump = k.local_map().dump()
    k.close()
    kc = oracle.load_port().Kiss(voxel_size=voxel, max_range=max_range, cap=cap, deskew=deskew, icp_max_iteration=max_iter)
    if mode:
        kc.set_mode(mode)
    staged = [torch.from_numpy(s).cuda() for s in seq]
    torch.cuda.synchronize()
    k = ctx.KissICP(speculate=True, **cfg)
    for i, t in enumerate(staged):
        if i + 1 < len(staged):
            k.hint_next_dev(staged[i + 1].data_ptr(), len(seq[i + 1]))
        p = k.register_frame_dev(t.data_ptr(), len(seq[i]))
        np.testing.assert_allclose(p, ref[i][2], rtol=0, atol=1e-9, err_msg=f"{what}, scan {i}")
        assert (k.stats.icp.iterations, k.stats.n_down, k.stats.n_keypoints) == (ref[i][3], len(ref[i][0]), len(ref[i][1])), (what, i)
        dc, sc, pc = kc.register_cloud(np.ascontiguousarray(seq[i][:, :3]), seq[i][:, 3].astype(np.float64))
        assert (len(dc), len(sc), kc.last_iterations()) == (k.stats.n_down, k.stats.n_keypoints, k.stats.icp.iterations), (what, i)
        assert np.abs(p[4:] - pc[4:]).max() < 1e-5 and np.abs(p[:4] - pc[:4]).max() < 1e-6, (what, i, p, pc)
    dump = k.local_map().dump()
    assert np.array_equal(dump[0], ref_dump[0]) and np.array_equal(dump[1], ref_dump[1]), what
    np.testing.assert_allclose(dump[2], ref_dump[2], rtol=0, atol=1e-9, err_msg=what)
    pd = kc.map().dump()
    if mode == 0:   # (poses equal to ~1e-15 under the reference's rules: the port's map holds the same voxels after the last eviction)
        assert np.array_equal(pd[0], dump[0]) and np.array_equal(pd[1], dump[1]), (what, len(pd[0]), len(dump[0]))
    k.close()


def _random_seeds_c():
    """4 seeds in the suite; LIMU_RANDOM_SEEDS_C="lo-hi" widens the campaign (profiles/r2_random_campaign.json)."""
    import os
    spec = os.environ.get("LIMU_RANDOM_SEEDS_C", "")
    if "-" in spec:
        lo, hi = spec.split("-")
        return range(int(lo), int(hi))
    return range(2000, 2004)


@pytest.mark.parametrize("seed", _random_seeds_c())
def test_random_configurations_through_the_host_pointer_entries(ctx, pkg, seed):
    """Third family: the entries a host application calls -- limu_odom_register_frame (packed x, y, z, t; pinned or pageable memory) with
    limu_odom_prefetch, or limu_odom_register_cloud (48-byte point records + FP64 stamps) with limu_odom_prefetch_cloud -- on ragged scan
    sizes, with a prefetch left out now and then. Pipelined against plain (1e-9, same clouds, same final map) and against the C port."""
    import oracle
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    rng = np.random.default_rng(seed)
    voxel = float(rng.choice([0.5, 1.0, 2.0]))
    cap = int(rng.choice([1, 10, 20]))
    deskew = bool(rng.integers(0, 2))
    beams = int(rng.choice([8, 16, 32]))
    az = int(rng.integers(300, 1800))
    max_iter = int(rng.choice([30, 100]))
    step = float(rng.choice([0.1, 0.5, 1.0]))
    cloud_api = bool(rng.integers(0, 2))
    pinned = bool(rng.integers(0, 2))
    scene = synth.Scene(seed=seed, n_boxes=int(rng.integers(10, 80)), n_cyl=int(rng.integers(5, 40)))
    n = 8
    traj = synth.loop_trajectory(n + 1, radius=30.0, step=step)
    seq = []
    for i in range(n):
        s = synth.cast_scan(scene, traj[i], traj[i + 1], beams=beams, azimuth_steps=az, seed=40 * seed + i, device="cuda:0")
        seq.append(np.ascontiguousarray(s[: max(1, int(len(s) * rng.uniform(0.4, 1.0)))]))   # ragged sizes
    skip = set(int(x) for x in np.nonzero(rng.random(n) < 0.2)[0])                           # scans whose prefetch is left out
    cfg = dict(voxel_size=voxel, cap=cap, deskew=deskew, icp_max_iteration=max_iter)
    what = f"seed {seed}: {cfg}, {beams} x {az}, {step} m/scan, {'cloud records' if cloud_api else 'packed scans'}, {'pinned' if pinned else 'pageable'}, no prefetch of {sorted(skip)}"
    bufs = []

    def hold(shape, dtype, fill):
        if pinned:
            b = pkg.PinnedArray(shape, dtype)
            bufs.append(b)
            b.array[...] = fill
            return b.array
        return np.ascontiguousarray(fill, dtype=dtype)

    if cloud_api:
        recs, tss = [], []
        for s in seq:
            r = np.zeros((len(s), 12), np.float32)
            r[:, :3] = s[:, :3]
            r[:, 4:] = rng.random((len(s), 8), dtype=np.float32)      # intensity / normal / curvature fields: must be ignored
            recs.append(hold(r.shape, np.float32, r))
            tss.append(hold((len(s),), np.float64, s[:, 3].astype(np.float64)))
    else:
        packed = [hold(s.shape, np.float32, s) for s in seq]

    def run(spec):
        k = ctx.KissICP(speculate=spec, **cfg)
        out = []
        for i in range(n):
            if spec and i + 1 < n and (i + 1) not in skip:
                if cloud_api:
                    k.prefetch_cloud(recs[i + 1], 48, tss[i + 1])
                else:
                    k.prefetch(packed[i + 1])
            d, sr, p = k.register_cloud(recs[i], 48, tss[i]) if cloud_api else k.register_frame(packed[i])
            out.append((d, sr, p.copy(), k.stats.icp.iterations))
        dump = k.local_map().dump()
        k.close()
        return out, dump

    (a, da), (b, db) = run(False), run(True)
    close_enough(b, a)
    assert np.array_equal(da[0], db[0]) and np.array_equal(da[1], db[1]), what
    kc = oracle.load_port().Kiss(voxel_size=voxel, max_range=100.0, cap=cap, deskew=deskew, icp_max_iteration=max_iter)
    for i, s in enumerate(seq):
        dc, sc, pc = kc.register_cloud(np.ascontiguousarray(s[:, :3]), s[:, 3].astype(np.float64))
        assert (len(dc), len(sc), kc.last_iterations()) == (len(b[i][0]), len(b[i][1]), b[i][3]), (what, i)
        assert np.abs(b[i][2][4:] - pc[4:]).max() < 1e-5 and np.abs(b[i][2][:4] - pc[:4]).max() < 1e-6, (what, i)
    for x in bufs:
        x.free()
