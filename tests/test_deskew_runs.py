"""P1 of k_voxelize computes one deskew transform per run of equal timestamp bits in a 1024-point tile (a shared table of VX_RUNS poses) and
falls back to one transform per point for a tile with more runs. Both must give exactly the frames of the per-point computation: the same
operations on the same operands. Checked bit for bit through the odometry handle:

* plain path (k_voxelize_full, twist taken on the host): the handle's downsampled and keypoint clouds against limu_deskew[_cloud] with the
  handle's last two poses (the same host log), then limu_voxel_downsample at 0.5 v and 1.5 v and limu_iqr_filter -- the per-point kernels;
* pipelined path (k_voxelize_lean beside the map update, twist left on the device by the loop kernel, which the ABI cannot hand out): the same
  scan twice, once with its timestamps as they are and once with every +0.0 of it turned into an alternation of +0.0 / -0.0 -- the same
  value, so the same transform, but a run per point, which sends those tiles down the per-point path. The two runs' clouds must be equal.

Every case asserts which branch its tiles take (the run count per tile, against VX_RUNS as the kernel source defines it)."""
import os
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = open(os.path.join(ROOT, "lidar-imu-slam_b200", "csrc", "voxelize.cu")).read()
R = int(re.search(r"constexpr int VX_RUNS = (\d+);", SRC).group(1))
BLOCK = int(re.search(r"constexpr int VX_BLOCK = (\d+);", SRC).group(1))
VOXEL = 1.0


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
def world(pkg):
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    scene = synth.Scene(seed=42)
    traj = synth.loop_trajectory(6, radius=30.0, step=1.0)
    warm = [synth.cast_scan(scene, traj[i], traj[i + 1], beams=16, azimuth_steps=500, seed=900 + i) for i in range(3)]
    full = synth.cast_scan(scene, traj[3], traj[4], seed=903)          # the bench's sensor: 64 beams x 2000 azimuth steps
    return synth, warm, full


def tiles_runs(t):
    """Runs of equal timestamp bits in each tile, as P1 counts them."""
    b = np.ascontiguousarray(t, np.float64).view(np.uint64)
    head = np.ones(len(b), bool)
    head[1:] = b[1:] != b[:-1]
    head[::BLOCK] = True
    return np.add.reduceat(head.astype(np.int64), np.arange(0, len(b), BLOCK))


def branches(t):
    r = tiles_runs(t)
    return {"table" if x <= R else "per-point" for x in r}


def runs_of_length(n, L):
    return (np.arange(n) // L).astype(np.float64) / (n // L + 1)


def runs_per_tile(n, k):
    """Exactly k runs in every full tile."""
    j = np.arange(n)
    ids = (j // BLOCK) * k + ((j % BLOCK) * k) // BLOCK
    return ids.astype(np.float64) / (ids.max() + 1)


def case_times(name, n, own_t, rng):
    if name == "bench":                # the scan's own times: 64 beams per azimuth step at 128 k points and above; a subsample has fewer
        return own_t, {"table"} if n >= 100000 or n <= R else {"per-point"}
    if name == "distinct":
        return (np.arange(n) + 0.5) / n, {"per-point"}
    if name.startswith("run"):
        L = int(name[3:])
        return runs_of_length(n, L), {"per-point"} if L == 1 else {"table"}
    if name == "R":
        return runs_per_tile(n, R), {"table"}
    if name == "R+1":
        return runs_per_tile(n, R + 1), {"per-point"}
    if name == "unsorted":
        v = np.repeat(np.arange(n // 64 + 1) / (n // 64 + 1), 64)[:n]
        return rng.permutation(v), {"per-point"}
    if name == "signed_zeros":        # +0 / -0 / the smallest denormal in runs of 100, then sorted times: equal values, distinct bits
        t = runs_of_length(n, 64)
        for k, z in enumerate((0.0, -0.0, 5e-324, -5e-324)):
            t[k * 100:(k + 1) * 100] = z
        return t, {"table"}
    raise KeyError(name)


CASES = [("bench", 128000), ("distinct", 5000), ("run1", 3000), ("run31", 20000), ("run32", 20000), ("run33", 20000), ("run1023", 20000),
         ("run1024", 20000), ("run1025", 20000), ("R", 10240), ("R+1", 10240), ("unsorted", 20000), ("signed_zeros", 30000),
         ("bench", 20), ("bench", 3000), ("bench", 160000), ("distinct", 160000)]


def scan_of(synth, full, n, name, seed):
    s = synth.pad_scan(full, n, seed=seed).copy()
    t, expect = case_times(name, n, s[:, 3].astype(np.float64), np.random.default_rng(seed))
    return s, t, expect


def plain_handle(ctx, warm):
    k = ctx.KissICP(voxel_size=VOXEL, deskew=True, icp_max_iteration=60, speculate=False)
    for w in warm:
        k.register_frame(w)
    return k


def reference(ctx, k, frame_fn):
    T = k.poses()
    frame = frame_fn(T[-2], T[-1])
    down = ctx.voxel_downsample(frame, 0.5 * VOXEL)
    src0 = ctx.voxel_downsample(down, 1.5 * VOXEL)
    return down, ctx.iqr_processing(src0)


@pytest.mark.parametrize("name,n", CASES)
def test_plain_path_equals_per_point_deskew_float4(ctx, world, name, n):
    synth, warm, full = world
    s, t, expect = scan_of(synth, full, n, name, seed=n)
    s[:, 3] = t.astype(np.float32)
    assert branches(s[:, 3]) == expect, (name, tiles_runs(s[:, 3]))
    k = plain_handle(ctx, warm)
    ref_down, ref_kp = reference(ctx, k, lambda T0, T1: ctx.deskew_scan(s, T0, T1))
    down, kp, _ = k.register_frame(s)
    assert k.stats.deskewed == 1
    assert np.array_equal(down, ref_down) and np.array_equal(kp, ref_kp), name
    k.close()


@pytest.mark.parametrize("name,n", [("bench", 128000), ("distinct", 20000), ("run33", 20000), ("R", 10240), ("R+1", 10240), ("unsorted", 20000),
                                    ("signed_zeros", 30000), ("bench", 160000)])
def test_plain_path_equals_per_point_deskew_records(ctx, world, name, n):
    """Mode 1: 48-byte point records + FP64 timestamps (the FP64 times are not rounded to float: runs are of the double bits)."""
    synth, warm, full = world
    s, t, expect = scan_of(synth, full, n, name, seed=n + 1)
    assert branches(t) == expect, (name, tiles_runs(t))
    rec = np.zeros((n, 12), np.float32)
    rec[:, :3] = s[:, :3]
    k = plain_handle(ctx, warm)
    ref_down, ref_kp = reference(ctx, k, lambda T0, T1: ctx.deskew_cloud(rec, 48, t, T0, T1))
    down, kp, _ = k.register_cloud(rec, 48, t)
    assert k.stats.deskewed == 1
    assert np.array_equal(down, ref_down) and np.array_equal(kp, ref_kp), name
    k.close()


def test_nonfinite_timestamps_fail_like_the_per_point_path(ctx, world, pkg):
    """NaN / +-inf timestamps give non-finite frames: the handle reports the out-of-range voxel key as the per-point path does."""
    synth, warm, full = world
    s = synth.pad_scan(full, 20000, seed=5).copy()
    s[:, 3] = runs_of_length(20000, 64)
    s[1000:1010, 3] = np.nan
    s[3000:3010, 3] = np.inf
    s[5000:5010, 3] = -np.inf
    assert branches(s[:, 3]) == {"table"}
    k = plain_handle(ctx, warm)
    T = k.poses()
    frame = ctx.deskew_scan(s, T[-2], T[-1])
    assert not np.isfinite(frame[1000:1010]).any() and np.isfinite(frame[:1000]).all()
    with pytest.raises(pkg.LimuError):
        ctx.voxel_downsample(frame, 0.5 * VOXEL)
    with pytest.raises(pkg.LimuError):
        k.register_frame(s)
    k.close()


def zeros_alternating(t):
    """The same values, a run per point wherever t is +0."""
    u = t.copy()
    z = np.flatnonzero(u == 0.0)
    u[z[1::2]] = -0.0
    return u


@pytest.mark.parametrize("mode", ["float4", "records"])
@pytest.mark.parametrize("n", [3000, 128000, 160000])
def test_pipelined_path_table_equals_per_point(ctx, pkg, world, mode, n):
    """k_voxelize_lean: the first half of every tile fired at t = 0, the rest in runs of 64 equal times. As they are, every tile
    has one run of zeros + the others (table); with the zeros' signs alternating, every tile has hundreds of runs (per-point path)."""
    synth, warm, full = world
    s = synth.pad_scan(full, n, seed=n + 2).copy()
    t = runs_of_length(n, 64)
    t[(np.arange(n) % BLOCK) < BLOCK // 2] = 0.0
    variants = [t, zeros_alternating(t)]
    assert branches(variants[0]) == {"table"} and branches(variants[1]) == {"per-point"}
    out = []
    for tv in variants:
        k = ctx.KissICP(voxel_size=VOXEL, deskew=True, icp_max_iteration=60, speculate=True)
        bufs = []
        seq = list(warm) + [None]
        for i in range(len(seq)):
            if mode == "float4":
                x = pkg.PinnedArray((len(seq[i]) if seq[i] is not None else n, 4), np.float32)
                if seq[i] is None:
                    x.array[:, :3] = s[:, :3]; x.array[:, 3] = tv.astype(np.float32)
                else:
                    x.array[...] = seq[i]
                bufs.append((x,))
            else:
                m = len(seq[i]) if seq[i] is not None else n
                r = pkg.PinnedArray((m, 12), np.float32); r.array[...] = 0
                ts = pkg.PinnedArray((m,), np.float64)
                src = s if seq[i] is None else seq[i]
                r.array[:, :3] = src[:, :3]
                ts.array[...] = tv if seq[i] is None else seq[i][:, 3]
                bufs.append((r, ts))
        poses = []
        for i in range(len(seq)):
            if i + 1 < len(seq):
                if mode == "float4":
                    k.prefetch(bufs[i + 1][0].array)
                else:
                    k.prefetch_cloud(bufs[i + 1][0].array, 48, bufs[i + 1][1].array)
            if mode == "float4":
                d, kp, p = k.register_frame(bufs[i][0].array)
            else:
                d, kp, p = k.register_cloud(bufs[i][0].array, 48, bufs[i][1].array)
            poses.append(p.copy())
        assert k.stats.reserved0 == 1 and k.stats.deskewed == 1      # the last scan ran ahead, beside the map update, deskewed
        out.append((np.array(poses[:-1]), d, kp))
        k.close()
        for b in bufs:
            for x in b:
                x.free()
    (pa, da, ka), (pb, db, kb) = out
    assert np.array_equal(pa, pb)              # the same poses before the scan: the same twist on the device
    assert np.array_equal(da, db) and np.array_equal(ka, kb)
