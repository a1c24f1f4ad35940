"""limu_map_score_poses and limu_relocalize: the fitness of limu_icp_multi at many poses without a Gauss-Newton loop, and global relocalization
over a planar grid of candidate poses (score every candidate on the device, keep the best n_refine, refine them with limu_icp_multi).

A pose's score is held to the C port: inliers = correspondences of port.Map.closest under the tau^2 test from the port's own transformed
points, exactly; rms within 1e-12 relative -- and its inliers equal what limu_icp_multi reports after 0 iterations. The selection is held to
a full sort of every candidate's score by (inliers desc, rms asc, index asc), the refinement to limu_icp_multi from the returned coarse poses,
bit for bit."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_icp_multi import STUB_COMMON, STUB_SOPHUS, guess_grid, port_fitness, scene

NN27, PLANE = 1, 2
IDENT = np.array([0, 0, 0, 1.0, 0, 0, 0])
LIMU_ERR_INVALID, LIMU_ERR_NOMEM = -1, -5


# ---------------------------------------------------------------------------------------------------------------- CPU
CONSUMER = """#include "limu/sensors/lidar/helpers/registration.hpp"
int main() {
    lidar::VoxelHashMap map(1.0, 100.0, 10);
    utils::Vec3dVector pts{utils::Vec3d(1, 2, 3)};
    Sophus::SE3d center;
    lidar::RelocalizeResult r = lidar::relocalize(map, pts, center, 21, 21, 36, 1.0, 0.17453292519943295, 32, 1.0, 0.5, 100, 1e-4);
    return r.best + (int)r.poses.size() + (int)r.candidates[0].coarse_inliers + (int)r.candidates[0].icp.inliers;
}
"""


def test_dropin_relocalize_compiles(tmp_path):
    """The drop-in header's lidar::relocalize compiles in a C++ consumer with -Wall -Werror against the stand-in Sophus / utils headers."""
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    stub = tmp_path / "stub"
    (stub / "sophus").mkdir(parents=True)
    (stub / "sophus" / "se3.hpp").write_text(STUB_SOPHUS)
    (stub / "common.hpp").write_text(STUB_COMMON)
    (tmp_path / "main.cpp").write_text(CONSUMER)
    inc = os.path.join(ROOT, "include")
    r = subprocess.run([gxx, "-std=c++17", "-fsyntax-only", "-Wall", "-Werror", "-I" + os.path.join(inc, "limu_dropin"), "-I" + inc,
                        "-I" + str(stub), str(tmp_path / "main.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


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


def grid_pose(port, center, nx, ny, nyaw, step_xy, step_yaw, index):
    """Candidate `index` of the planar grid, restated from the header's definition."""
    i, r = index % nx, index // nx
    j, l = r % ny, r // ny
    t = (l - (nyaw - 1) / 2) * step_yaw
    d = np.array([0.0, 0.0, np.sin(t / 2), np.cos(t / 2), (i - (nx - 1) / 2) * step_xy, (j - (ny - 1) / 2) * step_xy, 0.0])
    return port.se3_mul(center, d)


def ranking(inliers, rms):
    """Every candidate, ordered by (inliers desc, rms asc, index asc)."""
    return np.lexsort((np.arange(len(inliers)), rms, -inliers))


SCORE_CASES = [
    # (cap, n, k, mode): every lookup path of the loop (eight lanes per query up to cap 64 with 1, 2, 3 register rounds; one lane per query
    # beyond), n on both sides of 16384, k from 1 to beyond 10^5
    (1, 500, 1, 0), (10, 2000, 300, 0), (20, 3000, 37, NN27), (25, 1200, 64, 0), (64, 2000, 100_000, 0), (65, 1500, 50, NN27),
    (100, 1500, 50, 0), (10, 16384, 20, 0), (10, 16385, 20, NN27), (20, 16385, 120_000, NN27), (16, 900, 7, 0), (100, 700, 9, NN27),
]


@pytest.mark.gpu
@pytest.mark.parametrize("cap,n,k,mode", SCORE_CASES)
def test_score_poses_matches_the_port(ctx, port, cap, n, k, mode):
    rng = np.random.default_rng(17 * cap + n % 991 + 5 * k + mode)
    gm, om, src = scene(port, ctx, rng, cap, n, mode=mode)
    try:
        poses = guess_grid(port, rng, k, 1.0, 0.2)
        tau = 0.6
        res = gm.score_poses(src, poses, tau, icp_mode=mode)
        assert res["inliers"].shape == (k,) and res["rms"].shape == (k,)
        assert (res["inliers"] > 0).any()
        idx = np.arange(k) if k <= 300 else np.unique(np.concatenate([np.arange(20), rng.choice(k, 30, replace=False), [k - 1]]))
        for i in idx[:300 if n <= 3000 else 12]:   # the port is slow at 16 k points
            inl, rms = port_fitness(om, port.transform(poses[i], src), tau)
            assert res["inliers"][i] == inl, (i, res["inliers"][i], inl)
            assert abs(res["rms"][i] - rms) <= 1e-12 * rms, (i, res["rms"][i], rms)
        sub = idx[:60] if n <= 16384 else idx[:4]   # limu_icp_multi runs the loop kernel once per guess beyond 16384 points
        multi = gm.icp_multi(src, poses[sub], tau, 0.2, 0, 1e-4, icp_mode=mode)
        assert np.array_equal(multi["inliers"], res["inliers"][sub])
        np.testing.assert_allclose(multi["rms"], res["rms"][sub], rtol=1e-12, atol=0)
    finally:
        gm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cap,n,mode", [(10, 2000, 0), (20, 3137, NN27), (65, 1500, 0), (10, 16385, 0)])
def test_score_is_independent_of_k_and_position(ctx, port, cap, n, mode):
    rng = np.random.default_rng(5 + cap + n)
    gm, om, src = scene(port, ctx, rng, cap, n, mode=mode)
    try:
        poses = guess_grid(port, rng, 5000, 1.0, 0.2)
        probe = poses[5]
        alone = gm.score_poses(src, probe[None], 0.6, icp_mode=mode)
        for k, pos in ((2, 1), (7, 0), (149, 148), (5000, 5), (5000, 4321)):
            p = poses[:k].copy()
            p[pos] = probe
            res = gm.score_poses(src, p, 0.6, icp_mode=mode)
            assert res["inliers"][pos] == alone["inliers"][0] and res["rms"][pos].tobytes() == alone["rms"][0].tobytes(), (k, pos)
    finally:
        gm.close()


@pytest.mark.gpu
def test_score_isolation_and_degenerate_calls(ctx, port, pkg):
    rng = np.random.default_rng(99)
    gm, om, src = scene(port, ctx, rng, 10, 1000)
    empty, oempty = ctx.VoxelHashMap(1.0, 100.0, 10), port.Map(1.0, 100.0, 10)
    try:
        poses = guess_grid(port, rng, 40, 0.5, 0.1)
        ref = gm.score_poses(src, poses, 0.6)
        bad = poses.copy()
        bad[3, 4] = np.nan          # NaN translation
        bad[11, :4] = np.nan        # NaN rotation
        bad[17, 4:] = [1000.0, -800.0, 300.0]   # 1 km away
        res = gm.score_poses(src, bad, 0.6)
        keep = np.setdiff1d(np.arange(40), [3, 11, 17])
        assert np.array_equal(res["inliers"][keep], ref["inliers"][keep]) and np.array_equal(res["rms"][keep], ref["rms"][keep])
        for i in (3, 11, 17):
            inl, rms = port_fitness(om, port.transform(bad[i], src), 0.6)
            assert res["inliers"][i] == inl == 0 and res["rms"][i] == rms == 0.0
        multi = gm.icp_multi(src, bad[[3, 11, 17]], 0.6, 0.2, 0, 1e-4)
        assert np.array_equal(multi["inliers"], res["inliers"][[3, 11, 17]])
        r = empty.score_poses(src, poses, 0.6)                                   # empty map: nothing found -> (0,0,0), range-tested
        for p, inl, rms in zip(poses, r["inliers"], r["rms"]):
            assert (inl, rms) == pytest.approx(port_fitness(oempty, port.transform(p, src), 0.6), rel=1e-12)
        assert np.array_equal(r["inliers"], empty.icp_multi(src, poses, 0.6, 0.2, 0, 1e-4)["inliers"])
        r = gm.score_poses(src[:0], poses, 0.6)                                  # n = 0
        assert (r["inliers"] == 0).all() and (r["rms"] == 0).all()
        r = gm.score_poses(src, poses[:0], 0.6)                                  # k = 0
        assert r["inliers"].shape == (0,) and r["rms"].shape == (0,)
        with pytest.raises(pkg.LimuError, match="point-to-plane") as e:
            gm.score_poses(src, poses, 0.6, icp_mode=PLANE)
        assert e.value.status == LIMU_ERR_INVALID
    finally:
        gm.close()
        empty.close()


def small_grid_scene(port, ctx, rng, cap=10, n=1500, mode=0):
    gm, om, src = scene(port, ctx, rng, cap, n, mode=mode)
    lo, hi = om.dump()[2].min(0), om.dump()[2].max(0)
    center = IDENT.copy()
    center[4:6] = (lo[:2] + hi[:2]) / 2 + [0.3, -0.2]
    center[6] = 0.1
    return gm, om, src, center


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, NN27])
def test_full_ranking_and_prefixes(ctx, port, mode):
    """n_refine >= K: every grid index once, in (inliers desc, rms asc, index asc) order, coarse scores bit-equal to score_poses at the
    returned coarse poses, coarse poses within 1e-12 of center * D(i, j, l); a smaller n_refine returns the prefix of that ranking."""
    rng = np.random.default_rng(2024 + mode)
    gm, om, src, center = small_grid_scene(port, ctx, rng, mode=mode)
    try:
        nx, ny, nyaw, sxy, syaw = 13, 11, 24, 0.7, np.radians(15.0)
        K = nx * ny * nyaw
        args = (0.6, 0.2, 6, 1e-4)
        full = gm.relocalize(src, center, nx, ny, nyaw, sxy, syaw, 4096, *args, icp_mode=mode)
        assert len(full["index"]) == K and np.array_equal(np.sort(full["index"]), np.arange(K))
        inl, rms, idx = full["coarse_inliers"], full["coarse_rms"], full["index"]
        assert all((inl[a], -rms[a], -idx[a]) > (inl[a + 1], -rms[a + 1], -idx[a + 1]) for a in range(K - 1))
        assert inl[0] > 0 and (inl == 0).any()
        want = np.array([grid_pose(port, center, nx, ny, nyaw, sxy, syaw, int(i)) for i in idx])
        np.testing.assert_allclose(full["coarse_poses"], want, rtol=0, atol=1e-12)
        sc = gm.score_poses(src, full["coarse_poses"], 0.6, icp_mode=mode)
        assert np.array_equal(sc["inliers"], inl) and sc["rms"].tobytes() == rms.tobytes()
        for m in (1, 7, 100, K - 1):
            part = gm.relocalize(src, center, nx, ny, nyaw, sxy, syaw, m, *args, icp_mode=mode)
            for key in ("index", "coarse_poses", "coarse_inliers", "coarse_rms", "poses", "iters", "converged", "inliers", "rms"):
                assert part[key].tobytes() == full[key][:m].tobytes(), (m, key)
    finally:
        gm.close()


@pytest.mark.gpu
def test_selection_boundary_inside_a_huge_tie_class(ctx, port):
    """A grid of 13 448 candidates over +-60 m around a map 8 m across: more than 10^4 candidates see nothing within range (0 inliers, rms 0)
    and the selection boundary falls inside that class, where the index decides; a second call with max_corresp_dist so small that every
    candidate ties takes the n_refine lowest indices."""
    rng = np.random.default_rng(7)
    gm, om, src, center = small_grid_scene(port, ctx, rng)
    try:
        nx, ny, nyaw, sxy, syaw = 41, 41, 8, 3.0, np.radians(45.0)
        K = nx * ny * nyaw
        allp = np.array([grid_pose(port, center, nx, ny, nyaw, sxy, syaw, i) for i in range(K)])
        sc = gm.score_poses(src, allp, 0.6)
        hits = int((sc["inliers"] > 0).sum())
        assert (sc["inliers"] == 0).sum() > 10_000 and 0 < hits
        order = ranking(sc["inliers"], sc["rms"])
        for m in (hits + 1, hits + 777, 4096):
            r = gm.relocalize(src, center, nx, ny, nyaw, sxy, syaw, m, 0.6, 0.2, 0, 1e-4)
            assert np.array_equal(r["index"], order[:m]), m
            assert np.array_equal(r["coarse_inliers"], sc["inliers"][order[:m]]) and np.array_equal(r["coarse_rms"], sc["rms"][order[:m]])
        if hits > 2:   # a boundary inside a class of nonzero rms values as well
            r = gm.relocalize(src, center, nx, ny, nyaw, sxy, syaw, hits // 2, 0.6, 0.2, 0, 1e-4)
            assert np.array_equal(r["index"], order[: hits // 2])
        r = gm.relocalize(src, center, nx, ny, nyaw, sxy, syaw, 50, 1e-9, 0.2, 0, 1e-4)
        assert np.array_equal(r["index"], np.arange(50)) and (r["coarse_inliers"] == 0).all()
    finally:
        gm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cap,n,mode", [(10, 1500, 0), (20, 2500, NN27), (65, 1200, 0), (10, 16385, 0)])
def test_refinement_is_icp_multi_from_the_coarse_poses(ctx, port, cap, n, mode):
    rng = np.random.default_rng(300 + cap + mode)
    gm, om, src, center = small_grid_scene(port, ctx, rng, cap, n, mode)
    try:
        m = 3 if n > 16384 else 40
        r = gm.relocalize(src, center, 9, 9, 12, 1.0, np.radians(30.0), m, 0.6, 0.2, 30, 1e-4, icp_mode=mode)
        multi = gm.icp_multi(src, r["coarse_poses"], 0.6, 0.2, 30, 1e-4, icp_mode=mode)
        assert r["poses"].tobytes() == multi["poses"].tobytes()
        for key in ("iters", "converged", "inliers", "rms", "best"):
            assert np.array_equal(r[key], multi[key]), key
    finally:
        gm.close()


@pytest.mark.gpu
def test_invalid_arguments(ctx, port, pkg):
    rng = np.random.default_rng(3)
    gm, om, src, center = small_grid_scene(port, ctx, rng)
    try:
        ok = dict(nx=3, ny=3, nyaw=4, step_xy=1.0, step_yaw=0.5, n_refine=4)
        for change in (dict(n_refine=0), dict(n_refine=4097), dict(step_xy=0.0), dict(step_yaw=-0.1), dict(step_xy=np.nan), dict(nx=0),
                       dict(ny=0), dict(nyaw=0), dict(nyaw=-2)):
            a = {**ok, **change}
            with pytest.raises(pkg.LimuError) as e:
                gm.relocalize(src, center, a["nx"], a["ny"], a["nyaw"], a["step_xy"], a["step_yaw"], a["n_refine"], 0.6, 0.2, 5, 1e-4)
            assert e.value.status == LIMU_ERR_INVALID, change
        with pytest.raises(pkg.LimuError, match="point-to-plane") as e:
            gm.relocalize(src, center, 3, 3, 4, 1.0, 0.5, 4, 0.6, 0.2, 5, 1e-4, icp_mode=PLANE)
        assert e.value.status == LIMU_ERR_INVALID
        for nx, ny, nyaw in ((2**31 - 1, 2**31 - 1, 2**31 - 1), (2**20, 2**20, 2**10)):   # beyond int64, and 2^50 candidates
            with pytest.raises(pkg.LimuError) as e:
                gm.relocalize(src, center, nx, ny, nyaw, 1.0, 0.5, 4, 0.6, 0.2, 5, 1e-4)
            assert e.value.status == LIMU_ERR_NOMEM
        r = gm.relocalize(src, center, 1, 1, 1, 1.0, 0.5, 4096, 0.6, 0.2, 5, 1e-4)   # one candidate: the center itself
        assert np.array_equal(r["index"], [0]) and r["best"] == 0
        np.testing.assert_allclose(r["coarse_poses"][0], center, rtol=0, atol=1e-15)
    finally:
        gm.close()


@pytest.mark.gpu
def test_global_relocalization_without_a_prior(ctx, port):
    """The structure-rich scene of test_best_relocalizes_and_breaks_ties_by_index, searched over +-10 m at 1 m with 36 yaw steps around a
    center that is NOT near the truth: the truth is 4.4 m and 17 deg from the center, between grid points. best converges within 0.05 m /
    0.5 deg of the truth."""
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    sc = synth.Scene(seed=31, n_boxes=150, n_cyl=60)
    traj = synth.loop_trajectory(12, radius=30.0, step=0.5)
    built = ctx.VoxelHashMap(0.5, 100.0, 20)
    m = ctx.VoxelHashMap(0.5, 100.0, 20)
    try:
        for i in range(8):
            scan = synth.cast_scan(sc, traj[i], traj[i], beams=64, azimuth_steps=1800, elev=(-10.0, 30.0), noise=0.005, seed=500 + i)
            built.insert_points(port.transform(synth.pose7_of(traj[i]), scan[:, :3].astype(np.float64)))
        m.insert_points(built.pointcloud())
        truth = synth.pose7_of(traj[10])
        scan = synth.cast_scan(sc, traj[10], traj[10], beams=64, azimuth_steps=1800, elev=(-10.0, 30.0), noise=0.005, seed=600)
        kp, _ = ctx.voxelize(scan[:, :3].astype(np.float64), 0.25)
        center = port.se3_mul(truth, port.se3_exp(np.array([-3.37, 2.71, 0.0, 0.0, 0.0, np.radians(-17.3)])))
        r = m.relocalize(kp, center, 21, 21, 36, 1.0, np.radians(10.0), 32, 1.0, 0.5, 100, 1e-4)
        assert len(r["index"]) == 32
        b = r["best"]
        err = port.se3_log(port.se3_mul(port.se3_inv(truth), r["poses"][b]))
        assert r["converged"][b], (b, r["iters"][b])
        assert np.linalg.norm(err[:3]) < 0.05 and np.degrees(np.linalg.norm(err[3:])) < 0.5, (b, err)
    finally:
        built.close()
        m.close()


@pytest.mark.gpu
def test_calls_on_a_pipelined_handles_map(ctx, port):
    """relocalize and score_poses on local_map() between the register calls of a pipelined handle: the handle's poses, iteration counts and
    map are those of the same run without the calls, and the calls return what they return on a plain handle's (bit-identical) map."""
    import torch
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    sc = synth.Scene(seed=21)
    traj = synth.loop_trajectory(11, radius=30.0, step=0.7)
    scans = [synth.cast_scan(sc, traj[i], traj[i + 1], beams=16, azimuth_steps=700, seed=300 + i) for i in range(8)]
    rng = np.random.default_rng(8)
    query = scans[3][:, :3].astype(np.float64)[::3]
    poses = guess_grid(port, rng, 3000, 3.0, 0.3)
    center = synth.pose7_of(traj[3])

    def run(spec, calls):
        staged = [torch.from_numpy(s).cuda() for s in scans]
        torch.cuda.synchronize()
        k = ctx.KissICP(deskew=False, icp_max_iteration=60, speculate=spec)
        out, got = [], []
        for i, t in enumerate(staged):
            if spec and i + 1 < len(staged):
                k.hint_next_dev(staged[i + 1].data_ptr(), len(scans[i + 1]))
            p = k.register_frame_dev(t.data_ptr(), len(scans[i]))
            out.append((p.copy(), k.stats.icp.iterations))
            if calls and i >= 2:
                got.append((k.local_map().relocalize(query, center, 9, 9, 12, 1.0, np.radians(30.0), 16, 1.5, 0.5, 30, 1e-4),
                            k.local_map().score_poses(query, poses, 1.5), k.local_map().dump()))
        k.flush()
        dump = k.local_map().dump()
        k.close()
        return out, dump, got

    a, da, _ = run(True, False)
    b, db, gb = run(True, True)
    c, dc, gc = run(False, True)
    for (pa, ia), (pb, ib) in zip(a, b):
        assert ia == ib and np.array_equal(pa, pb)
    assert all(np.array_equal(x, y) for x, y in zip(da, db))
    for (rb, sb, mapb), (rc, sc_, mapc) in zip(gb, gc):
        assert all(np.array_equal(x, y) for x, y in zip(mapb, mapc))
        for key in rb:
            assert np.array_equal(rb[key], rc[key]), key
        assert np.array_equal(sb["inliers"], sc_["inliers"]) and sb["rms"].tobytes() == sc_["rms"].tobytes()


CPP_RUNNER = """#include <cstdio>
#include "limu/sensors/lidar/helpers/registration.hpp"
static std::vector<double> read_block(FILE *f) {
    long long n = 0;
    if (fread(&n, 8, 1, f) != 1) return {};
    std::vector<double> v((size_t)n);
    if (n && fread(v.data(), 8, (size_t)n, f) != (size_t)n) v.clear();
    return v;
}
static utils::Vec3dVector points(const std::vector<double> &v) {
    utils::Vec3dVector out;
    for (size_t i = 0; i + 2 < v.size(); i += 3) out.emplace_back(v[i], v[i + 1], v[i + 2]);
    return out;
}
int main(int argc, char **argv) {
    FILE *f = fopen(argv[1], "rb");
    const std::vector<double> world = read_block(f), query = read_block(f), c = read_block(f);
    fclose(f);
    lidar::VoxelHashMap map(1.0, 100.0, 10);
    map.insert_points(points(world));
    Sophus::SE3d center;
    std::copy(c.begin(), c.begin() + 7, center.data());
    const lidar::RelocalizeResult r = lidar::relocalize(map, points(query), center, 9, 7, 12, 0.8, 0.5, 25, 0.6, 0.2, 20, 1e-4);
    FILE *o = fopen(argv[2], "wb");
    for (size_t i = 0; i < r.candidates.size(); ++i) {
        const limu_reloc_candidate &x = r.candidates[i];
        double row[24] = {(double)x.index, (double)x.coarse_inliers, x.coarse_rms, (double)x.icp.iterations, (double)x.icp.converged,
                          (double)x.icp.inliers, x.icp.rms};
        std::copy(x.coarse_pose, x.coarse_pose + 7, row + 7);
        std::copy(r.poses[i].data(), r.poses[i].data() + 7, row + 14);
        row[21] = row[22] = row[23] = 0.0;
        fwrite(row, 8, 24, o);
    }
    const double best = r.best;
    fwrite(&best, 8, 1, o);
    fclose(o);
    return 0;
}
"""


@pytest.mark.gpu
def test_dropin_relocalize_runs(ctx, port, tmp_path):
    """lidar::relocalize from a C++ program linked against the library returns what VoxelHashMap.relocalize returns, bit for bit."""
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    import __graft_entry__ as g
    pkg = g.load_package()
    rng = np.random.default_rng(4711)
    gm, om, src, center = small_grid_scene(port, ctx, rng)
    world = gm.pointcloud()
    try:
        want = gm.relocalize(src, center, 9, 7, 12, 0.8, 0.5, 25, 0.6, 0.2, 20, 1e-4)
    finally:
        gm.close()
    stub = tmp_path / "stub"
    (stub / "sophus").mkdir(parents=True)
    (stub / "sophus" / "se3.hpp").write_text(STUB_SOPHUS)
    (stub / "common.hpp").write_text(STUB_COMMON)
    (tmp_path / "main.cpp").write_text(CPP_RUNNER)
    inc, libdir = os.path.join(ROOT, "include"), os.path.dirname(pkg.LIB_PATH)
    exe = tmp_path / "runner"
    r = subprocess.run([gxx, "-std=c++17", "-O1", "-I" + os.path.join(inc, "limu_dropin"), "-I" + inc, "-I" + str(stub), str(tmp_path / "main.cpp"),
                        "-o", str(exe), "-L" + libdir, "-llimu_cuda", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    with open(tmp_path / "in.bin", "wb") as f:
        for a in (world, src, center):
            a = np.ascontiguousarray(a, np.float64).ravel()
            f.write(np.int64(a.size).tobytes())
            f.write(a.tobytes())
    r = subprocess.run([str(exe), str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    got = np.fromfile(tmp_path / "out.bin", np.float64)
    rows = got[:-1].reshape(-1, 24)
    assert len(rows) == 25
    assert np.array_equal(rows[:, 0], want["index"]) and np.array_equal(rows[:, 1], want["coarse_inliers"])
    assert rows[:, 2].tobytes() == want["coarse_rms"].tobytes()
    assert np.array_equal(rows[:, 3], want["iters"]) and np.array_equal(rows[:, 4], want["converged"]) and np.array_equal(rows[:, 5], want["inliers"])
    assert rows[:, 6].tobytes() == want["rms"].tobytes()
    assert rows[:, 7:14].tobytes() == want["coarse_poses"].tobytes() and rows[:, 14:21].tobytes() == want["poses"].tobytes()
    assert got[-1] == want["best"]
