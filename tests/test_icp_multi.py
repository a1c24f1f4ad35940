"""limu_icp_multi: lidar::ICP (registration.cpp:94-130) from many initial guesses in one launch (relocalization).

Every hypothesis is held to the bar of stand-alone ICP against the C port (oracle/limu_oracle.c lo_icp) from the same guess: equal iteration
count, pose within 1e-9, and a fitness computed from the port's own src_after -- inliers = correspondences of port.Map.closest under the
tau^2 test, exactly; rms within 1e-12 relative.
A hypothesis's result must not depend on how many others run beside it or where it sits in the list (bit for bit), and a hypothesis that
fails (NaN guess, iteration cap) must not disturb the others."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_voxel_caps import make_queries, slab_world

NN27, PLANE = 1, 2
IDENT = np.array([0, 0, 0, 1.0, 0, 0, 0])


# ---------------------------------------------------------------------------------------------------------------- CPU
STUB_SOPHUS = """#pragma once
namespace Sophus { struct SE3d { double d[7] = {0, 0, 0, 1, 0, 0, 0}; double *data() { return d; } const double *data() const { return d; } }; }
"""
STUB_COMMON = """#pragma once
#include <tuple>
#include <vector>
namespace utils {
struct Vec3d { double v[3] = {0, 0, 0}; Vec3d() = default; Vec3d(double a, double b, double c) : v{a, b, c} {}
               double *data() { return v; } const double *data() const { return v; } };
using Vec3dVector = std::vector<Vec3d>;
struct Voxel { int x, y, z; Voxel(int a, int b, int c) : x(a), y(b), z(c) {} };
using Vec3_Vec3Tuple = std::tuple<Vec3dVector, Vec3dVector>;
}
"""
CONSUMER = """#include "limu/sensors/lidar/helpers/registration.hpp"
int main() {
    lidar::VoxelHashMap map(1.0, 100.0, 10);
    utils::Vec3dVector pts{utils::Vec3d(1, 2, 3)};
    std::vector<Sophus::SE3d> guesses(3);
    lidar::ICPMultiResult r = lidar::ICP_multi(map, pts, guesses, 3.0, 1.0, 50, 1e-4);
    return r.best + (int)r.poses.size() + (int)r.hypotheses[0].inliers;
}
"""


def test_dropin_icp_multi_compiles(tmp_path):
    """The drop-in header compiles in a C++ consumer with the include-path swap of INTEGRATION.md (our headers first). The reference's type
    headers (Sophus, utils) are replaced by minimal stand-ins here: what is checked is our header's own code against the C ABI."""
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


def test_map_rebuilt_from_pointcloud_has_equal_dump(port, rng):
    """The relocalization recipe's first step: a saved map's pointcloud() inserted into a fresh map of the same voxel size and cap gives the
    same voxels, counts, points and creation order."""
    for cap, vox in ((10, 1.0), (1, 0.5), (20, 2.0)):
        a = port.Map(vox, 100.0 * vox, cap)
        for _ in range(4):   # several batches, with points beyond the cap
            a.insert(rng.normal(size=(3000, 3)) * 6 * vox)
        keys, counts, pts = a.dump()
        b = port.Map(vox, 100.0 * vox, cap)
        b.insert(pts)
        kb, cb, pb = b.dump()
        assert np.array_equal(keys, kb) and np.array_equal(counts, cb) and np.array_equal(pts, pb)


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


def guess_grid(port, rng, k, trans=0.4, rot=0.05):
    """k guesses around the identity: translations up to `trans`, rotations up to `rot` rad about every axis."""
    out = np.empty((k, 7))
    for i in range(k):
        out[i] = port.se3_exp(np.concatenate([rng.uniform(-trans, trans, 3), rng.uniform(-rot, rot, 3)]))
    return out


def scene(port, ctx, rng, cap, nq, vox=1.0, mode=0):
    world = slab_world(rng, cap, vox)
    src = port.transform(port.se3_inv(port.se3_exp(np.array([0.06, -0.04, 0.02, 0.004, -0.003, 0.01]))), make_queries(rng, world, nq, vox))
    gm, om = ctx.VoxelHashMap(vox, 100.0 * vox, cap), port.Map(vox, 100.0 * vox, cap)
    gm.insert_points(world)
    om.insert(world)
    om.set_mode(mode)
    return gm, om, src


def port_fitness(om, after, tau):
    if len(after) == 0:
        return 0, 0.0
    d2 = ((om.closest(after) - after) ** 2).sum(axis=1)
    inl = d2 < tau * tau
    n = int(inl.sum())
    return n, (float(np.sqrt(d2[inl].sum() / n)) if n else 0.0)


def check_against_port(om, src, guesses, res, tau, th, max_iter, eps, what):
    for i, g in enumerate(guesses):
        port_icp = om.api.icp(om, src, g, tau, th, max_iter, eps, trace=True)
        w = f"{what}, hypothesis {i}"
        assert res["iters"][i] == port_icp["iters"], w
        np.testing.assert_allclose(res["poses"][i], port_icp["pose"], rtol=0, atol=1e-9, err_msg=w)
        if om.empty():
            continue
        inl, rms = port_fitness(om, port_icp["src_after"], tau)
        assert res["inliers"][i] == inl, w
        assert abs(res["rms"][i] - rms) <= 1e-12 * rms, w


MULTI_CASES = [
    # (cap, n, k, mode): n on either side of the group-size steps (G = ceil(8 n / 3584): 448 | 449, 3136 | 3137) and of 16384; caps 1 ... 64
    # in the latency shape, 65 (and n > 16384) through the loop kernel once per guess; K below, at and above one wave
    (10, 448, 7, 0), (10, 449, 148, 0), (1, 3136, 2, 0), (20, 3137, 149, 0), (64, 2000, 7, 0), (10, 16384, 7, 0),
    (10, 16385, 2, 0), (65, 1500, 7, 0), (10, 2000, 600, 0), (10, 2000, 1, 0),
    (10, 449, 7, NN27), (20, 3137, 149, NN27), (65, 1500, 2, NN27), (10, 16385, 2, NN27),
]


@pytest.mark.gpu
@pytest.mark.parametrize("cap,n,k,mode", MULTI_CASES)
def test_every_hypothesis_matches_the_port(ctx, port, cap, n, k, mode):
    rng = np.random.default_rng(1000 * cap + n % 997 + 7 * k + mode)
    gm, om, src = scene(port, ctx, rng, cap, n, mode=mode)
    try:
        guesses = guess_grid(port, rng, k)
        tau, th, max_iter, eps = 0.6, 0.2 / 3, 40, 1e-4
        res = gm.icp_multi(src, guesses, tau, th, max_iter, eps, icp_mode=mode)
        assert res["poses"].shape == (k, 7) and 0 <= res["best"] < k
        assert (res["inliers"] > 0).all()
        # the port is slow at 600 x 2000 points: every hypothesis up to 160, then a sample
        idx = np.arange(k) if k <= 160 else np.unique(np.concatenate([np.arange(40), rng.choice(k, 60, replace=False), [k - 1]]))
        sub = {key: (v[idx] if isinstance(v, np.ndarray) else v) for key, v in res.items()}
        check_against_port(om, src, guesses[idx], sub, tau, th, max_iter, eps, f"cap {cap}, n {n}, k {k}, mode {mode}")
    finally:
        gm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cap,n,mode", [(10, 2000, 0), (20, 3137, NN27), (65, 1500, 0)])
def test_result_is_independent_of_k_and_position(ctx, port, cap, n, mode):
    rng = np.random.default_rng(77 + cap + n)
    gm, om, src = scene(port, ctx, rng, cap, n, mode=mode)
    try:
        guesses = guess_grid(port, rng, 300)
        probe = guesses[5]
        args = (0.6, 0.2 / 3, 40, 1e-4)
        alone = gm.icp_multi(src, probe[None], *args, icp_mode=mode)
        keys = ("poses", "iters", "converged", "inliers", "rms")
        for k, pos in ((2, 1), (7, 0), (149, 148), (300, 5), (300, 211)):
            g = guesses[:k].copy()
            g[pos] = probe
            res = gm.icp_multi(src, g, *args, icp_mode=mode)
            for key in keys:
                assert np.array_equal(res[key][pos], alone[key][0]), (k, pos, key)
    finally:
        gm.close()


@pytest.mark.gpu
def test_isolation_of_failing_hypotheses(ctx, port):
    """Converging guesses, far guesses that hit a small iteration cap, and a NaN guess in one batch: every finite hypothesis equals its
    stand-alone port result, the NaN one equals what limu_icp_ex returns for it."""
    rng = np.random.default_rng(4242)
    gm, om, src = scene(port, ctx, rng, 10, 2500)
    try:
        near, far = guess_grid(port, rng, 20, 0.05, 0.005), guess_grid(port, rng, 20, 1.5, 0.3)
        nan = IDENT.copy()
        nan[4] = np.nan
        guesses = np.concatenate([near[:10], far[:10], nan[None], near[10:], far[10:]])
        fin = np.isfinite(guesses).all(axis=1)
        tau, th, eps = 0.6, 0.2 / 3, 1e-4
        free = [port.icp(om, src, g, tau, th, 100, eps)["iters"] for g in guesses[fin]]
        max_iter = (min(free) + max(free)) // 2   # an iteration cap that some hypotheses of the batch reach and others do not
        assert min(free) < max_iter < max(free)
        res = gm.icp_multi(src, guesses, tau, th, max_iter, eps)
        assert (res["iters"][fin] == max_iter).any() and (res["iters"][fin] < max_iter).any()
        check_against_port(om, src, guesses[fin], {key: (v[fin] if isinstance(v, np.ndarray) else v) for key, v in res.items()},
                           tau, th, max_iter, eps, "isolation")
        single = gm.icp(src, nan, tau, th, max_iter, eps)
        i = int(np.flatnonzero(~fin)[0])
        np.testing.assert_array_equal(res["poses"][i], single["pose"])   # (NaN == NaN here)
        assert res["iters"][i] == single["iters"] and res["converged"][i] == single["converged"]
    finally:
        gm.close()


@pytest.mark.gpu
def test_degenerate_calls(ctx, port):
    rng = np.random.default_rng(99)
    gm, om, src = scene(port, ctx, rng, 10, 1000)
    empty, oempty = ctx.VoxelHashMap(1.0, 100.0, 10), port.Map(1.0, 100.0, 10)
    try:
        guesses = guess_grid(port, rng, 5)
        args = (0.6, 0.2 / 3, 40, 1e-4)
        r = gm.icp_multi(src, guesses[:0], *args)                                 # k = 0
        assert r["poses"].shape == (0, 7) and r["best"] == -1
        r = empty.icp_multi(src, guesses, *args)                                  # empty map: the guesses, 0 iterations
        assert np.array_equal(r["poses"], guesses) and (r["iters"] == 0).all()
        for g, inl, rms in zip(guesses, r["inliers"], r["rms"]):                 # (nothing found -> (0,0,0), range-tested like a real point)
            assert (inl, rms) == pytest.approx(port_fitness(oempty, port.transform(g, src), 0.6), rel=1e-12)
        r = gm.icp_multi(src, guesses, 0.6, 0.2 / 3, 0, 1e-4)                    # max_iter = 0
        assert np.array_equal(r["poses"], guesses) and (r["iters"] == 0).all()
        for g, inl, rms in zip(guesses, r["inliers"], r["rms"]):
            assert (inl, rms) == pytest.approx(port_fitness(om, port.transform(g, src), 0.6), rel=1e-12)
        r = gm.icp_multi(src[:0], guesses, *args)                                 # n = 0
        check_against_port(om, src[:0], guesses, r, *args, "n = 0")
        assert (r["inliers"] == 0).all() and (r["rms"] == 0).all() and r["best"] == 0
        with pytest.raises(RuntimeError, match="point-to-plane"):
            gm.icp_multi(src, guesses, *args, icp_mode=PLANE)
    finally:
        gm.close()
        empty.close()


@pytest.mark.gpu
def test_best_relocalizes_and_breaks_ties_by_index(ctx, port):
    """A saved map (scans placed at their true poses) rebuilt by inserting its pointcloud() into a fresh map, a later scan's keypoints, a
    grid of +-1.5 m / +-20 deg around its true pose: the best hypothesis converged within 0.05 m / 0.5 deg of the truth. Identical guesses
    tie; the lower index wins. (max_corresp_dist 1 m: with 2 m a hypothesis stopped unconverged at the iteration cap 8 cm off the truth
    keeps a few more points within range than the converged ones -- the inlier count rewards the range, not convergence.)
    (A structure-rich scene seen mostly above the horizon: on a ground-dominated one the reference's point-to-point rule gives a
    hypothesis that slid along the ground as many inliers as the true pose.)"""
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
        guesses = np.array([port.se3_mul(truth, port.se3_exp(np.array([dx, dy, 0.0, 0.0, 0.0, np.radians(yaw)])))
                            for dx in (-1.5, 0.0, 1.5) for dy in (-1.5, 0.0, 1.5) for yaw in (-20.0, 0.0, 20.0)])
        res = m.icp_multi(kp, guesses, 1.0, 0.5, 100, 1e-4)
        b = res["best"]
        # best is the lexicographic maximum of (inliers, -rms, -index)
        order = sorted(range(len(guesses)), key=lambda i: (-res["inliers"][i], res["rms"][i], i))
        assert b == order[0]
        err = port.se3_log(port.se3_mul(port.se3_inv(truth), res["poses"][b]))
        assert res["converged"][b], (b, res["iters"][b])
        assert np.linalg.norm(err[:3]) < 0.05 and np.degrees(np.linalg.norm(err[3:])) < 0.5, (b, err)
        tie = m.icp_multi(kp, np.stack([guesses[0], guesses[b], guesses[b]]), 1.0, 0.5, 100, 1e-4)
        assert tie["inliers"][1] == tie["inliers"][2] and tie["rms"][1] == tie["rms"][2] and tie["best"] == 1
        assert tie["inliers"][1] > tie["inliers"][0] or (tie["inliers"][1] == tie["inliers"][0] and tie["rms"][1] <= tie["rms"][0])
    finally:
        built.close()
        m.close()


@pytest.mark.gpu
def test_calls_on_a_pipelined_handles_map(ctx, port):
    """icp_multi on local_map() between the register calls of a pipelined handle: the handle's poses, iteration counts and map are those of the
    same run without the calls (the multi loop only reads the map), and the calls return what they return on a plain handle's map."""
    import torch
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    sc = synth.Scene(seed=21)
    traj = synth.loop_trajectory(11, radius=30.0, step=0.7)
    scans = [synth.cast_scan(sc, traj[i], traj[i + 1], beams=16, azimuth_steps=700, seed=300 + i) for i in range(8)]
    rng = np.random.default_rng(8)
    query = scans[3][:, :3].astype(np.float64)[::3]
    guesses = guess_grid(port, rng, 40, 1.0, 0.1)

    def run(spec, calls):
        staged = [torch.from_numpy(s).cuda() for s in scans]
        torch.cuda.synchronize()
        k = ctx.KissICP(deskew=False, icp_max_iteration=60, speculate=spec)
        out, multi = [], []
        for i, t in enumerate(staged):
            if spec and i + 1 < len(staged):
                k.hint_next_dev(staged[i + 1].data_ptr(), len(scans[i + 1]))
            p = k.register_frame_dev(t.data_ptr(), len(scans[i]))
            out.append((p.copy(), k.stats.icp.iterations))
            if calls and i >= 2:
                multi.append((k.local_map().icp_multi(query, guesses, 1.5, 0.5, 30, 1e-4), k.local_map().dump()))
        k.flush()
        dump = k.local_map().dump()
        k.close()
        return out, dump, multi

    a, da, _ = run(True, False)
    b, db, mb = run(True, True)
    c, dc, mc = run(False, True)
    for (pa, ia), (pb, ib) in zip(a, b):
        assert ia == ib and np.array_equal(pa, pb)
    assert all(np.array_equal(x, y) for x, y in zip(da, db))
    # without deskew the pipelined and the plain handle build bit-identical maps, so everything icp_multi returns on them is bit-identical
    for (rb, mapb), (rc, mapc) in zip(mb, mc):
        assert all(np.array_equal(x, y) for x, y in zip(mapb, mapc))
        for key in ("poses", "iters", "converged", "inliers", "rms", "best"):
            assert np.array_equal(rb[key], rc[key]), key


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
    const std::vector<double> world = read_block(f), query = read_block(f), g = read_block(f);
    fclose(f);
    lidar::VoxelHashMap map(1.0, 100.0, 10);
    map.insert_points(points(world));
    std::vector<Sophus::SE3d> guesses(g.size() / 7);
    for (size_t i = 0; i < guesses.size(); ++i) std::copy(g.begin() + 7 * i, g.begin() + 7 * i + 7, guesses[i].data());
    const lidar::ICPMultiResult r = lidar::ICP_multi(map, points(query), guesses, 0.6, 0.2 / 3, 40, 1e-4);
    FILE *o = fopen(argv[2], "wb");
    for (size_t i = 0; i < r.poses.size(); ++i) {
        const limu_icp_hypothesis &h = r.hypotheses[i];
        const double row[11] = {r.poses[i].data()[0], r.poses[i].data()[1], r.poses[i].data()[2], r.poses[i].data()[3], r.poses[i].data()[4],
                                r.poses[i].data()[5], r.poses[i].data()[6], (double)h.iterations, (double)h.converged, (double)h.inliers, h.rms};
        fwrite(row, 8, 11, o);
    }
    const double best = r.best;
    fwrite(&best, 8, 1, o);
    fclose(o);
    return 0;
}
"""


@pytest.mark.gpu
def test_dropin_icp_multi_runs(ctx, port, tmp_path):
    """lidar::ICP_multi from a C++ program linked against the library (reference types replaced by the stand-ins above) returns what
    VoxelHashMap.icp_multi returns for the same map, points and guesses, bit for bit."""
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    import __graft_entry__ as g
    pkg = g.load_package()
    rng = np.random.default_rng(31337)
    gm, om, src = scene(port, ctx, rng, 10, 1500)
    world = gm.pointcloud()
    guesses = guess_grid(port, rng, 20)
    try:
        want = gm.icp_multi(src, guesses, 0.6, 0.2 / 3, 40, 1e-4)
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
        for a in (world, src, guesses):
            a = np.ascontiguousarray(a, np.float64).ravel()
            f.write(np.int64(a.size).tobytes())
            f.write(a.tobytes())
    r = subprocess.run([str(exe), str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    got = np.fromfile(tmp_path / "out.bin", np.float64)
    rows = got[:-1].reshape(len(guesses), 11)
    assert np.array_equal(rows[:, :7], want["poses"])
    assert np.array_equal(rows[:, 7], want["iters"]) and np.array_equal(rows[:, 8], want["converged"]) and np.array_equal(rows[:, 9], want["inliers"])
    assert np.array_equal(rows[:, 10], want["rms"]) and got[-1] == want["best"]
