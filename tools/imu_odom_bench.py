"""Constant-velocity versus IMU-deskewed registration on the c2 workload of bench.py (128 000 points per scan, 48-byte pcl::PointXYZINormal
records in pinned host memory, voxel 1.0 m, cap 10), all through the pipelined path with the next cloud prefetched:
  cv           : limu_odom_register_cloud     + limu_odom_prefetch_cloud      (records + FP64 timestamps, deskew on)
  imu          : limu_odom_register_cloud_imu + limu_odom_prefetch_cloud_imu  (records + an IMU pose table per scan, no timestamps)
  imu_rest     : the same with the IMU windows of a platform at rest (the same per-point work; the motion is left uncompensated)
  cv_no_deskew : cv with deskew off -- the control for imu_rest: nearly the same clouds, so nearly the same Gauss-Newton work
Per arm: R windows on a fresh handle (W warm-up scans, K timed scans between two device synchronisations), the arms alternating window by
window; the median is reported. A separate run with the per-stage event timing on gives the downsample stage (the fused deskew +
voxelize kernel) per scan. The card's name and power limit come from a read-only nvidia-smi query in the same run.

    python tools/imu_odom_bench.py [--steps 150 --warmup 5 --repeats 5] [--out profiles/imu_odom_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else f"nvidia-smi failed: {q.stderr.strip()}"


def imu_tables(pkg, traj, recs, seed, moving=True, dt=0.005, scan_dt=0.1, t_begin=50.0):
    """IMU samples (moving: along the trajectory -- yaw rate, centripetal acceleration; else a platform at rest; gravity and noise of
    0.002 rad/s / 0.03 m/s^2 in both) through limu_imu_forward_pass, one window per scan, state carried over.
    -> [(table, rot_end, pos_lidar_end, p_imu_lidar)]."""
    rng = np.random.default_rng(seed)
    n = len(recs)
    T = t_begin - 0.004 + np.arange(int((scan_dt * n + 0.06) / dt) + 2) * dt
    k = np.clip(((T - t_begin) / scan_dt).astype(int), 0, n - 1)
    yaw_rate = np.diff(traj[: n + 1, 2]) / scan_dt
    speed = np.linalg.norm(np.diff(traj[: n + 1, :2], axis=0), axis=1) / scan_dt
    if not moving:
        yaw_rate, speed = yaw_rate * 0.0, speed * 0.0
    z = np.zeros(len(T))
    gyr = np.stack([z, z, yaw_rate[k]], 1) + rng.normal(size=(len(T), 3)) * 0.002
    acc = np.stack([z, speed[k] * yaw_rate[k], z + 9.81], 1) + rng.normal(size=(len(T), 3)) * 0.03
    imu = np.concatenate([T[:, None], gyr, acc], 1)
    pil = np.array([0.1, -0.05, 0.2])
    st = pkg.ImuState()
    st.quat[:], st.bat[:], st.grav[:], st.p_imu_lidar[:] = [1, 0, 0, 0], [1, 1, 1], [0, 0, -9.81], pil
    st.mean_acc_norm, st.gravity_norm = float(np.linalg.norm(acc.mean(0))), 9.81
    st.acc_s_last[:], st.ang_vel_last[:] = acc[0], gyr[0]
    out, start = [], 0
    for i, r in enumerate(recs):
        beg, last_ms = t_begin + i * scan_dt, float(r[-1, 9])
        end = max(int(np.searchsorted(T, beg + last_ms / 1000.0)), start + 1)
        table, rot_end, ple = pkg.imu_forward_pass(st, imu[start:end + 1], beg, last_ms)
        st.pos[:], st.vel[:], st.quat[:] = st.tracker_pos[:], st.tracker_vel[:], st.tracker_quat[:]
        out.append((table, rot_end, ple, pil))
        start = end
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=150)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "imu_odom_bench.json"))
    a = ap.parse_args()
    import bench
    import __graft_entry__ as g
    pkg = g.load_package()
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    W, K, R = a.warmup, a.steps, a.repeats
    bargs = bench.parse([])                                        # the c2 workload: 128 000 points, 64 beams x 2000, 1 m/scan, voxel 1.0, cap 10
    scans = bench.make_scans(bargs, W + K, 42, "cuda:0")
    traj = synth.loop_trajectory(W + K + 1, radius=30.0, step=bargs.step_m)
    n_pts = bargs.points
    rec = [pkg.PinnedArray((n_pts, 12), np.float32) for _ in scans]
    tss = [pkg.PinnedArray((n_pts,), np.float64) for _ in scans]
    for r_, t_, s in zip(rec, tss, scans):
        r_.array[...] = 0
        r_.array[:, :3] = s[:, :3]
        r_.array[:, 3] = 1.0
        r_.array[:, 9] = (s[:, 3].astype(np.float64) * 100.0).astype(np.float32)   # curvature = offset time in ms (100 ms sweep)
        t_.array[...] = s[:, 3]
    imu_arms = {"imu": imu_tables(pkg, traj, [r_.array for r_ in rec], 11), "imu_rest": imu_tables(pkg, traj, [r_.array for r_ in rec], 11, moving=False)}
    ctx = pkg.Context(0)
    cfg = dict(voxel_size=bargs.voxel, cap=bargs.cap, icp_max_iteration=bargs.max_iter, speculate=True)

    def step(o, arm, i, last):
        if arm.startswith("cv"):
            if not last:
                o.prefetch_cloud(rec[i + 1].array, 48, tss[i + 1].array)
            o.register_cloud(rec[i].array, 48, tss[i].array, copy=False)
        else:
            imus = imu_arms[arm]
            if not last:
                o.prefetch_cloud_imu(rec[i + 1].array, 48, 36, *imus[i + 1])
            o.register_cloud_imu(rec[i].array, 48, 36, *imus[i], copy=False)

    def window(arm, profile=False):
        o = ctx.KissICP(deskew=arm != "cv_no_deskew", **cfg)
        for i in range(W):
            step(o, arm, i, False)
        o.flush()
        ctx.sync()
        if profile:
            ctx.set_profiling(True)
        t0 = time.perf_counter()
        hits = iters = 0
        for i in range(W, W + K):
            step(o, arm, i, i + 1 == W + K)
            hits += o.stats.reserved0
            iters += o.stats.icp.iterations
        o.flush()
        ctx.sync()
        sec = time.perf_counter() - t0
        prof = ctx.profile() if profile else None
        if profile:
            ctx.set_profiling(False)
        o.close()
        return sec, hits, iters / K, prof

    arms = ("cv", "imu", "imu_rest", "cv_no_deskew")
    res = {arm: [] for arm in arms}
    hits, iters = {}, {}
    for _ in range(R):
        for arm in arms:
            sec, h, it, _ = window(arm)
            res[arm].append(K / sec)
            hits[arm], iters[arm] = h, it
    stage = {}
    for arm in arms:
        _, _, _, (ms, frames) = window(arm, profile=True)
        stage[arm] = {k: v / max(frames, 1) for k, v in ms.items()}
    out = {
        "gpu": gpu_info(),
        "workload": bench.workload_text(bargs, "c2") + f"; 48-byte records from pinned host memory; K = {K}, W = {W}, {R} fresh-handle windows per arm, arms alternating",
        "scans_per_s": {arm: float(np.median(v)) for arm, v in res.items()},
        "windows_scans_per_s": res,
        "prepared_ahead_per_window": hits,
        "icp_iterations_per_scan": iters,
        "imu_vs_cv": float(np.median(res["imu"]) / np.median(res["cv"])),
        "imu_rest_vs_cv_no_deskew": float(np.median(res["imu_rest"]) / np.median(res["cv_no_deskew"])),
        "arms": {"cv": "register_cloud + prefetch_cloud, constant-velocity deskew on", "imu": "register_cloud_imu + prefetch_cloud_imu, IMU windows along the trajectory",
                 "imu_rest": "the same with the IMU windows of a platform at rest: the same per-point work, the motion left uncompensated",
                 "cv_no_deskew": "register_cloud + prefetch_cloud with deskew off: the control for imu_rest (the same clouds up to rounding, so the same "
                                 "Gauss-Newton work)"},
        "stage_ms_per_scan": stage,
        "stage_note": "separate run with limu_ctx_set_profiling on: CUDA events around each launch; downsample = the fused deskew + voxelize kernel "
                      "(k_voxelize_lean / k_voxelize_imu_lean beside the map update); its events sit in the pipe stream",
        "h2d_bytes_per_scan": {"cv": n_pts * 56, "imu": n_pts * 48 + int(np.mean([len(t[0]) for t in imu_arms["imu"]])) * 176},
        "source_hash": pkg.source_hash(),
    }
    print(json.dumps(out, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    for x in rec + tss:
        x.free()
    ctx.close()


if __name__ == "__main__":
    main()
