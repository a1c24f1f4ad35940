"""Multi-hypothesis ICP (limu_icp_multi, one launch) against a host loop of limu_icp_ex calls, one per guess: the relocalization workload.

Scenes (bench.py's workloads): "c2" = configs[1] (64-beam LiDAR, 128 000 points per scan, voxel 1.0 m, cap 10) and "c3" = a configs[2]-sized
case (128-beam urban canyon, 512 000 points per scan, voxel 0.5 m, cap 20). An odometry handle runs over the first scans; its local map is
saved with pointcloud() and rebuilt in a fresh map (the relocalization recipe of INTEGRATION.md); a later scan's keypoints (the cloud the
handle registered) are the query and the handle's pose of that scan the truth. Guesses: a grid of x, y (+-3 m) and yaw (+-45 deg) around it.
For every K both arms are timed with a host clock around work that ends in a device synchronisation, after a warm-up of both, alternating
arm by arm, R repeats; median and spread (min, max) are reported, as relocalizations per second and hypotheses per second. The card's name
and power limit come from a read-only nvidia-smi query in the same run.

    python tools/icp_multi_bench.py [--repeats 5] [--ks 1,8,32,128,512] [--out profiles/icp_multi_bench.json]
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

SCENES = {
    "c2": dict(scene=dict(), elev=(-25.0, 2.0), beams=64, azimuth_steps=2000, voxel=1.0, cap=10, step=1.0, map_scans=20, query_scan=24),
    "c3": dict(scene=dict(street=True, n_boxes=60, n_cyl=30), elev=(-25.0, 15.0), beams=128, azimuth_steps=4000, voxel=0.5, cap=20, step=1.0,
               map_scans=12, query_scan=15),
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else f"nvidia-smi failed: {q.stderr.strip()}"


def guess_grid(port, truth, k, seed):
    """k guesses: x, y in +-3 m and yaw in +-45 deg around the truth (a regular grid for perfect cubes, else seeded uniform draws)."""
    rng = np.random.default_rng(seed)
    side = round(k ** (1.0 / 3.0))
    if side ** 3 == k:
        lin = np.linspace(-1.0, 1.0, side) if side > 1 else np.zeros(1)
        d = np.array([(x, y, z) for x in lin for y in lin for z in lin])
    else:
        d = rng.uniform(-1.0, 1.0, size=(k, 3))
    return np.array([port.se3_mul(truth, port.se3_exp(np.array([3.0 * a, 3.0 * b, 0.0, 0.0, 0.0, np.radians(45.0) * c]))) for a, b, c in d])


def prepare(pkg, ctx, synth, name):
    w = SCENES[name]
    scene = synth.Scene(seed=42, **w["scene"])
    traj = synth.loop_trajectory(w["query_scan"] + 2, radius=30.0, step=w["step"])
    cast = lambda i: synth.cast_scan(scene, traj[i], traj[i + 1], beams=w["beams"], azimuth_steps=w["azimuth_steps"], elev=w["elev"],
                                     seed=1000 + i, device="cuda")
    k = ctx.KissICP(voxel_size=w["voxel"], cap=w["cap"], deskew=True, icp_max_iteration=500, speculate=False)
    for i in range(w["map_scans"]):
        k.register_frame(cast(i))
    saved = k.local_map().pointcloud()
    for i in range(w["map_scans"], w["query_scan"]):
        k.register_frame(cast(i))
    _, kp, truth = k.register_frame(cast(w["query_scan"]))
    k.close()
    m = ctx.VoxelHashMap(w["voxel"], 100.0, w["cap"])
    m.insert_points(saved)
    return m, kp, truth, w


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return time.perf_counter() - t0, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--ks", default="1,8,32,128,512")
    ap.add_argument("--scenes", default="c2,c3")
    ap.add_argument("--max-iter", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "icp_multi_bench.json"))
    a = ap.parse_args()
    import __graft_entry__ as g
    import oracle
    pkg = g.load_package()
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    port = oracle.load_port()
    ctx = pkg.Context(0)
    ks = [int(x) for x in a.ks.split(",")]
    record = {"gpu": gpu_info(), "repeats": a.repeats, "max_iter": a.max_iter, "scenes": {}}
    for name in a.scenes.split(","):
        m, kp, truth, w = prepare(pkg, ctx, synth, name)
        tau, th, eps = 3.0 * w["voxel"], w["voxel"], 1e-4
        seq = lambda gs: [m.icp(kp, q, tau, th, a.max_iter, eps) for q in gs]
        multi = lambda gs: m.icp_multi(kp, gs, tau, th, a.max_iter, eps)
        nv, npts = m.size()
        rows = []
        for k in ks:
            gs = guess_grid(port, truth, k, seed=k)
            rs, rm = seq(gs), multi(gs)   # warm-up of both arms (and the scratch they grow)
            ts, tm = [], []
            for _ in range(a.repeats):
                ts.append(timed(lambda: seq(gs))[0])
                tm.append(timed(lambda: multi(gs))[0])
            it_s = np.array([r["iters"] for r in rs])
            dpose = max(float(np.abs(np.array([r["pose"] for r in rs]) - rm["poses"]).max()), 0.0)
            b = rm["best"]
            err = port.se3_log(port.se3_mul(port.se3_inv(truth), rm["poses"][b]))
            row = {"k": k, "seq_s": {"median": float(np.median(ts)), "min": float(min(ts)), "max": float(max(ts))},
                   "multi_s": {"median": float(np.median(tm)), "min": float(min(tm)), "max": float(max(tm))},
                   "speedup_median": float(np.median(ts) / np.median(tm)),
                   "relocalizations_per_s": {"seq": float(1.0 / np.median(ts)), "multi": float(1.0 / np.median(tm))},
                   "hypotheses_per_s": {"seq": float(k / np.median(ts)), "multi": float(k / np.median(tm))},
                   "iters_per_hypothesis": {"mean": float(rm["iters"].mean()), "max": int(rm["iters"].max())},
                   "iters_equal_to_seq": bool(np.array_equal(it_s, rm["iters"])), "max_pose_diff_vs_seq": dpose,
                   "best": int(b), "best_inliers": int(rm["inliers"][b]), "best_rms": float(rm["rms"][b]),
                   "best_err_m": float(np.linalg.norm(err[:3])), "best_err_deg": float(np.degrees(np.linalg.norm(err[3:])))}
            rows.append(row)
            print(json.dumps({"scene": name, **row}), flush=True)
        record["scenes"][name] = {"keypoints": int(len(kp)), "map_voxels": int(nv), "map_points": int(npts), "voxel": w["voxel"], "cap": w["cap"],
                                  "beams": w["beams"], "azimuth_steps": w["azimuth_steps"], "max_corresp_dist": tau, "kernel": th, "rows": rows}
        m.close()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(record, f, indent=1)
    print("gpu:", record["gpu"])


if __name__ == "__main__":
    main()
