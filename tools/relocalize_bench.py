"""Pose scoring (limu_map_score_poses) against limu_icp_multi with 0 iterations on the same poses, and global relocalization (limu_relocalize)
end to end: the workload of a relocalization without a coarse pose.

Scenes: "c2" and "c3" of tools/icp_multi_bench.py, prepared by its `prepare` (an odometry handle's local map saved with pointcloud() and
rebuilt in a fresh map; a later scan's keypoints are the query, the handle's pose of that scan the truth).
Score throughput: K poses drawn uniformly over x, y in +-10 m and yaw in +-180 deg around the truth; both arms get the same poses (host
arrays in, scores out), are warmed up, then alternated arm by arm for R repeats; median and spread (min, max) of a host clock around the
synchronised call, as candidate-points per second (K x keypoints / s). The inlier counts of the two arms must be equal. Beyond the K the
loop arm can take in reasonable time, the scoring arm runs alone.
End to end: limu_relocalize over +-10 m / 1 m / 36 yaw steps and +-25 m / 0.5 m / 72 yaw steps around a center 3.4 m and 17 deg off the truth
(between grid points), n_refine 32, at max_corresp_dist 1 m (the 1 m grid step) and at the throughput arms' 3 voxels: the host-clock
time of the call (median and spread of R repeats after a warm-up), then one more call
under torch.profiler whose kernel times are summed by phase (score: k_score_poses; select: k_select_*, k_grid_poses; refine: k_icp_*),
and the winner's error against the truth. The card's name and power limit come from a read-only nvidia-smi query in the same run.

    python tools/relocalize_bench.py [--repeats 5] [--out profiles/relocalize_bench.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from icp_multi_bench import gpu_info, prepare  # noqa: E402


def qmul(a, b):
    """Hamilton product of [k, 4] (x, y, z, w) quaternion arrays."""
    ax, ay, az, aw = a.T
    bx, by, bz, bw = b.T
    return np.stack([aw * bx + ax * bw + ay * bz - az * by, aw * by + ay * bw + az * bx - ax * bz,
                     aw * bz + az * bw + ax * by - ay * bx, aw * bw - ax * bx - ay * by - az * bz], axis=1)


def planar_poses(truth, k, seed):
    """k poses truth * {yaw, (x, y, 0)} with x, y uniform in +-10 m and yaw uniform in +-180 deg (vectorised: the bench needs millions)."""
    rng = np.random.default_rng(seed)
    x, y, t = rng.uniform(-10, 10, k), rng.uniform(-10, 10, k), rng.uniform(-np.pi, np.pi, k)
    q = qmul(np.broadcast_to(truth[:4], (k, 4)), np.stack([np.zeros(k), np.zeros(k), np.sin(t / 2), np.cos(t / 2)], axis=1))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    v = np.stack([x, y, np.zeros(k)], axis=1)   # rotate (x, y, 0) by truth's rotation, then add its translation
    qv, w = truth[:3], truth[3]
    uv = 2.0 * np.cross(qv, v)
    tr = v + w * uv + np.cross(qv, uv) + truth[4:]
    return np.concatenate([q, tr], axis=1)


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return time.perf_counter() - t0, r


def stats(ts):
    return {"median": float(np.median(ts)), "min": float(min(ts)), "max": float(max(ts))}


def phase_split(fn):
    """Device time of one call by phase, from torch.profiler's CUDA kernel records."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {"score": 0.0, "select": 0.0, "refine": 0.0, "other": 0.0}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        name, us = e.name, e.device_time
        key = ("score" if "k_score_poses" in name else "select" if ("k_select" in name or "k_grid_poses" in name)
               else "refine" if "k_icp" in name else "other")
        out[key] += us / 1e3
    return {k + "_ms": v for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--ks", default="1024,4096,16384,65536")
    ap.add_argument("--ks-alone", default="262144,1048576,4194304")
    ap.add_argument("--scenes", default="c2,c3")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "relocalize_bench.json"))
    a = ap.parse_args()
    import __graft_entry__ as g
    import oracle
    pkg = g.load_package()
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    port = oracle.load_port()
    ctx = pkg.Context(0)
    record = {"gpu": gpu_info(), "repeats": a.repeats, "scenes": {}}
    for name in a.scenes.split(","):
        m, kp, truth, w = prepare(pkg, ctx, synth, name)
        tau, th, eps, max_iter = 3.0 * w["voxel"], w["voxel"], 1e-4, 50
        n = len(kp)
        score = lambda p: m.score_poses(kp, p, tau)
        loop0 = lambda p: m.icp_multi(kp, p, tau, th, 0, eps)
        rows = []
        for k in [int(x) for x in a.ks.split(",") if x] + [-int(x) for x in a.ks_alone.split(",") if x]:
            alone, k = k < 0, abs(k)
            p = planar_poses(truth, k, seed=k)
            rs = score(p)
            rl = None if alone else loop0(p)   # warm-up of both arms (and the scratch they grow)
            tsc, tlo = [], []
            for _ in range(a.repeats):
                tsc.append(timed(lambda: score(p))[0])
                if not alone:
                    tlo.append(timed(lambda: loop0(p))[0])
            row = {"k": k, "score_s": stats(tsc), "score_candidate_points_per_s": float(k * n / np.median(tsc))}
            if not alone:
                row.update({"icp_multi0_s": stats(tlo), "icp_multi0_candidate_points_per_s": float(k * n / np.median(tlo)),
                            "speedup_median": float(np.median(tlo) / np.median(tsc)),
                            "inliers_equal": bool(np.array_equal(rs["inliers"], rl["inliers"])),
                            "max_rms_rel_diff": float(np.max(np.abs(rs["rms"] - rl["rms"]) / np.maximum(rl["rms"], 1e-300)))})
            rows.append(row)
            print(json.dumps({"scene": name, **row}), flush=True)
        center = port.se3_mul(truth, port.se3_exp(np.array([-3.37, 2.71, 0.0, 0.0, 0.0, np.radians(-17.3)])))
        e2e = []
        for (half, step, nyaw), dist in [(g_, d_) for g_ in ((10.0, 1.0, 36), (25.0, 0.5, 72)) for d_ in (1.0, tau)]:
            nxy = int(round(2 * half / step)) + 1
            call = lambda: m.relocalize(kp, center, nxy, nxy, nyaw, step, 2 * np.pi / nyaw, 32, dist, th, max_iter, eps)
            r = call()
            ts = [timed(call)[0] for _ in range(a.repeats)]
            b = r["best"]
            err = port.se3_log(port.se3_mul(port.se3_inv(truth), r["poses"][b]))
            row = {"half_extent_m": half, "step_xy_m": step, "nyaw": nyaw, "candidates": nxy * nxy * nyaw, "n_refine": 32, "max_corresp_dist": dist,
                   "time_s": stats(ts),
                   "candidate_points_per_s": float(nxy * nxy * nyaw * n / np.median(ts)), **phase_split(call),
                   "best": int(b), "best_index": int(r["index"][b]), "best_converged": bool(r["converged"][b]),
                   "best_err_m": float(np.linalg.norm(err[:3])), "best_err_deg": float(np.degrees(np.linalg.norm(err[3:]))),
                   "top_coarse_inliers": int(r["coarse_inliers"][0])}
            e2e.append(row)
            print(json.dumps({"scene": name, **row}), flush=True)
        nv, npts = m.size()
        record["scenes"][name] = {"keypoints": int(n), "map_voxels": int(nv), "map_points": int(npts), "voxel": w["voxel"], "cap": w["cap"],
                                  "max_corresp_dist": tau, "kernel": th, "max_iter": max_iter, "score": rows, "relocalize": e2e}
        m.close()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(record, f, indent=1)
    print("gpu:", record["gpu"])


if __name__ == "__main__":
    main()
