#!/usr/bin/env python
"""bench.py -- LiDAR odometry hot path throughput (BASELINE.json metric) on B200.

Workload (BASELINE.json configs[1], SURVEY section 8d "C2"): synthetic 64-beam spinning LiDAR, 128 000
points per scan, loop trajectory of radius 30 m at 1 m/scan, voxel 1.0 m, max_points_per_voxel 10,
deskew on. One STEP = one scan through KissICP::register_frame (deskew -> 0.5v/1.5v first-wins
downsample -> IQR -> fused correspondence + normal-equation + Gauss-Newton loop -> map insert/evict).

  python bench.py [--gpus N] [--steps K] [--warmup W]            the B200 path (liblimu_cuda.so)
  python bench.py --impl reference ...                           the reference's own CPU code (oracle/_ref)

A timed WINDOW = a fresh odometry handle, W untimed warm-up scans, then exactly K timed scans bracketed by
stream sync + barrier on both sides. The window is repeated --repeats times on fresh handles; `value` is the
MEDIAN window (max over ranks inside each window), the spread is printed next to it.

N > 1 (torchrun): one independent sequence per GPU (configs[3], "fleet replay"): weak scaling, no
data-path collective; torch.distributed is used only for barriers and for gathering the per-rank times.
After the replica windows the ranks run configs[4] (one 4 M-point scan point-sharded over the N GPUs,
fused NVLink exchange inside the registration kernel) and print it as the `sharded` record.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "deskew+ICP+GN-loop odometry throughput at 128k pts/scan"
UNIT = "scans/s"

# Synthetic sequences (lidar-imu-slam_b200/synth.py). "c2" is SURVEY's C2 scene: ground plane + 28 boxes + 14 cylinders seen by a
# -25..+2 degree sensor. On it the reference's own-voxel-only, point-to-point rule barely moves (sensor-centric ground rings pull the
# estimate to zero motion) -- both arms alike. "tracking" is a structure-rich scene without ground returns (+0.5..+30 degrees, 150
# boxes + 60 cylinders) on which the reference's rule follows the true trajectory, so the local map grows along the loop, the eviction
# fires and k-bar / f_miss are those of a moving sensor.
WORKLOADS = {
    "c2": dict(scene=dict(), elev=(-25.0, 2.0), beams=64, azimuth_steps=2000,
               text="configs[1]: synthetic {beams}-beam LiDAR, {points} pts/scan, loop r=30 m at {step} m/scan, voxel {voxel} m, cap {cap}, deskew on"),
    "c3": dict(scene=dict(street=True, n_boxes=60, n_cyl=30), elev=(-25.0, 15.0), beams=128, azimuth_steps=4000,
               text="configs[2]: synthetic {beams}-beam LiDAR in an urban canyon (two facade rows + ground + clutter), {points} pts/scan, loop r=30 m at {step} m/scan, "
                    "voxel {voxel} m, cap {cap}, deskew on, local map of ~45 M points resident in HBM"),
    "tracking": dict(scene=dict(n_boxes=150, n_cyl=60), elev=(0.5, 30.0), beams=64, azimuth_steps=3000,
                     text="tracking regime: {beams}-beam LiDAR looking up (+0.5..+30 deg, no ground returns), 150 boxes + 60 cylinders, {points} pts/scan, "
                          "loop r=30 m at {step} m/scan, voxel {voxel} m, cap {cap}, deskew on"),
}


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=150, help="scans timed per window; the loop of radius 30 m closes after ~188 scans at 1 m/scan, where the reference's "
                    "Gauss-Newton loop stops converging and runs to its 500-iteration cap (both arms alike): W + K <= 180 stays in the converging regime")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=5, help="timed windows per arm (fresh handle each); the median is reported")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--points", type=int, default=128000)
    ap.add_argument("--beams", type=int, default=64)
    ap.add_argument("--azimuth-steps", type=int, default=2000)
    ap.add_argument("--step-m", type=float, default=1.0, help="metres travelled per scan (10 m/s at 10 Hz)")
    ap.add_argument("--voxel", type=float, default=1.0)
    ap.add_argument("--cap", type=int, default=10)
    ap.add_argument("--max-iter", type=int, default=500)
    ap.add_argument("--icp-mode", type=int, default=0, help="0 = the reference's registration rules (the parity configuration, default); 1 = nearest of the "
                    "27-cell neighbourhood, 2 = point-to-plane, 3 = both (opt-in variants, SURVEY 8f N2; the CPU arm is then the C oracle)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--ref-seconds", type=float, default=150.0, help="budget of the --impl reference run")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary records (tracking workload, icp_mode 3, e2e_cloud, loop closure, kernel mode, sharded)")
    ap.add_argument("--no-speculate", action="store_true", help="LIMU_OPT_SPECULATE off (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed windows of `value`, write what their last timed step returned "
                    "(rank 0) as DIR/pose.npy and DIR/frame_stats.npy (float64), to compare two builds on the same seeded inputs; "
                    "needs --impl b200 and --steps >= 1")
    args = ap.parse_args(argv)
    if args.dump_outputs and (args.impl != "b200" or args.steps < 1):
        ap.error("--dump-outputs writes the last timed step of the b200 path: it needs --impl b200 and --steps >= 1")
    return args


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def pin_cpus(local_rank, world):
    """One core set per rank: by default every rank of the node inherits the same affinity mask, so eight launch loops (and their
    helper threads) compete for whatever cores the scheduler picks. Returns the cores this rank now owns."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        if world <= 1 or len(cpus) < 2 * world:
            return cpus
        per = len(cpus) // world
        mine = cpus[local_rank * per:(local_rank + 1) * per]
        os.sched_setaffinity(0, mine)
        return mine
    except Exception:
        return []


def workload_text(args, name="c2", n_gpus=1):
    w = WORKLOADS[name]
    beams = args.beams if name == "c2" else w["beams"]
    t = w["text"].format(beams=beams, points=args.points, step=args.step_m, voxel=args.voxel, cap=args.cap)
    return t + (f"; configs[3]: {n_gpus} independent sequences, one per GPU (same world, per-vehicle sensor-noise realisation)" if n_gpus > 1 else "")


def make_config(args, n_gpus):
    """Both arms print the SAME object (the driver compares the two configs); what is specific to an arm goes to `arm_note`."""
    return {
        "workload": workload_text(args, "c2", n_gpus),
        "l2": "B200 arm: L2 flushed (512 MB write) after staging, every step reads a different scan, none re-read, the local map is persistent state; reference arm: host caches as they come",
        "timing": "B200 arm: window = fresh handle, W warm-up scans, K timed scans bracketed by stream sync + barrier; per rank max(host wall, CUDA events on the library stream); max over ranks; median of the windows. Reference arm: K consecutive scans after W warm-up scans, host wall clock",
        "icp_max_iteration": args.max_iter,
        "icp_mode": args.icp_mode,
    }


def make_scans(args, n_scans, seed, device, workload="c2", first=0, vehicle=0):
    """The sequence of one vehicle: scans first .. first+n_scans-1 along the loop, each resized to exactly --points rows.
    `seed` picks the world, `vehicle` the realisation of the sensor noise (fleet replay: N vehicles in the same world)."""
    import __graft_entry__ as g
    g.load_package()
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    w = WORKLOADS[workload]
    scene = synth.Scene(seed=seed, **w["scene"])
    traj = synth.loop_trajectory(first + n_scans + 1, radius=30.0, step=args.step_m)
    beams = args.beams if workload == "c2" else w["beams"]
    az = args.azimuth_steps if workload == "c2" else w["azimuth_steps"]
    scans = []
    for i in range(first, first + n_scans):
        s = synth.cast_scan(scene, traj[i], traj[i + 1], beams=beams, azimuth_steps=az, elev=w["elev"], seed=(seed + 7919 * vehicle) * 100003 + i, device=device)
        scans.append(synth.pad_scan(s, args.points, seed=i + 1000003 * vehicle))
    return scans


def true_pose_xy(args, i):
    import __graft_entry__ as g
    g.load_package()
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    return synth.loop_trajectory(i + 2, radius=30.0, step=args.step_m)[i + 1][:2]


class ClockSampler:
    """SM clock and throttle reasons of this rank's GPU DURING the timed windows, read in-process through NVML every 10 ms.
    (Round 1 spawned one `nvidia-smi -lms 100` per rank: its start-up enumerates every GPU of the node under the driver's global
    lock, inside a 4 ms window -- one of the suspects of the 1 -> 8 collapse -- and 100 ms polling saw 0-1 samples per window.)"""

    def __init__(self, torch, local_rank):
        self.rows, self.stop_flag, self.in_window, self.h, self.err = [], False, False, None, None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            p = torch.cuda.get_device_properties(local_rank)
            try:
                bus = f"{getattr(p, 'pci_domain_id', 0):08X}:{p.pci_bus_id:02X}:{p.pci_device_id:02X}.0"
                self.h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                idx = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
                self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:   # noqa: BLE001
            self.err = repr(e)

    def start(self):
        if self.h is None:
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                self.rows.append((self.in_window, float(mhz), int(rs)))
            except Exception:
                pass
            time.sleep(0.010)

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"NVML unavailable: {self.err}"], "samples": 0}
        self.stop_flag = True
        self.t.join(timeout=1.0)
        nv = self.nv
        names = [("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)]
        inw = [r for r in self.rows if r[0]]
        use = inw if inw else self.rows
        reasons = [n for n, bit in names if any(r[2] & bit for r in use)]
        return {"sm_mhz": float(np.median([r[1] for r in use])) if use else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(use), "samples_inside_timed_windows": len(inw), "how": "NVML in-process, 10 ms period, samples taken while a timed window was open"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def profiled_traffic(pkg):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, per launch, from the committed ncu --set full capture of this
    command -- ONLY if that capture was taken from the library that is loaded now (same source hash); otherwise null with the reason."""
    path = os.path.join(ROOT, "profiles", "r2_frame_kernels_ncu.json")
    try:
        d = json.load(open(path))
    except Exception:
        return None, "no ncu capture committed for this round (profiles/r2_frame_kernels_ncu.json)"
    have = pkg.source_hash()
    if d.get("source_hash") != have:
        return None, f"stale: the committed capture is of source hash {d.get('source_hash')}, the loaded library is {have}"
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    vals = []
    for l in d.get("launches", []):
        if "k_icp_persistent" in l["kernel"]:
            r, ru = l["dram__bytes_read.sum"].split()
            w, wu = l["dram__bytes_write.sum"].split()
            vals.append(float(r) * unit[ru] + float(w) * unit[wu])
    return (float(np.mean(vals)) if vals else None), "ncu --set full, cold cache, per launch (profiles/r2_frame_kernels_ncu.json)"


def k4_bytes(n_q, iters, kbar, fmiss):
    """Algorithmic bytes of the fused registration loop (SURVEY section 8d): per query per iteration
    24 B query + 16 B own-voxel slot + 24*kbar B candidate points + fmiss * 27 * 16 B fallback probes."""
    return iters * n_q * (24.0 + 16.0 + 24.0 * kbar + fmiss * 27 * 16.0)


def frame_kernel_bytes(n_q, iters, kbar, fmiss, n_src0, n_down, map_voxels):
    """SURVEY section 8d for what the persistent frame kernel does: the loop above + the IQR filter (24 B per candidate keypoint) + the map
    insert (K3: 64 B per inserted point) + the eviction over the OCCUPIED voxels (4 B list entry + 16 B slot each), as the reference does."""
    return k4_bytes(n_q, iters, kbar, fmiss) + 24.0 * n_src0 + 64.0 * n_down + 20.0 * map_voxels


def cpu_reference_api(icp_mode=0, mt=True):
    import oracle
    if icp_mode == 0 and os.path.exists(oracle.REF_MT_SO if mt else oracle.REF_SO):
        return oracle.load_ref(mt=mt), "reference"
    return oracle.load_port(), "port"   # the opt-in variants do not exist in the reference: the C oracle defines them


def time_cpu(args, scans, warmup, max_steps, budget_s, mt=True, keep=False):
    """The reference's own register_frame on the host cores over a bounded prefix of the same sequence."""
    api, kind = cpu_reference_api(args.icp_mode, mt)
    k = api.Kiss(voxel_size=args.voxel, max_range=getattr(args, "max_range", 100.0), cap=args.cap, deskew=True, icp_max_iteration=args.max_iter)
    if args.icp_mode:
        k.set_mode(args.icp_mode)
    xyz = [np.ascontiguousarray(s[:, :3]) for s in scans]
    ts = [s[:, 3].astype(np.float64) for s in scans]
    sizes = []
    for i in range(min(warmup, len(scans))):
        d, s, _ = k.register_cloud(xyz[i], ts[i])
        sizes.append((len(d), len(s)))
    done, t0 = 0, time.perf_counter()
    for i in range(warmup, min(len(scans), warmup + max_steps)):
        d, s, _ = k.register_cloud(xyz[i], ts[i])
        sizes.append((len(d), len(s)))
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    out = {"done": done, "dt": dt, "kind": kind, "cores": api.num_threads() if mt else 1}
    if keep:
        out["poses"], out["sizes"] = k.poses(), sizes
    return out


def cpu_stage_split(args, scan, mt=True):
    """BASELINE.md section 4: the reference's stages timed one by one on one representative scan of the sequence (same inputs, stand-alone
    calls of the reference's own functions): downsample = voxelize (2 x voxel_downsample + IQR), correspondences / align / transform = ONE
    Gauss-Newton iteration's share, insert = VoxelHashMap::insert_points of the downsampled scan."""
    api, kind = cpu_reference_api(0, mt)
    xyz = scan[:, :3].astype(np.float64)
    t = {}
    t0 = time.perf_counter(); src, down = api.voxelize(xyz, args.voxel); t["downsample_ms"] = 1e3 * (time.perf_counter() - t0)
    m = api.Map(args.voxel, 100.0, args.cap)
    t0 = time.perf_counter(); m.insert(down); t["insert_ms"] = 1e3 * (time.perf_counter() - t0)
    sigma = 2.0
    t0 = time.perf_counter(); s_, t_ = m.correspondences(src, 3.0 * sigma); t["correspondences_ms_per_iteration"] = 1e3 * (time.perf_counter() - t0)
    t0 = time.perf_counter(); api.align(s_, t_, sigma / 3.0); t["align_ms_per_iteration"] = 1e3 * (time.perf_counter() - t0)
    T = np.array([0.0, 0.0, 0.0, 1.0, 0.01, 0.0, 0.0])
    t0 = time.perf_counter(); api.transform(T, src); t["transform_ms_per_iteration"] = 1e3 * (time.perf_counter() - t0)
    t.update({"kind": kind, "n_down": len(down), "n_keypoints": len(src), "n_correspondences": len(s_),
              "note": "fresh map holding only this scan: the sequence's map is larger, its insert and eviction slower (std::next(map.begin(), k) is O(V) per voxel)"})
    return {k: (round(v, 3) if isinstance(v, float) else v) for k, v in t.items()}


def parity_record(args, scans, gpu_poses, gpu_frames, cpu):
    """Poses / sizes of the CUDA path against the compiled reference over the scans the CPU leg covered, iterations against the C port
    (the reference does not export its iteration count; the port is pinned to it by tests/test_oracle_pin.py)."""
    import oracle
    n = min(len(cpu["poses"]), len(gpu_poses))
    if n == 0:
        return None
    dp = np.abs(np.asarray(gpu_poses[:n]) - cpu["poses"][:n])
    port = oracle.load_port()
    k = port.Kiss(voxel_size=args.voxel, max_range=getattr(args, "max_range", 100.0), cap=args.cap, deskew=True, icp_max_iteration=args.max_iter)
    its = []
    for i in range(n):
        k.register_cloud(np.ascontiguousarray(scans[i][:, :3]), scans[i][:, 3].astype(np.float64))
        its.append(k.last_iterations())
    g_it = [int(f[1]) for f in gpu_frames[:n]]
    return {"scans": n, "max_dt_m": float(dp[:, 4:].max()), "max_dq": float(dp[:, :4].max()),
            "iters_equal": bool(g_it == its), "n_down_equal": bool([int(f[4]) for f in gpu_frames[:n]] == [s[0] for s in cpu["sizes"][:n]]),
            "n_keypoints_equal": bool([int(f[0]) for f in gpu_frames[:n]] == [s[1] for s in cpu["sizes"][:n]]),
            "tolerance": "1e-5 m / 1e-6 (quaternion components) per update (north star)", "ok": bool(dp[:, 4:].max() < 1e-5 and dp[:, :4].max() < 1e-6 and g_it == its),
            "against": f"oracle/_ref ({cpu['kind']}: the reference's own sources compiled) for poses and cloud sizes; oracle C port for iterations"}


FRAME_STATS_ORDER = ("n_points", "n_down", "n_keypoints", "sigma", "icp.iterations", "icp.converged", "icp.last_ncorr", "icp.mean_candidates",
                     "icp.miss_fraction", "deskewed")


def dump_outputs(out_dir, pose, stats):
    """What one register_frame_dev call hands its caller: the pose {qx,qy,qz,qw,tx,ty,tz} and the FrameStats it fills, as FRAME_STATS_ORDER."""
    os.makedirs(out_dir, exist_ok=True)
    row = [getattr(stats.icp, k[4:]) if k.startswith("icp.") else getattr(stats, k) for k in FRAME_STATS_ORDER]
    np.save(os.path.join(out_dir, "pose.npy"), np.asarray(pose, np.float64))
    np.save(os.path.join(out_dir, "frame_stats.npy"), np.asarray(row, np.float64))


# ------------------------------------------------------------------------------------------------------------------------ GPU side
class Bench:
    def __init__(self, args, torch, pkg, ctx, rank, local_rank, world):
        self.args, self.torch, self.pkg, self.ctx = args, torch, pkg, ctx
        self.rank, self.local_rank, self.world = rank, local_rank, world
        self.ext = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local_rank))
        self.dist = None
        if world > 1:
            import torch.distributed as dist
            self.dist = dist
        self.sampler = None

    def barrier(self):
        self.torch.cuda.synchronize()
        self.ctx.sync()
        if self.dist:
            self.dist.barrier()

    def gather(self, vals):
        """[vals of rank 0, vals of rank 1, ...] on every rank."""
        if not self.dist:
            return [list(vals)]
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device="cuda")
        out = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [o.tolist() for o in out]

    def new_odom(self, icp_mode=None, speculate=None, args=None, map_capacity_voxels=0):
        a = args or self.args
        spec = (not a.no_speculate) if speculate is None else speculate
        return self.ctx.KissICP(voxel_size=a.voxel, max_range=getattr(a, "max_range", 100.0), cap=a.cap, deskew=True, icp_max_iteration=a.max_iter,
                                icp_mode=a.icp_mode if icp_mode is None else icp_mode, speculate=spec, map_capacity_voxels=map_capacity_voxels)

    def window(self, step, n_warm, n_timed, odom, after_warmup=None):
        """W untimed + K timed calls of step(odom, i, last_of_phase). Returns this window's per-rank (time, wall, dev, closing barrier) rows."""
        for i in range(n_warm):
            step(odom, i, i == n_warm - 1)
        if after_warmup:
            after_warmup()
        self.barrier()
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        if self.sampler:
            self.sampler.in_window = True
        e0.record(self.ext)
        t0 = time.perf_counter()
        for i in range(n_warm, n_warm + n_timed):
            step(odom, i, i == n_warm + n_timed - 1)
        e1.record(self.ext)
        self.ctx.sync()
        t1 = time.perf_counter()
        if self.sampler:
            self.sampler.in_window = False
        self.barrier()
        t2 = time.perf_counter()
        wall, dev = t1 - t0, e0.elapsed_time(e1) / 1e3
        return self.gather([max(wall, dev), wall, dev, t2 - t1])

    def run_windows(self, make_step, n_warm, n_timed, repeats, icp_mode=None, keep_last=False, after_warmup=None):
        """`repeats` windows on fresh handles. Returns (summary, last odom or None)."""
        rows, odom = [], None
        for r in range(repeats):
            if odom is not None:
                odom.close()
            odom = self.new_odom(icp_mode)
            rows.append(self.window(make_step(), n_warm, n_timed, odom, after_warmup))
        if not keep_last:
            odom.close()
            odom = None
        per_window = [max(rk[0] for rk in w) for w in rows]               # max over ranks, per window
        order = np.argsort(per_window)
        med = int(order[len(order) // 2])
        n_g = max(self.args.gpus, self.world)
        summary = {"seconds": per_window[med], "value": n_g * n_timed / per_window[med],
                   "windows_scans_per_s": [round(n_g * n_timed / t, 1) for t in per_window],
                   "per_rank_median_window": {"wall_s": [rk[1] for rk in rows[med]], "dev_s": [rk[2] for rk in rows[med]], "closing_barrier_s": [rk[3] for rk in rows[med]]}}
        return summary, odom


def kernel_mode_record(torch, pkg, ctx, queries=(524288, 4194304), voxels=2.5e6, fill=20.0, voxel=0.5, cap=20, iters=10, reps=5):
    """The HBM-bound shape of the fused registration kernel (configs[2] / SURVEY C3 and the per-GPU work of C5): every point of a large scan
    is an ICP query against a ~45 M-point map (1.1 GB of stored points >> L2), fixed iteration count, one launch per ICP call."""
    ext = torch.cuda.ExternalStream(ctx.stream())
    side = float(np.sqrt(voxels) * voxel)
    gen = torch.Generator(device="cuda").manual_seed(1)
    m = ctx.VoxelHashMap(voxel, 1e9, cap, capacity_voxels=int(voxels * 1.3))
    total, done = int(voxels * fill), 0
    while done < total:
        n = min(1 << 20, total - done)
        p = torch.empty((n, 3), dtype=torch.float64, device="cuda")
        p[:, :2] = (torch.rand((n, 2), generator=gen, device="cuda", dtype=torch.float64) - 0.5) * side
        p[:, 2] = torch.randn(n, generator=gen, device="cuda", dtype=torch.float64) * 0.02 + 0.1
        torch.cuda.synchronize()
        m.insert_points_dev(p.data_ptr(), n)
        done += n
    nv, npts = m.size()
    peak, peak_src = measured_peak()
    init = pkg.se3_exp(np.array([0.03, -0.02, 0.01, 0.0005, -0.0003, 0.001]))
    out = []
    for nq in queries:
        q = torch.empty((nq, 3), dtype=torch.float64, device="cuda")
        q[:, :2] = (torch.rand((nq, 2), generator=gen, device="cuda", dtype=torch.float64) - 0.5) * side * 0.98
        q[:, 2] = torch.randn(nq, generator=gen, device="cuda", dtype=torch.float64) * 0.02 + 0.1
        torch.cuda.synchronize()
        times = []
        for rep in range(reps + 2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(ext)
            r = m.icp_dev(q.data_ptr(), nq, init, 1.5, 0.5, iters, 0.0)
            e1.record(ext)
            torch.cuda.synchronize()
            if rep >= 2:
                times.append(e0.elapsed_time(e1))
        ms = float(np.median(times))
        us_it = ms * 1e3 / max(r["iters"], 1)
        kb, fm = r["mean_candidates"], r["miss_fraction"]
        alg = nq * (24 + 16 + 24 * kb + fm * 27 * 16)
        alg_wb = alg + nq * 24.0   # + the in-place source update the reference also does every iteration (registration.cpp:119)
        out.append({"queries": nq, "iters": r["iters"], "us_per_iter": round(us_it, 2), "us_per_iter_min": round(min(times) * 1e3 / max(r["iters"], 1), 2),
                    "k_bar": round(kb, 3), "f_miss": round(fm, 4), "alg_bytes_per_iter": alg, "achieved_GBs": round(alg / (us_it * 1e-6) / 1e9, 1),
                    "frac": round(alg / (us_it * 1e-6) / 1e9 / peak, 4), "frac_with_source_writeback": round(alg_wb / (us_it * 1e-6) / 1e9 / peak, 4), "ncorr": r["last_ncorr"]})
    m.close()
    return {"map_voxels": nv, "map_points": npts, "map_point_bytes": npts * 24, "voxel": voxel, "cap": cap, "peak_GBs": peak, "peak_source": peak_src,
            "bytes_formula": "SURVEY 8d K4: per query per iteration 24 + 16 + 24*k_bar + f_miss*27*16 B (measured k_bar, f_miss); frac_with_source_writeback adds the 24 B/query source update",
            "timing": "CUDA events on the library stream around limu_icp_dev (one cooperative launch = the whole loop + one 104-byte D2H), median of 5 after 2 warm-ups; queries and map >> L2",
            "cases": out}


def c3_record(b, args, device, W3=3, K3=12, R3=3, bg_points=46_000_000):
    """configs[2] / SURVEY C3 in PIPELINE mode: the whole register_frame path on 512 000-point scans (128 beams x 4000 azimuth steps, urban
    canyon), voxel 0.5 m, cap 20, against a local map of ~45 M points resident in HBM. The map's bulk is a background slab (800 x 800 x 4
    voxels at z = 150..152 m, inserted through limu_map_insert_dev BEHIND warm-up scan 0, outside the timed region): it makes the table and
    the block array large (lookups of the scene's own voxels are scattered over ~4 GB) and is walked by every eviction sweep, but no query
    comes within 100 m of it, so the poses are those of the same sequence without it -- which is what the CPU arm (the reference's
    register_frame, no background) checks. max_range (= the map's max_distance) is 1000 m on both arms so the slab is never evicted."""
    import copy
    torch, ctx = b.torch, b.ctx
    a3 = copy.copy(args)
    a3.points, a3.beams, a3.azimuth_steps, a3.voxel, a3.cap, a3.max_range, a3.icp_mode = 512000, 128, 4000, 0.5, 20, 1000.0, 0
    n3 = a3.points
    scans = make_scans(a3, W3 + K3, 42, device, workload="c3")
    devs = [torch.from_numpy(s).cuda() for s in scans]
    gen = torch.Generator(device="cuda").manual_seed(3)
    bg = torch.empty((bg_points, 3), dtype=torch.float64, device="cuda")
    bg[:, :2] = (torch.rand((bg_points, 2), generator=gen, device="cuda", dtype=torch.float64) - 0.5) * 400.0
    bg[:, 2] = 150.0 + torch.rand(bg_points, generator=gen, device="cuda", dtype=torch.float64) * 2.0
    torch.cuda.synchronize()

    def prefill(o):
        m = o.local_map()
        for lo in range(0, bg_points, 1 << 20):
            m.insert_points_dev(bg[lo:lo + (1 << 20)].data_ptr(), min(1 << 20, bg_points - lo))

    def mk(rec):
        def step(o, i, last):
            if i > 0 and not last and i + 1 < len(devs):
                o.hint_next_dev(devs[i + 1].data_ptr(), n3)
            o.register_frame_dev(devs[i].data_ptr(), n3)
            st = o.stats
            rec.append((st.n_keypoints, st.icp.iterations, st.icp.mean_candidates, st.icp.miss_fraction, st.n_down))
            if i == 0:
                prefill(o)
        return step

    rows, frames, odom = [], [], None
    for r in range(R3):
        if odom is not None:
            odom.close()
        frames = []
        odom = b.new_odom(args=a3, map_capacity_voxels=3_400_000)
        rows.append(b.window(mk(frames), W3, K3, odom)[0])
    poses = odom.poses()
    nv, npts = odom.local_map().size()
    odom.close()
    # stage split (and the k_voxelize roofline at this size) from one more window with the stage events on
    ctx.set_profiling(True)
    odom = b.new_odom(args=a3, map_capacity_voxels=3_400_000)
    pfr = []
    b.window(mk(pfr), W3, K3, odom, after_warmup=lambda: ctx.set_profiling(True))
    prof, nfr = ctx.profile()
    ctx.set_profiling(False)
    odom.close()
    del bg
    torch.cuda.empty_cache()
    times = sorted(max(rw[0], rw[2]) for rw in rows)
    sec = times[len(times) // 2]
    f = np.array(frames[W3:], dtype=np.float64)
    peak, peak_src = measured_peak()
    nd, nk = float(f[:, 4].mean()), float(f[:, 0].mean())
    vox_bytes = 40.0 * n3 + 40.0 * (n3 + nd) + 24.0 * (nd + nk * 1.05)      # SURVEY 8d: K1*N + K2*(N + N_d), K2 = 40 B/point + 24 B/winner
    vox_ms = prof["downsample"] / max(nfr, 1)
    loop_bytes = float(np.mean([k4_bytes(x[0], x[1], x[2], x[3]) for x in pfr[W3:]]))
    loop_ms = prof["icp"] / max(nfr, 1)
    cpu = time_cpu(a3, scans, W3, K3, min(args.cpu_seconds, 12.0), mt=True, keep=True)
    return {
        "workload": workload_text(a3, "c3"), "value": K3 / sec, "unit": UNIT, "mpoints_per_s": K3 / sec * n3 / 1e6, "ms_per_step": 1e3 * sec / K3,
        "windows_scans_per_s": [round(K3 / t, 1) for t in times], "steps": K3, "warmup": W3,
        "iterations_per_scan": float(f[:, 1].mean()), "keypoints_per_scan": nk, "downsampled_per_scan": nd, "k_bar": float(f[:, 2].mean()), "f_miss": float(f[:, 3].mean()),
        "map_voxels": int(nv), "map_points": int(npts), "map_block_bytes": int(nv) * 512,
        "stage_ms_per_step": {k: v / max(nfr, 1) for k, v in prof.items()},
        "roofline_k_voxelize": {"bound": "hbm", "achieved": vox_bytes / (vox_ms * 1e-3) / 1e9 if vox_ms > 0 else 0.0, "peak": peak, "unit": "GB/s",
                                "frac": vox_bytes / (vox_ms * 1e-3) / 1e9 / peak if vox_ms > 0 else 0.0, "algorithmic_bytes_per_launch": vox_bytes,
                                "avg_launch_ms": vox_ms, "bytes_formula": "SURVEY 8d: K1*N + K2*(N + N_d) = 40 N + 40 (N + N_d) + 24 B per stage winner"},
        "roofline_loop_kernel": {"bound": "hbm", "achieved": loop_bytes / (loop_ms * 1e-3) / 1e9 if loop_ms > 0 else 0.0, "peak": peak, "unit": "GB/s",
                                 "frac": loop_bytes / (loop_ms * 1e-3) / 1e9 / peak if loop_ms > 0 else 0.0, "algorithmic_bytes_per_launch": loop_bytes,
                                 "avg_launch_ms": loop_ms, "note": "pipeline mode: the queries are the ~N_k keypoints, not the 512 k points (kernel mode: roofline_kernel_mode)"},
        "cpu_baseline": {"value": cpu["done"] / cpu["dt"] if cpu["done"] else None, "unit": UNIT, "cores": cpu["cores"], "kind": cpu["kind"],
                         "sample": f"first {cpu['done']} timed scans of the same sequence (no background slab: it cannot be matched)"},
        "parity": parity_record(a3, scans, poses, frames, cpu),
        "timing": "windows on fresh handles (background re-inserted each time, behind warm-up scan 0); per window max(host wall, CUDA events); median of the windows",
    }


def sharded_record(b, voxels=2.5e6, fill=20.0, nq=4194304, iters=20, reps=3):
    """configs[4] / SURVEY C5: one 4 M-point scan point-sharded over the ranks; every rank holds a replica of the ~45 M-point map and a
    contiguous shard of the queries; the per-iteration exchange of the 20-double row is fused into the registration kernel (NVLink stores
    into peer mailboxes). Compared with the same job on one GPU (every rank runs it, so the 1-GPU time is the max over ranks too)."""
    torch, pkg, ctx, dist = b.torch, b.pkg, b.ctx, b.dist
    from importlib import import_module
    sh = import_module("limu_b200.sharding")
    sh.connect(ctx, nccl_baseline=False)
    ext = b.ext
    voxel, cap = 0.5, 20
    side = float(np.sqrt(voxels) * voxel)
    gen = torch.Generator(device="cuda").manual_seed(1)
    m = ctx.VoxelHashMap(voxel, 1e9, cap, capacity_voxels=int(voxels * 1.3))
    total, done = int(voxels * fill), 0
    while done < total:
        n = min(1 << 20, total - done)
        p = torch.empty((n, 3), dtype=torch.float64, device="cuda")
        p[:, :2] = (torch.rand((n, 2), generator=gen, device="cuda", dtype=torch.float64) - 0.5) * side
        p[:, 2] = torch.randn(n, generator=gen, device="cuda", dtype=torch.float64) * 0.02 + 0.1
        torch.cuda.synchronize()
        m.insert_points_dev(p.data_ptr(), n)
        done += n
    gq = torch.Generator(device="cuda").manual_seed(7)
    q = torch.empty((nq, 3), dtype=torch.float64, device="cuda")
    q[:, :2] = (torch.rand((nq, 2), generator=gq, device="cuda", dtype=torch.float64) - 0.5) * side * 0.98
    q[:, 2] = torch.randn(nq, generator=gq, device="cuda", dtype=torch.float64) * 0.02 + 0.1
    torch.cuda.synchronize()
    lo, hi = sh.shard_range(nq, b.rank, b.world)
    shard = q[lo:hi].contiguous()
    init = pkg.se3_exp(np.array([0.03, -0.02, 0.01, 0.0005, -0.0003, 0.001]))

    def timed(fn):
        ts, out = [], None
        for rep in range(reps + 1):
            b.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(ext)
            out = fn()
            e1.record(ext)
            torch.cuda.synchronize()
            allr = b.gather([e0.elapsed_time(e1)])
            if rep >= 1:
                ts.append(max(x[0] for x in allr))
        return float(np.median(ts)), out

    t_single, single = timed(lambda: m.icp_dev(q.data_ptr(), nq, init, 1.5, 0.5, iters, 1e-9))
    t_fused, fused = timed(lambda: m.icp_sharded_dev(shard.data_ptr(), hi - lo, init, 1.5, 0.5, iters, 1e-9, mode=0))
    poses = [None] * b.world
    dist.all_gather_object(poses, fused["pose"].tolist())
    it = max(fused["iters"], 1)
    rec = {"ranks": b.world, "queries": nq, "map_points": m.size()[1], "iters": fused["iters"], "iters_single_gpu": single["iters"],
           "us_per_iter": round(t_fused * 1e3 / it, 2), "us_per_iter_single_gpu": round(t_single * 1e3 / max(single["iters"], 1), 2),
           "speedup_vs_1gpu": round(t_single / t_fused, 3),
           "pose_diff": float(np.abs(fused["pose"] - single["pose"]).max()), "ncorr_equal": bool(fused["last_ncorr"] == single["last_ncorr"]),
           "bit_identical": bool(all(p == poses[0] for p in poses)),
           "exchange": "fused: 20-double row stored into every peer's mailbox over NVLink inside k_icp_persistent (no NCCL launch, no host in the loop)",
           "timing": "CUDA events on the library stream, max over ranks, median of 3 after 1 warm-up"}
    m.close()
    ctx.comm_destroy()
    return rec


def main():
    args = parse()
    rank, local_rank, world = dist_env()
    n_gpus = max(args.gpus, world)
    W, K = args.warmup, args.steps
    cores = pin_cpus(local_rank, world)
    if world > 1:
        os.environ.setdefault("OMP_NUM_THREADS", str(max(1, len(cores) or 1)))
    import torch

    if args.impl == "reference":
        if rank != 0:
            return 0
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        est_steps = max(1, min(K, 2000))
        scans = make_scans(args, W + est_steps, 42, dev)
        r = time_cpu(args, scans, W, est_steps, args.ref_seconds)
        done, dt, kind = r["done"], r["dt"], r["kind"]
        val = done / dt
        note = ("the reference's unmodified register_frame (oracle/_ref: its own .cpp files compiled against vendored Eigen/Sophus; oneTBB, Boost.Thread, tsl::robin_map, "
                "PCL and ROS are absent here and shimmed -- thread-pool TBB shim, insertion-ordered robin_map shim) on the host cores; rank 0 only"
                if kind == "reference" else "C oracle (single thread): the opt-in registration variant has no counterpart in the reference")
        line = {
            "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": n_gpus, "steps": done, "steps_requested": K, "warmup": W,
            "ms_per_step": 1e3 * dt / done, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": make_config(args, n_gpus), "arm_note": note,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": r["cores"], "kind": kind, "sample": f"{done} consecutive scans after {W} warm-up scans (budget {args.ref_seconds:.0f} s)"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "mpoints_per_s": val * args.points / 1e6,
        }
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------- the B200 path
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the B200 path has no CPU fallback"}))
        return 2
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import __graft_entry__ as g
    pkg = g.load_package()
    ctx = pkg.Context(local_rank)
    b = Bench(args, torch, pkg, ctx, rank, local_rank, world)
    extras = not args.no_extras
    n_pts = args.points
    R = max(1, args.repeats)

    def stage(scans):
        pinned = [pkg.PinnedArray((n_pts, 4), np.float32) for _ in scans]
        for p, s in zip(pinned, scans):
            p.array[...] = s
        dev = [torch.from_numpy(s).cuda() for s in scans]
        return pinned, dev

    # configs[3]: one independent sequence per GPU. Weak scaling needs EQUAL work per GPU, so every rank replays the same world (scene seed 42)
    # with its own sensor-noise realisation. (Round 1 gave rank r scene seed 42 + r: on scene 45 the reference's Gauss-Newton loop runs to its
    # 500-iteration cap on some of the first 25 scans, that rank did ~6x the work and the max-over-ranks time followed it: profiles/r2_multi_gpu_n8.json.)
    scans = make_scans(args, W + K, 42, f"cuda:{local_rank}", vehicle=rank)
    pinned, dev_scans = stage(scans)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    flush.fill_(1)                                                      # push the staged scans out of L2
    torch.cuda.synchronize()
    b.sampler = ClockSampler(torch, local_rank)
    b.sampler.start()

    # -- arm 1: end to end through the host-pointer API (H2D of the scan + D2H of pose and both clouds every step)
    d2h = [0]

    def host_step_factory(pins):
        def mk():
            def step(o, i, last):
                if not last and i + 1 < len(pins):
                    o.prefetch(pins[i + 1].array)      # replay mode: the next scan's H2D (and, speculatively, its voxelize) overlaps this scan's kernels
                down, key, _pose = o.register_frame(pins[i].array, want_clouds=True, copy=False)
                d2h[0] += 56 + 16 + down.nbytes + key.nbytes
            return step
        return mk

    e2e, _ = b.run_windows(host_step_factory(pinned), W, K, R)
    e2e_d2h = d2h[0] / (R * (W + K))

    # -- arm 2: inputs resident in HBM (the `value`)
    frames = []

    def dev_step_factory(devs, rec=None, returned=None):
        def mk():
            if rec is not None:
                rec.clear()

            def step(o, i, last):
                if not last and i + 1 < len(devs):
                    o.hint_next_dev(devs[i + 1].data_ptr(), n_pts)   # replay hint (LIMU_OPT_SPECULATE): never across the warm-up / timed boundary
                pose = o.register_frame_dev(devs[i].data_ptr(), n_pts)
                if returned is not None:
                    returned["pose"] = pose
                if rec is not None:
                    st = o.stats
                    rec.append((st.n_keypoints, st.icp.iterations, st.icp.mean_candidates, st.icp.miss_fraction, st.n_down))
            return step
        return mk

    flush.fill_(2)
    launches0 = pkg.kernel_launches()
    returned = {}
    val, odom = b.run_windows(dev_step_factory(dev_scans, frames, returned), W, K, R, keep_last=True)
    launches = (pkg.kernel_launches() - launches0) // R
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, returned["pose"], odom.stats)
    gpu_poses = odom.poses()
    gpu_frames = list(frames)
    map_voxels, map_points = odom.local_map().size()
    last_pose = gpu_poses[-1]
    odom.close()

    # -- one more window with per-stage event timing switched on (NOT part of `value`): the frame kernel's own duration for the roofline
    ctx.set_profiling(True)
    prof_frames = []
    # (the sums restart behind the warm-up scans: a fresh handle's first k_voxelize has its scratch allocated between the two events)
    b.run_windows(dev_step_factory(dev_scans, prof_frames), W, K, 1, after_warmup=lambda: ctx.set_profiling(True))
    prof, nframes = ctx.profile()
    ctx.set_profiling(False)
    clocks = b.sampler.stop()
    b.sampler = None

    fr = np.array(gpu_frames[W:], dtype=np.float64)
    iters_total = float(fr[:, 1].sum())
    rank_work = b.gather([float(fr[:, 1].mean()), float(fr[:, 1].max()), float(fr[:, 0].mean())])   # equal work per GPU? (weak scaling)
    # bytes per launch over the profiled frames (the K timed scans of that window)
    pf = prof_frames[W:] if prof_frames else gpu_frames[W:]
    # LIMU_OPT_SPECULATE on (pipelined path): the loop kernel carries IQR + Gauss-Newton loop only, the map update is a launch of its own
    pipelined = not args.no_speculate
    if pipelined:
        alg_bytes = float(sum(k4_bytes(nk, it, kb, fm) + 24.0 * nk * 1.05 for nk, it, kb, fm, nd in pf))
    else:
        alg_bytes = float(sum(frame_kernel_bytes(nk, it, kb, fm, nk * 1.05, nd, map_voxels) for nk, it, kb, fm, nd in pf))
    icp_only_bytes = float(sum(k4_bytes(nk, it, kb, fm) for nk, it, kb, fm, _ in pf))
    icp_ms = prof["icp"]
    peak, peak_src = measured_peak()
    achieved = alg_bytes / (icp_ms * 1e-3) / 1e9 if icp_ms > 0 else 0.0
    stage_share = {k: round(v / max(sum(prof.values()), 1e-9), 4) for k, v in prof.items()}
    traffic, traffic_note = profiled_traffic(pkg)

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": val["value"], "unit": UNIT, "n_gpus": n_gpus, "steps": K, "warmup": W, "ms_per_step": 1e3 * val["seconds"] / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": make_config(args, n_gpus), "arm_note": "liblimu_cuda.so through its C ABI; LIMU_OPT_SPECULATE " + ("off" if args.no_speculate else "on"),
            "repeats": R, "windows_scans_per_s": val["windows_scans_per_s"],
            "per_rank": dict(val["per_rank_median_window"], iterations_per_scan=[round(r_[0], 2) for r_ in rank_work], max_iterations=[int(r_[1]) for r_ in rank_work],
                             keypoints_per_scan=[round(r_[2], 1) for r_ in rank_work]),
            "cpu_cores_per_rank": len(cores),
            "mpoints_per_s": val["value"] * n_pts / 1e6,
            "iterations_per_scan": iters_total / K, "scans_at_iteration_cap": int((fr[:, 1] >= args.max_iter).sum()),
            "keypoints_per_scan": float(fr[:, 0].mean()), "downsampled_per_scan": float(fr[:, 4].mean()),
            "k_bar": float(fr[:, 2].mean()), "f_miss": float(fr[:, 3].mean()), "map_voxels": int(map_voxels), "map_points": int(map_points),
            "e2e": {"value": e2e["value"], "unit": UNIT, "h2d_bytes_per_step": n_pts * 16, "d2h_bytes_per_step": int(e2e_d2h),
                    "windows_scans_per_s": e2e["windows_scans_per_s"], "per_rank": e2e["per_rank_median_window"],
                    "api": "limu_odom_register_frame (host pointers, pinned) with limu_odom_prefetch of the following scan: every step uploads one 2 MB scan (overlapped with the previous step's kernels) and reads back pose + downsampled + keypoint clouds"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": ("k_icp_persistent<latency> (one launch per scan: IQR filter + fused correspondence/residual/Jacobian/normal-equation Gauss-Newton loop; "
                                                    "the map insert + eviction is k_frame_update, launched beside the next scan's k_voxelize)") if pipelined else
                         "k_icp_persistent<latency> (one launch per scan: IQR filter + fused correspondence/residual/Jacobian/normal-equation Gauss-Newton loop + map insert + eviction)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes / max(nframes, 1), "avg_launch_ms": icp_ms / max(nframes, 1),
                         "share_of_step": stage_share.get("icp"),
                         "share_of_step_note": "its share of the SUM of the kernels' own durations (what a serialised ncu launch list shows); in the pipelined path k_voxelize and k_frame_update overlap each other, so the sum exceeds ms_per_step",
                         "share_of_period": (icp_ms / max(nframes, 1)) / (1e3 * val["seconds"] / K),
                         "registration_loop_bytes_per_launch": icp_only_bytes / max(nframes, 1),
                         "bytes_formula": "SURVEY 8d: I*K4*N_q (K4 = 24 + 16 + 24*k_bar + f_miss*27*16 B) + 24 B/IQR candidate" + ("" if pipelined else " + K3 = 64 B/inserted point + 20 B/occupied voxel (eviction)"),
                         "note": "pipeline mode: ~2.4k keypoint queries per iteration -> latency bound by construction (SURVEY H3): each Gauss-Newton iteration is a grid-wide dependency chain; the HBM-bound shape of the same kernel is `roofline_kernel_mode` below"},
            "stage_ms_per_step": {k: v / max(nframes, 1) for k, v in prof.items()}, "stage_share": stage_share,
            "clocks": clocks,
            "last_pose": [round(float(x), 6) for x in last_pose],
            "library": {"source_hash": pkg.source_hash(), "speculate": not args.no_speculate},
        }

    # ---------------------------------------------------------------- secondary records
    if extras and n_gpus == 1 and rank == 0:
        # e2e through what the drop-in's lidar::KissICP::register_frame(cloud, timestamps) really sends: 48-byte PCL records + FP64 timestamps
        rec = [pkg.PinnedArray((n_pts, 12), np.float32) for _ in scans]
        tss = [pkg.PinnedArray((n_pts,), np.float64) for _ in scans]
        for r_, t_, s in zip(rec, tss, scans):
            r_.array[...] = 0
            r_.array[:, :3] = s[:, :3]
            t_.array[...] = s[:, 3]
        bytes_out = [0]

        def cloud_mk(prefetch):
            def mk():
                def step(o, i, last):
                    if prefetch and not last and i + 1 < len(rec):
                        o.prefetch_cloud(rec[i + 1].array, 48, tss[i + 1].array)   # what the drop-in's KissICP::prefetch(cloud, timestamps) sends
                    down, key, _ = o.register_cloud(rec[i].array, 48, tss[i].array, copy=False)
                    bytes_out[0] += 56 + 16 + down.nbytes + key.nbytes
                return step
            return mk
        ec, _ = b.run_windows(cloud_mk(False), W, K, min(R, 3))
        d2h_cloud = int(bytes_out[0] / (min(R, 3) * (W + K)))
        ecp, _ = b.run_windows(cloud_mk(True), W, K, min(R, 3))
        line["e2e_cloud"] = {"value": ec["value"], "unit": UNIT, "h2d_bytes_per_step": n_pts * 56, "d2h_bytes_per_step": d2h_cloud,
                             "windows_scans_per_s": ec["windows_scans_per_s"],
                             "api": "limu_odom_register_cloud: 48-byte pcl::PointXYZINormal records + FP64 timestamps from pinned host memory (what include/limu_dropin's lidar::KissICP::register_frame sends), no prefetch",
                             "with_prefetch": {"value": ecp["value"], "windows_scans_per_s": ecp["windows_scans_per_s"],
                                               "api": "the same with limu_odom_prefetch_cloud of the following cloud (the drop-in's KissICP::prefetch): the 7.2 MB upload overlaps the registration of the current cloud"}}
        for x in rec + tss:
            x.free()

        # the opt-in variant that tracks on this scene (nearest of 27 cells + point-to-plane), same sequence
        m3 = []
        v3, o3 = b.run_windows(dev_step_factory(dev_scans, m3), W, K, min(R, 3), icp_mode=3, keep_last=True)
        p3 = o3.poses()[-1]
        o3.close()
        f3 = np.array(m3[W:], dtype=np.float64)
        line["icp_mode_3"] = {"value": v3["value"], "unit": UNIT, "windows_scans_per_s": v3["windows_scans_per_s"], "iterations_per_scan": float(f3[:, 1].mean()),
                              "last_pose_xy": [round(float(p3[4]), 3), round(float(p3[5]), 3)], "true_xy": [round(float(x), 3) for x in true_pose_xy(args, W + K - 1)],
                              "note": "LIMU_ICP_NN27 | LIMU_ICP_PLANE (SURVEY 8f N2, no counterpart in the reference: parity unpinned, defined by the C oracle)"}

    if extras and n_gpus == 1 and rank == 0:
        # second workload: a scene on which the REFERENCE's rule tracks (map grows, eviction fires)
        for p_ in pinned:
            p_.free()
        del dev_scans
        tscans = make_scans(args, W + K, 42, f"cuda:{local_rank}", workload="tracking")
        tpin, tdev = stage(tscans)
        tfr = []
        tv, to = b.run_windows(dev_step_factory(tdev, tfr), W, K, min(R, 3), keep_last=True)
        tposes = to.poses()
        tnv, tnp = to.local_map().size()
        to.close()
        te, _ = b.run_windows(host_step_factory(tpin), W, K, min(R, 3))
        tf = np.array(tfr[W:], dtype=np.float64)
        tcpu = time_cpu(args, tscans, W, K, min(args.cpu_seconds, 10.0), mt=True, keep=True)
        tpar = parity_record(args, tscans, tposes, tfr, tcpu)
        line["workload_tracking"] = {
            "workload": workload_text(args, "tracking"), "value": tv["value"], "unit": UNIT, "windows_scans_per_s": tv["windows_scans_per_s"],
            "e2e": te["value"], "iterations_per_scan": float(tf[:, 1].mean()), "scans_at_iteration_cap": int((tf[:, 1] >= args.max_iter).sum()),
            "keypoints_per_scan": float(tf[:, 0].mean()), "downsampled_per_scan": float(tf[:, 4].mean()), "k_bar": float(tf[:, 2].mean()), "f_miss": float(tf[:, 3].mean()),
            "map_voxels": int(tnv), "map_points": int(tnp), "inserted_points_total": int(np.array(tfr)[:, 4].sum()),
            "last_pose_xy": [round(float(tposes[-1][4]), 3), round(float(tposes[-1][5]), 3)], "true_xy": [round(float(x), 3) for x in true_pose_xy(args, W + K - 1)],
            "cpu_baseline": {"value": tcpu["done"] / tcpu["dt"], "unit": UNIT, "cores": tcpu["cores"], "kind": tcpu["kind"], "sample": f"first {tcpu['done']} timed scans"},
            "parity": tpar}
        for p_ in tpin:
            p_.free()
        del tdev

    if extras and n_gpus == 1 and rank == 0 and args.icp_mode == 0 and abs(args.step_m - 1.0) < 1e-9:
        # configs[1] as worded is a 1000-scan loop: after the loop closes (scan ~188) the reference's Gauss-Newton loop runs to its cap on
        # almost every scan. Replay scans 0..199 once and time the last 10 (the capped regime) separately.
        n_all, n_tail = 200, 10
        lscans = make_scans(args, n_all, 42, f"cuda:{local_rank}")
        ldev = [torch.from_numpy(s).cuda() for s in lscans]
        lfr = []
        lv, _ = b.run_windows(dev_step_factory(ldev, lfr), n_all - n_tail, n_tail, 1)
        lf = np.array(lfr[n_all - n_tail:], dtype=np.float64)
        line["loop_closure_regime"] = {"scans_timed": [n_all - n_tail, n_all], "value": lv["value"], "unit": UNIT, "iterations_per_scan": float(lf[:, 1].mean()),
                                       "scans_at_iteration_cap": int((lf[:, 1] >= args.max_iter).sum()),
                                       "note": "the reference's loop stops converging here (C oracle and CUDA agree scan by scan: tests/test_bench_parity.py); one window"}
        del ldev

    if extras and n_gpus == 1 and rank == 0:
        torch.cuda.empty_cache()
        line["roofline_kernel_mode"] = kernel_mode_record(torch, pkg, ctx)
        try:
            line["workload_c3"] = c3_record(b, args, f"cuda:{local_rank}")
        except Exception as e:   # noqa: BLE001
            line["workload_c3"] = {"error": repr(e)}

    if rank == 0 and n_gpus == 1:
        cpu = time_cpu(args, scans, W, K, args.cpu_seconds, mt=True, keep=True)
        line["cpu_baseline"] = {"value": cpu["done"] / cpu["dt"], "unit": UNIT, "cores": cpu["cores"], "kind": cpu["kind"],
                                "sample": f"first {cpu['done']} timed scans of the same sequence after {W} warm-up scans ({cpu['dt']:.1f} s of host time)",
                                "caveat": "oracle/_ref = the reference's unmodified sources against SHIMS for what this image lacks: std::thread-pool oneTBB, null-lock Boost.Thread, insertion-ordered tsl::robin_map (upstream iterates in bucket order), PCL/ROS structs"}
        if args.icp_mode == 0:
            line["parity"] = parity_record(args, scans, gpu_poses, gpu_frames, cpu)
            ser = time_cpu(args, scans, W, K, min(6.0, args.cpu_seconds), mt=False)
            line["cpu_baseline"]["serial_1_core"] = {"value": ser["done"] / ser["dt"], "unit": UNIT, "cores": 1, "kind": ser["kind"], "sample": f"first {ser['done']} timed scans, serial TBB shim (the parity oracle)"}
            try:
                line["cpu_baseline"]["stages"] = cpu_stage_split(args, scans[min(len(scans) - 1, W + 3)])
            except Exception as e:   # noqa: BLE001
                line["cpu_baseline"]["stages"] = {"error": repr(e)}

    if extras and n_gpus > 1:
        try:
            srec = sharded_record(b)
        except Exception as e:   # noqa: BLE001
            srec = {"error": repr(e)}
        if rank == 0:
            line["sharded"] = srec

    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
