"""Developer tool: where the time goes inside the fused frame kernel (IQR | ICP loop | insert claim | insert place |
eviction sweep) on the bench workload. Needs the instrumented build:
  LIMU_LIB=lidar-imu-slam_b200/build/liblimu_pt.so python tools/frame_phase_timing.py"""
import ctypes
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as g

pkg = g.load_package()
from importlib import import_module
synth = import_module("limu_b200.synth")
ctx = pkg.Context(0)
WL = os.environ.get("LIMU_PT_WORKLOAD", "c2")     # c2: the bench workload; c3: configs[2] in pipeline mode (512 k points/scan, voxel 0.5 m, cap 20)
if WL == "c3":
    import copy
    import bench
    a3 = copy.copy(bench.parse([]))
    a3.points, a3.beams, a3.azimuth_steps, a3.voxel, a3.cap, a3.max_range = 512000, 128, 4000, 0.5, 20, 1000.0
    K = 14
    scans = bench.make_scans(a3, K, 42, "cuda", workload="c3")
    KW = dict(voxel_size=0.5, cap=20, max_range=1000.0, map_capacity_voxels=3_400_000 if os.environ.get("LIMU_PT_BG") else 0)
else:
    scene = synth.Scene(seed=42)
    K = 40
    traj = synth.loop_trajectory(K + 1, radius=30.0, step=1.0)
    scans = [synth.pad_scan(synth.cast_scan(scene, traj[i], traj[i + 1], seed=42 * 100003 + i, device="cuda"), 128000, seed=i) for i in range(K)]
    KW = dict(voxel_size=1.0, cap=10)
odo = ctx.KissICP(deskew=True, icp_max_iteration=500, **KW)


def background(o):
    """configs[2]: the ~45 M-point slab bench.py's workload_c3 keeps resident (LIMU_PT_BG=1)."""
    import torch
    n = 46_000_000
    gen = torch.Generator(device="cuda").manual_seed(3)
    bg = torch.empty((n, 3), dtype=torch.float64, device="cuda")
    bg[:, :2] = (torch.rand((n, 2), generator=gen, device="cuda", dtype=torch.float64) - 0.5) * 400.0
    bg[:, 2] = 150.0 + torch.rand(n, generator=gen, device="cuda", dtype=torch.float64) * 2.0
    torch.cuda.synchronize()
    m = o.local_map()
    for lo in range(0, n, 1 << 20):
        m.insert_points_dev(bg[lo:lo + (1 << 20)].data_ptr(), min(1 << 20, n - lo))
    ctx.sync()
marks = np.zeros(72)
vmarks = np.zeros(8)
have_vox = hasattr(pkg.lib(), "limu_debug_vox_marks")
rows, iters, rounds, vrows = [], [], [], []
for i, s in enumerate(scans):
    odo.register_frame(s, want_clouds=False)
    if i == 0 and WL == "c3" and os.environ.get("LIMU_PT_BG"):
        background(odo)
    pkg.lib().limu_debug_frame_marks(marks.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
    if i >= (3 if WL == "c3" else 5):
        rows.append(np.diff(marks[:6]) / 1e3)
        iters.append(odo.stats.icp.iterations)
        nr = min(odo.stats.icp.iterations, 47)              # round j starts at marks[24 + j]; the last one has no successor
        d = np.diff(marks[24:24 + nr]) / 1.965e3
        rounds.append(np.pad(d, (0, max(0, 12 - len(d))), constant_values=np.nan)[:12])
        if have_vox:
            pkg.lib().limu_debug_vox_marks(vmarks.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
            vrows.append(np.diff(vmarks[:4]) / 1e3)
r = np.array(rows)
names = ["iqr", "icp_loop", "insert_claim", "insert_place", "evict_sweep"]
print({n: round(float(v), 2) for n, v in zip(names, r.mean(axis=0))}, "total_us", round(float(r.sum(axis=1).mean()), 2), "iters/scan", np.mean(iters),
      "icp_us_per_iter", round(float(r[:, 1].mean() / np.mean(iters)), 2))
cyc = lambda a, b: int(marks[b] - marks[a])
print("iteration 2 of the last scan (SM cycles of CTA 0, 1965 MHz): pass of warp 0", cyc(6, 7), "| pass end -> S1", cyc(7, 11), "| CTA row + grid barrier", cyc(11, 12),
      "| fold", cyc(12, 8), "| ldlt", cyc(8, 9), "| exp", cyc(9, 10), "| -> S2", cyc(10, 15), "| whole round (pass start -> S2)", cyc(6, 15),
      "| tail of the solver warp (its own clock)", cyc(13, 14))
print("rounds of the Gauss-Newton loop (us, CTA 0, mean over scans; nan = fewer rounds):", [round(float(x), 2) for x in np.nanmean(np.array(rounds), axis=0)])
if vrows:
    print("k_voxelize phases (us; plain launch, 1024-thread CTAs): P1 deskew + claim | P2 flags, counts, scatter, claim 2 | P3 un-claim, flags, counts, scatter:", [round(float(x), 2) for x in np.mean(np.array(vrows), axis=0)], "total", round(float(np.sum(np.mean(np.array(vrows), axis=0))), 2))
if hasattr(pkg.lib(), "limu_debug_cta_marks"):
    cm = np.zeros(640)
    pkg.lib().limu_debug_cta_marks(cm.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
    cm = cm.reshape(4, 160)
    live = cm[0] > cm[0].max() - 5e4          # (marks of CTAs that only took part in an earlier, larger launch are stale)
    cm = cm[:, live]
    nb = cm.shape[1]
    t0 = cm[0, :nb].min()
    q = lambda a: "min %.2f / median %.2f / max %.2f" % (np.min(a), np.median(a), np.max(a))
    print("round 3 of the last scan over the %d CTAs of the loop (us after the first CTA started the round): round start %s | pass over (S1) %s | rows folded %s | S2 %s"
          % (nb, q((cm[0, :nb] - t0) / 1e3), q((cm[1, :nb] - t0) / 1e3), q((cm[2, :nb] - t0) / 1e3), q((cm[3, :nb] - t0) / 1e3)))
    print("  pass duration per CTA (S1 - round start):", q((cm[1, :nb] - cm[0, :nb]) / 1e3), "| ten slowest CTAs:", np.argsort(cm[1, :nb] - cm[0, :nb])[-10:].tolist())
if hasattr(pkg.lib(), "limu_debug_warp_pass"):
    wp = np.zeros(1280, np.uint32)
    pkg.lib().limu_debug_warp_pass(wp.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)))
    wflags = (wp.reshape(160, 8)[:, :7] >> 24)
    wp = (wp.reshape(160, 8)[:, :7] & 0xFFFFFF).astype(np.float64) / 1.965e3
    if hasattr(pkg.lib(), "limu_debug_cta_marks"):
        wp = wp[:len(live)][live]
        wflags = wflags[:len(live)][live]
    for name, sel in (("all four lookups repeats", wflags == 0), ("a first-time lookup on the common path", wflags == 1), ("a lookup off the common path", wflags >= 2),
                      ("  ... a displaced voxel (linear probing)", (wflags & 8) != 0), ("  ... an absent voxel (neighbour fallback)", (wflags & 4) != 0)):
        if sel.any():
            print("    warps with %-40s %4d: median %.2f  max %.2f us" % (name + ":", int(sel.sum()), np.median(wp[sel]), wp[sel].max()))
    print("pass of round 3 per warp (us, %d CTAs x 7 query warps): median %.2f | p90 %.2f | p99 %.2f | max %.2f | mean per warp index %s | slowest warp per CTA: median %.2f, max %.2f"
          % (len(wp), np.median(wp), np.percentile(wp, 90), np.percentile(wp, 99), wp.max(), [round(float(x), 2) for x in wp.mean(axis=0)], np.median(wp.max(axis=1)), wp.max()))
print("IQR phase of the last scan (SM cycles of CTA 0): squared ranges + ranking", cyc(16, 17), "| barrier of the loop CTAs", cyc(17, 18), "| local compaction (+ keypoints written out)", cyc(18, 19))

# ---- timeline of the pipelined path (hinted device replay): one ring of (id, globaltimer) records per translation unit, merged here
if hasattr(pkg.lib(), "limu_debug_trace_reg"):
    import torch
    odo.close()
    dev = [torch.from_numpy(s).cuda() if isinstance(s, np.ndarray) else s for s in scans]
    torch.cuda.synchronize()
    odo = ctx.KissICP(deskew=True, icp_max_iteration=500, speculate=True, **KW)
    for i, s in enumerate(dev):
        if i + 1 < len(dev) and i > 0:
            odo.hint_next_dev(dev[i + 1].data_ptr(), dev[i + 1].shape[0])
        odo.register_frame_dev(s.data_ptr(), s.shape[0])
        if i == 0 and WL == "c3" and os.environ.get("LIMU_PT_BG"):
            background(odo)
    odo.flush()
    names = {1: "loop kernel starts", 2: "IQR done", 3: "loop over (gate flag)", 4: "loop kernel ends", 10: "voxelize starts", 11: "voxelize P1 done", 12: "voxelize P2 done",
             13: "voxelize ends", 20: "update starts", 21: "update: claim done", 22: "update: place done", 23: "update ends", 30: "gate exits (update released)"}
    ev = []
    for fn in ("limu_debug_trace_reg", "limu_debug_trace_vox"):
        buf = np.zeros(2048, np.uint64)
        cnt = ctypes.c_uint(0)
        getattr(pkg.lib(), fn)(buf.ctypes.data_as(ctypes.POINTER(ctypes.c_ulonglong)), ctypes.byref(cnt))
        k = min(cnt.value, 2048)
        for w in buf[:k]:
            ev.append((int(w) & ((1 << 56) - 1), int(w) >> 56))
    ev.sort()
    starts = [i for i, e in enumerate(ev) if e[1] == 1]
    if len(starts) >= 8:
        # steady state: average the offsets of every record relative to the loop start of ITS scan, over the last scans
        rel = {}
        periods = []
        for a, b in zip(starts[-12:-1], starts[-11:]):
            t0 = ev[a][0]
            periods.append((ev[b][0] - t0) / 1e3)
            for t, idn in ev[a:b]:
                rel.setdefault(idn, []).append((t - t0) / 1e3)
        print("pipelined path, hinted device replay: period between loop starts %.1f us (last 11 scans: %s)" % (np.mean(periods), [round(p, 1) for p in periods]))
        for idn, v in sorted(rel.items(), key=lambda kv: np.mean(kv[1])):
            print("  +%7.2f us  %s" % (np.mean(v), names.get(idn, str(idn))))
