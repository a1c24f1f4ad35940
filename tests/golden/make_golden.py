"""Generates tests/golden/*.npz from the REFERENCE ITSELF (oracle/_ref/liblimu_ref.so = the unmodified
sources of Oreoluwa-Se/Lidar-Imu-Slam env_ws/src/limu compiled by oracle/Makefile with serial shims).

Run in the authoring container (where /root/reference exists):   python tests/golden/make_golden.py
The fixtures travel with the repo; tests/test_golden.py checks the C oracle (CPU) and the CUDA path (GPU)
against them, so parity is pinned to reference outputs even where oracle/_ref cannot be rebuilt.

Two families:
  fixtures_hash_map_test.npz  the six known-answer inputs of L/src/tests/hash_map_test.hpp (the reference's
                              only tests, SURVEY section 4) with the reference's outputs on them;
  fixtures_path_<i>.npz       seeded synthetic inputs through every function of the hot path
                              (SURVEY section 8a rows a1-a19) with the reference's outputs, in parts under 1 MB;
  fixtures_frame.npz          seeded PointCloud2 payloads through frame::Lidar::process_frame (SURVEY section 8f N3).
Regenerate a subset with:  python tests/golden/make_golden.py frame
"""
import ctypes
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402


def libc_rand_stream(n):
    """glibc rand() with the default seed (srand(1)), as the reference's tests draw their inputs."""
    libc = ctypes.CDLL("libc.so.6")
    libc.srand(1)
    return np.array([libc.rand() for _ in range(n)], dtype=np.float64)


RAND_MAX = 2147483647.0


def hash_map_test_fixtures(ref):
    out = {}
    # basic_test (hash_map_test.hpp:8-52): 10 points (i, i+1, i+2); VoxelHashMap(1, 1, 200) -> 10 voxels x 1 point
    pts = np.array([[i, i + 1.0, i + 2.0] for i in range(1, 11)], dtype=np.float64)
    m = ref.Map(1.0, 1.0, 200)
    m.insert(pts)
    k, c, p = m.dump()
    out.update(basic_in=pts, basic_keys=k, basic_counts=c, basic_pts=p)
    # test_insert_points (:53-100): lattice -10..10 step 1.1 (accumulated in double, as the for loop does) + 10 hand points
    axis = []
    x = -10.0
    while x <= 10:
        axis.append(x)
        x += 1.1
    axis = np.array(axis)
    lat = np.array([[a, b, c_] for a in axis for b in axis for c_ in axis])
    hand = np.array([[-0.5, -0.5, -0.5], [-0.5, -0.5, 0.5], [-0.5, 0.5, -0.5], [-0.5, 0.5, 0.5], [0.5, -0.5, -0.5], [0.5, -0.5, 0.5],
                     [0.5, 0.5, -0.5], [0.5, 0.5, 0.5], [1.6, 0.5, -1.1], [-1.6, -0.5, 1.1]])
    pts = np.concatenate([lat, hand])
    m = ref.Map(1.0, 1.0, 200)
    m.insert(pts)
    k, c, p = m.dump()
    out.update(insert_in=pts, insert_keys=k, insert_counts=c, insert_pts=p)
    # test_closest_neighbor (:102-128): map {(0,0,0),(2,2,2),(4,4,4)}; queries (0,0,0) and (1,1,1)
    m = ref.Map(1.0, 1.0, 200)
    m.insert(np.array([[0.0, 0, 0], [2.0, 2, 2], [4.0, 4, 4]]))
    q = np.array([[0.0, 0, 0], [1.0, 1, 1]])
    out.update(closest_q=q, closest_out=m.closest(q))
    # test_correspondences (:130-168): 1000 points rand()/RAND_MAX, VoxelHashMap(1, 0.2, 1000), tau 0.2
    r = libc_rand_stream(3000)
    pts = (1.0 * r / RAND_MAX).reshape(1000, 3)
    m = ref.Map(1.0, 0.2, 1000)
    m.insert(pts)
    s, t = m.correspondences(pts, 0.2)
    out.update(corr_in=pts, corr_src=s, corr_tgt=t)
    # test_correspondences2(cap) (:170-208): Vector3d::Random()*0.5 = (-1 + 2*rand()/RAND_MAX) * 0.5; caps {100,50,10,60,1000}
    # (6 000 of the reference's 100 000 points keep the fixture small; every point still falls in voxel (0,0,0))
    r = libc_rand_stream(18000)
    pts = ((-1.0 + (2.0 * r) / RAND_MAX) * 0.5).reshape(6000, 3)
    out["corr2_in"] = pts
    for cap in (100, 50, 10, 60, 1000):
        m = ref.Map(1.0, 1.0, cap)
        m.insert(pts)
        s, t = m.correspondences(pts, 0.1)
        out[f"corr2_n_{cap}"] = len(s)
        out[f"corr2_tgt_{cap}"] = t
        out[f"corr2_counts_{cap}"] = m.dump()[1]
    # test_remove_points_from_far(5.0) (:210-246): 1000 points Random()*100, v = 0.1, max_dist 5, cap 100
    r = libc_rand_stream(3000)
    pts = ((-1.0 + (2.0 * r) / RAND_MAX) * 100).reshape(1000, 3)
    m = ref.Map(0.1, 5.0, 100)
    m.insert(pts)
    m.remove_far(np.zeros(3))
    k, c, p = m.dump()
    out.update(far_in=pts, far_keys=k, far_counts=c, far_pts=p)
    return out


def path_fixtures(ref):
    rng = np.random.default_rng(20260101)
    out = {}
    pts = rng.normal(size=(6000, 3)) * np.array([25, 25, 3])
    pts[:50] = np.round(pts[:50])
    T = ref.se3_exp(np.array([1.5, -0.7, 0.2, 0.02, -0.03, 0.4]))
    out.update(pts=pts, T=T)
    for v in (1.0, 0.5, 1.5):
        out[f"keys_{v}"] = ref.vox_index(pts, v)
    out["transformed"] = ref.transform(T, pts)
    for s in (0.5, 1.5):
        out[f"ds_{s}"] = ref.voxel_downsample(pts, s)
    out["iqr"] = ref.iqr(pts)
    src, down = ref.voxelize(pts, 1.0)
    out.update(vox_src=src, vox_down=down)
    # map: three batches, cap 5
    m = ref.Map(1.0, 40.0, 5)
    batches = [rng.normal(size=(4000, 3)) * 12 for _ in range(3)]
    for b in batches:
        m.insert(b)
    k, c, p = m.dump()
    q = rng.normal(size=(5000, 3)) * 14
    out.update(map_b0=batches[0], map_b1=batches[1], map_b2=batches[2], map_keys=k, map_counts=c, map_pts=p, map_q=q, map_closest=m.closest(q))
    s, t = m.correspondences(q, 1.2)
    out.update(map_corr_src=s, map_corr_tgt=t)
    o = np.array([3.0, -2.0, 1.0])
    m.remove_far(o)
    k, c, p = m.dump()
    out.update(evict_origin=o, evict_keys=k, evict_counts=c, evict_pts=p)
    # align + ICP on a dense three-plane scene
    n = 30000
    a = rng.random((n // 3, 3)) * 40 - 20
    a[:, 2] = rng.normal(size=len(a)) * 0.02
    b = rng.random((n // 3, 3)) * 40 - 20
    b[:, 0] = 20 + rng.normal(size=len(b)) * 0.02
    c_ = rng.random((n // 3, 3)) * 40 - 20
    c_[:, 1] = -20 + rng.normal(size=len(c_)) * 0.02
    world = np.concatenate([a, b, c_])
    true = ref.se3_exp(np.array([0.3, -0.2, 0.05, 0.004, -0.003, 0.02]))
    srcp = ref.transform(ref.se3_inv(true), world[rng.choice(len(world), 3000, replace=False)])
    m = ref.Map(1.0, 100.0, 20)
    m.insert(world)
    init = np.array([0, 0, 0, 1.0, 0, 0, 0])
    r = ref.icp(m, srcp, init, 6.0, 2.0 / 3.0, 60, 1e-4, trace=True)
    s, t = m.correspondences(srcp, 6.0)
    out.update(icp_world=world.astype(np.float32).astype(np.float64), icp_src=srcp, icp_pose=r["pose"], icp_est=r["est"], icp_ncorr=r["ncorr"], icp_iters=r["iters"])
    # (the world is stored rounded to float32 to halve the file; recompute the reference on exactly what is stored)
    m = ref.Map(1.0, 100.0, 20)
    m.insert(out["icp_world"])
    r = ref.icp(m, srcp, init, 6.0, 2.0 / 3.0, 60, 1e-4, trace=True)
    s, t = m.correspondences(srcp, 6.0)
    out["icp_world"] = out["icp_world"].astype(np.float32)   # exact: values are float32-representable
    out.update(icp_pose=r["pose"], icp_est=r["est"], icp_ncorr=r["ncorr"], icp_iters=r["iters"], align_src=s[:2000], align_tgt=t[:2000],
               align_pose=ref.align(s[:2000], t[:2000], 2.0 / 3.0)["pose"])
    # deskew
    xyz = (rng.normal(size=(3000, 3)) * 30).astype(np.float32)
    ts = rng.random(3000)
    T0 = ref.se3_exp(np.array([4.0, 1.0, 0.0, 0.0, 0.01, 0.3]))
    T1 = ref.se3_mul(T0, ref.se3_exp(np.array([1.0, 0.1, -0.05, 0.01, -0.02, 0.1])))
    out.update(dk_xyz=xyz, dk_ts=ts, dk_T0=T0, dk_T1=T1, dk_out=ref.deskew(xyz, ts, T0, T1))
    # IMU-propagated backward deskew (kalman::EKF::motion_compensation_with_imu, ekf.cpp:292-469): 200 Hz IMU window,
    # turning + accelerating platform; the first point sits at t > 0 so the reference's repeated compensation of the
    # never-consumed first point (:455-456) is part of the fixture
    kimu, nimu = 22, 4000
    t0 = 100.0
    its = t0 - 0.004 + np.arange(kimu) * 0.005
    gyr = np.array([0.02, -0.01, 0.35]) + rng.normal(size=(kimu, 3)) * 0.002
    acc = np.array([0.3, -0.2, 9.81]) + rng.normal(size=(kimu, 3)) * 0.03
    imu = np.concatenate([its[:, None], gyr, acc], 1)
    curv = np.sort(rng.random(nimu) * 100.0).astype(np.float32)
    curv[0] = 0.37
    ixyz = (rng.normal(size=(nimu, 3)) * 25).astype(np.float32)
    pil = np.array([0.1, -0.05, 0.2])
    mean_acc, bg = np.array([0.3, -0.2, 9.81]), np.array([0.001, 0.002, -0.001])
    r = ref.imu_deskew_reference(ixyz, curv, imu, t0, mean_acc, pil, bg)
    out.update(imu_samples=imu, imu_t0=t0, imu_mean_acc=mean_acc, imu_bg=bg, imu_xyz=ixyz, imu_curv=curv, imu_table=r["table"], imu_rot_end=r["rot_end"], imu_pos_lidar_end=r["pos_lidar_end"], imu_pil=pil,
               imu_deskewed=r["deskewed"], imu_written_back=r["written_back"])
    # KissICP sequence (register_frame x 6, deskew on), scans from the package's own generator
    import __graft_entry__ as g
    g.load_package()
    from importlib import import_module
    synth = import_module("limu_b200.synth")
    scene = synth.Scene(seed=11)
    traj = synth.loop_trajectory(7, radius=30.0, step=0.5)
    k = ref.Kiss(voxel_size=1.0, max_range=100.0, cap=10, deskew=True, icp_max_iteration=100)
    for i in range(6):
        scan = synth.cast_scan(scene, traj[i], traj[i + 1], beams=16, azimuth_steps=360, seed=500 + i)
        d, s, p = k.register_cloud(scan[:, :3], scan[:, 3].astype(np.float64))
        out[f"kiss_scan_{i}"] = scan
        out[f"kiss_pose_{i}"] = p
        out[f"kiss_ndown_{i}"] = len(d)
        out[f"kiss_nsrc_{i}"] = len(s)
        if i == 5:
            out["kiss_down_5"] = d
            out["kiss_src_5"] = s
    return out


def frame_fixtures(ref):
    """frame::Lidar::process_frame (lidar/frame.cpp:101-193; SURVEY section 8f N3) on seeded PointCloud2 payloads in the layout the
    reference registers for its LidarPoint (lidar/frame.hpp:12-23). Offset times are distinct, so std::sort's tie order plays no role."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_preprocess import CFG, make_msg
    out = {}
    cases = [(101, 3000, "distinct", 1, 1), (102, 3001, "distinct", 3, 25), (103, 2500, "distinct", 4, 60), (104, 2000, "nooffset", 1, 5)]
    for k, (seed, n, kind, split, sc) in enumerate(cases):
        data, fields, mt = make_msg(seed, n, kind=kind)
        seg = ref.process_frame(data, fields, dict(CFG, frame_split_num=split), mt, sc)
        out[f"c{k}_data"], out[f"c{k}_mt"], out[f"c{k}_sc"], out[f"c{k}_split"], out[f"c{k}_nooffset"] = data, mt, sc, split, kind == "nooffset"
        out[f"c{k}_sizes"] = np.array([len(s["points"]) for s in seg], np.int64)
        out[f"c{k}_points"] = np.concatenate([s["points"] for s in seg])
        out[f"c{k}_ts"] = np.concatenate([s["ts"] for s in seg])
        out[f"c{k}_times"] = np.array([s["time"] for s in seg])
    out["n_cases"] = len(cases)
    return out


def ekf_fixtures():
    """kalman::EKF (ekf.cpp) stepped by oracle/ref_ekf_driver.cpp through the script of tests/test_ekf.py (trail 5 keeps the file small):
    the state and covariance after every augmentation / zero-velocity update / undo, after the last predict, and after a few early predicts."""
    sys.path.insert(0, os.path.dirname(HERE))
    import test_ekf as T
    seed, trail, noise_scale = 11, 5, 1.5
    steps = T.script(np.random.default_rng(seed))
    f = oracle.RefEkf(lidar_pose_trail=trail, noise_scale=noise_scale)
    m0, P0, _ = f.state()
    m0[3:6] = [0.8, -0.3, 0.05]
    q = np.array([0.98, 0.05, -0.12, 0.1]); m0[6:10] = q / np.linalg.norm(q)
    m0[10:13] = [1e-3, -2e-3, 5e-4]; m0[13:16] = [0.02, -0.01, 0.03]; m0[16:19] = [1.01, 0.99, 1.02]; m0[19:22] = T.GRAV
    P0[6:10, 6:10] = np.diag([1e-6, 1e-6, 1e-6, 0.0]) * noise_scale ** 2
    f.set_state(m0, P0)
    states = T.run_script(f, steps, T.GRAV, T.TRANS, T.ROT)
    idx = [i for i, s_ in enumerate(steps) if s_[0] in ("augment", "zupt", "undo")] + [1, 2, 7, len(steps) - 1]
    idx = sorted(set(idx))
    return {"seed": seed, "trail": trail, "noise_scale": noise_scale, "m0": m0, "P0": P0, "idx": np.array(idx), "m": np.array([states[i][0] for i in idx]),
            "P": np.array([states[i][1] for i in idx])}


def save_parts(stem, arrays, max_bytes=900_000):
    """Write `arrays` (in order) as stem_0.npz, stem_1.npz, ...: a new part starts before max_bytes of array data, so no stored file
    reaches 1 MB. tests/test_golden.py merges the parts back into one mapping."""
    for f in os.listdir(HERE):
        if f.startswith(stem + "_") and f.endswith(".npz"):
            os.remove(os.path.join(HERE, f))
    parts, size = [{}], 0
    for k, v in arrays.items():
        v = np.asarray(v)
        if parts[-1] and size + v.nbytes > max_bytes:
            parts.append({})
            size = 0
        parts[-1][k] = v
        size += v.nbytes
    names = [f"{stem}_{i}.npz" for i in range(len(parts))]
    for name, part in zip(names, parts):
        np.savez_compressed(os.path.join(HERE, name), **part)
        assert os.path.getsize(os.path.join(HERE, name)) < 1 << 20, f"{name}: one array of {list(part)} alone reaches 1 MB; sample it"
    return names


if __name__ == "__main__":
    oracle.build_ref()
    ref = oracle.load_ref()
    which = sys.argv[1:] or ["hash_map", "path", "frame", "ekf"]
    made = []
    if "hash_map" in which:
        np.savez_compressed(os.path.join(HERE, "fixtures_hash_map_test.npz"), **hash_map_test_fixtures(ref))
        made.append("fixtures_hash_map_test.npz")
    if "path" in which:
        made += save_parts("fixtures_path", path_fixtures(ref))
    if "frame" in which:
        np.savez_compressed(os.path.join(HERE, "fixtures_frame.npz"), **frame_fixtures(ref))
        made.append("fixtures_frame.npz")
    if "ekf" in which:
        np.savez_compressed(os.path.join(HERE, "fixtures_ekf.npz"), **ekf_fixtures())
        made.append("fixtures_ekf.npz")
    for f in made:
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")
