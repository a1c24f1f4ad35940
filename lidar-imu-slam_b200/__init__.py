"""limu_b200 -- Python face of liblimu_cuda.so (the C ABI in include/limu_cuda.h).

A thin ctypes binding used by the tests, bench.py and __graft_entry__.py. Class and method names follow
the reference's C++ surface (lidar::VoxelHashMap, lidar::ICP, lidar::KissICP in
Oreoluwa-Se/Lidar-Imu-Slam env_ws/src/limu) so parity tests read like the reference's own
hash_map_test.hpp. There is NO CPU fallback: importing works anywhere (so CPU-only checks can verify the
exported symbols), but creating a Context without a usable B200 raises LimuError.

The directory name has a hyphen, so import it through ``__graft_entry__.load_package()`` (or
``importlib`` with this file's path); the module registers itself as ``limu_b200``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import weakref

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LIMU_LIB", os.path.join(HERE, "liblimu_cuda.so"))   # LIMU_LIB: instrumented builds (tools/)
HEADER = os.path.join(os.path.dirname(HERE), "include", "limu_cuda.h")

_dp, _fp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_float), C.POINTER(C.c_int32)
_lp = C.POINTER(C.c_int64)
_vp = C.c_void_p


ICP_REFERENCE, ICP_NN27, ICP_PLANE = 0, 1, 2   # limu_cuda.h LIMU_ICP_*: opt-in registration variants (SURVEY section 8f N2)


class LimuError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"limu status {status}: {msg}")
        self.status = status


class IcpStats(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("converged", C.c_int32), ("last_ncorr", C.c_int64),
                ("mean_candidates", C.c_double), ("miss_fraction", C.c_double)]


class IcpHypothesis(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("converged", C.c_int32), ("inliers", C.c_int64), ("rms", C.c_double)]


class RelocGrid(C.Structure):
    _fields_ = [("center", C.c_double * 7), ("nx", C.c_int32), ("ny", C.c_int32), ("nyaw", C.c_int32), ("reserved0", C.c_int32),
                ("step_xy", C.c_double), ("step_yaw", C.c_double)]


class RelocCandidate(C.Structure):
    _fields_ = [("index", C.c_int64), ("coarse_pose", C.c_double * 7), ("coarse_inliers", C.c_int64), ("coarse_rms", C.c_double),
                ("pose", C.c_double * 7), ("icp", IcpHypothesis)]


class OdomConfig(C.Structure):
    _fields_ = [("voxel_size", C.c_double), ("max_range", C.c_double), ("max_points_per_voxel", C.c_int32),
                ("deskew", C.c_int32), ("min_motion_th", C.c_double), ("icp_max_iteration", C.c_int32),
                ("icp_mode", C.c_int32), ("initial_threshold", C.c_double), ("estimation_threshold", C.c_double),
                ("map_capacity_voxels", C.c_int64), ("max_points_per_scan", C.c_int64)]


class FrameStats(C.Structure):
    _fields_ = [("n_points", C.c_int64), ("n_down", C.c_int64), ("n_keypoints", C.c_int64), ("sigma", C.c_double),
                ("icp", IcpStats), ("deskewed", C.c_int32), ("reserved0", C.c_int32)]


class CloudFields(C.Structure):
    """Where a PointCloud2 payload keeps the members of the reference's LidarPoint (lidar/frame.hpp:12-23); -1 = absent."""
    _fields_ = [("point_step", C.c_int32), ("off_x", C.c_int32), ("off_y", C.c_int32), ("off_z", C.c_int32), ("off_intensity", C.c_int32),
                ("off_ring", C.c_int32), ("off_timestamp", C.c_int32), ("off_time_field", C.c_int32), ("time_field_is_f64", C.c_int32)]


class LidarConfig(C.Structure):
    """frame::Lidar::ProcessingInfo's sensor fields (lidar/frame.hpp:39-45)."""
    _fields_ = [("min_range", C.c_double), ("max_range", C.c_double), ("min_angle", C.c_double), ("max_angle", C.c_double),
                ("frame_rate", C.c_double), ("num_scan_lines", C.c_int32), ("frame_split_num", C.c_int32)]


class ImuSample(C.Structure):
    _fields_ = [("t", C.c_double), ("gyr", C.c_double * 3), ("acc", C.c_double * 3)]


class ImuState(C.Structure):
    """The EKF state entries kalman::EKF::motion_compensation_with_imu reads (limu_cuda.h limu_imu_state)."""
    _fields_ = [("pos", C.c_double * 3), ("vel", C.c_double * 3), ("quat", C.c_double * 4), ("bga", C.c_double * 3), ("baa", C.c_double * 3),
                ("bat", C.c_double * 3), ("grav", C.c_double * 3), ("p_imu_lidar", C.c_double * 3), ("mean_acc_norm", C.c_double), ("gravity_norm", C.c_double),
                ("last_lidar_end_time", C.c_double), ("acc_s_last", C.c_double * 3), ("ang_vel_last", C.c_double * 3), ("tracker_vel", C.c_double * 3),
                ("tracker_pos", C.c_double * 3), ("tracker_quat", C.c_double * 4)]


class EkfParams(C.Structure):
    """limu_ekf_params == kalman::EKF_PARAMETERS (ekf.hpp:62-86)."""
    _fields_ = [("lidar_pose_trail", C.c_int32), ("reserved0", C.c_int32)] + [(n, C.c_double) for n in (
        "noise_scale", "init_pos_noise", "init_vel_noise", "init_ori_noise", "init_bga_noise", "init_baa_noise", "init_bat_noise",
        "acc_process_noise", "gyro_process_noise", "acc_process_noise_rev", "gyro_process_noise_rev",
        "init_lidar_imu_time_noise", "init_pos_trail_noise", "init_ori_trail_noise", "visualZuptR")]


def imu_forward_pass(state: ImuState, imu, lidar_beg_time, last_point_curvature_ms):
    """IMU forward pass of EKF::motion_compensation_with_imu (ekf.cpp:292-418), host code. imu: [k,7] rows {t, gyr xyz, acc xyz}, row 0 = the last
    sample of the previous window. Returns (table [M,22], rot_end [9], pos_lidar_end [3]); `state` is updated in place."""
    imu = np.ascontiguousarray(imu, np.float64).reshape(-1, 7)
    k = len(imu)
    table = np.zeros((k + 2, 22))
    rot_end, ple = np.zeros(9), np.zeros(3)
    n = C.c_int32(0)
    _chk(lib().limu_imu_forward_pass(C.byref(state), imu.ctypes.data_as(_vp), k, float(lidar_beg_time), float(last_point_curvature_ms),
                                     table.ctypes.data_as(_vp), len(table), C.byref(n), _d(rot_end), _d(ple)))
    return table[: n.value].copy(), rot_end, ple


def cloud_fields(fields, point_step) -> CloudFields:
    """fields: [(name, offset, PointField datatype, count)] -> the selection frame::Lidar::process_frame makes of them."""
    names = b"".join(f[0].encode() + b"\0" for f in fields)
    offs = np.array([f[1] for f in fields], np.int32)
    dts = np.array([f[2] for f in fields], np.int32)
    cnts = np.array([f[3] for f in fields], np.int32)
    out = CloudFields()
    _chk(lib().limu_cloud_fields_from_pointfields(len(fields), names, offs.ctypes.data_as(_ip), dts.ctypes.data_as(_ip), cnts.ctypes.data_as(_ip),
                                                  int(point_step), C.byref(out)))
    return out


def lidar_config(**kw) -> LidarConfig:
    cfg = LidarConfig()
    lib().limu_lidar_default_config(C.byref(cfg))
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


def build(force: bool = False) -> str:
    """Compile liblimu_cuda.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    srcs = [os.path.join(HERE, "csrc", f) for f in os.listdir(os.path.join(HERE, "csrc"))] + [HEADER]
    stale = not os.path.exists(LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        subprocess.check_call(["make", "-s", "-j8", "-C", HERE])
    return LIB_PATH


_lib = None


def lib():
    """Load the shared library (fails loudly if it was not built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LimuError(-2, f"{LIB_PATH} is missing: run __graft_entry__.build() (nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.limu_last_error.restype = C.c_char_p
        L.limu_source_hash.restype = C.c_char_p
        L.limu_kernel_launches.restype = C.c_uint64
        L.limu_host_alloc.restype = _vp
        L.limu_host_alloc.argtypes = [C.c_size_t]
        L.limu_host_free.argtypes = [_vp]
        L.limu_ctx_stream.restype = _vp
        L.limu_ctx_stream.argtypes = [_vp]
        L.limu_odom_map.restype = _vp
        L.limu_odom_map.argtypes = [_vp]
        sig = {
            "limu_ctx_create": [C.c_int, C.POINTER(_vp)], "limu_ctx_destroy": [_vp], "limu_ctx_sync": [_vp],
            "limu_ctx_set_profiling": [_vp, C.c_int], "limu_ctx_get_profile": [_vp, _dp, _lp],
            "limu_voxel_keys": [_vp, _dp, C.c_int64, C.c_double, _ip],
            "limu_transform_points": [_vp, _dp, _dp, C.c_int64],
            "limu_deskew": [_vp, _fp, C.c_int64, _dp, _dp, _dp],
            "limu_deskew_cloud": [_vp, _vp, C.c_int32, _dp, C.c_int64, _dp, _dp, _dp],
            "limu_deskew_imu": [_vp, _vp, C.c_int32, C.c_int32, C.c_int64, _dp, C.c_int32, _dp, _dp, _dp, _dp, C.c_int32],
            "limu_odom_register_cloud": [_vp, _vp, C.c_int32, _dp, C.c_int64, _dp, _dp, _lp, _dp, _lp, C.POINTER(FrameStats)],
            "limu_voxel_downsample": [_vp, _dp, C.c_int64, C.c_double, _dp, _lp, _lp],
            "limu_iqr_filter": [_vp, _dp, C.c_int64, _dp, _lp, _dp],
            "limu_voxelize": [_vp, _dp, C.c_int64, C.c_double, _dp, _lp, _dp, _lp],
            "limu_align": [_vp, _dp, _dp, C.c_int64, C.c_double, _dp, _dp, _dp, _dp],
            "limu_map_create": [_vp, C.c_double, C.c_double, C.c_int, C.c_int64, C.POINTER(_vp)],
            "limu_map_destroy": [_vp], "limu_map_clear": [_vp], "limu_map_empty": [_vp, C.POINTER(C.c_int)],
            "limu_map_size": [_vp, _lp, _lp],
            "limu_map_insert": [_vp, _dp, C.c_int64], "limu_map_insert_dev": [_vp, _vp, C.c_int64],
            "limu_map_update": [_vp, _dp, C.c_int64, _dp], "limu_map_update_origin": [_vp, _dp, C.c_int64, _dp],
            "limu_map_remove_far": [_vp, _dp],
            "limu_map_closest": [_vp, _dp, C.c_int64, _dp, _ip, _ip],
            "limu_map_correspondences": [_vp, _dp, C.c_int64, C.c_double, _dp, _dp, _lp, _lp],
            "limu_map_pointcloud": [_vp, _dp, C.c_int64, _lp],
            "limu_map_dump": [_vp, _ip, _ip, _dp, C.c_int64, C.c_int64, _lp, _lp],
            "limu_icp": [_vp, _dp, C.c_int64, _dp, C.c_double, C.c_double, C.c_int, C.c_double, _dp, C.POINTER(IcpStats), _dp, _lp, _dp],
            "limu_icp_ex": [_vp, _dp, C.c_int64, _dp, C.c_double, C.c_double, C.c_int, C.c_double, C.c_int32, _dp, C.POINTER(IcpStats), _dp, _lp, _dp],
            "limu_icp_multi": [_vp, _dp, C.c_int64, _dp, C.c_int32, C.c_double, C.c_double, C.c_int, C.c_double, C.c_int32, _dp, C.POINTER(IcpHypothesis),
                               C.POINTER(C.c_int32)],
            "limu_map_score_poses": [_vp, _dp, C.c_int64, _dp, C.c_int64, C.c_double, C.c_int32, _lp, _dp],
            "limu_relocalize": [_vp, _dp, C.c_int64, C.POINTER(RelocGrid), C.c_int32, C.c_double, C.c_double, C.c_int, C.c_double, C.c_int32,
                                C.POINTER(RelocCandidate), C.POINTER(C.c_int32), C.POINTER(C.c_int32)],
            "limu_map_closest_ex": [_vp, _dp, C.c_int64, C.c_int32, _dp, _ip, _ip],
            "limu_icp_dev": [_vp, _vp, C.c_int64, _dp, C.c_double, C.c_double, C.c_int, C.c_double, _dp, C.POINTER(IcpStats)],
            "limu_comm_create": [_vp, C.c_int, C.c_int, C.c_char_p], "limu_comm_connect": [_vp, C.c_char_p], "limu_comm_destroy": [_vp],
            "limu_comm_nccl_unique_id": [C.c_char_p], "limu_comm_nccl_init": [_vp, C.c_char_p],
            "limu_icp_sharded_dev": [_vp, _vp, C.c_int64, _dp, C.c_double, C.c_double, C.c_int, C.c_double, C.c_int, _dp, C.POINTER(IcpStats)],
            "limu_odom_default_config": [C.POINTER(OdomConfig)],
            "limu_odom_create": [_vp, C.POINTER(OdomConfig), C.POINTER(_vp)], "limu_odom_destroy": [_vp],
            "limu_odom_register_frame": [_vp, _fp, C.c_int64, _dp, _dp, _lp, _dp, _lp, C.POINTER(FrameStats)],
            "limu_odom_register_frame_dev": [_vp, _vp, C.c_int64, _dp, C.POINTER(FrameStats)],
            "limu_odom_prefetch": [_vp, _fp, C.c_int64],
            "limu_odom_prefetch_cloud": [_vp, _vp, C.c_int32, _dp, C.c_int64],
            "limu_odom_register_cloud_imu": [_vp, _vp, C.c_int32, C.c_int32, C.c_int64, _dp, C.c_int32, _dp, _dp, _dp, _dp, _dp, _lp, _dp, _lp, C.POINTER(FrameStats)],
            "limu_odom_prefetch_cloud_imu": [_vp, _vp, C.c_int32, C.c_int32, C.c_int64, _dp, C.c_int32, _dp, _dp, _dp],
            "limu_odom_hint_next_dev": [_vp, _vp, C.c_int64],
            "limu_odom_set_option": [_vp, C.c_int32, C.c_int64],
            "limu_odom_flush": [_vp],
            "limu_odom_register_points": [_vp, _dp, C.c_int64, _dp, _dp, _lp, _dp, _lp, C.POINTER(FrameStats)],
            "limu_odom_num_poses": [_vp, _lp], "limu_odom_pose": [_vp, C.c_int64, _dp],
            "limu_odom_adaptive_threshold": [_vp, _dp], "limu_odom_prediction": [_vp, _dp], "limu_odom_has_moved": [_vp, C.POINTER(C.c_int)],
            "limu_cloud_fields_from_pointfields": [C.c_int32, C.c_char_p, _ip, _ip, _ip, C.c_int32, C.POINTER(CloudFields)],
            "limu_lidar_default_config": [C.POINTER(LidarConfig)],
            "limu_preprocess_frame": [_vp, _vp, C.c_int64, C.POINTER(CloudFields), C.POINTER(LidarConfig), C.c_double, C.c_int32, _vp, _dp, C.c_int32, _lp, _dp,
                                      C.POINTER(C.c_int32)],
            "limu_odom_register_msg": [_vp, _vp, C.c_int64, C.POINTER(CloudFields), C.POINTER(LidarConfig), C.c_double, C.c_int32, C.c_int32, _dp, _lp, _dp,
                                       C.POINTER(C.c_int32), C.POINTER(FrameStats)],
            "limu_imu_forward_pass": [C.POINTER(ImuState), _vp, C.c_int32, C.c_double, C.c_double, _vp, C.c_int32, C.POINTER(C.c_int32), _dp, _dp],
            "limu_ekf_default_params": [C.POINTER(EkfParams)], "limu_ekf_create": [C.POINTER(EkfParams), C.POINTER(_vp)], "limu_ekf_destroy": [_vp],
            "limu_ekf_state_dim": [_vp, C.POINTER(C.c_int32)], "limu_ekf_get_state": [_vp, _dp, _dp, _dp], "limu_ekf_set_state": [_vp, _dp, _dp],
            "limu_ekf_initialize_orientation": [_vp, _dp, _dp], "limu_ekf_predict": [_vp, C.c_double, _dp, _dp, _dp, _dp, _dp],
            "limu_ekf_normalize_quaternions": [_vp, C.c_int], "limu_ekf_zero_velocity_update": [_vp, C.c_double], "limu_ekf_augment_pose_trail": [_vp],
            "limu_ekf_undo_augmentation": [_vp], "limu_ekf_update_and_propagate": [_vp], "limu_ekf_update_lidar_pose": [_vp, _dp, C.c_double, C.c_double],
            "limu_se3_exp": [_dp, _dp], "limu_se3_log": [_dp, _dp], "limu_se3_mul": [_dp, _dp, _dp], "limu_se3_inverse": [_dp, _dp],
        }
        for name, args in sig.items():
            getattr(L, name).argtypes = args
        _lib = L
    return _lib


def _chk(st):
    if st != 0:
        raise LimuError(st, lib().limu_last_error().decode())


def _d(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def _pts(x):
    return np.ascontiguousarray(x, dtype=np.float64).reshape(-1, 3)


def _pose(p):
    p = np.ascontiguousarray(p, dtype=np.float64)
    assert p.shape == (7,)
    return p


def source_hash() -> str:
    """Identity of the sources the LOADED library was built from (limu_source_hash)."""
    return lib().limu_source_hash().decode()


def kernel_launches() -> int:
    return int(lib().limu_kernel_launches())


def device_count() -> int:
    return int(lib().limu_device_count())


# ---- host-side SE(3) helpers -----------------------------------------------------------------------
def se3_exp(x6):
    x6 = np.ascontiguousarray(x6, np.float64)
    out = np.empty(7)
    lib().limu_se3_exp(_d(x6), _d(out))
    return out


def se3_log(p7):
    out = np.empty(6)
    lib().limu_se3_log(_d(_pose(p7)), _d(out))
    return out


def se3_mul(a, b):
    out = np.empty(7)
    lib().limu_se3_mul(_d(_pose(a)), _d(_pose(b)), _d(out))
    return out


def se3_inverse(a):
    out = np.empty(7)
    lib().limu_se3_inverse(_d(_pose(a)), _d(out))
    return out


class PinnedArray:
    """numpy view over cudaHostAlloc memory (limu_host_alloc)."""

    def __init__(self, shape, dtype):
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self.ptr = lib().limu_host_alloc(max(self.nbytes, 1))
        if not self.ptr:
            raise LimuError(-5, lib().limu_last_error().decode())
        buf = (C.c_char * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self.ptr:
            self.array = None
            lib().limu_host_free(self.ptr)
            self.ptr = None


class Context:
    """One GPU + one stream (limu_ctx)."""

    def __init__(self, device: int = 0):
        self.h = _vp()
        self._children = weakref.WeakSet()   # maps / odometry handles must die before their context
        _chk(lib().limu_ctx_create(device, C.byref(self.h)))
        self.device = device

    def close(self):
        if self.h:
            for child in list(self._children):
                child.close()
            lib().limu_ctx_destroy(self.h)
            self.h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        _chk(lib().limu_ctx_sync(self.h))

    def stream(self) -> int:
        return int(lib().limu_ctx_stream(self.h) or 0)

    # ---- multi-GPU (one process per GPU): mailbox handles are exchanged by the caller's transport ------------------
    def comm_init(self, rank, nranks, all_gather_bytes, broadcast_bytes=None, nccl_baseline=False):
        """all_gather_bytes(b) -> [b_rank0, b_rank1, ...]; broadcast_bytes(b_or_None) -> bytes from rank 0."""
        buf = C.create_string_buffer(64)
        _chk(lib().limu_comm_create(self.h, int(rank), int(nranks), buf))
        handles = all_gather_bytes(buf.raw)
        assert len(handles) == nranks and all(len(h) == 64 for h in handles)
        _chk(lib().limu_comm_connect(self.h, b"".join(handles)))
        if nccl_baseline:
            idb = C.create_string_buffer(128)
            if rank == 0:
                _chk(lib().limu_comm_nccl_unique_id(idb))
            idr = broadcast_bytes(idb.raw if rank == 0 else None)
            _chk(lib().limu_comm_nccl_init(self.h, idr))
        self.rank, self.nranks = rank, nranks

    def comm_destroy(self):
        lib().limu_comm_destroy(self.h)

    STAGES = ("prepare", "downsample", "iqr", "icp", "map_update")

    def set_profiling(self, enabled: bool):
        _chk(lib().limu_ctx_set_profiling(self.h, int(enabled)))

    def profile(self):
        """{stage: accumulated device ms} and the number of frames folded in."""
        ms = np.zeros(len(self.STAGES))
        fr = np.zeros(1, np.int64)
        _chk(lib().limu_ctx_get_profile(self.h, _d(ms), fr.ctypes.data_as(_lp)))
        return dict(zip(self.STAGES, ms.tolist())), int(fr[0])

    # utils::get_vox_index
    def voxel_keys(self, xyz, v):
        xyz = _pts(xyz)
        keys = np.empty((len(xyz), 3), np.int32)
        _chk(lib().limu_voxel_keys(self.h, _d(xyz), len(xyz), float(v), keys.ctypes.data_as(_ip)))
        return keys

    # utils::transform_points
    def transform_points(self, pose7, xyz):
        out = _pts(xyz).copy()
        _chk(lib().limu_transform_points(self.h, _d(_pose(pose7)), _d(out), len(out)))
        return out

    # MotionCompensator::deskew_scan
    def deskew_scan(self, xyzt_f32, T0, T1):
        x = np.ascontiguousarray(xyzt_f32, np.float32).reshape(-1, 4)
        out = np.empty((len(x), 3))
        _chk(lib().limu_deskew(self.h, x.ctypes.data_as(_fp), len(x), _d(_pose(T0)), _d(_pose(T1)), _d(out)))
        return out

    def deskew_cloud(self, records, stride_bytes, timestamps, T0, T1):
        """MotionCompensator::deskew_scan on strided point records (float x,y,z first) + float64 timestamps."""
        rec = np.ascontiguousarray(records)
        ts = np.ascontiguousarray(timestamps, np.float64)
        out = np.empty((len(ts), 3))
        _chk(lib().limu_deskew_cloud(self.h, rec.ctypes.data_as(_vp), int(stride_bytes), _d(ts), len(ts), _d(_pose(T0)), _d(_pose(T1)), _d(out)))
        return out

    def deskew_imu(self, xyzc_f32, table, rot_end, pos_lidar_end, p_imu_lidar):
        """EKF::motion_compensation_with_imu's per-point loop. xyzc = float32 [n,4] rows (x, y, z, curvature_ms) sorted by time;
        table = [M,22] kalman::Pose6D rows. Returns (deskewed float64 [n,3], written-back float32 [n,3])."""
        rec = np.ascontiguousarray(xyzc_f32, np.float32).reshape(-1, 4).copy()
        t = np.ascontiguousarray(table, np.float64).reshape(-1, 22)
        out = np.empty((len(rec), 3))
        re, pe, pil = (np.ascontiguousarray(v, np.float64) for v in (rot_end, pos_lidar_end, p_imu_lidar))
        _chk(lib().limu_deskew_imu(self.h, rec.ctypes.data_as(_vp), 16, 12, len(rec), _d(t), len(t), _d(re), _d(pe), _d(pil), _d(out), 1))
        return out, rec[:, :3].copy()

    def process_frame(self, data, fields, cfg, message_time, scan_count, max_segments=16):
        """frame::Lidar::process_frame (lidar/frame.cpp:101-193) on one PointCloud2 payload. data: uint8 [n, point_step];
        fields: [(name, offset, datatype, count)] or a CloudFields; cfg: LidarConfig or dict. Returns a list of segments
        dict(points [m,5] f32 = x,y,z,intensity,curvature; records [m,12] f32 = the 48-byte PCL rows; ts [m] f64; time)."""
        data = np.ascontiguousarray(data, np.uint8)
        n, step = data.shape
        cf = fields if isinstance(fields, CloudFields) else cloud_fields(fields, step)
        lc = cfg if isinstance(cfg, LidarConfig) else lidar_config(**cfg)
        rec = np.zeros((max(n, 1), 12), np.float32)
        ts = np.zeros(max(n, 1))
        sizes = np.zeros(max(max_segments, 1), np.int64)
        times = np.zeros(max(max_segments, 1))
        ns = C.c_int32(0)
        _chk(lib().limu_preprocess_frame(self.h, data.ctypes.data_as(_vp), n, C.byref(cf), C.byref(lc), float(message_time), int(scan_count),
                                         rec.ctypes.data_as(_vp), _d(ts), int(max_segments), sizes.ctypes.data_as(_lp), _d(times), C.byref(ns)))
        out, at = [], 0
        for k in range(ns.value):
            m = int(sizes[k])
            r = rec[at:at + m]
            out.append({"points": np.ascontiguousarray(r[:, [0, 1, 2, 8, 9]]), "records": r.copy(), "ts": ts[at:at + m].copy(), "time": float(times[k])})
            at += m
        return out

    def voxel_downsample(self, xyz, s, with_index=False):
        xyz = _pts(xyz)
        out = np.empty((max(len(xyz), 1), 3))
        idx = np.empty(max(len(xyz), 1), np.int64)
        n = C.c_int64(0)
        _chk(lib().limu_voxel_downsample(self.h, _d(xyz), len(xyz), float(s), _d(out), idx.ctypes.data_as(_lp), C.byref(n)))
        return (out[: n.value].copy(), idx[: n.value].copy()) if with_index else out[: n.value].copy()

    def iqr_processing(self, xyz, with_bounds=False):
        xyz = _pts(xyz)
        out = np.empty((max(len(xyz), 1), 3))
        n = C.c_int64(0)
        b = np.zeros(2)
        _chk(lib().limu_iqr_filter(self.h, _d(xyz), len(xyz), _d(out), C.byref(n), _d(b)))
        return (out[: n.value].copy(), b) if with_bounds else out[: n.value].copy()

    def voxelize(self, xyz, v):
        xyz = _pts(xyz)
        src = np.empty((max(len(xyz), 1), 3))
        down = np.empty((max(len(xyz), 1), 3))
        ns, nd = C.c_int64(0), C.c_int64(0)
        _chk(lib().limu_voxelize(self.h, _d(xyz), len(xyz), float(v), _d(src), C.byref(ns), _d(down), C.byref(nd)))
        return src[: ns.value].copy(), down[: nd.value].copy()

    # lidar::align_clouds
    def align_clouds(self, src, tgt, th):
        src, tgt = _pts(src), _pts(tgt)
        H, g, x, pose = np.empty((6, 6)), np.empty(6), np.empty(6), np.empty(7)
        _chk(lib().limu_align(self.h, _d(src), _d(tgt), len(src), float(th), _d(H), _d(g), _d(x), _d(pose)))
        return {"pose": pose, "H": H, "g": g, "x": x}

    def VoxelHashMap(self, vox_size, max_distance, max_points_per_voxel, capacity_voxels=0):
        return VoxelHashMap(self, vox_size, max_distance, max_points_per_voxel, capacity_voxels)

    def KissICP(self, **cfg):
        return KissICP(self, **cfg)


class VoxelHashMap:
    """lidar::VoxelHashMap (helpers/voxel_hash_map.hpp:14-48) resident in HBM."""

    def __init__(self, ctx, vox_size, max_distance, max_points_per_voxel, capacity_voxels=0, handle=None):
        self.ctx, self.cap = ctx, max_points_per_voxel
        self.owned = handle is None
        if handle is None:
            self.h = _vp()
            _chk(lib().limu_map_create(ctx.h, float(vox_size), float(max_distance), int(max_points_per_voxel), int(capacity_voxels), C.byref(self.h)))
            ctx._children.add(self)
        else:
            self.h = handle

    def close(self):
        if self.owned and self.h:
            lib().limu_map_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def insert_points(self, xyz):
        xyz = _pts(xyz)
        _chk(lib().limu_map_insert(self.h, _d(xyz), len(xyz)))

    def update(self, xyz, pose_or_origin):
        xyz = _pts(xyz)
        p = np.ascontiguousarray(pose_or_origin, np.float64)
        if p.shape == (7,):
            _chk(lib().limu_map_update(self.h, _d(xyz), len(xyz), _d(p)))
        else:
            _chk(lib().limu_map_update_origin(self.h, _d(xyz), len(xyz), _d(p)))

    def remove_points_from_far(self, origin):
        o = np.ascontiguousarray(origin, np.float64)
        _chk(lib().limu_map_remove_far(self.h, _d(o)))

    def clear(self):
        _chk(lib().limu_map_clear(self.h))

    def empty(self):
        e = C.c_int(0)
        _chk(lib().limu_map_empty(self.h, C.byref(e)))
        return bool(e.value)

    def size(self):
        nv, npt = C.c_int64(0), C.c_int64(0)
        _chk(lib().limu_map_size(self.h, C.byref(nv), C.byref(npt)))
        return nv.value, npt.value

    def get_closest_neighbour(self, xyz, with_index=False, icp_mode=0):
        """icp_mode: 0 = the reference's rule; ICP_NN27 = nearest point of the 27-cell neighbourhood (opt-in, SURVEY section 8f N2)."""
        xyz = _pts(xyz)
        out = np.empty((len(xyz), 3))
        key = np.empty((len(xyz), 3), np.int32)
        rank = np.empty(len(xyz), np.int32)
        _chk(lib().limu_map_closest_ex(self.h, _d(xyz), len(xyz), int(icp_mode), _d(out), key.ctypes.data_as(_ip), rank.ctypes.data_as(_ip)))
        return (out, key, rank) if with_index else out

    def get_correspondences(self, xyz, max_correspondance, with_index=False):
        xyz = _pts(xyz)
        n = max(len(xyz), 1)
        src, tgt, idx = np.empty((n, 3)), np.empty((n, 3)), np.empty(n, np.int64)
        k = C.c_int64(0)
        _chk(lib().limu_map_correspondences(self.h, _d(xyz), len(xyz), float(max_correspondance), _d(src), _d(tgt), idx.ctypes.data_as(_lp), C.byref(k)))
        k = k.value
        return (src[:k].copy(), tgt[:k].copy(), idx[:k].copy()) if with_index else (src[:k].copy(), tgt[:k].copy())

    def pointcloud(self):
        n = C.c_int64(0)
        _chk(lib().limu_map_pointcloud(self.h, None, 0, C.byref(n)))
        out = np.empty((max(n.value, 1), 3))
        _chk(lib().limu_map_pointcloud(self.h, _d(out), n.value, C.byref(n)))
        return out[: n.value]

    def dump(self):
        """(keys [V,3], counts [V], points [sum(counts),3]) in voxel creation order."""
        nv, npt = C.c_int64(0), C.c_int64(0)
        _chk(lib().limu_map_dump(self.h, None, None, None, 0, 0, C.byref(nv), C.byref(npt)))
        keys = np.empty((max(nv.value, 1), 3), np.int32)
        counts = np.empty(max(nv.value, 1), np.int32)
        pts = np.empty((max(npt.value, 1), 3))
        _chk(lib().limu_map_dump(self.h, keys.ctypes.data_as(_ip), counts.ctypes.data_as(_ip), _d(pts), nv.value, npt.value, C.byref(nv), C.byref(npt)))
        return keys[: nv.value], counts[: nv.value], pts[: npt.value]

    # lidar::ICP(local_map, points, init_guess, max_corresp_dist, kernel, icp_max_iteration, est_threshold)
    def icp(self, xyz, init_guess, max_corresp_dist, kernel, icp_max_iteration, est_threshold, trace=False, icp_mode=0):
        xyz = _pts(xyz)
        pose = np.empty(7)
        st = IcpStats()
        it = max(int(icp_max_iteration), 1)
        est = np.zeros((it, 7)) if trace else None
        nc = np.zeros(it, np.int64) if trace else None
        hg = np.zeros((it, 42)) if trace else None
        _chk(lib().limu_icp_ex(self.h, _d(xyz), len(xyz), _d(_pose(init_guess)), float(max_corresp_dist), float(kernel), int(icp_max_iteration),
                               float(est_threshold), int(icp_mode), _d(pose), C.byref(st), _d(est), nc.ctypes.data_as(_lp) if trace else None, _d(hg)))
        r = {"pose": pose, "iters": st.iterations, "converged": bool(st.converged), "last_ncorr": st.last_ncorr,
             "mean_candidates": st.mean_candidates, "miss_fraction": st.miss_fraction}
        if trace:
            r.update(est=est[: st.iterations], ncorr=nc[: st.iterations], hg=hg[: st.iterations])
        return r

    def icp_multi(self, xyz, guesses, max_corresp_dist, kernel, icp_max_iteration, est_threshold, icp_mode=0):
        """lidar::ICP from every row of guesses [k, 7] in one launch (limu_icp_multi): relocalization against this map.
        Returns dict(poses [k,7], iters [k], converged [k], inliers [k], rms [k], best); best = most inliers, then smaller rms, then lower index."""
        xyz = _pts(xyz)
        g = np.ascontiguousarray(np.asarray(guesses, np.float64).reshape(-1, 7))
        k = len(g)
        poses = np.empty((max(k, 1), 7))
        hyp = (IcpHypothesis * max(k, 1))()
        best = C.c_int32(-1)
        _chk(lib().limu_icp_multi(self.h, _d(xyz), len(xyz), _d(g), k, float(max_corresp_dist), float(kernel), int(icp_max_iteration),
                                  float(est_threshold), int(icp_mode), _d(poses), hyp, C.byref(best)))
        return {"poses": poses[:k].copy(), "iters": np.array([hyp[i].iterations for i in range(k)], np.int32),
                "converged": np.array([bool(hyp[i].converged) for i in range(k)], bool),
                "inliers": np.array([hyp[i].inliers for i in range(k)], np.int64), "rms": np.array([hyp[i].rms for i in range(k)]),
                "best": best.value}

    def score_poses(self, xyz, poses, max_corresp_dist, icp_mode=0):
        """Fitness of xyz at every row of poses [k, 7] without a Gauss-Newton loop (limu_map_score_poses): what icp_multi reports for a
        hypothesis run for 0 iterations. Returns dict(inliers [k], rms [k])."""
        xyz = _pts(xyz)
        p = np.ascontiguousarray(np.asarray(poses, np.float64).reshape(-1, 7))
        k = len(p)
        inl, rms = np.zeros(max(k, 1), np.int64), np.zeros(max(k, 1))
        _chk(lib().limu_map_score_poses(self.h, _d(xyz), len(xyz), _d(p), k, float(max_corresp_dist), int(icp_mode),
                                        inl.ctypes.data_as(_lp), _d(rms)))
        return {"inliers": inl[:k].copy(), "rms": rms[:k].copy()}

    def relocalize(self, xyz, center, nx, ny, nyaw, step_xy, step_yaw, n_refine, max_corresp_dist, kernel, icp_max_iteration, est_threshold,
                   icp_mode=0):
        """Global relocalization (limu_relocalize): score the planar grid of nx x ny x nyaw candidates around center (index (l * ny + j) * nx + i),
        keep the n_refine best by (inliers desc, rms asc, index asc) and run icp_multi from them. Returns dict of arrays in that order --
        index, coarse_poses, coarse_inliers, coarse_rms, poses, iters, converged, inliers, rms -- and best (icp_multi's rule)."""
        xyz = _pts(xyz)
        g = RelocGrid()
        g.center[:] = [float(v) for v in _pose(center)]
        g.nx, g.ny, g.nyaw, g.step_xy, g.step_yaw = int(nx), int(ny), int(nyaw), float(step_xy), float(step_yaw)
        cand = (RelocCandidate * max(1, min(int(n_refine), 4096)))()
        n_out, best = C.c_int32(0), C.c_int32(-1)
        _chk(lib().limu_relocalize(self.h, _d(xyz), len(xyz), C.byref(g), int(n_refine), float(max_corresp_dist), float(kernel),
                                   int(icp_max_iteration), float(est_threshold), int(icp_mode), cand, C.byref(n_out), C.byref(best)))
        c = cand[:n_out.value]
        return {"index": np.array([x.index for x in c], np.int64), "coarse_poses": np.array([list(x.coarse_pose) for x in c]).reshape(-1, 7),
                "coarse_inliers": np.array([x.coarse_inliers for x in c], np.int64), "coarse_rms": np.array([x.coarse_rms for x in c]),
                "poses": np.array([list(x.pose) for x in c]).reshape(-1, 7), "iters": np.array([x.icp.iterations for x in c], np.int32),
                "converged": np.array([bool(x.icp.converged) for x in c], bool), "inliers": np.array([x.icp.inliers for x in c], np.int64),
                "rms": np.array([x.icp.rms for x in c]), "best": best.value}

    def icp_dev(self, xyz_dev_ptr, n, init_guess, max_corresp_dist, kernel, icp_max_iteration, est_threshold):
        pose = np.empty(7)
        st = IcpStats()
        _chk(lib().limu_icp_dev(self.h, _vp(xyz_dev_ptr), int(n), _d(_pose(init_guess)), float(max_corresp_dist), float(kernel),
                                int(icp_max_iteration), float(est_threshold), _d(pose), C.byref(st)))
        return {"pose": pose, "iters": st.iterations, "converged": bool(st.converged), "last_ncorr": st.last_ncorr,
                "mean_candidates": st.mean_candidates, "miss_fraction": st.miss_fraction}

    def icp_sharded_dev(self, xyz_dev_ptr, n_local, init_guess, max_corresp_dist, kernel, icp_max_iteration, est_threshold, mode=0):
        """Point-sharded lidar::ICP: this rank's shard of the queries against the replicated map (mode 0 fused peer exchange, 1 NCCL baseline)."""
        pose = np.empty(7)
        st = IcpStats()
        _chk(lib().limu_icp_sharded_dev(self.h, _vp(xyz_dev_ptr), int(n_local), _d(_pose(init_guess)), float(max_corresp_dist), float(kernel),
                                        int(icp_max_iteration), float(est_threshold), int(mode), _d(pose), C.byref(st)))
        return {"pose": pose, "iters": st.iterations, "converged": bool(st.converged), "last_ncorr": st.last_ncorr,
                "candidates_total": st.mean_candidates, "misses_total": st.miss_fraction}

    def insert_points_dev(self, xyz_dev_ptr, n):
        _chk(lib().limu_map_insert_dev(self.h, _vp(xyz_dev_ptr), int(n)))


class KissICP:
    """lidar::KissICP (sensors/lidar/icp.hpp:31-68); config = frame::Lidar::ProcessingInfo fields."""

    def __init__(self, ctx, voxel_size=1.0, max_range=100.0, cap=10, deskew=False, min_motion_th=0.1, icp_max_iteration=500,
                 initial_threshold=2.0, estimation_threshold=1e-4, map_capacity_voxels=0, icp_mode=0, speculate=None):
        self.ctx = ctx
        cfg = OdomConfig()
        lib().limu_odom_default_config(C.byref(cfg))
        cfg.voxel_size, cfg.max_range, cfg.max_points_per_voxel, cfg.deskew = voxel_size, max_range, cap, int(deskew)
        cfg.min_motion_th, cfg.icp_max_iteration = min_motion_th, icp_max_iteration
        cfg.initial_threshold, cfg.estimation_threshold = initial_threshold, estimation_threshold
        cfg.map_capacity_voxels = map_capacity_voxels
        cfg.icp_mode = icp_mode
        self.cfg = cfg
        self.h = _vp()
        _chk(lib().limu_odom_create(ctx.h, C.byref(cfg), C.byref(self.h)))
        ctx._children.add(self)
        self.stats = FrameStats()
        if speculate is not None:
            self.set_speculate(speculate)

    def set_speculate(self, on: bool):
        """LIMU_OPT_SPECULATE: pipeline consecutive scans when the next one is known (hint_next_dev / prefetch; see limu_cuda.h)."""
        _chk(lib().limu_odom_set_option(self.h, 1, int(bool(on))))

    def flush(self):
        """Wait for what the handle has in flight; raises what a deferred map update had to report."""
        _chk(lib().limu_odom_flush(self.h))

    def close(self):
        if self.h:
            lib().limu_odom_destroy(self.h)
            self.h = None
            for b in getattr(self, "_outs", []):
                b.free()
            self._outs, self._out_n = [], -1

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _out_buffers(self, n):
        """Persistent pinned output buffers (grown on demand) so D2H copies are plain DMA."""
        if getattr(self, "_out_n", -1) < n:
            for b in getattr(self, "_outs", []):
                b.free()
            self._outs = [PinnedArray((max(n, 1), 3), np.float64), PinnedArray((max(n, 1), 3), np.float64)]
            self._out_n = n
        return self._outs[0].array, self._outs[1].array

    def register_frame(self, xyzt_f32, want_clouds=True, copy=True):
        """register_frame(cloud, timestamps): xyzt = float32 [n,4] (x,y,z,t in [0,1]). -> (down, keypoints, pose).
        With copy=False the clouds are views into pinned buffers that the next call overwrites."""
        x = xyzt_f32 if isinstance(xyzt_f32, np.ndarray) and xyzt_f32.dtype == np.float32 and xyzt_f32.flags.c_contiguous else np.ascontiguousarray(xyzt_f32, np.float32)
        x = x.reshape(-1, 4)
        n = len(x)
        pose = np.empty(7)
        if not want_clouds:
            _chk(lib().limu_odom_register_frame(self.h, x.ctypes.data_as(_fp), n, _d(pose), None, None, None, None, C.byref(self.stats)))
            return None, None, pose
        down, src = self._out_buffers(n)
        nd, ns = C.c_int64(0), C.c_int64(0)
        _chk(lib().limu_odom_register_frame(self.h, x.ctypes.data_as(_fp), n, _d(pose), _d(down), C.byref(nd), _d(src), C.byref(ns), C.byref(self.stats)))
        if copy:
            return down[: nd.value].copy(), src[: ns.value].copy(), pose
        return down[: nd.value], src[: ns.value], pose

    def prefetch(self, xyzt_f32):
        """Start the H2D copy of the NEXT scan (pinned float32 [n,4]); pass the same array to the next register_frame."""
        assert isinstance(xyzt_f32, np.ndarray) and xyzt_f32.dtype == np.float32 and xyzt_f32.flags.c_contiguous
        _chk(lib().limu_odom_prefetch(self.h, xyzt_f32.ctypes.data_as(_fp), xyzt_f32.size // 4))

    def prefetch_cloud(self, records, stride_bytes, timestamps):
        """Start the H2D copy of the NEXT cloud (contiguous records + float64 timestamps, ideally pinned); pass the same arrays to the next register_cloud."""
        assert isinstance(records, np.ndarray) and records.flags.c_contiguous
        assert isinstance(timestamps, np.ndarray) and timestamps.dtype == np.float64 and timestamps.flags.c_contiguous
        _chk(lib().limu_odom_prefetch_cloud(self.h, records.ctypes.data_as(_vp), int(stride_bytes), _d(timestamps), len(timestamps)))

    def register_cloud(self, records, stride_bytes, timestamps, copy=True):
        """register_frame(cloud, timestamps) on strided point records + float64 timestamps (the reference's layout).
        With copy=False the clouds are views into pinned buffers that the next call overwrites."""
        rec = records if isinstance(records, np.ndarray) and records.flags.c_contiguous else np.ascontiguousarray(records)
        ts = timestamps if isinstance(timestamps, np.ndarray) and timestamps.dtype == np.float64 and timestamps.flags.c_contiguous else np.ascontiguousarray(timestamps, np.float64)
        n = len(ts)
        pose = np.empty(7)
        down, src = self._out_buffers(n)
        nd, ns = C.c_int64(0), C.c_int64(0)
        _chk(lib().limu_odom_register_cloud(self.h, rec.ctypes.data_as(_vp), int(stride_bytes), _d(ts), n, _d(pose), _d(down), C.byref(nd), _d(src), C.byref(ns), C.byref(self.stats)))
        if copy:
            return down[: nd.value].copy(), src[: ns.value].copy(), pose
        return down[: nd.value], src[: ns.value], pose

    @staticmethod
    def _imu_args(table, rot_end, pos_lidar_end, p_imu_lidar):
        t = np.ascontiguousarray(table, np.float64).reshape(-1, 22)
        return (t,) + tuple(np.ascontiguousarray(v, np.float64).reshape(n) for v, n in ((rot_end, 9), (pos_lidar_end, 3), (p_imu_lidar, 3)))

    def register_cloud_imu(self, records, stride_bytes, curvature_offset, table, rot_end, pos_lidar_end, p_imu_lidar, copy=True):
        """EKF::motion_compensation_with_imu + register_frame(Vec3dVector) in one call (limu_odom_register_cloud_imu): records = contiguous point
        records (float x,y,z first, float curvature in ms at curvature_offset), table = [M,22] pose rows of imu_forward_pass. -> (down, keypoints,
        pose) in the scan-end lidar frame. With copy=False the clouds are views into pinned buffers that the next call overwrites."""
        rec = records if isinstance(records, np.ndarray) and records.flags.c_contiguous else np.ascontiguousarray(records)
        n = rec.nbytes // int(stride_bytes)
        t, re, pe, pil = self._imu_args(table, rot_end, pos_lidar_end, p_imu_lidar)
        pose = np.empty(7)
        down, src = self._out_buffers(n)
        nd, ns = C.c_int64(0), C.c_int64(0)
        _chk(lib().limu_odom_register_cloud_imu(self.h, rec.ctypes.data_as(_vp), int(stride_bytes), int(curvature_offset), n, _d(t), len(t), _d(re), _d(pe), _d(pil),
                                                _d(pose), _d(down), C.byref(nd), _d(src), C.byref(ns), C.byref(self.stats)))
        if copy:
            return down[: nd.value].copy(), src[: ns.value].copy(), pose
        return down[: nd.value], src[: ns.value], pose

    def prefetch_cloud_imu(self, records, stride_bytes, curvature_offset, table, rot_end, pos_lidar_end, p_imu_lidar):
        """Start the H2D copy of the NEXT cloud (contiguous records, ideally pinned) and its pose table; pass the same records and IMU arguments to
        the next register_cloud_imu."""
        assert isinstance(records, np.ndarray) and records.flags.c_contiguous
        t, re, pe, pil = self._imu_args(table, rot_end, pos_lidar_end, p_imu_lidar)
        _chk(lib().limu_odom_prefetch_cloud_imu(self.h, records.ctypes.data_as(_vp), int(stride_bytes), int(curvature_offset), records.nbytes // int(stride_bytes),
                                                _d(t), len(t), _d(re), _d(pe), _d(pil)))

    def register_msg(self, data, fields, cfg, message_time, scan_count, max_segments=16):
        """lidar_callback -> estimate_lidar_odometry for one PointCloud2 payload: preprocess + register every segment on the
        device. Returns (poses [k,7], segment sizes [k], segment times [k], [FrameStats] * k)."""
        data = np.ascontiguousarray(data, np.uint8)
        n, step = data.shape
        cf = fields if isinstance(fields, CloudFields) else cloud_fields(fields, step)
        lc = cfg if isinstance(cfg, LidarConfig) else lidar_config(**cfg)
        poses = np.zeros((max(max_segments, 1), 7))
        sizes = np.zeros(max(max_segments, 1), np.int64)
        times = np.zeros(max(max_segments, 1))
        stats = (FrameStats * max(max_segments, 1))()
        ns = C.c_int32(0)
        _chk(lib().limu_odom_register_msg(self.h, data.ctypes.data_as(_vp), n, C.byref(cf), C.byref(lc), float(message_time), int(scan_count),
                                          int(max_segments), _d(poses), sizes.ctypes.data_as(_lp), _d(times), C.byref(ns), stats))
        k = ns.value
        return poses[:k].copy(), sizes[:k].copy(), times[:k].copy(), [stats[j] for j in range(k)]

    def register_frame_dev(self, xyzt_dev_ptr, n):
        pose = np.empty(7)
        _chk(lib().limu_odom_register_frame_dev(self.h, _vp(xyzt_dev_ptr), int(n), _d(pose), C.byref(self.stats)))
        return pose

    def hint_next_dev(self, xyzt_dev_ptr, n):
        """Replay hint: the scan after the next register_frame_dev call already sits at this device address (see limu_cuda.h)."""
        _chk(lib().limu_odom_hint_next_dev(self.h, _vp(xyzt_dev_ptr), int(n)))

    def register_points(self, xyz):
        """register_frame(Vec3dVector)."""
        xyz = _pts(xyz)
        n = len(xyz)
        pose = np.empty(7)
        down, src = np.empty((max(n, 1), 3)), np.empty((max(n, 1), 3))
        nd, ns = C.c_int64(0), C.c_int64(0)
        _chk(lib().limu_odom_register_points(self.h, _d(xyz), n, _d(pose), _d(down), C.byref(nd), _d(src), C.byref(ns), C.byref(self.stats)))
        return down[: nd.value].copy(), src[: ns.value].copy(), pose

    def poses(self):
        n = C.c_int64(0)
        _chk(lib().limu_odom_num_poses(self.h, C.byref(n)))
        out = np.empty((n.value, 7))
        for i in range(n.value):
            _chk(lib().limu_odom_pose(self.h, i, _d(out[i])))
        return out

    def local_map(self):
        return VoxelHashMap(self.ctx, 0, 0, self.cfg.max_points_per_voxel, handle=_vp(lib().limu_odom_map(self.h)))

    def has_moved(self):
        e = C.c_int(0)
        _chk(lib().limu_odom_has_moved(self.h, C.byref(e)))
        return bool(e.value)

    def get_adaptive_threshold(self):
        """KissICP::get_adaptive_threshold (icp.cpp:138-144) -- with the reference's side effect: every call adds a sample to the model."""
        out = C.c_double(0.0)
        _chk(lib().limu_odom_adaptive_threshold(self.h, C.byref(out)))
        return out.value

    def get_prediction_model(self):
        out = np.empty(7)
        _chk(lib().limu_odom_prediction(self.h, _d(out)))
        return out


class Ekf:
    """kalman::EKF predict / update (L/src/kalman/ekf.cpp), host code inside the library (SURVEY section 8f N4)."""

    def __init__(self, **params):
        p = EkfParams()
        lib().limu_ekf_default_params(C.byref(p))
        for k, v in params.items():
            setattr(p, k, v)
        self.params = p
        self.h = _vp()
        _chk(lib().limu_ekf_create(C.byref(p), C.byref(self.h)))
        d = C.c_int32(0)
        _chk(lib().limu_ekf_state_dim(self.h, C.byref(d)))
        self.dim = d.value

    def close(self):
        if self.h:
            lib().limu_ekf_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def state(self):
        """(m [dim], P [dim, dim], current_time)."""
        m, P, t = np.empty(self.dim), np.empty((self.dim, self.dim)), np.empty(1)
        _chk(lib().limu_ekf_get_state(self.h, _d(m), _d(P), _d(t)))
        return m, P, float(t[0])

    def set_state(self, m=None, P=None):
        _chk(lib().limu_ekf_set_state(self.h, _d(np.ascontiguousarray(m, np.float64)) if m is not None else None,
                                      _d(np.ascontiguousarray(P, np.float64)) if P is not None else None))

    def initialize_orientation(self, xa, calc_grav):
        _chk(lib().limu_ekf_initialize_orientation(self.h, _d(np.ascontiguousarray(xa, np.float64)), _d(np.ascontiguousarray(calc_grav, np.float64))))

    def predict(self, t, xg, xa, calc_grav, trans_lidar_imu, rot_lidar_imu):
        a = [np.ascontiguousarray(x, np.float64) for x in (xg, xa, calc_grav, trans_lidar_imu, np.asarray(rot_lidar_imu, np.float64).reshape(9))]
        _chk(lib().limu_ekf_predict(self.h, float(t), *[_d(x) for x in a]))

    def normalize_quaternions(self, only_current=False):
        _chk(lib().limu_ekf_normalize_quaternions(self.h, int(only_current)))

    def zero_velocity_update(self, r):
        _chk(lib().limu_ekf_zero_velocity_update(self.h, float(r)))

    def augment_pose_trail(self):
        _chk(lib().limu_ekf_augment_pose_trail(self.h))

    def undo_augmentation(self):
        _chk(lib().limu_ekf_undo_augmentation(self.h))

    def update_and_propagate(self):
        _chk(lib().limu_ekf_update_and_propagate(self.h))

    def update_lidar_pose(self, pose7, pos_sigma, ori_sigma):
        _chk(lib().limu_ekf_update_lidar_pose(self.h, _d(_pose(pose7)), float(pos_sigma), float(ori_sigma)))
