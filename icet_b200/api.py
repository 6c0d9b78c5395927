"""ctypes binding of include/icet_b200.h and the Python mirror of the reference's `class ICET`."""
from __future__ import annotations

import ctypes as C
import os
import weakref
from dataclasses import dataclass

import numpy as np

from . import build as _build

_FP, _IP, _BP = C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_uint8)


class IcetError(RuntimeError):
    pass


class Params(C.Structure):
    """ctor arguments of the reference (include/icet.h:38-40)."""
    _fields_ = [("runlen", C.c_int32), ("bins_phi", C.c_int32), ("bins_theta", C.c_int32), ("n", C.c_int32),
                ("thresh", C.c_float), ("buff", C.c_float), ("flags", C.c_int32), ("reserved", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("X", C.c_float * 6), ("pred_stds", C.c_float * 6), ("Q", C.c_float * 36), ("status", C.c_int32),
                ("n_gauss1", C.c_int32), ("n_used", C.c_int32), ("n_dropped", C.c_int32), ("cond", C.c_float),
                ("reserved", C.c_int32 * 3)]


RESULT_DTYPE = np.dtype([("X", np.float32, 6), ("pred_stds", np.float32, 6), ("Q", np.float32, (6, 6)),
                         ("status", np.int32), ("n_gauss1", np.int32), ("n_used", np.int32),
                         ("n_dropped", np.int32), ("cond", np.float32), ("reserved", np.int32, 3)])
assert RESULT_DTYPE.itemsize == C.sizeof(Result) == 224

FLAG_FULL_EIG = 1
FLAG_UNFUSED_LOOP = 2
FLAG_PERSISTENT_LOOP = 4
FLAG_SHIPPED_ORDER = 16  # validation: cluster in the row order the reference's broken permutation loop leaves (single pair)
FLAG_EXACT_PASS = 32  # scan 2: the reference's per-point pipeline in every iteration (validation form)
FLAG_FULL_REBUILD = 64  # scan 2: incremental bookkeeping, every point re-evaluated in every iteration (diagnostic)
FLAG_VERIFY_INCREMENTAL = 128  # self-check: result["reserved"][0] counts stable points whose class changed (must be 0)
FLAG_CLUSTER_LOOP = 256  # the loop of every pair inside one thread-block cluster (default for single / chained pairs)
FLAG_CHAIN_X0 = 8  # odometry.cpp:82: pair k+1 starts from the solution of pair k; X0 = one seed (pair 0)

_DUMP_FIELDS = [("cnt1", _IP), ("bounds", _FP), ("nin1", _IP), ("has1", _BP), ("mu1", _FP), ("sigma1", _FP),
                ("evec1", _FP), ("eval1", _FP), ("lmask", _BP), ("cnt2", _IP), ("nin2", _IP), ("used2", _BP),
                ("mu2", _FP), ("sigma2", _FP), ("Xit", _FP), ("HTWH", _FP), ("HTWdz", _FP), ("TRit", _FP),
                ("testPoints", _FP)]


class OdometryParams(C.Structure):
    """icet_b200_odometry_params: the steps the reference's ROS nodes wrap around the constructor."""
    _fields_ = [("min_range", C.c_float), ("chain_x0", C.c_int32), ("rate_hz", C.c_float), ("guard_trans", C.c_float),
                ("guard_rot", C.c_float), ("reserved", C.c_int32 * 3)]


class Pose(C.Structure):
    _fields_ = [("X_homo", C.c_float * 16), ("position", C.c_float * 3), ("orientation", C.c_float * 4),
                ("covariance_diag", C.c_float * 6), ("twist", C.c_float * 6), ("X", C.c_float * 6),
                ("n_points", C.c_int32), ("guarded", C.c_int32), ("frame", C.c_int32), ("reserved", C.c_int32)]


POSE_DTYPE = np.dtype([("X_homo", np.float32, (4, 4)), ("position", np.float32, 3), ("orientation", np.float32, 4),
                       ("covariance_diag", np.float32, 6), ("twist", np.float32, 6), ("X", np.float32, 6),
                       ("n_points", np.int32), ("guarded", np.int32), ("frame", np.int32), ("reserved", np.int32)])
assert POSE_DTYPE.itemsize == C.sizeof(Pose) == 180


class KeyframePolicy(C.Structure):
    """icet_b200_keyframe_policy: when a scan of the keyframe odometry node becomes the next keyframe.  A scan is
    promoted when ||X_rel[:3]|| > max_trans, max |X_rel[3:]| > max_rot, n_used < min_overlap * n_gauss1 of the keyframe,
    max_interval scans have been registered against the keyframe, or its registration has status != 0.  A threshold
    <= 0 turns its test off.  The defaults are those DESIGN.md §13 chose from the drift measurement."""
    _fields_ = [("max_trans", C.c_float), ("max_rot", C.c_float), ("min_overlap", C.c_float),
                ("max_interval", C.c_int32), ("reserved", C.c_int32 * 4)]

    def __init__(self, max_trans=1.0, max_rot=0.1, min_overlap=0.5, max_interval=10):
        for name, v in (("max_trans", max_trans), ("max_rot", max_rot), ("min_overlap", min_overlap)):
            if not np.isfinite(v):
                raise ValueError("policy.%s must be finite" % name)
        if int(max_interval) != max_interval:
            raise ValueError("policy.max_interval must be an integer")
        super().__init__(float(max_trans), float(max_rot), float(min_overlap), int(max_interval))


KF_TRANS, KF_ROT, KF_OVERLAP, KF_INTERVAL, KF_STATUS = 1, 2, 4, 8, 16  # icet_b200_kf_info.reason bits


class KfInfo(C.Structure):
    _fields_ = [("keyframe", C.c_int32), ("promoted", C.c_int32), ("reason", C.c_int32), ("x0", C.c_float * 6),
                ("reserved", C.c_int32)]


KF_INFO_DTYPE = np.dtype([("keyframe", np.int32), ("promoted", np.int32), ("reason", np.int32), ("x0", np.float32, 6),
                          ("reserved", np.int32)])
assert KF_INFO_DTYPE.itemsize == C.sizeof(KfInfo) == 40


F32, F64, I32 = 0, 1, 2


class Cloud(C.Structure):
    """icet_b200_cloud: a caller's point buffer in its native layout (ingest, SURVEY.md 8f N3)."""
    _fields_ = [("data", C.c_void_p), ("n", C.c_int32), ("point_step", C.c_int32), ("off", C.c_int32 * 3),
                ("dtype", C.c_int32), ("divide", C.c_float), ("plane_stride", C.c_int32)]


def cloud_desc(a, divide: float = 0.0, point_step: int | None = None, offsets=None, dtype=None, n=None):
    """Describe a host buffer without touching its elements.  Returns (Cloud, keep-alive object).
      * N x 3 C-order float32 / float64 / int32 (records), N x 3 Fortran-order or 3 x N C-order (planes);
      * raw bytes of a sensor_msgs::PointCloud2 (`a` = data, point_step, offsets = field offsets of x, y, z)."""
    if point_step is not None:
        buf = np.frombuffer(a, dtype=np.uint8) if not isinstance(a, np.ndarray) else a.view(np.uint8).reshape(-1)
        cnt = buf.size // point_step if n is None else n
        c = Cloud(buf.ctypes.data, cnt, point_step, (C.c_int32 * 3)(*offsets), F32 if dtype is None else dtype,
                  divide, 0)
        return c, buf
    a = np.asarray(a)
    code = {np.dtype(np.float32): F32, np.dtype(np.float64): F64, np.dtype(np.int32): I32}.get(a.dtype)
    if code is None or a.ndim != 2:
        raise ValueError("cloud must be a 2-D float32 / float64 / int32 array")
    es = a.dtype.itemsize
    if a.shape[1] == 3 and a.shape[0] != 3 and a.flags["C_CONTIGUOUS"]:
        return Cloud(a.ctypes.data, a.shape[0], 3 * es, (C.c_int32 * 3)(0, es, 2 * es), code, divide, 0), a
    if a.shape[1] == 3 and a.shape[0] != 3 and a.flags["F_CONTIGUOUS"]:
        return Cloud(a.ctypes.data, a.shape[0], 0, (C.c_int32 * 3)(0, 0, 0), code, divide, a.shape[0]), a
    if a.shape[0] == 3 and a.flags["C_CONTIGUOUS"]:
        return Cloud(a.ctypes.data, a.shape[1], 0, (C.c_int32 * 3)(0, 0, 0), code, divide, a.shape[1]), a
    a = np.ascontiguousarray(a)
    return cloud_desc(a, divide)


class _Dump(C.Structure):
    _fields_ = _DUMP_FIELDS


EXPORTS = ["icet_b200_version", "icet_b200_last_error", "icet_b200_create", "icet_b200_destroy",
           "icet_b200_set_stream", "icet_b200_set_chunk", "icet_b200_set_host_chunk", "icet_b200_set_lanes", "icet_b200_debug_timeline", "icet_b200_register", "icet_b200_register_batch",
           "icet_b200_register_batch_device", "icet_b200_register_sequence_device", "icet_b200_synchronize",
           "icet_b200_set_dump", "icet_b200_get_dump", "icet_b200_get_points2", "icet_b200_spherical_bins",
           "icet_b200_classify_scan2",
           "icet_b200_synth_scans_device", "icet_b200_kernel_launches", "icet_b200_set_profile",
           "icet_b200_get_profile", "icet_b200_kernel_name",
           "icet_b200_node_create", "icet_b200_node_destroy", "icet_b200_node_push_device", "icet_b200_node_push",
           "icet_b200_node_current_scan", "icet_b200_node_last_result", "icet_b200_map_create",
           "icet_b200_map_destroy", "icet_b200_map_add_scan_device", "icet_b200_map_get", "icet_b200_map_get_device",
           "icet_b200_ingest", "icet_b200_register_clouds", "icet_b200_node_push_cloud",
           "icet_b200_transform_cloud_device", "icet_b200_transform_cloud",
           "icet_b200_multi_create", "icet_b200_multi_destroy", "icet_b200_multi_devices", "icet_b200_multi_context",
           "icet_b200_register_batch_multi", "icet_b200_register_sequence_multi_device", "icet_b200_multi_gathered",
           "icet_b200_multi_gathered_host", "icet_b200_keyframe_create", "icet_b200_keyframe_create_device",
           "icet_b200_keyframe_destroy", "icet_b200_keyframe_gaussians", "icet_b200_register_keyframe",
           "icet_b200_register_keyframe_batch_device", "icet_b200_kfnode_create", "icet_b200_kfnode_destroy",
           "icet_b200_kfnode_push_device", "icet_b200_kfnode_push", "icet_b200_kfnode_push_cloud",
           "icet_b200_kfnode_keyframe", "icet_b200_kfnode_create_local_map", "icet_b200_kfnode_local_map",
           "icet_b200_kfnode_local_map_host"]
NKERNELS = 11

_LIB = None


def lib_path() -> str:
    """The in-tree library; ICET_B200_LIB overrides it (A/B runs of two builds on the same GPU box)."""
    return os.environ.get("ICET_B200_LIB") or _build.LIB


def load_library() -> C.CDLL:
    """Load libicet_b200.so.  Fails loudly when it has not been built -- there is no fallback."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise IcetError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(icet_b200 has no CPU / PyTorch fallback)" % path)
    L = C.CDLL(path)
    vp = C.c_void_p
    L.icet_b200_version.restype = C.c_int
    L.icet_b200_last_error.restype = C.c_char_p
    L.icet_b200_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.icet_b200_destroy.argtypes = [vp]
    L.icet_b200_set_stream.argtypes = [vp, vp]
    L.icet_b200_set_chunk.argtypes = [vp, C.c_int32]
    L.icet_b200_set_host_chunk.argtypes = [vp, C.c_int32]
    L.icet_b200_set_lanes.argtypes = [vp, C.c_int32]
    L.icet_b200_debug_timeline.argtypes = [vp, vp, C.c_int32]
    L.icet_b200_register.argtypes = [vp, C.POINTER(Params), vp, C.c_int32, C.c_int32, vp, C.c_int32, C.c_int32,
                                     vp, C.POINTER(Result)]
    L.icet_b200_register_batch.argtypes = [vp, C.POINTER(Params), C.c_int32, vp, vp, vp, vp, vp, vp]
    L.icet_b200_register_batch_device.argtypes = [vp, C.POINTER(Params), C.c_int32, vp, vp, vp, vp, vp, vp]
    L.icet_b200_register_sequence_device.argtypes = [vp, C.POINTER(Params), C.c_int32, vp, C.c_int32, vp]
    L.icet_b200_synchronize.argtypes = [vp]
    L.icet_b200_set_dump.argtypes = [vp, C.c_int32]
    L.icet_b200_get_dump.argtypes = [vp, C.POINTER(_Dump)]
    L.icet_b200_get_points2.argtypes = [vp, vp, C.c_int32]
    L.icet_b200_classify_scan2.argtypes = [vp, C.c_int32, vp, vp, C.c_int32]
    L.icet_b200_spherical_bins.argtypes = [vp, C.POINTER(Params), vp, C.c_int32, C.c_int32, vp, vp]
    L.icet_b200_synth_scans_device.argtypes = [vp, C.c_uint64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp]
    L.icet_b200_kernel_launches.argtypes = [vp]
    L.icet_b200_kernel_launches.restype = C.c_int64
    L.icet_b200_set_profile.argtypes = [vp, C.c_int32]
    L.icet_b200_get_profile.argtypes = [vp, vp, vp]
    L.icet_b200_kernel_name.argtypes = [C.c_int]
    L.icet_b200_node_create.argtypes = [vp, C.POINTER(Params), C.POINTER(OdometryParams), C.c_int32, vp, vp,
                                        C.POINTER(vp)]
    L.icet_b200_node_destroy.argtypes = [vp]
    L.icet_b200_node_push_device.argtypes = [vp, C.c_int32, vp, C.c_int32, vp, vp]
    L.icet_b200_node_push.argtypes = [vp, vp, C.c_int32, C.c_int32, C.POINTER(Result), C.POINTER(Pose)]
    L.icet_b200_node_current_scan.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_int32)]
    L.icet_b200_node_last_result.argtypes = [vp, C.POINTER(vp)]
    L.icet_b200_map_create.argtypes = [vp, C.c_int32, C.POINTER(vp)]
    L.icet_b200_map_destroy.argtypes = [vp]
    L.icet_b200_map_add_scan_device.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, vp, C.c_int32, vp, C.c_float,
                                                C.c_float]
    L.icet_b200_map_get.argtypes = [vp, vp, C.c_int32, C.POINTER(C.c_int32)]
    L.icet_b200_map_get_device.argtypes = [vp, vp, C.c_int32, vp]
    L.icet_b200_transform_cloud_device.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, vp, C.c_int32, vp, C.c_int32]
    L.icet_b200_transform_cloud.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, C.c_int32, vp, C.c_int32]
    L.icet_b200_ingest.argtypes = [vp, C.POINTER(Cloud), vp, C.c_int32]
    L.icet_b200_register_clouds.argtypes = [vp, C.POINTER(Params), C.POINTER(Cloud), C.POINTER(Cloud), vp,
                                            C.POINTER(Result)]
    L.icet_b200_node_push_cloud.argtypes = [vp, C.POINTER(Cloud), C.POINTER(Result), C.POINTER(Pose)]
    L.icet_b200_kernel_name.restype = C.c_char_p
    L.icet_b200_multi_create.argtypes = [vp, C.c_int32, C.POINTER(vp)]
    L.icet_b200_multi_destroy.argtypes = [vp]
    L.icet_b200_multi_devices.argtypes = [vp]
    L.icet_b200_multi_context.argtypes = [vp, C.c_int32]
    L.icet_b200_multi_context.restype = vp
    L.icet_b200_register_batch_multi.argtypes = [vp, C.POINTER(Params), C.c_int32, vp, vp, vp, vp, vp, vp]
    L.icet_b200_register_sequence_multi_device.argtypes = [vp, C.POINTER(Params), C.c_int32, vp, C.c_int32]
    L.icet_b200_multi_gathered.argtypes = [vp, C.c_int32, C.POINTER(vp), C.POINTER(C.c_int32)]
    L.icet_b200_multi_gathered_host.argtypes = [vp, C.c_int32, vp]
    L.icet_b200_keyframe_create.argtypes = [vp, C.POINTER(Params), vp, C.c_int32, C.c_int32, C.POINTER(vp)]
    L.icet_b200_keyframe_create_device.argtypes = [vp, C.POINTER(Params), vp, C.c_int32, C.c_int32, C.POINTER(vp)]
    L.icet_b200_keyframe_destroy.argtypes = [vp]
    L.icet_b200_keyframe_gaussians.argtypes = [vp]
    L.icet_b200_register_keyframe.argtypes = [vp, C.POINTER(Params), vp, C.c_int32, C.c_int32, vp, C.POINTER(Result)]
    L.icet_b200_register_keyframe_batch_device.argtypes = [vp, C.POINTER(Params), C.c_int32, vp, vp, vp, vp]
    L.icet_b200_kfnode_create.argtypes = [vp, C.POINTER(Params), C.POINTER(OdometryParams), C.POINTER(KeyframePolicy),
                                          C.c_int32, vp, vp, C.POINTER(vp)]
    L.icet_b200_kfnode_destroy.argtypes = [vp]
    L.icet_b200_kfnode_push_device.argtypes = [vp, C.c_int32, vp, C.c_int32, vp, vp, vp]
    L.icet_b200_kfnode_push.argtypes = [vp, vp, C.c_int32, C.c_int32, C.POINTER(Result), C.POINTER(Pose),
                                        C.POINTER(KfInfo)]
    L.icet_b200_kfnode_push_cloud.argtypes = [vp, C.POINTER(Cloud), C.POINTER(Result), C.POINTER(Pose),
                                              C.POINTER(KfInfo)]
    L.icet_b200_kfnode_keyframe.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_int32)]
    L.icet_b200_kfnode_create_local_map.argtypes = [vp, C.POINTER(Params), C.POINTER(OdometryParams),
                                                    C.POINTER(KeyframePolicy), C.c_int32, C.c_int32, vp, vp,
                                                    C.POINTER(vp)]
    L.icet_b200_kfnode_local_map.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_int32)]
    L.icet_b200_kfnode_local_map_host.argtypes = [vp, vp, C.c_int32, C.POINTER(C.c_int32)]
    _LIB = L
    return L


def as_planes(cloud) -> np.ndarray:
    """N x 3 (any dtype/order) or 3 x N -> C-contiguous float32 [3, N] planes = the memory of a
    column-major Eigen::MatrixXf(N, 3)."""
    a = np.asarray(cloud)
    if a.ndim != 2:
        raise ValueError("cloud must be 2-D")
    if a.shape[1] == 3 and a.shape[0] != 3:
        a = a.T
    elif a.shape[0] != 3:
        raise ValueError("cloud must be N x 3 or 3 x N")
    return np.ascontiguousarray(a, dtype=np.float32)


def make_params(runlen=7, bins_phi=24, bins_theta=75, n=25, thresh=0.1, buff=0.1, flags=0) -> Params:
    return Params(runlen, bins_phi, bins_theta, n, thresh, buff, flags, 0)


class Context:
    """One device context (workspace + stream).  Not thread-safe; use one per host thread."""

    def __init__(self, device: int = -1):
        self._L = load_library()
        h = C.c_void_p()
        self._h = None
        self._keyframes = weakref.WeakSet()  # closed before the context: they live in its device memory
        self._check(self._L.icet_b200_create(device, C.byref(h)))
        self._h = h

    def _check(self, rc: int):
        if rc < 0:
            raise IcetError("icet_b200 error %d: %s" % (rc, self._L.icet_b200_last_error().decode()))
        return rc

    def close(self):
        if self._h is not None:
            for kf in list(self._keyframes):
                kf.close()
            self._L.icet_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- configuration -----------------------------------------------------------------------
    def set_stream(self, cuda_stream: int):
        self._check(self._L.icet_b200_set_stream(self._h, C.c_void_p(cuda_stream)))

    def set_chunk(self, pairs: int):
        self._check(self._L.icet_b200_set_chunk(self._h, pairs))

    def set_lanes(self, lanes: int):
        self._check(self._L.icet_b200_set_lanes(self._h, lanes))

    def set_host_chunk(self, pairs: int):
        self._check(self._L.icet_b200_set_host_chunk(self._h, pairs))

    def synchronize(self):
        self._check(self._L.icet_b200_synchronize(self._h))

    @property
    def kernel_launches(self) -> int:
        return int(self._L.icet_b200_kernel_launches(self._h))

    def set_profile(self, enable: bool):
        self._check(self._L.icet_b200_set_profile(self._h, 1 if enable else 0))

    def get_profile(self) -> dict:
        """{kernel name: (summed device ms, launches)} since profiling was enabled."""
        ms = np.zeros(NKERNELS, np.float64)
        cnt = np.zeros(NKERNELS, np.int64)
        self._check(self._L.icet_b200_get_profile(self._h, ms.ctypes.data, cnt.ctypes.data))
        return {self._L.icet_b200_kernel_name(k).decode(): (float(ms[k]), int(cnt[k])) for k in range(NKERNELS)}

    # -- host-buffer registration ------------------------------------------------------------
    def register(self, scan1, scan2, X0=None, params: Params | None = None, dump: bool = False):
        p = params or make_params()
        s1, s2 = as_planes(scan1), as_planes(scan2)
        x0 = np.zeros(6, np.float32) if X0 is None else np.ascontiguousarray(X0, np.float32)
        res = Result()
        self._check(self._L.icet_b200_set_dump(self._h, 1 if dump else 0))
        self._check(self._L.icet_b200_register(self._h, C.byref(p), s1.ctypes.data, s1.shape[1], s1.shape[1],
                                               s2.ctypes.data, s2.shape[1], s2.shape[1], x0.ctypes.data,
                                               C.byref(res)))
        out = np.frombuffer(bytes(res), dtype=RESULT_DTYPE)[0]
        if dump:
            return out, self.get_dump(p)
        return out

    def register_clouds(self, cloud1, cloud2, X0=None, params: Params | None = None, divide: float = 0.0):
        """`register` for clouds in their native layout (N x 3 float64 / float32 / int32 in either order, or Cloud
        descriptors): the raw bytes are uploaded and converted on the device -- no host-side astype / transpose."""
        p = params or make_params()
        c1, k1 = cloud1 if isinstance(cloud1, tuple) else cloud_desc(cloud1, divide)
        c2, k2 = cloud2 if isinstance(cloud2, tuple) else cloud_desc(cloud2, divide)
        x0 = np.zeros(6, np.float32) if X0 is None else np.ascontiguousarray(X0, np.float32)
        res = Result()
        self._check(self._L.icet_b200_set_dump(self._h, 0))
        self._check(self._L.icet_b200_register_clouds(self._h, C.byref(p), C.byref(c1), C.byref(c2), x0.ctypes.data,
                                                      C.byref(res)))
        return np.frombuffer(bytes(res), dtype=RESULT_DTYPE)[0]

    def transform_cloud_device(self, cloud_ptr: int, n: int, ld: int, X_ptr: int, mode: int, out_ptr: int, ld_out: int,
                               n_dev_ptr: int = 0):
        """mode 0: (cloud * R^-1) - t (scanMatcher.cpp:73); mode 1: (cloud - t) * R^-1 (simpleMapMaker.cpp:41);
        X (6 floats) in device memory."""
        self._check(self._L.icet_b200_transform_cloud_device(self._h, C.c_void_p(cloud_ptr), n, ld,
                                                             C.c_void_p(n_dev_ptr) if n_dev_ptr else None,
                                                             C.c_void_p(X_ptr), mode, C.c_void_p(out_ptr), ld_out))

    def ingest(self, cloud, out_ptr: int, ld: int, divide: float = 0.0):
        c, keep = cloud if isinstance(cloud, tuple) else cloud_desc(cloud, divide)
        self._check(self._L.icet_b200_ingest(self._h, C.byref(c), C.c_void_p(out_ptr), ld))

    def register_batch(self, scans1, scans2, X0=None, params: Params | None = None) -> np.ndarray:
        """scans1[i], scans2[i]: float32 [3, N_i] planes in HOST memory (pinned or pageable).  Passing the
        same array object as scans2[i] and scans1[i+1] uploads it once."""
        p = params or make_params()
        npairs = len(scans1)
        assert len(scans2) == npairs
        for a in list(scans1) + list(scans2):
            assert a.dtype == np.float32 and a.ndim == 2 and a.shape[0] == 3 and a.flags["C_CONTIGUOUS"]
        p1 = (C.c_void_p * npairs)(*[a.ctypes.data for a in scans1])
        p2 = (C.c_void_p * npairs)(*[a.ctypes.data for a in scans2])
        n1 = np.array([a.shape[1] for a in scans1], np.int32)
        n2 = np.array([a.shape[1] for a in scans2], np.int32)
        x0p = None
        if X0 is not None:
            x0 = np.ascontiguousarray(X0, np.float32).reshape(1 if (p.flags & FLAG_CHAIN_X0) else npairs, 6)
            x0p = x0.ctypes.data
        out = np.zeros(npairs, RESULT_DTYPE)
        self._check(self._L.icet_b200_register_batch(self._h, C.byref(p), npairs, p1, n1.ctypes.data, p2,
                                                     n2.ctypes.data, x0p, out.ctypes.data))
        return out

    def register_batch_ptrs(self, ptrs1, n1, ptrs2, n2, out_ptr: int, x0_ptr: int = 0, params=None, device=False):
        """Raw-pointer form (host or device pointers; `out_ptr` likewise)."""
        p = params or make_params()
        npairs = len(ptrs1)
        # pointer tables: a uint64 numpy array IS a `const float* const*` (pass one to skip the per-call conversion)
        a1 = ptrs1 if isinstance(ptrs1, np.ndarray) else np.array(ptrs1, np.uint64)
        a2 = ptrs2 if isinstance(ptrs2, np.ndarray) else np.array(ptrs2, np.uint64)
        assert a1.dtype == np.uint64 and a2.dtype == np.uint64 and a1.flags["C_CONTIGUOUS"] and a2.flags["C_CONTIGUOUS"]
        n1 = np.ascontiguousarray(n1, np.int32)
        n2 = np.ascontiguousarray(n2, np.int32)
        f = self._L.icet_b200_register_batch_device if device else self._L.icet_b200_register_batch
        self._check(f(self._h, C.byref(p), npairs, a1.ctypes.data, n1.ctypes.data, a2.ctypes.data, n2.ctypes.data,
                      C.c_void_p(x0_ptr) if x0_ptr else None, C.c_void_p(out_ptr)))

    # -- device-resident registration ----------------------------------------------------------
    def register_sequence_device(self, scans_ptr: int, nscans: int, n: int, out_ptr: int, params=None):
        """scans_ptr: device float32 [nscans, 3, n]; out_ptr: device buffer of (nscans-1)*224 bytes.
        Asynchronous on the context's stream."""
        p = params or make_params()
        self._check(self._L.icet_b200_register_sequence_device(self._h, C.byref(p), nscans, C.c_void_p(scans_ptr),
                                                               n, C.c_void_p(out_ptr)))

    def synth_scans_device(self, out_ptr: int, nscans: int, first_scan=0, seed=20240, rings=64, azim=2048):
        self._check(self._L.icet_b200_synth_scans_device(self._h, seed, first_scan, nscans, rings, azim,
                                                         C.c_void_p(out_ptr)))

    # -- parity-test helpers ---------------------------------------------------------------------
    def spherical_bins(self, scan, params=None):
        p = params or make_params()
        s = as_planes(scan)
        n = s.shape[1]
        sph = np.zeros((3, n), np.float32)
        cell = np.zeros(n, np.int32)
        self._check(self._L.icet_b200_spherical_bins(self._h, C.byref(p), s.ctypes.data, n, n, sph.ctypes.data,
                                                     cell.ctypes.data))
        return sph, cell

    def get_points2(self, n2: int) -> np.ndarray:
        """[3, n2] planes: the reference's public `points2` member of the last `register` call."""
        out = np.zeros((3, n2), np.float32)
        self._check(self._L.icet_b200_get_points2(self._h, out.ctypes.data, n2))
        return out

    def classify_scan2(self, it: int, n2: int):
        """(cell [n2] int32, in [n2] uint8): class of every point of scan 2 of the last dumped `register` call in
        iteration `it` by the per-point pipeline, in the caller's point order."""
        cell = np.zeros(n2, np.int32)
        inb = np.zeros(n2, np.uint8)
        self._check(self._L.icet_b200_classify_scan2(self._h, it, cell.ctypes.data, inb.ctypes.data, n2))
        return cell, inb

    def debug_timeline(self, runlen: int) -> np.ndarray:
        """%globaltimer stamps [runlen, 16] (ns) of the loop kernel for the last dumped single-pair call."""
        out = np.zeros(runlen * 16 + 6144, np.uint64)
        self._check(self._L.icet_b200_debug_timeline(self._h, out.ctypes.data, runlen))
        self.tile_stamps = out[runlen * 16: runlen * 16 + 4096].reshape(2048, 2)
        self.tile_mid = out[runlen * 16 + 4096:]  # end of phase A of those tiles  # begin / end of the tiles of iteration 3 (debug)
        return out[: runlen * 16].reshape(runlen, 16)

    def get_dump(self, p: Params) -> dict:
        ncell, rl = p.bins_phi * p.bins_theta, p.runlen
        shapes = {"cnt1": ((ncell,), np.int32), "bounds": ((ncell, 6), np.float32), "nin1": ((ncell,), np.int32),
                  "has1": ((ncell,), np.uint8), "mu1": ((ncell, 3), np.float32), "sigma1": ((ncell, 3, 3), np.float32),
                  "evec1": ((ncell, 3, 3), np.float32), "eval1": ((ncell, 3), np.float32),
                  "lmask": ((ncell, 3), np.uint8), "cnt2": ((rl, ncell), np.int32), "nin2": ((rl, ncell), np.int32),
                  "used2": ((rl, ncell), np.uint8), "mu2": ((rl, ncell, 3), np.float32),
                  "sigma2": ((rl, ncell, 3, 3), np.float32), "Xit": ((rl, 6), np.float32),
                  "HTWH": ((rl, 6, 6), np.float32), "HTWdz": ((rl, 6), np.float32),
                  "TRit": ((rl, 12), np.float32), "testPoints": ((ncell * 6, 3), np.float32)}
        arrs = {k: np.zeros(s, d) for k, (s, d) in shapes.items()}
        d = _Dump()
        for name, ct in _DUMP_FIELDS:
            setattr(d, name, arrs[name].ctypes.data_as(ct))
        self._check(self._L.icet_b200_get_dump(self._h, C.byref(d)))
        return arrs


class MultiContext:
    """icet_b200_multi: one process, one context per device, batches sharded by contiguous pair range, one
    ncclAllGather of 48 floats per pair at the end (include/icet_b200.h "multi-GPU")."""

    def __init__(self, devices=None, ndev=None):
        self._L = load_library()
        devs = list(devices) if devices is not None else list(range(ndev or 1))
        arr = np.array(devs, np.int32)
        h = C.c_void_p()
        self._h = None
        rc = self._L.icet_b200_multi_create(arr.ctypes.data, len(devs), C.byref(h))
        if rc < 0:
            raise IcetError("icet_b200 error %d: %s" % (rc, self._L.icet_b200_last_error().decode()))
        self._h = h
        self.devices = devs

    def _check(self, rc):
        if rc < 0:
            raise IcetError("icet_b200 error %d: %s" % (rc, self._L.icet_b200_last_error().decode()))
        return rc

    def close(self):
        if self._h is not None:
            self._L.icet_b200_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def register_batch(self, scans1, scans2, X0=None, params: Params | None = None) -> np.ndarray:
        """HOST planes, like Context.register_batch; pairs [P d / G, P (d+1) / G) run on device slot d."""
        p = params or make_params()
        npairs = len(scans1)
        p1 = np.array([a.ctypes.data for a in scans1], np.uint64)
        p2 = np.array([a.ctypes.data for a in scans2], np.uint64)
        n1 = np.array([a.shape[1] for a in scans1], np.int32)
        n2 = np.array([a.shape[1] for a in scans2], np.int32)
        x0p = None
        if X0 is not None:
            x0 = np.ascontiguousarray(X0, np.float32).reshape(npairs, 6)
            x0p = x0.ctypes.data
        out = np.zeros(npairs, RESULT_DTYPE)
        self._check(self._L.icet_b200_register_batch_multi(self._h, C.byref(p), npairs, p1.ctypes.data, n1.ctypes.data,
                                                           p2.ctypes.data, n2.ctypes.data, x0p, out.ctypes.data))
        return out

    def register_sequence_device(self, shard_ptrs, nscans: int, n: int, params: Params | None = None):
        """shard_ptrs[d]: device pointer (on device slot d) to that device's scans of the sequence."""
        p = params or make_params()
        ptrs = np.array(shard_ptrs, np.uint64)
        self._check(self._L.icet_b200_register_sequence_multi_device(self._h, C.byref(p), nscans, ptrs.ctypes.data, n))

    def gathered(self, d: int):
        """(device pointer to [ndev][rows_per_shard][48] floats on device slot d, rows_per_shard)"""
        ptr, rows = C.c_void_p(), C.c_int32()
        self._check(self._L.icet_b200_multi_gathered(self._h, d, C.byref(ptr), C.byref(rows)))
        return ptr.value, rows.value

    def gathered_host(self, d: int) -> np.ndarray:
        """[ndev, rows_per_shard, 48] float32: the all-gathered rows (X 6 | pred_stds 6 | Q 36) as device slot d holds them"""
        _, rows = self.gathered(d)
        out = np.zeros((len(self.devices), rows, 48), np.float32)
        self._check(self._L.icet_b200_multi_gathered_host(self._h, d, out.ctypes.data))
        return out


_DEFAULT_CTX: Context | None = None


def default_context() -> Context:
    global _DEFAULT_CTX
    if _DEFAULT_CTX is None:
        _DEFAULT_CTX = Context()
    return _DEFAULT_CTX


class ICET:
    """Python mirror of the reference's `class ICET` (include/icet.h:36-116): all the work happens in the
    constructor (src/icet.cpp:29-63); results are public attributes.

        it = ICET(scan1, scan2, runlen, X0, num_bins_phi, num_bins_theta, n=25, thresh=0.1, buff=0.1)
        it.X, it.pred_stds            # what odometry.cpp:77-79 / simpleMapMaker.cpp:120-122 read
        it.Q                          # 6x6 error-bound covariance (noise_mat, src/icet.cpp:411)

    scan1/scan2: N x 3 arrays (as Eigen::MatrixXf rows) or [3, N] planes.
    """

    def __init__(self, scan1, scan2, runlen, X0, num_bins_phi, num_bins_theta, n=25, thresh=0.1, buff=0.1,
                 ctx: Context | None = None, debug: bool = False, shipped_row_order: bool = False):
        self.rl, self.numBinsPhi, self.numBinsTheta = runlen, num_bins_phi, num_bins_theta
        self.n, self.thresh, self.buff = n, thresh, buff
        ctx = ctx or default_context()
        # shipped_row_order: cluster in the row order the reference's broken permutation loop leaves (validation
        # against an unmodified reference build); default: the sorted order its comments intend
        p = make_params(runlen, num_bins_phi, num_bins_theta, n, thresh, buff,
                        flags=FLAG_SHIPPED_ORDER if shipped_row_order else 0)
        r = ctx.register(scan1, scan2, X0, p, dump=debug)
        if debug:
            r, self.debug = r
            self.clusterBounds = self.debug["bounds"]
        if r["status"] < 0:
            raise IcetError("registration failed with status %d" % r["status"])
        self.X = r["X"].copy()
        self.pred_stds = r["pred_stds"].copy()
        self.Q = r["Q"].copy()
        self.status = int(r["status"])
        self.result = r


class Keyframe:
    """Scan 1 fitted once (icet_b200_keyframe_create): register any number of scans against it without refitting it --
    a scan against an accumulated map, one pair from several initial guesses, scans k+1 .. k+m against keyframe k.
    Results are bit-identical to `Context.register(scan1, scan2, ...)` with the same settings.

        kf = Keyframe(map_points)                       # N x 3 or [3, N] host cloud
        r = kf.register(scan, X0)                       # one RESULT_DTYPE record
        kf.register_batch_device(ptrs2, n2, out_ptr)    # device scans, asynchronous

    The bins, n, thresh, buff and the row-order mode are those of the keyframe; runlen and the loop / scan-2 flags are
    chosen per call."""

    def __init__(self, scan1, num_bins_phi=24, num_bins_theta=75, n=25, thresh=0.1, buff=0.1, ctx: Context | None = None,
                 shipped_row_order=False, _device=None):
        self._h = None
        self._ctx = ctx or default_context()
        self._L = self._ctx._L
        self.shipped_row_order = bool(shipped_row_order)
        self._p = make_params(0, num_bins_phi, num_bins_theta, n, thresh, buff,
                              flags=FLAG_SHIPPED_ORDER if shipped_row_order else 0)
        h = C.c_void_p()
        if _device is None:
            s1 = as_planes(scan1)
            rc = self._L.icet_b200_keyframe_create(self._ctx._h, C.byref(self._p), s1.ctypes.data, s1.shape[1],
                                                   s1.shape[1], C.byref(h))
        else:
            ptr, n1, ld1 = _device
            rc = self._L.icet_b200_keyframe_create_device(self._ctx._h, C.byref(self._p), C.c_void_p(ptr), n1, ld1,
                                                          C.byref(h))
        self._ctx._check(rc)
        self._h = h
        self._ctx._keyframes.add(self)

    @classmethod
    def from_device(cls, ptr: int, n1: int, ld1: int | None = None, **kw) -> "Keyframe":
        """scan 1 as float32 planes in DEVICE memory (leading dimension ld1, default n1)."""
        return cls(None, _device=(ptr, n1, n1 if ld1 is None else ld1), **kw)

    def _handle(self):
        if self._h is None:
            raise IcetError("keyframe is closed")
        return self._h

    def params(self, runlen=7, flags=0) -> Params:
        """icet_b200_params of a registration against this keyframe."""
        p = make_params(runlen, self._p.bins_phi, self._p.bins_theta, self._p.n, self._p.thresh, self._p.buff, flags)
        p.flags |= self._p.flags
        return p

    @property
    def n_gauss1(self) -> int:
        h = self._handle()
        return self._ctx._check(self._L.icet_b200_keyframe_gaussians(h))

    def register(self, scan2, X0=None, runlen=7, flags=0):
        """One HOST scan 2 against the keyframe (blocking); returns one RESULT_DTYPE record."""
        h = self._handle()
        p = self.params(runlen, flags)
        s2 = as_planes(scan2)
        x0 = np.zeros(6, np.float32) if X0 is None else np.ascontiguousarray(X0, np.float32)
        res = Result()
        self._ctx._check(self._L.icet_b200_register_keyframe(h, C.byref(p), s2.ctypes.data, s2.shape[1], s2.shape[1],
                                                             x0.ctypes.data, C.byref(res)))
        return np.frombuffer(bytes(res), dtype=RESULT_DTYPE)[0]

    def register_batch_device(self, ptrs2, n2, out_ptr: int, x0_ptr: int = 0, runlen=7, flags=0):
        """DEVICE scans ptrs2[i] (n2[i] points each) against the keyframe; x0 (npairs x 6 or 0) and out (npairs
        records) in DEVICE memory.  Asynchronous on the context's stream."""
        h = self._handle()
        p = self.params(runlen, flags)
        a2 = ptrs2 if isinstance(ptrs2, np.ndarray) else np.array(ptrs2, np.uint64)
        assert a2.dtype == np.uint64 and a2.flags["C_CONTIGUOUS"]
        n2 = np.ascontiguousarray(n2, np.int32)
        assert n2.shape == a2.shape
        self._ctx._check(self._L.icet_b200_register_keyframe_batch_device(
            h, C.byref(p), len(a2), a2.ctypes.data, n2.ctypes.data, C.c_void_p(x0_ptr) if x0_ptr else None,
            C.c_void_p(out_ptr)))

    def close(self):
        if self._h is not None:
            self._L.icet_b200_keyframe_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
