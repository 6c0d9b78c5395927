"""Host-side mirror of the reference's two ROS nodes, minus ROS (SURVEY.md 8f rows N1, N2):

    OdometryNode   reference src/odometry.cpp:23-214       scan in -> pose / covariance diagonal / twist out
    ScanMatcherNode reference src/scanMatcher.cpp:18-150    scan in -> scan 2 in the frame of scan 1 + snail trail out
    MapMakerNode   reference src/simpleMapMaker.cpp:60-291  scan in -> pose + 600 000-point FIFO map out

Both are thin: every step between two scans (min-range filter, registration, seeding of the next registration, pose
accumulation, map re-expression) runs on the device behind the C ABI (include/icet_b200.h, "callers either side of
the path"); the host only hands scans in and reads the published values back.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import api
from .api import Context, IcetError, OdometryParams, Params, Pose, POSE_DTYPE, RESULT_DTYPE, Result, as_planes


class Node:
    """icet_b200_node: device-resident prev_pcl_matrix / X0 / X_homo of one node."""

    def __init__(self, ctx: Context, params: Params, op: OdometryParams, max_points: int, X_homo0=None, X0=None):
        self.ctx, self._L = ctx, ctx._L
        self.params, self.op = params, op
        h = C.c_void_p()
        xh = None if X_homo0 is None else np.ascontiguousarray(X_homo0, np.float32).reshape(16)
        x0 = None if X0 is None else np.ascontiguousarray(X0, np.float32).reshape(6)
        self._h = None
        ctx._check(self._L.icet_b200_node_create(ctx._h, C.byref(params), C.byref(op), max_points,
                                                 None if xh is None else xh.ctypes.data,
                                                 None if x0 is None else x0.ctypes.data, C.byref(h)))
        self._h = h

    def close(self):
        if self._h is not None:
            self._L.icet_b200_node_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def push(self, scan):
        """One scan from host memory (N x 3 or [3, N]).  Returns None for the very first scan, else (result, pose)
        as numpy records."""
        s = as_planes(scan)
        res, pose = Result(), Pose()
        n = s.shape[1]
        rc = self.ctx._check(self._L.icet_b200_node_push(self._h, s.ctypes.data, n, n, C.byref(res), C.byref(pose)))
        if rc == 0:
            return None
        return (np.frombuffer(bytes(res), dtype=RESULT_DTYPE)[0], np.frombuffer(bytes(pose), dtype=POSE_DTYPE)[0])

    def push_cloud(self, cloud, divide: float = 0.0):
        """`push` for a cloud in its native layout (see api.cloud_desc): e.g. the bytes of a PointCloud2 message."""
        c, keep = cloud if isinstance(cloud, tuple) else api.cloud_desc(cloud, divide)
        res, pose = Result(), Pose()
        rc = self.ctx._check(self._L.icet_b200_node_push_cloud(self._h, C.byref(c), C.byref(res), C.byref(pose)))
        if rc == 0:
            return None
        return (np.frombuffer(bytes(res), dtype=RESULT_DTYPE)[0], np.frombuffer(bytes(pose), dtype=POSE_DTYPE)[0])

    def push_device(self, scans_ptr: int, nscans: int, n: int, res_ptr: int, pose_ptr: int) -> int:
        """nscans consecutive scans in device memory [nscans, 3, n]; asynchronous.  Returns the number of
        registrations whose result / pose will be written to the device arrays."""
        return self.ctx._check(self._L.icet_b200_node_push_device(self._h, nscans, C.c_void_p(scans_ptr), n,
                                                                  C.c_void_p(res_ptr), C.c_void_p(pose_ptr)))

    def current_scan(self):
        """(device pointer of the filtered current scan planes, device pointer of its row count, leading dim)."""
        p, q, ld = C.c_void_p(), C.c_void_p(), C.c_int32()
        self.ctx._check(self._L.icet_b200_node_current_scan(self._h, C.byref(p), C.byref(q), C.byref(ld)))
        return p.value, q.value, ld.value

    def last_result_ptr(self):
        p = C.c_void_p()
        self.ctx._check(self._L.icet_b200_node_last_result(self._h, C.byref(p)))
        return p.value


class PointMap:
    """icet_b200_map: the reference's EigenQueue (src/simpleMapMaker.cpp:18-58) on the device."""

    def __init__(self, ctx: Context, capacity: int = 600_000):
        self.ctx, self._L, self.capacity = ctx, ctx._L, capacity
        h = C.c_void_p()
        self._h = None
        ctx._check(self._L.icet_b200_map_create(ctx._h, capacity, C.byref(h)))
        self._h = h

    def close(self):
        if self._h is not None:
            self._L.icet_b200_map_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def add_scan_device(self, scan_ptr: int, n: int, ld: int, X_ptr: int, idx=None, count: int | None = None,
                        n_dev_ptr: int = 0, guard_trans: float = 0.0, guard_rot: float = 0.0):
        ix = None if idx is None else np.ascontiguousarray(idx, np.int32)
        cnt = (len(ix) if ix is not None else n) if count is None else count
        self.ctx._check(self._L.icet_b200_map_add_scan_device(
            self._h, C.c_void_p(scan_ptr), n, ld, C.c_void_p(n_dev_ptr) if n_dev_ptr else None,
            None if ix is None else ix.ctypes.data, cnt, C.c_void_p(X_ptr), guard_trans, guard_rot))

    def get(self) -> np.ndarray:
        """EigenQueue::getQueue: rows oldest first, as an [n, 3] array."""
        out = np.zeros((3, self.capacity), np.float32)
        n = C.c_int32()
        self.ctx._check(self._L.icet_b200_map_get(self._h, out.ctypes.data, self.capacity, C.byref(n)))
        return np.ascontiguousarray(out[:, : n.value].T)


class OdometryNode:
    """Mirror of OdometryNode (src/odometry.cpp:23-214): `callback(scan)` is pointcloudCallback without the ROS
    plumbing.  Parameters are the node's constants: minD = 2 (:57), run_length 7, 24 x 75 bins (:73-75), X0 seeded with
    the previous solution (:82), 10 Hz twist (:134-139)."""

    def __init__(self, ctx: Context | None = None, max_points: int = 131072, min_range: float = 2.0, runlen: int = 7,
                 num_bins_phi: int = 24, num_bins_theta: int = 75, rate_hz: float = 10.0):
        self.ctx = ctx or api.default_context()
        self.node = Node(self.ctx, api.make_params(runlen, num_bins_phi, num_bins_theta),
                         OdometryParams(min_range, 1, rate_hz, 0.0, 0.0), max_points)
        self.X_homo = np.eye(4, dtype=np.float32)
        self.X0 = np.zeros(6, np.float32)
        self.frameCount = 0

    def callback(self, scan):
        self.frameCount += 1
        out = self.node.push(scan)
        if out is None:
            return None
        res, pose = out
        self.X0 = res["X"].copy()
        self.X_homo = pose["X_homo"].copy()
        return {"X": res["X"].copy(), "pred_stds": res["pred_stds"].copy(), "position": pose["position"].copy(),
                "orientation": pose["orientation"].copy(), "covariance_diag": pose["covariance_diag"].copy(),
                "twist": pose["twist"].copy(), "X_homo": pose["X_homo"].copy(), "n_points": int(pose["n_points"])}


class KeyframeOdometryNode:
    """Keyframe odometry (include/icet_b200.h "keyframe odometry", DESIGN.md §13): every filtered scan is registered
    against the node's current keyframe instead of its predecessor, so the registration errors of the scans between
    two keyframes do not add up.

    * The first scan is stored unfiltered and is keyframe 0 with pose X_homo0.
    * Scan k is filtered (||p|| > min_range) and registered against keyframe f, seeded with x0_k; its X is X_rel,
      scan k relative to f.  Pose: X_homo_k = X_homo_f @ Hi(X_rel) (the float product of OdometryNode).
    * Frame step: X_rel verbatim when f = k-1, else params(Hi(X_rel,k-1)^-1 Hi(X_rel,k)); twist = rate_hz * step.
      params(H): translation column verbatim, angles from the inverse of R() (double precision).
    * Next seed (chain_x0): params(Hi(X_rel,k) Hi(step_k)), or step_k when scan k was promoted; else 0.
    * Scan k becomes the keyframe of scan k+1 when a test of `policy` (api.KeyframePolicy) fires or its registration
      has status != 0.  KeyframePolicy(max_interval=1, max_trans=0, max_rot=0, min_overlap=0) reproduces
      OdometryNode bit for bit.

    `callback(scan)` returns None for the first scan, else (result, pose, info) as dicts of numpy values, info being
    {keyframe, promoted, reason (api.KF_* bits), x0 (the seed used)}.  Nothing returns to the host between the scans of
    one `push_device` call.

    Local map (DESIGN.md §14): with `map_keyframes=M` (1 <= M <= 16) scan 1 of every registration is the local map
    instead of the keyframe alone: the filtered clouds of the last M keyframes in the frame of the newest keyframe f.
    Its rows are f's cloud (bit for bit), then the older keyframes, newest to oldest, without gaps.  On a promotion of
    scan k a point q of f's frame becomes q R(X_rel)^-1 - t(X_rel) in k's frame (Context.transform_cloud_device mode
    0); each keyframe keeps its original filtered cloud and its transform into the current frame, composed in double
    on the device, so a map is never re-expressed twice.  Pose, seeds, policy and info are those above; the overlap
    test uses the map's n_gauss1.  The window slides once M keyframes exist.  M = 1 is the plain node byte for byte;
    `None` (the default) creates the plain node through icet_b200_kfnode_create."""

    def __init__(self, ctx: Context | None = None, max_points: int = 131072, min_range: float = 2.0, runlen: int = 7,
                 num_bins_phi: int = 24, num_bins_theta: int = 75, rate_hz: float = 10.0, chain_x0: bool = True,
                 policy: api.KeyframePolicy | None = None, X_homo0=None, X0=None, flags: int = 0,
                 map_keyframes: int | None = None):
        policy = api.KeyframePolicy() if policy is None else policy
        if not isinstance(policy, api.KeyframePolicy):
            raise TypeError("policy must be an icet_b200.api.KeyframePolicy")
        if any(policy.reserved):
            raise ValueError("policy.reserved must be 0")
        if flags & api.FLAG_CHAIN_X0:
            raise ValueError("flags: FLAG_CHAIN_X0 is not supported by the keyframe odometry node (it seeds every "
                             "registration itself; use chain_x0)")
        if flags & api.FLAG_SHIPPED_ORDER:
            raise ValueError("flags: FLAG_SHIPPED_ORDER is not supported by the keyframe odometry node (its scan-1 fit "
                             "needs a host round trip)")
        if max_points < 1:
            raise ValueError("max_points must be >= 1")
        if map_keyframes is not None and not 1 <= map_keyframes <= 16:
            raise ValueError("map_keyframes must be in 1 .. 16")
        xh = None if X_homo0 is None else np.ascontiguousarray(X_homo0, np.float32).reshape(16)
        x0 = None if X0 is None else np.ascontiguousarray(X0, np.float32).reshape(6)
        self.ctx = ctx or api.default_context()
        self._L = self.ctx._L
        self.params = api.make_params(runlen, num_bins_phi, num_bins_theta, flags=flags)
        self.op = OdometryParams(min_range, 1 if chain_x0 else 0, rate_hz, 0.0, 0.0)
        self.policy = policy
        self.max_points = max_points
        self.map_keyframes = map_keyframes
        h = C.c_void_p()
        self._h = None
        pointers = (None if xh is None else xh.ctypes.data, None if x0 is None else x0.ctypes.data, C.byref(h))
        if map_keyframes is None:
            rc = self._L.icet_b200_kfnode_create(self.ctx._h, C.byref(self.params), C.byref(self.op), C.byref(policy),
                                                 max_points, *pointers)
        else:
            rc = self._L.icet_b200_kfnode_create_local_map(self.ctx._h, C.byref(self.params), C.byref(self.op),
                                                           C.byref(policy), map_keyframes, max_points, *pointers)
        self.ctx._check(rc)
        self._h = h
        self.X_homo = np.eye(4, dtype=np.float32) if xh is None else xh.reshape(4, 4).copy()
        self.frameCount = 0

    def _handle(self):
        if self._h is None:
            raise IcetError("node is closed")
        return self._h

    def close(self):
        if self._h is not None:
            self._L.icet_b200_kfnode_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _unpack(res, pose, info):
        r = np.frombuffer(bytes(res), dtype=RESULT_DTYPE)[0]
        p = np.frombuffer(bytes(pose), dtype=POSE_DTYPE)[0]
        i = np.frombuffer(bytes(info), dtype=api.KF_INFO_DTYPE)[0]
        return ({k: r[k].copy() for k in RESULT_DTYPE.names}, {k: p[k].copy() for k in POSE_DTYPE.names},
                {k: i[k].copy() for k in api.KF_INFO_DTYPE.names})

    def callback(self, scan):
        """One scan from host memory (N x 3 or [3, N]), blocking."""
        h = self._handle()
        s = as_planes(scan)
        res, pose, info = Result(), Pose(), api.KfInfo()
        n = s.shape[1]
        self.frameCount += 1
        rc = self.ctx._check(self._L.icet_b200_kfnode_push(h, s.ctypes.data, n, n, C.byref(res), C.byref(pose),
                                                           C.byref(info)))
        if rc == 0:
            return None
        out = self._unpack(res, pose, info)
        self.X_homo = out[1]["X_homo"].copy()
        return out

    def callback_cloud(self, cloud, divide: float = 0.0):
        """`callback` for a cloud in its native layout (see api.cloud_desc)."""
        h = self._handle()
        c, keep = cloud if isinstance(cloud, tuple) else api.cloud_desc(cloud, divide)
        res, pose, info = Result(), Pose(), api.KfInfo()
        self.frameCount += 1
        rc = self.ctx._check(self._L.icet_b200_kfnode_push_cloud(h, C.byref(c), C.byref(res), C.byref(pose),
                                                                 C.byref(info)))
        if rc == 0:
            return None
        out = self._unpack(res, pose, info)
        self.X_homo = out[1]["X_homo"].copy()
        return out

    def push_device(self, scans_ptr: int, nscans: int, n: int, res_ptr: int, pose_ptr: int, info_ptr: int = 0) -> int:
        """nscans consecutive scans in device memory [nscans, 3, n]; results (RESULT_DTYPE), poses (POSE_DTYPE) and
        infos (KF_INFO_DTYPE, optional) to device arrays.  Asynchronous.  Returns the number of registrations."""
        h = self._handle()
        if nscans < 0 or n < 0 or n > self.max_points:
            raise ValueError("nscans / n out of range")
        return self.ctx._check(self._L.icet_b200_kfnode_push_device(h, nscans, C.c_void_p(scans_ptr), n,
                                                                    C.c_void_p(res_ptr), C.c_void_p(pose_ptr),
                                                                    C.c_void_p(info_ptr) if info_ptr else None))

    def keyframe_device(self):
        """(device pointer of the keyframe's filtered cloud planes, device pointer of its row count, leading dim)."""
        p, q, ld = C.c_void_p(), C.c_void_p(), C.c_int32()
        self.ctx._check(self._L.icet_b200_kfnode_keyframe(self._handle(), C.byref(p), C.byref(q), C.byref(ld)))
        return p.value, q.value, ld.value

    def keyframe_cloud(self) -> np.ndarray:
        """The current keyframe's filtered cloud as an [n, 3] host array (blocking; for visualisation)."""
        return self._host_cloud(*self.keyframe_device())

    def local_map_device(self):
        """(device pointer of the local map's planes, device pointer of its row count, leading dim): scan 1 of the next
        registration, valid until the next push.  The keyframe cloud for a node made without map_keyframes."""
        p, q, ld = C.c_void_p(), C.c_void_p(), C.c_int32()
        self.ctx._check(self._L.icet_b200_kfnode_local_map(self._handle(), C.byref(p), C.byref(q), C.byref(ld)))
        return p.value, q.value, ld.value

    def local_map_cloud(self) -> np.ndarray:
        """The local map as an [n, 3] host array (blocking)."""
        return self._host_cloud(*self.local_map_device())

    def _host_cloud(self, p, q, ld) -> np.ndarray:
        import torch
        self.ctx.synchronize()
        n = int(torch.as_tensor(_DeviceArray(q, (1,), "<i4"), device="cuda").cpu()[0])
        planes = torch.as_tensor(_DeviceArray(p, (3, ld), "<f4"), device="cuda")[:, :n].cpu().numpy()
        return np.ascontiguousarray(planes.T)


class _DeviceArray:
    """A library-owned device buffer seen through __cuda_array_interface__ (a view, no copy; only read here)."""

    def __init__(self, ptr: int, shape, typestr: str):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 2}


class MapMakerNode:
    """Mirror of MapMakerNode (src/simpleMapMaker.cpp:60-291): min range 0.2 (:100), run_length 12 (:115), X0 = 0 for
    every pair (:124), divergence guard 0.3 / 0.3 (:128-137, :241-242), 2000-point random sample of every scan
    (:150-159) pushed into a 600 000-point FIFO that is re-expressed in the newest sensor frame (EigenQueue, :18-58).
    The sample is `rng.permutation(rows)[:downsample]` (the reference shuffles with a default-seeded std::mt19937;
    the C++ mirror in icet_b200/host/nodes.h uses exactly that)."""

    def __init__(self, ctx: Context | None = None, max_points: int = 131072, min_range: float = 0.2, runlen: int = 12,
                 num_bins_phi: int = 24, num_bins_theta: int = 75, capacity: int = 600_000, downsample: int = 2000,
                 trans_thresh: float = 0.3, rot_thresh: float = 0.3, seed: int = 5489):
        self.ctx = ctx or api.default_context()
        self.trans_thresh, self.rot_thresh, self.downsample = trans_thresh, rot_thresh, downsample
        self.node = Node(self.ctx, api.make_params(runlen, num_bins_phi, num_bins_theta),
                         OdometryParams(min_range, 0, 10.0, trans_thresh, rot_thresh), max_points)
        self.q = PointMap(self.ctx, capacity)
        self.rng = np.random.RandomState(seed)
        self.X_homo = np.eye(4, dtype=np.float32)
        self.frameCount = 0

    def callback(self, scan):
        self.frameCount += 1
        out = self.node.push(scan)
        if out is None:
            return None
        res, pose = out
        rows = int(pose["n_points"])
        idx = self.rng.permutation(rows)[: min(self.downsample, rows)].astype(np.int32)
        scan_ptr, n_ptr, ld = self.node.current_scan()
        self.q.add_scan_device(scan_ptr, rows, ld, self.node.last_result_ptr(), idx=idx, n_dev_ptr=n_ptr,
                               guard_trans=self.trans_thresh, guard_rot=self.rot_thresh)
        self.X_homo = pose["X_homo"].copy()
        return {"X": pose["X"].copy(), "pred_stds": res["pred_stds"].copy(), "X_homo": pose["X_homo"].copy(),
                "guarded": bool(pose["guarded"]), "n_points": rows, "sample": idx}

    def map_points(self) -> np.ndarray:
        return self.q.get()


class ScanMatcherNode:
    """Mirror of ScanMatcherNode (src/scanMatcher.cpp:18-150): every cloud is registered against its predecessor as it
    came (no range filter), X0 = 0 (:58-62), run_length 7, 24 x 75 bins (:55-57); publishes scan 2 re-expressed in
    the frame of scan 1, `(pcl_matrix * rot_mat.inverse()).rowwise() - trans` (:73), and the snail trail (:76-80).
    The re-expression of the cloud runs on the device from the device-resident result."""

    def __init__(self, ctx: Context | None = None, max_points: int = 131072, runlen: int = 7, num_bins_phi: int = 24,
                 num_bins_theta: int = 75):
        import torch
        self.ctx = ctx or api.default_context()
        self.node = Node(self.ctx, api.make_params(runlen, num_bins_phi, num_bins_theta),
                         OdometryParams(-1.0, 0, 10.0, 0.0, 0.0), max_points)
        self._torch = torch
        self._out = torch.empty((3, max_points), dtype=torch.float32, device="cuda")
        self.snailTrail = np.zeros((1, 3), np.float32)   # scanMatcher.cpp:25-26
        self.frameCount = 0

    def callback(self, scan):
        self.frameCount += 1
        s = as_planes(scan)
        if s.shape[1] == 0:           # "Received an empty point cloud" (:41-44)
            return None
        out = self.node.push(s)
        if out is None:               # "Previous point cloud is empty, skipping this frame" (:47-51)
            return None
        res, pose = out
        X = res["X"].copy()
        scan_ptr, n_ptr, ld = self.node.current_scan()
        n = s.shape[1]
        self.ctx.transform_cloud_device(scan_ptr, n, ld, self.node.last_result_ptr(), 0, self._out.data_ptr(),
                                        self._out.shape[1])
        self.ctx.synchronize()
        aligned = self._out[:, :n].cpu().numpy().T.copy()
        # snail trail (:76-80): a handful of rows, host side like the reference
        from numpy.linalg import inv
        R = _rot_R(X[3], X[4], X[5])
        self.snailTrail = ((self.snailTrail @ inv(R.astype(np.float64)).astype(np.float32)) - X[:3]).astype(np.float32)
        self.snailTrail = np.vstack([self.snailTrail, np.zeros((1, 3), np.float32)])
        return {"X": X, "scan2_in_scan1_frame": aligned, "snailTrail": self.snailTrail.copy()}


def _rot_R(phi, theta, psi) -> np.ndarray:
    """utils::R (reference src/utils.cpp:144-152), float32, row-major."""
    f = np.float32
    sph, cph, sth, cth, sps, cps = (np.sin(f(phi)), np.cos(f(phi)), np.sin(f(theta)), np.cos(f(theta)),
                                    np.sin(f(psi)), np.cos(f(psi)))
    return np.array([[cth * cps, sps * cph + sph * sth * cps, sph * sps - sth * cph * cps],
                     [-sps * cth, cph * cps - sph * sth * sps, sph * cps + sth * sps * cph],
                     [sth, -sph * cth, cph * cth]], dtype=f)
