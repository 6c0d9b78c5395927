"""TEST INFRASTRUCTURE -- CPU restatement of the keyframe odometry node (include/icet_b200.h "keyframe odometry",
DESIGN.md §13): the pose / frame-step / seed / promotion rules in numpy, and a node that registers the same filtered
keyframe / scan pairs with oracle/pyoracle.run.

Only tests/ and tools/ may import this module; the product never does.  Clouds and poses are float32 like the node's;
frame steps and seeds are composed in double like the node's.
"""
from __future__ import annotations

import numpy as np

from . import pyoracle as po
from .nodes_oracle import F, homogeneous, min_range_filter  # noqa: F401  (re-exported for the tests)


# -- keyframe odometry node (include/icet_b200.h "keyframe odometry", DESIGN.md §13) -------------------------------
KF_TRANS, KF_ROT, KF_OVERLAP, KF_INTERVAL, KF_STATUS = 1, 2, 4, 8, 16


def kf_params(H) -> np.ndarray:
    """params(H): translation column verbatim, angles from the inverse of utils::R (|theta| < pi/2), double in, f32 out."""
    H = np.asarray(H, np.float64)
    return np.array([H[0, 3], H[1, 3], H[2, 3], np.arctan2(-H[2, 1], H[2, 2]), np.arcsin(np.clip(H[2, 0], -1.0, 1.0)),
                     np.arctan2(-H[1, 0], H[0, 0])], np.float64).astype(F)


def kf_homo64(X) -> np.ndarray:
    """Hi(X) built in float (homogeneous) and widened to double, as the node composes steps and seeds."""
    return homogeneous(X).astype(np.float64)


def kf_rigid_inv(H) -> np.ndarray:
    R, t = H[:3, :3], H[:3, 3]
    out = np.eye(4)
    out[:3, :3] = R.T
    out[:3, 3] = -R.T @ t
    return out


def kf_step(X_prev, X, keyframe_is_predecessor: bool) -> np.ndarray:
    """frame step of scan k: X_rel verbatim when its keyframe is scan k-1, else params(Hi(X_rel,k-1)^-1 Hi(X_rel,k))"""
    if keyframe_is_predecessor:
        return np.asarray(X, F).copy()
    return kf_params(kf_rigid_inv(kf_homo64(X_prev)) @ kf_homo64(X))


def kf_next_seed(X, step, promoted: bool, chain: bool) -> np.ndarray:
    """seed of scan k+1: constant velocity relative to the keyframe it will be registered against"""
    if not chain:
        return np.zeros(6, F)
    if promoted:
        return np.asarray(step, F).copy()
    return kf_params(kf_homo64(X) @ kf_homo64(step))


def kf_reason(X, status, n_used, n_gauss1, interval_before, max_trans=0.0, max_rot=0.0, min_overlap=0.0,
              max_interval=0) -> int:
    """The promotion tests of icet_b200_keyframe_policy in float32, as the device evaluates them.  interval_before:
    registrations against the keyframe before this one."""
    X = np.asarray(X, F)
    tn = np.sqrt(F(F(F(X[0] * X[0]) + F(X[1] * X[1])) + F(X[2] * X[2])))
    rm = np.abs(X[3:]).max()
    r = 0
    if max_trans > 0 and tn > F(max_trans):
        r |= KF_TRANS
    if max_rot > 0 and rm > F(max_rot):
        r |= KF_ROT
    if min_overlap > 0 and F(n_used) < F(F(min_overlap) * F(n_gauss1)):
        r |= KF_OVERLAP
    if max_interval > 0 and interval_before + 1 >= max_interval:
        r |= KF_INTERVAL
    if status != 0:
        r |= KF_STATUS
    return r


class KeyframeOdometryOracle:
    """The keyframe odometry node restated on the CPU: filtered scans registered against the filtered keyframe with
    oracle/pyoracle.run, the policy / step / seed / pose rules above.  `callback(cloud, x0=None)`: x0 replaces the
    node's own seed (to register the very pairs a device run registered)."""

    def __init__(self, min_d=2.0, runlen=7, bins_phi=24, bins_theta=75, chain=True, rate=10.0, policy=None, **kw):
        self.min_d, self.runlen, self.bins_phi, self.bins_theta = min_d, runlen, bins_phi, bins_theta
        self.chain, self.rate, self.kw = chain, F(rate), kw
        self.policy = dict(max_trans=2.0, max_rot=0.1, min_overlap=0.5, max_interval=10) if policy is None else policy
        self.kf = None
        self.kf_frame, self.interval, self.frames = 0, 0, 0
        self.H_f = np.eye(4, dtype=F)
        self.x0 = np.zeros(6, F)
        self.X_prev = np.zeros(6, F)

    def callback(self, cloud, x0=None):
        cloud = np.ascontiguousarray(np.asarray(cloud, F))
        if self.kf is None:
            self.kf = cloud
            return None
        cur = min_range_filter(cloud, self.min_d)
        seed = self.x0 if x0 is None else np.asarray(x0, F)
        it = po.run(self.kf, cur, runlen=self.runlen, X0=seed, bins_phi=self.bins_phi, bins_theta=self.bins_theta,
                    dumps=None, **self.kw)
        X = np.asarray(it.X, F).copy()
        frame = self.frames + 1
        step = kf_step(self.X_prev, X, self.kf_frame == frame - 1)
        # (pyoracle.run reports no voxel counts: the overlap test is left to kf_reason with the device's counts)
        reason = kf_reason(X, it.status, 0, 0, self.interval, **dict(self.policy, min_overlap=0.0))
        promoted = reason != 0
        X_homo = (self.H_f @ homogeneous(X)).astype(F)
        out = {"X": X, "pred_stds": np.asarray(it.pred_stds, F).copy(), "X_homo": X_homo, "step": step,
               "twist": (self.rate * step).astype(F), "keyframe": self.kf_frame, "promoted": promoted, "reason": reason,
               "x0": seed.copy(), "n_points": cur.shape[0], "cur": cur}
        self.x0 = kf_next_seed(X, step, promoted, self.chain)
        self.X_prev = X
        if promoted:
            self.H_f, self.kf, self.kf_frame, self.interval = X_homo, cur, frame, 0
        else:
            self.interval += 1
        self.frames = frame
        return out
