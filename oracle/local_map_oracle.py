"""TEST INFRASTRUCTURE -- CPU restatement of the local-map window of the keyframe odometry node
(icet_b200_kfnode_create_local_map, DESIGN.md §14): the slot transforms, their composition on a promotion, the sliding
window and the order in which the map lists its blocks.  It is driven by the node's own X_rel and promotion decisions.

Only tests/ and tools/ may import this module; the product never does.  Transforms are composed in double in the
summation order of the device's kf_mul; clouds are re-expressed in float32 with every product and sum rounded, as
k_transform_cloud mode 0 does.  R(X) comes from numpy's float trig, which may differ from the device's by an ulp.
"""
from __future__ import annotations

import numpy as np

from .nodes_oracle import F, homogeneous


def promotion_transform(X) -> np.ndarray:
    """The point map from keyframe f's frame into the frame of scan k, promoted after its registration X against f.
    The registration maps p of k into f as (p + t) R(X) (row vectors), so q of f is q R^-1 - t in k's frame; on column
    vectors, with R^-T = R for a rotation: [R t'; 0 1], t' = -t."""
    T = homogeneous(X).astype(np.float64)
    T[:3, 3] = -T[:3, 3]
    return T


def compose(A, B) -> np.ndarray:
    """A @ B in double, summed in the order of the device's kf_mul."""
    C = np.zeros((4, 4))
    for a in range(4):
        for b in range(4):
            s = A[a, 0] * B[0, b]
            for c in range(1, 4):
                s += A[a, c] * B[c, b]
            C[a, b] = s
    return C


def reexpress(cloud, T) -> np.ndarray:
    """cloud (N x 3 float32, original slot frame) in the current keyframe frame: `row * m - t'` in float32 with
    m = T[:3, :3]^T and t' = -T[:3, 3] rounded to float, every operation rounded (k_transform_cloud mode 0)."""
    c = np.asarray(cloud, F)
    m = T[:3, :3].T.astype(F)
    t = (-T[:3, 3]).astype(F)
    x, y, z = c[:, 0], c[:, 1], c[:, 2]
    out = np.empty_like(c)
    for j in range(3):
        out[:, j] = ((x * m[0, j] + y * m[1, j]) + z * m[2, j]) - t[j]
    return out


class LocalMapWindow:
    """The last M keyframes, newest first: (frame index, original filtered cloud, transform into the newest frame)."""

    def __init__(self, M: int):
        if not 1 <= M <= 16:
            raise ValueError("map_keyframes must be in 1 .. 16")
        self.M = M
        self.slots: list[tuple[int, np.ndarray, np.ndarray]] = []

    def promote(self, frame: int, cloud, X_rel=None, F_point=None):
        """Scan `frame` becomes the newest keyframe.  X_rel: its registration against the previous newest keyframe
        (None for keyframe 0); F_point: the point map into its frame given directly (instead of X_rel)."""
        if X_rel is not None or F_point is not None:
            Fp = promotion_transform(X_rel) if F_point is None else np.asarray(F_point, np.float64)
            self.slots = [(f, c, compose(Fp, T)) for f, c, T in self.slots]
        self.slots.insert(0, (frame, np.ascontiguousarray(cloud, F), np.eye(4)))
        del self.slots[self.M:]

    def frames(self) -> list[int]:
        return [f for f, _, _ in self.slots]

    def block_rows(self) -> list[int]:
        return [c.shape[0] for _, c, _ in self.slots]

    def map(self) -> np.ndarray:
        """The local map: the newest keyframe's rows verbatim, then the older ones re-expressed, newest to oldest."""
        blocks = [self.slots[0][1]] + [reexpress(c, T) for _, c, T in self.slots[1:]]
        return np.concatenate(blocks) if blocks else np.zeros((0, 3), F)
