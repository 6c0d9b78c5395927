"""GPU tests of the blocking host-memory entry points against their device-memory twins: every way of handing a node a
scan from the host (packed planes, planes with a leading dimension, N x 3 records) gives the records push_device gives
on the same scans, byte for byte; a keyframe made or registered from planes with a leading dimension equals the packed
call and the device batch."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PAD = 37  # extra columns of the padded planes (ld = n + PAD); the padding holds NaN, which no route may read


@pytest.fixture(scope="module")
def scans():
    """five consecutive synthetic 64-channel scans as N x 3 arrays (the fixture of test_gpu_nodes.py, shorter)"""
    from tools import synth_host
    s = synth_host.scans(5, first_scan=3, seed=20240, rings=64, azim=2048)
    return [np.ascontiguousarray(a.T) for a in s]


def _padded(scan):
    """[3, n + PAD] planes: the scan in the first n columns, NaN behind it."""
    out = np.full((3, scan.shape[0] + PAD), np.nan, np.float32)
    out[:, : scan.shape[0]] = scan.T
    return out


def _make_node(ctx, kind, n):
    from icet_b200 import KeyframeOdometryNode, Node, api
    if kind == "node":
        return Node(ctx, api.make_params(), api.OdometryParams(2.0, 1, 10.0, 0.0, 0.0), n)
    policy = api.KeyframePolicy(max_trans=0.0, max_rot=0.0, min_overlap=0.0, max_interval=2)
    return KeyframeOdometryNode(ctx, max_points=n, policy=policy, map_keyframes=2 if kind == "kfnode_map2" else None)


def _push_host(ctx, node, kind, route, scan):
    """One blocking host push through the C entry point; returns the raw result / pose / info records (b"" for the
    first scan, which registers nothing)."""
    from icet_b200 import api
    L, h = ctx._L, node._h
    res, pose, info = api.Result(), api.Pose(), api.KfInfo()
    n = scan.shape[0]
    if route == "cloud":
        c, keep = api.cloud_desc(np.ascontiguousarray(scan, np.float32))
        assert c.point_step == 12 and c.plane_stride == 0     # N x 3 records, not planes
        args = (C.byref(c),)
    else:
        planes = api.as_planes(scan) if route == "packed" else _padded(scan)
        keep = planes
        args = (planes.ctypes.data, n, planes.shape[1])
    if kind == "node":
        fn = L.icet_b200_node_push_cloud if route == "cloud" else L.icet_b200_node_push
        k = ctx._check(fn(h, *args, C.byref(res), C.byref(pose)))
        recs = (bytes(res), bytes(pose))
    else:
        fn = L.icet_b200_kfnode_push_cloud if route == "cloud" else L.icet_b200_kfnode_push
        k = ctx._check(fn(h, *args, C.byref(res), C.byref(pose), C.byref(info)))
        recs = (bytes(res), bytes(pose), bytes(info))
    del keep
    return recs if k else b""


@pytest.mark.parametrize("kind", ["node", "kfnode", "kfnode_map2"])
def test_host_pushes_equal_device_pushes(ctx, scans, kind):
    """node / kfnode push with packed planes, with planes of leading dimension ld > n and push_cloud with N x 3 records
    each give the records of push_device of the same scans, byte for byte, over a stream of scans (with keyframe
    promotions for the keyframe nodes)."""
    import torch
    from icet_b200 import api
    n = scans[0].shape[0]
    got = {}
    for route in ("packed", "padded", "cloud"):
        node = _make_node(ctx, kind, n)
        got[route] = [_push_host(ctx, node, kind, route, s) for s in scans]
        node.close()
    node = _make_node(ctx, kind, n)
    dev = []
    for s in scans:
        planes = torch.from_numpy(api.as_planes(s)).cuda()
        res = torch.zeros(56, dtype=torch.float32, device="cuda")
        pose = torch.zeros(45, dtype=torch.float32, device="cuda")
        info = torch.zeros(10, dtype=torch.float32, device="cuda")
        if kind == "node":
            k = node.push_device(planes.data_ptr(), 1, n, res.data_ptr(), pose.data_ptr())
            recs = (res, pose)
        else:
            k = node.push_device(planes.data_ptr(), 1, n, res.data_ptr(), pose.data_ptr(), info.data_ptr())
            recs = (res, pose, info)
        ctx.synchronize()
        dev.append(tuple(r.cpu().numpy().tobytes() for r in recs) if k else b"")
    node.close()
    assert dev[0] == b"" and all(d != b"" for d in dev[1:])
    for route, recs in got.items():
        assert recs == dev, (kind, route)
    if kind != "node":
        promoted = [np.frombuffer(d[2], api.KF_INFO_DTYPE)[0]["promoted"] for d in dev[1:]]
        assert any(promoted) and not all(promoted)


def test_keyframe_create_with_leading_dimension(ctx, scans):
    """icet_b200_keyframe_create from planes with ld1 > n1 == the packed create: the same Gaussian count and the same
    registrations against it."""
    from icet_b200 import Keyframe, api
    L = ctx._L
    s1 = scans[0]
    packed = Keyframe(s1, ctx=ctx)
    planes = _padded(s1)
    p = api.make_params(0)
    h = C.c_void_p()
    ctx._check(L.icet_b200_keyframe_create(ctx._h, C.byref(p), planes.ctypes.data, s1.shape[0], planes.shape[1],
                                           C.byref(h)))
    try:
        assert L.icet_b200_keyframe_gaussians(h) == packed.n_gauss1 > 0
        x0 = np.array([0.3, 0, 0, 0, 0, 0.01], np.float32)
        for s2 in scans[1:3]:
            want = packed.register(s2, X0=x0)
            q = packed.params()
            s = api.as_planes(s2)
            res = api.Result()
            ctx._check(L.icet_b200_register_keyframe(h, C.byref(q), s.ctypes.data, s.shape[1], s.shape[1],
                                                     x0.ctypes.data, C.byref(res)))
            assert bytes(res) == want.tobytes()
    finally:
        L.icet_b200_keyframe_destroy(h)
        packed.close()


@pytest.mark.parametrize("seeded", [True, False])
def test_register_keyframe_with_leading_dimension(ctx, scans, seeded):
    """icet_b200_register_keyframe from planes with ld2 > n2 == the packed call == register_keyframe_batch_device of the
    same scan, with a seed and with none (NULL)."""
    import torch
    from icet_b200 import Keyframe, api
    L = ctx._L
    kf = Keyframe(scans[0], ctx=ctx)
    x0 = np.array([0.3, 0, 0, 0, 0, 0.01], np.float32) if seeded else None

    def register(planes, n):
        res = api.Result()
        ctx._check(L.icet_b200_register_keyframe(kf._h, C.byref(kf.params()), planes.ctypes.data, n, planes.shape[1],
                                                 None if x0 is None else x0.ctypes.data, C.byref(res)))
        return bytes(res)

    for s2 in scans[1:3]:
        n = s2.shape[0]
        packed = register(api.as_planes(s2), n)
        assert register(_padded(s2), n) == packed
        d2 = torch.from_numpy(api.as_planes(s2)).cuda()
        out = torch.zeros(56, dtype=torch.float32, device="cuda")
        dx = torch.from_numpy(x0).cuda() if seeded else None
        kf.register_batch_device([d2.data_ptr()], [n], out.data_ptr(), dx.data_ptr() if seeded else 0)
        ctx.synchronize()
        assert out.cpu().numpy().tobytes() == packed
    kf.close()
