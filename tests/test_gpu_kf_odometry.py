"""GPU tests of the keyframe odometry node (include/icet_b200.h "keyframe odometry", DESIGN.md §13): the frame-to-frame
limit against the odometry node, batched against streamed callbacks, replay of every registration against a keyframe
built from the same filtered cloud, the promotion tests one at a time, the CPU oracle, and drift against the
generator's ground truth."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL_M, TOL_RAD = 1e-4, 1e-5
OFF = dict(max_trans=0.0, max_rot=0.0, min_overlap=0.0, max_interval=0)


@pytest.fixture(scope="module")
def scans():
    """seven consecutive synthetic 64-channel scans as N x 3 arrays (the fixture of test_gpu_nodes.py)"""
    from tools import synth_host
    s = synth_host.scans(7, first_scan=3, seed=20240, rings=64, azim=2048)
    return [np.ascontiguousarray(a.T) for a in s]


def _policy(**kw):
    from icet_b200 import api
    return api.KeyframePolicy(**dict(OFF, **kw))


def _run(ctx, scans, policy, chain=True, runlen=7):
    from icet_b200 import KeyframeOdometryNode
    node = KeyframeOdometryNode(ctx, max_points=scans[0].shape[0], runlen=runlen, chain_x0=chain, policy=policy)
    out = [node.callback(s) for s in scans]
    node.close()
    assert out[0] is None
    return out[1:]


@pytest.mark.parametrize("chain", [1, 0])
def test_one_scan_per_keyframe_reproduces_the_odometry_node(ctx, scans, chain):
    """max_interval = 1 with every other test off: every scan is the keyframe of the next one, seeds are the previous
    solution (chain_x0) or 0 -- the odometry node, byte for byte in results and poses."""
    from icet_b200 import Node, api
    ref = Node(ctx, api.make_params(), api.OdometryParams(2.0, chain, 10.0, 0.0, 0.0), scans[0].shape[0])
    want = [ref.push(s) for s in scans][1:]
    ref.close()
    got = _run(ctx, scans, _policy(max_interval=1), chain=bool(chain))
    for k, ((r, p), (gr, gp, gi)) in enumerate(zip(want, got), start=1):
        for f in ("X", "Q", "status", "pred_stds", "n_gauss1", "n_used"):
            assert np.asarray(gr[f]).tobytes() == np.asarray(r[f]).tobytes(), (chain, k, f)
        for f in ("X_homo", "orientation", "position", "twist", "covariance_diag", "n_points", "frame"):
            assert np.asarray(gp[f]).tobytes() == np.asarray(p[f]).tobytes(), (chain, k, f)
        assert gi["keyframe"] == k - 1 and gi["promoted"] == 1 and gi["reason"] == api.KF_INTERVAL


@pytest.mark.parametrize("policy", [dict(max_interval=2), dict(max_interval=3), dict()],
                         ids=["promotes_mid_call", "promotes_first_scan_of_call", "never"])
def test_batched_equals_streamed(ctx, scans, policy):
    """push_device of all scans in two calls (3 + 4) == one blocking callback per scan, byte for byte."""
    import torch
    from icet_b200 import KeyframeOdometryNode, api
    streamed = _run(ctx, scans, _policy(**policy))
    planes = np.stack([np.ascontiguousarray(s.T) for s in scans])
    dev = torch.from_numpy(planes).cuda()
    ns, n = planes.shape[0], planes.shape[2]
    node = KeyframeOdometryNode(ctx, max_points=n, policy=_policy(**policy))
    res = torch.zeros((ns, 56), dtype=torch.float32, device="cuda")
    pose = torch.zeros((ns, 45), dtype=torch.float32, device="cuda")
    info = torch.zeros((ns, 10), dtype=torch.float32, device="cuda")
    k1 = node.push_device(dev.data_ptr(), 3, n, res.data_ptr(), pose.data_ptr(), info.data_ptr())
    k2 = node.push_device(dev[3:].data_ptr(), ns - 3, n, res[k1:].data_ptr(), pose[k1:].data_ptr(), info[k1:].data_ptr())
    ctx.synchronize()
    assert (k1, k2) == (2, ns - 3)
    r = res.cpu().numpy().view(api.RESULT_DTYPE).reshape(-1)
    p = pose.cpu().numpy().view(api.POSE_DTYPE).reshape(-1)
    i = info.cpu().numpy().view(api.KF_INFO_DTYPE).reshape(-1)
    for k, (sr, sp, si) in enumerate(streamed):
        for rec, ref, dt in ((r[k], sr, api.RESULT_DTYPE), (p[k], sp, api.POSE_DTYPE), (i[k], si, api.KF_INFO_DTYPE)):
            for f in dt.names:
                assert rec[f].tobytes() == np.asarray(ref[f]).tobytes(), (policy, k, f)
    promoted = [int(x["promoted"]) for x in i[: ns - 1]]
    if policy.get("max_interval") == 2:
        assert promoted == [0, 1, 0, 1, 0, 1]     # scan 4 is promoted in the middle of the second call
    elif policy.get("max_interval") == 3:
        assert promoted == [0, 0, 1, 0, 0, 1]     # scan 3 is the first scan of the second call
    else:
        assert not any(promoted) and (i["keyframe"][: ns - 1] == 0).all()
    # the keyframe cloud the node exposes: the filtered last keyframe
    from oracle import kf_odometry_oracle as no
    last = max([0] + [k + 1 for k in range(ns - 1) if promoted[k]])
    want = scans[0] if last == 0 else no.min_range_filter(scans[last], 2.0)
    assert node.keyframe_cloud().tobytes() == np.ascontiguousarray(want, np.float32).tobytes()
    node.close()


def test_replay_against_keyframes(ctx, scans):
    """Every registration == Keyframe(filtered keyframe scan).register(filtered scan, x0 = info.x0) byte for byte;
    promotions == the numpy restatement of the policy on the node's own results; seeds and poses == their numpy
    restatements (double seeds to 1e-6, float poses to 1e-5 relative)."""
    from icet_b200 import Keyframe
    from oracle import kf_odometry_oracle as no
    pol = dict(max_trans=0.9, max_rot=0.02, min_overlap=0.5, max_interval=3)
    got = _run(ctx, scans, _policy(**pol))
    filt = [np.ascontiguousarray(scans[0], np.float32)] + [no.min_range_filter(s, 2.0) for s in scans[1:]]
    kf_frame, interval, H_f, X_prev, x0 = 0, 0, np.eye(4, dtype=np.float32), np.zeros(6, np.float32), np.zeros(6, np.float32)
    kfs = {}
    for k, (r, p, i) in enumerate(got, start=1):
        assert i["keyframe"] == kf_frame
        np.testing.assert_allclose(i["x0"], x0, rtol=0, atol=1e-6)
        if kf_frame not in kfs:
            kfs[kf_frame] = Keyframe(filt[kf_frame], ctx=ctx)
        rr = kfs[kf_frame].register(filt[k], X0=i["x0"])
        for f in ("X", "Q", "status", "n_gauss1", "n_used"):
            assert np.asarray(rr[f]).tobytes() == np.asarray(r[f]).tobytes(), (k, f)
        reason = no.kf_reason(r["X"], int(r["status"]), int(r["n_used"]), int(r["n_gauss1"]), interval, **pol)
        assert int(i["reason"]) == reason and int(i["promoted"]) == int(reason != 0), k
        H = (H_f.astype(np.float64) @ no.homogeneous(r["X"]).astype(np.float64))
        np.testing.assert_allclose(p["X_homo"], H, rtol=1e-5, atol=1e-5)
        step = no.kf_step(X_prev, r["X"], kf_frame == k - 1)
        np.testing.assert_allclose(p["twist"], 10.0 * step, rtol=1e-5, atol=1e-6)
        x0 = no.kf_next_seed(r["X"], step, reason != 0, True)
        X_prev = r["X"]
        if reason:
            kf_frame, interval, H_f = k, 0, p["X_homo"]
        else:
            interval += 1
    assert len(kfs) >= 2   # the policy promoted at least once
    for kf in kfs.values():
        kf.close()


@pytest.mark.parametrize("name,kw,bit", [("translation", dict(max_trans=1e-3), 1), ("rotation", dict(max_rot=1e-7), 2),
                                         ("interval", dict(max_interval=2), 8), ("overlap", dict(min_overlap=1.0), 4)])
def test_each_trigger_alone(ctx, scans, name, kw, bit):
    """One test on, the others off: it promotes, its bit alone is the reason, and the reason equals the restatement."""
    from oracle import kf_odometry_oracle as no
    got = _run(ctx, scans, _policy(**kw))
    interval, fired = 0, 0
    for r, p, i in got:
        want = no.kf_reason(r["X"], int(r["status"]), int(r["n_used"]), int(r["n_gauss1"]), interval, **dict(OFF, **kw))
        assert int(i["reason"]) == want and (want & ~16) in (0, bit), (name, want)
        fired += int((want & bit) != 0)
        interval = 0 if want else interval + 1
    assert fired >= 1, name
    # a registration that did not converge promotes whatever the policy says
    for r, p, i in got:
        if int(r["status"]) != 0:
            assert int(i["reason"]) & 16 and int(i["promoted"]) == 1


def test_matches_oracle(ctx, scans):
    """5 scans, keyframe every second scan: X of every registration within the tolerances of
    test_odometry_node_matches_oracle, the oracle registering the same filtered keyframe / scan pairs from the same seeds."""
    from oracle import kf_odometry_oracle as no
    got = _run(ctx, scans[:5], _policy(max_interval=2))
    orc = no.KeyframeOdometryOracle(policy=dict(OFF, max_interval=2))
    assert orc.callback(scans[0]) is None
    for k, (r, p, i) in enumerate(got, start=1):
        o = orc.callback(scans[k], x0=i["x0"])
        assert o["keyframe"] == int(i["keyframe"]) and o["promoted"] == bool(i["promoted"])
        assert o["n_points"] == int(p["n_points"])
        assert np.abs(r["X"][:3] - o["X"][:3]).max() < TOL_M
        assert np.abs(r["X"][3:] - o["X"][3:]).max() < TOL_RAD
        assert np.abs(p["X_homo"] - o["X_homo"]).max() < 2 * TOL_M * k


# measured on one B200 (1000 W power limit) with this test: median 0.0060 m, p99 0.0345 m, max 0.0593 m of translation
# error per keyframe-relative registration over 240 scans with the default policy (91 keyframes); bounds at 2x that
KF_ERR_MEDIAN, KF_ERR_P99 = 0.012, 0.07


def test_drift_against_ground_truth(ctx):
    """>= 200 scans with the default policy: the translation error of every keyframe-relative registration against the
    generator's motion composed from the keyframe to the scan, in the mapping test_full_size_sequence_properties uses
    for single steps."""
    import torch
    from icet_b200 import KeyframeOdometryNode, api
    from oracle import kf_odometry_oracle as no
    from tools import synth_host
    ns, n = 241, 64 * 2048
    dev = torch.empty((ns, 3, n), dtype=torch.float32, device="cuda")
    for c0 in range(0, ns, 64):
        m = min(64, ns - c0)
        dev[c0:c0 + m] = torch.from_numpy(synth_host.scans(m, first_scan=c0))
    node = KeyframeOdometryNode(ctx, max_points=n)
    res = torch.zeros((ns, 56), dtype=torch.float32, device="cuda")
    pose = torch.zeros((ns, 45), dtype=torch.float32, device="cuda")
    info = torch.zeros((ns, 10), dtype=torch.float32, device="cuda")
    assert node.push_device(dev.data_ptr(), ns, n, res.data_ptr(), pose.data_ptr(), info.data_ptr()) == ns - 1
    ctx.synchronize()
    node.close()
    r = res.cpu().numpy().view(api.RESULT_DTYPE).reshape(-1)[: ns - 1]
    i = info.cpu().numpy().view(api.KF_INFO_DTYPE).reshape(-1)[: ns - 1]
    gt = synth_host.motions(0, ns - 1)
    err = []
    for k in range(1, ns):
        f = int(i[k - 1]["keyframe"])
        H = np.eye(4)
        for j in range(f, k):
            H = H @ no.homogeneous(gt[j]).astype(np.float64)
        err.append(np.abs(r[k - 1]["X"][:3] - H[:3, 3]).max())
    err = np.array(err)
    print("keyframe registrations vs ground truth: median %.4f p99 %.4f max %.4f m; keyframes %d"
          % (np.median(err), np.percentile(err, 99), err.max(), int(i["promoted"].sum())))
    assert np.median(err) < KF_ERR_MEDIAN and np.percentile(err, 99) < KF_ERR_P99


def test_cpp_example_prints_the_python_poses(ctx, scans, tmp_path):
    """examples/kf_odometry_headless.cpp (include/icet_nodes.h KeyframeOdometryNode) replays the scans: same library,
    same bits as the Python node, same keyframe decisions."""
    import json
    import os
    import subprocess
    from conftest import ROOT
    r = subprocess.run(["make", "-C", os.path.join(ROOT, "examples"), "_build/kf_odometry_headless"], capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    f = tmp_path / "seq.f32"
    np.stack([np.ascontiguousarray(s.T) for s in scans]).tofile(f)
    n = scans[0].shape[0]
    out = subprocess.run([os.path.join(ROOT, "examples", "_build", "kf_odometry_headless"), str(n), str(f), "0.9", "0.02",
                          "0.5", "3"], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    rows = [l for l in out.stdout.splitlines() if l.startswith("POSE")]
    py = _run(ctx, scans, _policy(max_trans=0.9, max_rot=0.02, min_overlap=0.5, max_interval=3))
    assert len(rows) == len(py) == len(scans) - 1
    for l, (r, p, i) in zip(rows, py):
        x = np.float32(json.loads(l[l.index("X [") + 2: l.index("] pos") + 1]))
        pos = np.float32(json.loads(l[l.index("pos [") + 4: l.index("] quat") + 1]))
        q = np.float32(json.loads(l[l.index("quat [") + 5: l.index("] points") + 1]))
        np.testing.assert_array_equal(x, p["X"])
        np.testing.assert_array_equal(pos, p["position"])
        np.testing.assert_array_equal(q, p["orientation"])
        tail = l.split("points ")[1].split()
        assert int(tail[0]) == int(p["n_points"]) and int(tail[2]) == int(i["keyframe"])
        assert int(tail[4]) == int(i["promoted"]) and int(tail[6]) == int(i["reason"])
