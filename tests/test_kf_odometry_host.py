"""CPU tests of the keyframe odometry node (include/icet_b200.h "keyframe odometry"): the C entry points reject bad
arguments and unsupported flags with a message naming the field (no device needed: the arguments are checked before
the context), the Python class validates the same, and the numpy restatement of its pose / seed / policy rules
(oracle/kf_odometry_oracle.py) behaves on hand-made cases."""
import ctypes as C

import numpy as np
import pytest


def _lib():
    import icet_b200
    icet_b200.build()
    return icet_b200.load_library()


def _create(L, p=None, op=None, kp=None, max_points=1024):
    from icet_b200 import api
    p = p or api.make_params()
    op = op or api.OdometryParams(2.0, 1, 10.0, 0.0, 0.0)
    kp = kp or api.KeyframePolicy()
    h = C.c_void_p()
    rc = L.icet_b200_kfnode_create(None, C.byref(p), C.byref(op), C.byref(kp), max_points, None, None, C.byref(h))
    return rc, L.icet_b200_last_error().decode()


def test_create_rejects_unsupported_arguments_naming_the_field():
    from icet_b200 import api
    L = _lib()
    cases = [
        (dict(p=api.make_params(flags=api.FLAG_SHIPPED_ORDER)), "ICET_B200_FLAG_SHIPPED_ORDER"),
        (dict(p=api.make_params(flags=api.FLAG_CHAIN_X0)), "ICET_B200_FLAG_CHAIN_X0"),
        (dict(op=api.OdometryParams(2.0, 1, 10.0, 0.3, 0.0)), "guard_trans"),
        (dict(op=api.OdometryParams(2.0, 1, 10.0, 0.0, 0.3)), "guard_rot"),
        (dict(max_points=0), "max_points"),
        (dict(p=api.make_params(bins_phi=0)), "bins_phi"),
    ]
    kp = api.KeyframePolicy()
    kp.reserved[2] = 1
    cases.append((dict(kp=kp), "reserved"))
    nan = api.KeyframePolicy()
    nan.max_rot = float("nan")
    cases.append((dict(kp=nan), "max_rot"))
    for kw, field in cases:
        rc, msg = _create(L, **kw)
        assert rc == -1 and field in msg, (kw, msg)
    rc, msg = _create(L)  # valid arguments: only the missing context is left
    assert rc == -1 and "ctx is NULL" in msg


def test_entry_points_reject_null_arguments():
    from icet_b200 import api
    L = _lib()
    res, pose, info = api.Result(), api.Pose(), api.KfInfo()
    pts = np.zeros((3, 8), np.float32)
    assert L.icet_b200_kfnode_push(None, pts.ctypes.data, 8, 8, C.byref(res), C.byref(pose), C.byref(info)) == -1
    assert b"node is NULL" in L.icet_b200_last_error()
    assert L.icet_b200_kfnode_push_device(None, 1, pts.ctypes.data, 8, None, None, None) == -1
    assert L.icet_b200_kfnode_push_cloud(None, None, None, None, None) == -1
    assert L.icet_b200_kfnode_keyframe(None, None, None, None) == -1
    assert L.icet_b200_kfnode_destroy(None) == 0  # like free(NULL)
    p, op = api.make_params(), api.OdometryParams(2.0, 1, 10.0, 0.0, 0.0)
    h = C.c_void_p()
    assert L.icet_b200_kfnode_create(None, C.byref(p), C.byref(op), None, 16, None, None, C.byref(h)) == -1
    assert b"NULL" in L.icet_b200_last_error()


def test_python_node_validates_before_touching_the_device():
    import icet_b200
    from icet_b200 import api
    with pytest.raises(ValueError, match="FLAG_CHAIN_X0"):
        icet_b200.KeyframeOdometryNode(flags=api.FLAG_CHAIN_X0)
    with pytest.raises(ValueError, match="FLAG_SHIPPED_ORDER"):
        icet_b200.KeyframeOdometryNode(flags=api.FLAG_SHIPPED_ORDER)
    with pytest.raises(ValueError, match="max_points"):
        icet_b200.KeyframeOdometryNode(max_points=0)
    with pytest.raises(TypeError):
        icet_b200.KeyframeOdometryNode(policy=dict(max_interval=3))
    with pytest.raises(ValueError, match="max_trans"):
        api.KeyframePolicy(max_trans=float("inf"))
    kp = api.KeyframePolicy()
    kp.reserved[0] = 7
    with pytest.raises(ValueError, match="reserved"):
        icet_b200.KeyframeOdometryNode(policy=kp)
    assert api.KF_INFO_DTYPE.itemsize == C.sizeof(api.KfInfo) == 40 and C.sizeof(api.KeyframePolicy) == 32


def test_params_inverts_homogeneous():
    """params(Hi(X)) == X over random angles inside the valid range (|theta| < pi/2)."""
    from oracle import kf_odometry_oracle as no
    rng = np.random.default_rng(7)
    for _ in range(500):
        X = np.concatenate([rng.uniform(-20, 20, 3), rng.uniform(-3.0, 3.0, 1), rng.uniform(-1.5, 1.5, 1),
                            rng.uniform(-3.0, 3.0, 1)]).astype(np.float32)
        Y = no.kf_params(no.kf_homo64(X))
        assert np.array_equal(Y[:3], X[:3])
        np.testing.assert_allclose(Y[3:], X[3:], rtol=0, atol=5e-6)


def test_step_and_seed_restatement():
    """A constant motion m: the step between two scans that share a keyframe is m again, the seed after a promotion is
    the step, and without one it is the keyframe-relative prediction Hi(X) Hi(step)."""
    from oracle import kf_odometry_oracle as no
    m = np.array([0.5, 0.02, -0.01, 0.001, -0.002, 0.03], np.float32)
    X1 = m
    X2 = no.kf_params(no.kf_homo64(m) @ no.kf_homo64(m))
    np.testing.assert_array_equal(no.kf_step(np.zeros(6, np.float32), X1, True), X1)
    np.testing.assert_allclose(no.kf_step(X1, X2, False), m, atol=2e-6)
    np.testing.assert_array_equal(no.kf_next_seed(X2, m, True, True), m)
    np.testing.assert_allclose(no.kf_next_seed(X1, m, False, True), X2, atol=1e-7)
    assert not no.kf_next_seed(X1, m, False, False).any()


def test_policy_restatement_on_hand_made_cases():
    from oracle import kf_odometry_oracle as no
    X = np.array([1.2, 1.6, 0.0, 0.01, -0.2, 0.0], np.float32)   # |t| = 2.0 exactly, max |angle| = 0.2
    off = dict(max_trans=0.0, max_rot=0.0, min_overlap=0.0, max_interval=0)
    assert no.kf_reason(X, 0, 100, 100, 0, **off) == 0
    assert no.kf_reason(X, 0, 100, 100, 0, **dict(off, max_trans=2.0)) == 0          # `>`, not `>=`
    assert no.kf_reason(X, 0, 100, 100, 0, **dict(off, max_trans=1.99)) == no.KF_TRANS
    assert no.kf_reason(X, 0, 100, 100, 0, **dict(off, max_rot=0.1)) == no.KF_ROT
    assert no.kf_reason(X, 0, 49, 100, 0, **dict(off, min_overlap=0.5)) == no.KF_OVERLAP
    assert no.kf_reason(X, 0, 50, 100, 0, **dict(off, min_overlap=0.5)) == 0
    assert no.kf_reason(X, 0, 100, 100, 8, **dict(off, max_interval=10)) == 0
    assert no.kf_reason(X, 0, 100, 100, 9, **dict(off, max_interval=10)) == no.KF_INTERVAL
    assert no.kf_reason(X, 1, 100, 100, 0, **off) == no.KF_STATUS                     # status promotes, policy or not
    assert no.kf_reason(X, 1, 0, 100, 9, max_trans=1.0, max_rot=0.1, min_overlap=0.5, max_interval=10) == 31


@pytest.mark.parametrize("eigen", ["tests/stubs", "oracle/eigen_shim"])
def test_cpp_class_compiles_against_both_eigen_stand_ins(eigen):
    import os
    import subprocess
    from conftest import ROOT
    r = subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-Wall", "-Werror", "-fsyntax-only",
                        "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, eigen),
                        os.path.join(ROOT, "icet_b200", "host", "nodes.cpp"),
                        os.path.join(ROOT, "examples", "kf_odometry_headless.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
