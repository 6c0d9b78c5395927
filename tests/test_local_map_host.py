"""CPU tests of the local-map keyframe odometry node (icet_b200_kfnode_create_local_map, DESIGN.md §14): the C entry
points reject bad arguments with a message naming the field (no device needed), the Python keyword maps None to the
plain entry point, and the numpy restatement of the window (oracle/local_map_oracle.py) composes and slides as stated."""
import ctypes as C

import numpy as np
import pytest


def _lib():
    import icet_b200
    icet_b200.build()
    return icet_b200.load_library()


def _create(L, M=3, max_points=1024, p=None, op=None, kp=None):
    from icet_b200 import api
    p = p or api.make_params()
    op = op or api.OdometryParams(2.0, 1, 10.0, 0.0, 0.0)
    kp = kp or api.KeyframePolicy()
    h = C.c_void_p()
    rc = L.icet_b200_kfnode_create_local_map(None, C.byref(p), C.byref(op), C.byref(kp), M, max_points, None, None,
                                             C.byref(h))
    return rc, L.icet_b200_last_error().decode()


def test_create_local_map_rejects_bad_arguments_naming_the_field():
    from icet_b200 import api
    L = _lib()
    cases = [
        (dict(M=0), "map_keyframes"),
        (dict(M=17), "map_keyframes"),
        (dict(M=-1), "map_keyframes"),
        (dict(M=16, max_points=(1 << 24) + 1), "map_keyframes * max_points"),
        (dict(M=2, max_points=(1 << 27) + 1), "map_keyframes * max_points"),
        # everything icet_b200_kfnode_create rejects
        (dict(p=api.make_params(flags=api.FLAG_SHIPPED_ORDER)), "ICET_B200_FLAG_SHIPPED_ORDER"),
        (dict(p=api.make_params(flags=api.FLAG_CHAIN_X0)), "ICET_B200_FLAG_CHAIN_X0"),
        (dict(op=api.OdometryParams(2.0, 1, 10.0, 0.3, 0.0)), "guard_trans"),
        (dict(max_points=0), "max_points"),
        (dict(p=api.make_params(bins_phi=0)), "bins_phi"),
    ]
    kp = api.KeyframePolicy()
    kp.reserved[1] = 1
    cases.append((dict(kp=kp), "reserved"))
    for kw, field in cases:
        rc, msg = _create(L, **kw)
        assert rc == -1 and field in msg, (kw, msg)
    for M, mp in ((1, 1024), (16, 1 << 24), (2, 1 << 27)):   # valid arguments: only the missing context is left
        rc, msg = _create(L, M=M, max_points=mp)
        assert rc == -1 and "ctx is NULL" in msg, (M, mp, msg)


def test_local_map_entry_points_reject_null_arguments():
    L = _lib()
    assert L.icet_b200_kfnode_local_map(None, None, None, None) == -1
    n = C.c_int32()
    assert L.icet_b200_kfnode_local_map_host(None, None, 0, C.byref(n)) == -1


class _FakeLib:
    """records which create entry point the Python node calls, then fails it"""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def f(*args):
            self.calls.append((name, args))
            return -1
        return f


class _FakeCtx:
    def __init__(self):
        self._L, self._h = _FakeLib(), None

    def _check(self, rc):
        if rc < 0:
            raise RuntimeError("create failed")
        return rc


@pytest.mark.parametrize("M,entry", [(None, "icet_b200_kfnode_create"), (1, "icet_b200_kfnode_create_local_map"),
                                     (4, "icet_b200_kfnode_create_local_map")])
def test_python_keyword_selects_the_entry_point(M, entry):
    import icet_b200
    ctx = _FakeCtx()
    with pytest.raises(RuntimeError, match="create failed"):
        icet_b200.KeyframeOdometryNode(ctx, max_points=4096, map_keyframes=M)
    (name, args), = [c for c in ctx._L.calls if c[0].startswith("icet_b200_kfnode_create")]
    assert name == entry
    if M is not None:
        assert args[4] == M and args[5] == 4096


def test_python_node_validates_map_keyframes():
    import icet_b200
    for M in (0, 17):
        with pytest.raises(ValueError, match="map_keyframes"):
            icet_b200.KeyframeOdometryNode(_FakeCtx(), map_keyframes=M)


def _X(rng):
    return np.concatenate([rng.uniform(-1.5, 1.5, 3), rng.uniform(-0.05, 0.05, 3)]).astype(np.float32)


def test_promotion_transform_inverts_the_registration():
    """The registration maps p of scan k into keyframe f as (p + t) R(X); the promotion transform takes it back."""
    from oracle import local_map_oracle as lo
    from oracle.nodes_oracle import rot_R
    rng = np.random.default_rng(3)
    for _ in range(50):
        X = _X(rng)
        p = rng.uniform(-80, 80, (20, 3))
        pf = (p + X[:3].astype(np.float64)) @ rot_R(X[3], X[4], X[5]).astype(np.float64)
        T = lo.promotion_transform(X)
        back = pf @ T[:3, :3].T + T[:3, 3]
        np.testing.assert_allclose(back, p, rtol=0, atol=1e-4)   # R in float: orthonormal to ~1e-7, |p| <= 140 m


def test_a_promotion_followed_by_its_inverse_is_the_identity():
    from oracle import local_map_oracle as lo
    rng = np.random.default_rng(5)
    for _ in range(20):
        A = lo.promotion_transform(_X(rng))
        w = lo.LocalMapWindow(3)
        w.promote(0, np.zeros((1, 3), np.float32))
        w.promote(1, np.zeros((1, 3), np.float32), F_point=A)
        w.promote(2, np.zeros((1, 3), np.float32), F_point=np.linalg.inv(A))
        assert w.frames() == [2, 1, 0]
        np.testing.assert_allclose(w.slots[2][2], np.eye(4), rtol=0, atol=1e-12)
        np.testing.assert_allclose(w.slots[1][2], np.linalg.inv(A), rtol=0, atol=1e-12)


def test_composition_order():
    """Two promotions A then B: the oldest keyframe's points reach the newest frame as B(A(p)), not A(B(p))."""
    from oracle import local_map_oracle as lo
    rng = np.random.default_rng(11)
    XA, XB = _X(rng), _X(rng)
    A, B = lo.promotion_transform(XA), lo.promotion_transform(XB)
    w = lo.LocalMapWindow(3)
    p = rng.uniform(-50, 50, (16, 3)).astype(np.float32)
    w.promote(0, p)
    w.promote(1, p + 1, X_rel=XA)
    w.promote(2, p + 2, X_rel=XB)
    P = np.c_[p.astype(np.float64), np.ones(16)]
    want = (B @ (A @ P.T)).T[:, :3]
    got = w.map()[32:]
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-4)
    assert np.abs((A @ (B @ P.T)).T[:, :3] - want).max() > 1e-2   # the other order is far off
    np.testing.assert_array_equal(w.map()[:16], p + 2)            # the newest block verbatim


@pytest.mark.parametrize("M", [1, 2, 3, 5])
def test_window_slides_newest_first(M):
    """M + 2 promotions of clouds of distinct sizes: the map lists the last M keyframes newest first, no gaps."""
    from oracle import local_map_oracle as lo
    rng = np.random.default_rng(M)
    w = lo.LocalMapWindow(M)
    sizes = {}
    for k in range(M + 3):
        n = 10 + 7 * k
        sizes[k] = n
        w.promote(k, rng.uniform(-20, 20, (n, 3)).astype(np.float32), X_rel=None if k == 0 else _X(rng))
        want = list(range(k, max(-1, k - M), -1))
        assert w.frames() == want, (k, w.frames())
        assert w.block_rows() == [sizes[f] for f in want]
        assert w.map().shape == (sum(sizes[f] for f in want), 3)
    with pytest.raises(ValueError, match="map_keyframes"):
        lo.LocalMapWindow(17)
