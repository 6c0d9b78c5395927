"""GPU tests of keyframe registration (include/icet_b200.h "keyframes", icet_b200.Keyframe): scan 1 fitted once and
registered against many scans gives, byte for byte, what registering the same pairs with that cloud as scan 1 gives --
in batches of every chunking, lane count and loop form, in single calls, for many seeds of one pair, for the 2 M-point
map of BASELINE.json configs[4] and in shipped row order."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SCAN1_KERNELS = ("k_scan1_bin", "k_scatter", "k_cluster", "k_pass<scan1>", "k_fit1")


@pytest.fixture(scope="module")
def kctx():
    import icet_b200
    icet_b200.build()
    c = icet_b200.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def seq(kctx):
    """synthetic 64-channel scans 0 .. 8 on the device: scan 0 is the keyframe"""
    return synth_device(kctx, 9)


def synth_device(ctx, nscans, first=0, rings=64, azim=2048, seed=20240):
    import torch
    t = torch.empty((nscans, 3, rings * azim), dtype=torch.float32, device="cuda")
    ctx.synth_scans_device(t.data_ptr(), nscans, first_scan=first, seed=seed, rings=rings, azim=azim)
    ctx.synchronize()
    return t


def mixed_x0(npairs, seed=3):
    """zeros for the even pairs, small seeded offsets for the odd ones"""
    rng = np.random.default_rng(seed)
    x0 = np.zeros((npairs, 6), np.float32)
    x0[1::2, :3] = rng.uniform(-0.05, 0.05, (len(x0[1::2]), 3))
    x0[1::2, 3:] = rng.uniform(-0.01, 0.01, (len(x0[1::2]), 3))
    return x0


def as_results(t):
    from icet_b200 import api
    return t.cpu().numpy().view(api.RESULT_DTYPE).reshape(-1)


def batch_both(ctx, kf, scan1, scans2, x0, runlen=7, flags=0):
    """(keyframe batch, ordinary batch with scan1 repeated) over device scans2[i], DEVICE x0 and results"""
    import torch
    from icet_b200 import api
    P = len(scans2)
    ptr2 = np.array([s.data_ptr() for s in scans2], np.uint64)
    n2 = np.array([s.shape[1] for s in scans2], np.int32)
    x0d = torch.from_numpy(np.ascontiguousarray(x0, np.float32)).cuda()
    out_k = torch.zeros((P, 56), dtype=torch.float32, device="cuda")
    out_b = torch.zeros((P, 56), dtype=torch.float32, device="cuda")
    kf.register_batch_device(ptr2, n2, out_k.data_ptr(), x0d.data_ptr(), runlen=runlen, flags=flags)
    p = kf.params(runlen, flags)
    ptr1 = np.full(P, scan1.data_ptr(), np.uint64)
    n1 = np.full(P, scan1.shape[1], np.int32)
    ctx.register_batch_ptrs(ptr1, n1, ptr2, n2, out_b.data_ptr(), x0d.data_ptr(), params=p, device=True)
    ctx.synchronize()
    return as_results(out_k), as_results(out_b)


@pytest.mark.parametrize("chunk,lanes,flag", [
    (0, 0, 0), (3, 0, 0), (0, 1, 0), (0, 2, 0),
    (0, 0, "UNFUSED_LOOP"), (0, 0, "PERSISTENT_LOOP"), (0, 0, "CLUSTER_LOOP"), (0, 0, "EXACT_PASS")])
def test_keyframe_batch_equals_batch(kctx, seq, chunk, lanes, flag):
    import icet_b200
    from icet_b200 import api
    flags = getattr(api, "FLAG_" + flag) if flag else 0
    kf = icet_b200.Keyframe.from_device(seq[0].data_ptr(), seq.shape[2], ctx=kctx)
    kctx.set_chunk(chunk)
    kctx.set_lanes(lanes)
    try:
        k, b = batch_both(kctx, kf, seq[0], [seq[i] for i in range(1, 9)], mixed_x0(8), flags=flags)
    finally:
        kctx.set_chunk(0)
        kctx.set_lanes(0)
    assert k.tobytes() == b.tobytes()
    assert np.all(k["status"] == 0) and np.all(k["n_gauss1"] == kf.n_gauss1) and kf.n_gauss1 > 100
    kf.close()


def test_keyframe_register_equals_register(kctx, frame_pair, sample_pair):
    import icet_b200
    from icet_b200 import api
    s1, s2 = frame_pair
    kf = icet_b200.Keyframe(s1.T, ctx=kctx)  # N x 3 as well as planes
    for x0 in (np.zeros(6, np.float32), np.array([1, 0, 0, 0, 0, 0], np.float32)):
        r = kf.register(s2, x0)
        assert r.tobytes() == kctx.register(s1, s2, x0).tobytes()
    assert r["n_gauss1"] == kf.n_gauss1
    kf.close()
    s1, s2 = sample_pair
    kf = icet_b200.Keyframe(s1, ctx=kctx)
    assert kf.register(s2).tobytes() == kctx.register(s1, s2).tobytes()
    kf.close()
    # BASELINE.json configs[3]: 128 x 2048 points, 150 x 48 voxels, 10 iterations
    host = synth_device(kctx, 2, rings=128, azim=2048, first=3).cpu().numpy()
    kf = icet_b200.Keyframe(host[0], num_bins_phi=48, num_bins_theta=150, ctx=kctx)
    p = api.make_params(runlen=10, bins_phi=48, bins_theta=150)
    assert kf.register(host[1], runlen=10).tobytes() == kctx.register(host[0], host[1], params=p).tobytes()


def test_many_seeds_of_one_pair(kctx, seq):
    import icet_b200
    rng = np.random.default_rng(11)
    x0 = np.zeros((16, 6), np.float32)
    x0[:, :3] = rng.normal(0, 0.1, (16, 3))
    x0[:, 3:] = rng.normal(0, 0.02, (16, 3))
    kf = icet_b200.Keyframe.from_device(seq[0].data_ptr(), seq.shape[2], ctx=kctx)
    k, b = batch_both(kctx, kf, seq[0], [seq[1]] * 16, x0)
    assert k.tobytes() == b.tobytes()
    h0, h1 = seq[0].cpu().numpy(), seq[1].cpu().numpy()
    for i in range(16):
        assert k[i].tobytes() == kctx.register(h0, h1, x0[i]).tobytes()
    assert len({r.tobytes() for r in k}) > 1
    kf.close()


def test_submap_keyframe_full_size(kctx):
    """BASELINE.json configs[4]: the 2 002 756-point accumulated map as the keyframe."""
    import os
    import icet_b200
    from conftest import GOLDEN
    from tools import synth_host
    mp, cur = synth_host.submap()
    kf = icet_b200.Keyframe(mp, ctx=kctx)
    r = kf.register(cur)
    assert r.tobytes() == kctx.register(mp, cur).tobytes()
    assert r["status"] == 0 and r["n_gauss1"] == kf.n_gauss1
    gold = np.load(os.path.join(GOLDEN, "golden_submap_2M.npz"))
    assert kf.n_gauss1 == int((gold["has1"] > 0).sum())
    # the map registered against many scans: every result as its direct counterpart
    r2 = kf.register(cur, np.array([0.02, -0.01, 0, 0, 0, 0.003], np.float32))
    assert r2.tobytes() == kctx.register(mp, cur, np.array([0.02, -0.01, 0, 0, 0, 0.003], np.float32)).tobytes()
    kf.close()


def test_shipped_order_keyframe(kctx, frame_pair):
    import icet_b200
    from icet_b200 import api
    s1, s2 = frame_pair
    kf = icet_b200.Keyframe(s1, ctx=kctx, shipped_row_order=True)
    r = kf.register(s2)
    assert r.tobytes() == kctx.register(s1, s2, params=api.make_params(flags=api.FLAG_SHIPPED_ORDER)).tobytes()
    assert r["n_gauss1"] < icet_b200.Keyframe(s1, ctx=kctx).n_gauss1  # the shipped order finds fewer clusters
    kf.close()


def test_verify_incremental_keyframe_batch(kctx, seq):
    import icet_b200
    from icet_b200 import api
    kf = icet_b200.Keyframe.from_device(seq[0].data_ptr(), seq.shape[2], ctx=kctx)
    k, b = batch_both(kctx, kf, seq[0], [seq[i] for i in range(1, 9)], mixed_x0(8), flags=api.FLAG_VERIFY_INCREMENTAL)
    assert k.tobytes() == b.tobytes()
    assert np.all(k["reserved"][:, 0] == 0) and np.all(k["reserved"][:, 1] == 0)
    kf.close()


def test_two_keyframes_on_one_context(kctx, seq, frame_pair):
    """Keyframes of different bins stay valid while other registrations re-initialise the context's bin tables."""
    import icet_b200
    from icet_b200 import api
    h = seq.cpu().numpy()
    big = synth_device(kctx, 2, rings=128, azim=2048, first=3).cpu().numpy()
    p_big = api.make_params(runlen=10, bins_phi=48, bins_theta=150)
    p_odd = api.make_params(bins_phi=20, bins_theta=64)
    want_a = [kctx.register(h[0], h[k]) for k in (1, 2)]
    want_b = kctx.register(big[0], big[1], params=p_big)
    want_o = kctx.register(frame_pair[0], frame_pair[1], params=p_odd)
    a = icet_b200.Keyframe(h[0], ctx=kctx)
    b = icet_b200.Keyframe(big[0], num_bins_phi=48, num_bins_theta=150, ctx=kctx)
    for _ in range(2):
        assert a.register(h[1]).tobytes() == want_a[0].tobytes()
        assert kctx.register(frame_pair[0], frame_pair[1], params=p_odd).tobytes() == want_o.tobytes()
        assert b.register(big[1], runlen=10).tobytes() == want_b.tobytes()
        assert kctx.register(frame_pair[0], frame_pair[1], params=p_odd).tobytes() == want_o.tobytes()
        assert a.register(h[2]).tobytes() == want_a[1].tobytes()
    a.close()
    b.close()


def test_keyframe_launches_no_scan1_kernels(kctx, seq):
    import icet_b200
    kf = icet_b200.Keyframe.from_device(seq[0].data_ptr(), seq.shape[2], ctx=kctx)
    h = seq.cpu().numpy()
    want = kctx.register(h[0], h[1])
    kctx.set_profile(True)
    try:
        r = kf.register(h[1])
        k, b = batch_both(kctx, kf, seq[0], [seq[i] for i in range(1, 9)], mixed_x0(8))
        kctx.set_profile(False)
        kctx.set_profile(True)  # (resets the sums)
        kf.register(h[1])
        prof = kctx.get_profile()
    finally:
        kctx.set_profile(False)
    assert r.tobytes() == want.tobytes() and k.tobytes() == b.tobytes()
    for name in SCAN1_KERNELS:
        assert prof[name][1] == 0, name
    assert prof["k_cell_scan"][1] == 1  # k_kf_attach
    kf.close()


def test_keyframe_rejects_mismatched_params(kctx, seq):
    import icet_b200
    from icet_b200 import api
    kf = icet_b200.Keyframe.from_device(seq[0].data_ptr(), seq.shape[2], ctx=kctx)
    s2 = np.ascontiguousarray(seq[1].cpu().numpy())
    res = api.Result()
    L = kctx._L
    for field, value in (("bins_phi", 48), ("bins_theta", 150), ("n", 20), ("thresh", 0.2), ("buff", 0.3)):
        p = kf.params()
        setattr(p, field, value)
        with pytest.raises(icet_b200.IcetError, match=field):
            kctx._check(L.icet_b200_register_keyframe(kf._h, C.byref(p), s2.ctypes.data, s2.shape[1], s2.shape[1],
                                                      None, C.byref(res)))
        with pytest.raises(icet_b200.IcetError, match=field):
            kctx._check(L.icet_b200_register_keyframe_batch_device(kf._h, C.byref(p), 0, None, None, None, None))
    with pytest.raises(icet_b200.IcetError, match="SHIPPED_ORDER"):
        kf.register(s2, flags=api.FLAG_SHIPPED_ORDER)
    with pytest.raises(icet_b200.IcetError, match="CHAIN_X0"):
        kf.register(s2, flags=api.FLAG_CHAIN_X0)
    with pytest.raises(icet_b200.IcetError, match="CHAIN_X0"):
        kf.register_batch_device([seq[1].data_ptr()], [seq.shape[2]], 0, flags=api.FLAG_CHAIN_X0)
    # repeated batches: the same bytes
    a, _ = batch_both(kctx, kf, seq[0], [seq[i] for i in range(1, 9)], mixed_x0(8))
    b, _ = batch_both(kctx, kf, seq[0], [seq[i] for i in range(1, 9)], mixed_x0(8))
    assert a.tobytes() == b.tobytes()
    kf.close()
    with pytest.raises(icet_b200.IcetError, match="closed"):
        kf.register(s2)
