"""GPU tests of batches whose pairs differ in size (ragged batches): real scans cut to tail lengths, a random
subsample, an accumulated map on either side, the bundled pairs and degenerate clouds, all in one batch.

DESIGN.md 3.6 promises bit-identical results for any chunking, lane count, ordering and device split.  Uniform batches
cannot show whether a pair's result depends on its neighbours in the chunk (the fixed-point precision of the voxel
moments, the huge-cell clustering path) or whether a kernel stops at its own pair's n rather than at the chunk's
largest one.  Here:
  * every row of a ragged batch equals the single call of that pair, byte for byte, for device and host buffers, every
    chunk size, lane count, host pipeline ramp, ordering and loop form, with the incremental self-check, chained, against
    a keyframe and across devices;
  * the device scans sit in one allocation, each followed by a NaN guard of a whole CTA tile: a read past a pair's n
    turns into different numbers, not into the next scan's valid points.  The result rows are fenced the same way;
  * selected rows against the oracle, degenerate rows exactly;
  * scan-2 classes of the tail members per point (a dropped last tile shows up as a count off by the tail).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GUARD = 3072           # NaN floats behind every device scan: one CTA tile of k_pass2 / k_pass<true> (pass_tile_points)
ALIGN = 64             # scans start on 256-byte boundaries, like separate allocations
FENCE = 3              # sentinel result rows before and after the batch's rows
X0_DEG = np.array([0.1, 0, 0, 0, 0, 0.01], np.float32)
TAILS = (1, 3, 31, 33, 127, 129, 383, 385)


def fp_bits(n):
    """mirror of fp_bits (chunk.cuh): fixed-point bits of the voxel moments of a cloud of n points"""
    lg = 1
    while (1 << lg) < max(n, 2):
        lg += 1
    return max(12, min(23, (62 - lg) // 2))


def params(**kw):
    from icet_b200 import api
    return api.make_params(**kw)


class Member:
    def __init__(self, name, s1, s2, x0=None, kind="real"):
        self.name, self.kind = name, kind
        self.s1, self.s2 = np.ascontiguousarray(s1, np.float32), np.ascontiguousarray(s2, np.float32)
        self.x0 = np.zeros(6, np.float32) if x0 is None else np.asarray(x0, np.float32)

    @property
    def n1(self):
        return self.s1.shape[1]

    @property
    def n2(self):
        return self.s2.shape[1]


@pytest.fixture(scope="module")
def rctx():
    import icet_b200
    icet_b200.build()
    c = icet_b200.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def members():
    from conftest import load_pair
    from tools import synth_host
    f1, f2 = load_pair("frame")
    p1, p2 = load_pair("sample_pc")
    sc = synth_host.scans(5, first_scan=40)
    rng = np.random.default_rng(1)
    big = np.concatenate([sc[k] for k in range(4)], axis=1)            # 524 288-point map (4 scans, one frame)
    big = big[:, rng.permutation(big.shape[1])]
    m = [Member("frame", f1, f2), Member("sample_pc", p1, p2),
         Member("synth40", sc[0], sc[1]), Member("synth42", sc[2], sc[3]),
         Member("map_vs_scan", big, sc[4]), Member("scan_vs_map", sc[4], big)]
    for j, k in enumerate(TAILS):  # cut scan 2 only, or both scans
        m.append(Member("tail-%d%s" % (k, "-both" if j % 2 else ""), p1[:, :131072 - k] if j % 2 else p1,
                        p2[:, :131072 - k], kind="tail"))
    m.append(Member("tail65537", p1[:, :65537], p2[:, :65537], kind="tail"))
    m.append(Member("tail4097", f1, f2[:, :4097], kind="tail"))
    rs = np.random.default_rng(20011)
    i1, i2 = np.sort(rs.choice(65536, 20011, replace=False)), np.sort(rs.choice(65536, 20011, replace=False))
    m.append(Member("sub20011", f1[:, i1], f2[:, i2]))
    # degenerate members: too few points of scan 2 for a voxel (strided: no cell gets more than n of them), empty clouds,
    # only dropped returns
    for k in (1, 2, 3, 5, 31, 33):
        m.append(Member("n2=%d" % k, f1, f2[:, ::1999][:, :k], X0_DEG, "degenerate"))
    m.append(Member("n1=0", np.zeros((3, 0), np.float32), f2, X0_DEG, "degenerate"))
    m.append(Member("n2=0", f1, np.zeros((3, 0), np.float32), X0_DEG, "degenerate"))
    m.append(Member("zero4096", f1, np.zeros((3, 4096), np.float32), X0_DEG, "degenerate"))
    for side in ("n1", "n2"):
        classes = {fp_bits(getattr(x, side)) for x in m}
        assert len(classes) >= 3, (side, classes)
    return m


@pytest.fixture(scope="module")
def guarded(members):
    """every scan of the member set in ONE device allocation, each followed by a NaN guard of GUARD floats:
    {id(array): device pointer}"""
    import torch
    arrays = {}
    for x in members:
        for a in (x.s1, x.s2):
            arrays[id(a)] = a
    offs, tot = {}, 0
    for k, a in arrays.items():
        offs[k] = tot
        tot += -(-(a.size + GUARD) // ALIGN) * ALIGN
    host = np.full(tot, np.nan, np.float32)
    for k, a in arrays.items():
        host[offs[k]:offs[k] + a.size] = a.reshape(-1)
    buf = torch.from_numpy(host).cuda()
    base = buf.data_ptr()
    return buf, {k: base + 4 * o for k, o in offs.items()}


def sentinel_rows(P):
    import torch
    t = torch.empty((P + 2 * FENCE, 56), dtype=torch.float32, device="cuda")
    t.view(torch.int32).fill_(0x5A5AA5A5)
    return t


def check_fence(t, P):
    a = t.cpu().numpy().view(np.int32)
    assert (a[:FENCE] == 0x5A5AA5A5).all() and (a[FENCE + P:] == 0x5A5AA5A5).all(), "a result record outside the batch was written"


def rows(t, P):
    from icet_b200 import api
    check_fence(t, P)
    return t.cpu().numpy()[FENCE:FENCE + P].copy().view(api.RESULT_DTYPE).reshape(-1)


def device_batch(ctx, guarded, ms, p):
    import torch
    buf, ptr = guarded
    P = len(ms)
    out = sentinel_rows(P)
    x0 = torch.from_numpy(np.stack([x.x0 for x in ms])).cuda()
    ctx.register_batch_ptrs(np.array([ptr[id(x.s1)] for x in ms], np.uint64), [x.n1 for x in ms],
                            np.array([ptr[id(x.s2)] for x in ms], np.uint64), [x.n2 for x in ms],
                            out.data_ptr() + FENCE * 224, x0_ptr=x0.data_ptr(), params=p, device=True)
    ctx.synchronize()
    return rows(out, P)


def host_batch(ctx, ms, p):
    return ctx.register_batch([x.s1 for x in ms], [x.s2 for x in ms], np.stack([x.x0 for x in ms]), p)


_SINGLES = {}


def single(ctx, x, flags=0):
    k = (x.name, flags)
    if k not in _SINGLES:
        _SINGLES[k] = ctx.register(x.s1, x.s2, X0=x.x0, params=params(flags=flags)).copy()
    return _SINGLES[k]


def assert_rows_equal_singles(ctx, ms, out, flags=0):
    bad = [x.name for x, r in zip(ms, out) if r.tobytes() != single(ctx, x, flags).tobytes()]
    assert not bad, "rows differing from the single call of their pair: %s" % bad


def ordering(ms, order):
    if order == "reversed":
        return ms[::-1]
    if order == "rotated":
        return ms[len(ms) // 3:] + ms[:len(ms) // 3]
    return list(ms)


def flag_value(flag):
    from icet_b200 import api
    return getattr(api, "FLAG_" + flag) if flag else 0


# ---------------------------------------------------------------------------------------------------------
# 1. against the oracle
# ---------------------------------------------------------------------------------------------------------
ORACLE_MEMBERS = ("frame", "sample_pc", "synth40", "tail-385-both", "tail65537", "sub20011")


def test_ragged_batch_vs_oracle(rctx, po, guarded, members):
    from test_gpu_parity import check_final, oracle_with_gpu_signs
    out = device_batch(rctx, guarded, members, params())
    for x, r in zip(members, out):
        if x.name in ORACLE_MEMBERS:
            assert r["status"] == 0
            _, g = rctx.register(x.s1, x.s2, X0=x.x0, dump=True)
            o = po.run(x.s1, x.s2, X0=x.x0, dumps="small")
            o2, o64, nbad = oracle_with_gpu_signs(po, x.s1, x.s2, g, o, X0=x.x0)
            check_final(r, o2, o64, "ragged batch: %s" % x.name)
            assert r["n_used"] == int(o2.used2[-1].sum()), x.name
        elif x.kind == "degenerate":
            o = po.run(x.s1, x.s2, X0=x.x0, dumps=None)
            np.testing.assert_array_equal(r["X"], o.X, err_msg=x.name)
            np.testing.assert_array_equal(r["X"], x.x0, err_msg=x.name)
            assert np.all(r["Q"] == 0) and np.all(r["pred_stds"] == 0), x.name
            assert r["status"] == 0 and r["n_used"] == 0, x.name
        else:
            assert r["status"] == 0 and np.all(np.isfinite(r["X"])) and np.all(np.isfinite(r["Q"])), x.name
            assert r["n_used"] > 0, x.name


# ---------------------------------------------------------------------------------------------------------
# 2. batch = single, byte for byte
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chunk", [0, 1, 2, 3, 5])
@pytest.mark.parametrize("lanes", [1, 2, 3])
def test_device_batch_equals_single(rctx, guarded, members, chunk, lanes):
    rctx.set_chunk(chunk)
    rctx.set_lanes(lanes)
    try:
        out = device_batch(rctx, guarded, members, params())
    finally:
        rctx.set_chunk(0)
        rctx.set_lanes(0)
    assert_rows_equal_singles(rctx, members, out)


@pytest.mark.parametrize("order", ["built", "reversed", "rotated"])
@pytest.mark.parametrize("flag", [0, "PERSISTENT_LOOP", "UNFUSED_LOOP", "CLUSTER_LOOP", "EXACT_PASS"])
def test_device_batch_orders_and_loops(rctx, guarded, members, order, flag):
    ms = ordering(members, order)
    fl = flag_value(flag)
    rctx.set_chunk(3)
    try:
        out = device_batch(rctx, guarded, ms, params(flags=fl))
    finally:
        rctx.set_chunk(0)
    assert_rows_equal_singles(rctx, ms, out, fl)
    whole = device_batch(rctx, guarded, ms, params(flags=fl))   # one chunk
    assert_rows_equal_singles(rctx, ms, whole, fl)


@pytest.mark.parametrize("host_chunk", [1, 4])
@pytest.mark.parametrize("chunk", [0, 3])
@pytest.mark.parametrize("order", ["built", "reversed", "rotated"])
def test_host_batch_equals_single(rctx, members, host_chunk, chunk, order):
    ms = ordering(members, order)
    rctx.set_host_chunk(host_chunk)
    rctx.set_chunk(chunk)
    try:
        out = host_batch(rctx, ms, params())
    finally:
        rctx.set_host_chunk(0)
        rctx.set_chunk(0)
    assert_rows_equal_singles(rctx, ms, out)


@pytest.mark.parametrize("flag", ["PERSISTENT_LOOP", "UNFUSED_LOOP", "CLUSTER_LOOP", "EXACT_PASS"])
def test_host_batch_loops(rctx, members, flag):
    fl = flag_value(flag)
    out = host_batch(rctx, members, params(flags=fl))
    assert_rows_equal_singles(rctx, members, out, fl)


# ---------------------------------------------------------------------------------------------------------
# 3. incremental self-check
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flag", [0, "PERSISTENT_LOOP", "CLUSTER_LOOP"])
def test_ragged_verify_incremental(rctx, guarded, members, flag):
    from icet_b200 import api
    fl = flag_value(flag)
    plain = device_batch(rctx, guarded, members, params(flags=fl))
    v = device_batch(rctx, guarded, members, params(flags=fl | api.FLAG_VERIFY_INCREMENTAL))
    bad = [x.name for x, r in zip(members, v) if (r["reserved"][:2] != 0).any()]
    assert not bad, "stable points changed class / filtered evaluation differs in: %s" % bad
    assert v["X"].tobytes() == plain["X"].tobytes() and v["Q"].tobytes() == plain["Q"].tobytes()
    h = host_batch(rctx, members, params(flags=fl | api.FLAG_VERIFY_INCREMENTAL))
    assert (h["reserved"][:, :2] == 0).all()
    assert h["X"].tobytes() == plain["X"].tobytes()


# ---------------------------------------------------------------------------------------------------------
# 4. chained batch over a ragged sequence
# ---------------------------------------------------------------------------------------------------------
def test_chained_ragged_batch_equals_seeded_single_calls(rctx):
    import torch
    from icet_b200 import api
    from tools import synth_host
    sc = synth_host.scans(9, first_scan=60)
    lens = [131072, 131071, 65537, 131072 - 385, 20011, 131072, 4097, 131072 - 31, 65536 + 127]
    seq = [np.ascontiguousarray(sc[k][:, :n]) for k, n in enumerate(lens)]
    x = np.array([0.2, 0.0, 0.0, 0.0, 0.0, 0.01], np.float32)
    x0 = x.copy()
    ref = []
    for k in range(len(seq) - 1):
        r = rctx.register(seq[k], seq[k + 1], x)
        x = r["X"].copy()
        ref.append(r.copy())
    ref = np.array(ref)
    pc = api.make_params(flags=api.FLAG_CHAIN_X0)
    P = len(seq) - 1
    # device scans, each followed by a NaN guard; scan k + 1 is scan 2 of pair k and scan 1 of pair k + 1
    offs, tot = [], 0
    for s in seq:
        offs.append(tot)
        tot += -(-(s.size + GUARD) // ALIGN) * ALIGN
    host = np.full(tot, np.nan, np.float32)
    for o, s in zip(offs, seq):
        host[o:o + s.size] = s.reshape(-1)
    dev = torch.from_numpy(host).cuda()
    ptr = [dev.data_ptr() + 4 * o for o in offs]
    n = np.array(lens, np.int32)
    xs = torch.from_numpy(x0).cuda()
    try:
        rctx.set_chunk(3)
        hb = rctx.register_batch(seq[:-1], seq[1:], x0, pc)
        out = sentinel_rows(P)
        rctx.register_batch_ptrs(np.array(ptr[:-1], np.uint64), n[:-1], np.array(ptr[1:], np.uint64), n[1:],
                                 out.data_ptr() + FENCE * 224, x0_ptr=xs.data_ptr(), params=pc, device=True)
        rctx.synchronize()
        db = rows(out, P)
    finally:
        rctx.set_chunk(0)
    for k in range(P):
        for name, got in (("host", hb), ("device", db)):
            assert got[k]["X"].tobytes() == ref[k]["X"].tobytes(), (name, k)
            assert got[k]["Q"].tobytes() == ref[k]["Q"].tobytes(), (name, k)


# ---------------------------------------------------------------------------------------------------------
# 5. keyframe: scans 2 of mixed sizes
# ---------------------------------------------------------------------------------------------------------
def test_keyframe_ragged_batch(rctx, guarded, members):
    import torch
    import icet_b200
    by = {x.name: x for x in members}
    kf_cloud = by["sample_pc"].s1
    scans = [by[k].s2 for k in ("sample_pc", "tail-1", "tail-33-both", "tail-129-both", "tail-385-both", "tail65537",
                                "tail4097", "frame", "sub20011", "n2=5", "n2=0", "zero4096", "synth40")]
    P = len(scans)
    x0 = np.zeros((P, 6), np.float32)
    x0[1::2] = X0_DEG
    _, ptr = guarded
    kf = icet_b200.Keyframe(kf_cloud, ctx=rctx)
    try:
        for chunk in (0, 3):
            rctx.set_chunk(chunk)
            try:
                out = sentinel_rows(P)
                xd = torch.from_numpy(x0).cuda()
                kf.register_batch_device(np.array([ptr[id(s)] for s in scans], np.uint64), [s.shape[1] for s in scans],
                                         out.data_ptr() + FENCE * 224, xd.data_ptr())
                rctx.synchronize()
                k = rows(out, P)
            finally:
                rctx.set_chunk(0)
            for i, s in enumerate(scans):
                assert k[i].tobytes() == kf.register(s, x0[i]).tobytes(), (chunk, i, s.shape[1])
                assert k[i].tobytes() == rctx.register(kf_cloud, s, x0[i]).tobytes(), (chunk, i, s.shape[1])
    finally:
        kf.close()


# ---------------------------------------------------------------------------------------------------------
# 6. multi-GPU
# ---------------------------------------------------------------------------------------------------------
def test_multi_gpu_ragged_batch(rctx, members):
    import torch
    import icet_b200
    ndev = torch.cuda.device_count()
    ref = host_batch(rctx, members, params())
    assert_rows_equal_singles(rctx, members, ref)
    x0 = np.stack([x.x0 for x in members])
    for devs in ([0], list(range(min(ndev, 2))), list(range(ndev))):
        m = icet_b200.MultiContext(devs)
        try:
            out = m.register_batch([x.s1 for x in members], [x.s2 for x in members], x0)
        finally:
            m.close()
        for x, a, b in zip(members, out, ref):
            assert a["X"].tobytes() == b["X"].tobytes() and a["Q"].tobytes() == b["Q"].tobytes(), (devs, x.name)
            assert a["pred_stds"].tobytes() == b["pred_stds"].tobytes() and a["n_used"] == b["n_used"], (devs, x.name)


# ---------------------------------------------------------------------------------------------------------
# 7. tails, point by point
# ---------------------------------------------------------------------------------------------------------
def _ulps_to_edges(v, edges):
    v = v.astype(np.float32)
    d = np.abs(v.astype(np.float64)[:, None] - np.asarray(edges, np.float64)[None, :]).min(1)
    return d / np.spacing(np.abs(v)).astype(np.float64)


def test_tail_members_per_point(rctx, po, members):
    """For every tail member as a single pair: in every iteration the voxel counts of scan 2 are exactly the histogram of
    the per-point classes (classify_scan2); in iteration 0 (same transform on both sides) the classes equal the oracle's
    except for points within 2-3 ulp of an edge, which are listed."""
    p = params()
    nT, nP = p.bins_theta, p.bins_phi
    th_edges = (np.arange(nT + 1, dtype=np.float64) / nT) * 2 * np.pi
    ph_edges = (np.arange(nP + 1, dtype=np.float64) / nP) * np.pi
    for x in members:
        if x.kind != "tail":
            continue
        n2 = x.n2
        r, g = rctx.register(x.s1, x.s2, X0=x.x0, params=p, dump=True)
        assert r["status"] == 0 and r["n_used"] > 0, x.name
        for it in range(p.runlen):
            cell, inb = rctx.classify_scan2(it, n2)
            act = g["cnt2"][it] >= 0
            hist = np.bincount(cell, minlength=nT * nP)
            np.testing.assert_array_equal(hist[act], g["cnt2"][it][act], err_msg="%s iteration %d" % (x.name, it))
            gate = act & (g["cnt2"][it] > p.n)
            hin = np.bincount(cell[inb > 0], minlength=nT * nP)
            np.testing.assert_array_equal(hin[gate], g["nin2"][it][gate], err_msg="%s iteration %d" % (x.name, it))
            if it == 0:
                cell0, gin0 = cell, (inb > 0) & gate[cell]
        o = po.run(x.s1, x.s2, X0=x.x0, dumps="all")
        ocell, oin = o.cell2[0], o.in2[0]
        diff = np.where((cell0 != ocell) | (gin0 != (oin > 0)))[0]
        act = g["cnt2"][0] >= 0
        # each point that moved changes the counts of at most two cells by one
        assert np.abs(g["cnt2"][0] - o.cnt2[0])[act].sum() <= 2 * len(diff), x.name
        sph = o.sph2[0]
        for i in diff:
            rr, th, ph = sph[0, i], sph[1, i], sph[2, i]
            near = min(_ulps_to_edges(np.float32([th]), th_edges)[0], _ulps_to_edges(np.float32([ph]), ph_edges)[0])
            b = o.bounds[ocell[i]]
            if b[5] > 0:
                near = min(near, _ulps_to_edges(np.float32([rr]), [b[4], b[5]])[0])
            if near > 2.0 and cell0[i] == ocell[i]:
                assert (g["cnt2"][0][cell0[i]] > p.n) != (o.cnt2[0][cell0[i]] > p.n), \
                    "%s point %d: in-box differs, %.1f ulp from any edge" % (x.name, i, near)
            else:
                assert near <= 2.0, "%s point %d changed class but is %.1f ulp from an edge" % (x.name, i, near)
        assert len(diff) <= 12, (x.name, len(diff))
        print("%s: n1 %d n2 %d, %d scan-2 points differ from the oracle's class at iteration 0: %s"
              % (x.name, x.n1, n2, len(diff), diff.tolist()))
