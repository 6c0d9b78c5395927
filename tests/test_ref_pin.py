"""The oracle pinned against the REFERENCE ITSELF.

tests/golden/ref_*.npz hold the public members of the reference's own `class ICET` -- its unmodified src/icet.cpp,
src/utils.cpp, src/ThreadPool.cpp compiled by `make -C oracle ref` against oracle/eigen_shim (Eigen does not exist in
this image; see oracle/Makefile) -- written by tools/pin_against_ref.py.  The oracle restatement must reproduce them:
  * as shipped (REF_SHIPPED order): every member bit for bit;
  * with scan 1 pre-sorted by range (the reference's broken permutation loop is then a no-op, so the reference runs
    in the order its comments intend = the product's default): identical voxels / bounds / counts / Gaussians, X to
    1e-5 m / 1e-6 rad (the two sides then add the fp32 scan-2 sums in a different order).
Where the compiled reference is present (the build container, or a box that received oracle/_ref) the same
comparison also runs live.
"""
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN


def _inputs(name, g):
    from oracle import pyoracle as po
    from tools import synth_host
    if "scan1" in g:
        return g["scan1"], g["scan2"]
    base = name.split("_")[0]
    if base == "synth100":
        sc = synth_host.scans(2, first_scan=100)
        s1, s2 = sc[0], sc[1]
    else:
        d = np.load(os.path.join(GOLDEN, "inputs_%s.npz" % ("sample_pc" if name.startswith("sample_pc") else base)))
        s1, s2 = d["scan1"], d["scan2"]
    if "presorted" in name:
        s1 = po.presort_by_range(s1)
    return s1, s2


CASES = sorted(os.path.basename(f)[4:-4] for f in glob.glob(os.path.join(GOLDEN, "ref_*.npz")))


def _check(name, ref, o, shipped):
    has = ref["has1"] > 0
    np.testing.assert_array_equal(o.bounds, ref["clusterBounds"])
    np.testing.assert_array_equal(o.cnt1, ref["cnt1"])
    np.testing.assert_array_equal(o.has1, ref["has1"])
    np.testing.assert_array_equal(o.cnt2[-1], ref["cnt2"])
    assert int(has.sum()) == int(ref["n_ellipsoids"])
    np.testing.assert_array_equal(np.diagonal(ref["L"][has], axis1=1, axis2=2), o.lmask[has].astype(np.float32))
    if shipped:
        for a, b in ((o.X, ref["X"]), (o.pred_stds, ref["pred_stds"]), (o.mu1[has], ref["mu1"][has]),
                     (o.sigma1[has], ref["sigma1"][has]), (o.evec1[has].transpose(0, 2, 1), ref["U"][has]),
                     (o.HTWH[-1], ref["HTWH"]), (o.HTWdz[-1], ref["HTWdz"])):
            np.testing.assert_array_equal(a.view(np.int32), np.asarray(b, np.float32).view(np.int32))
    else:
        assert np.abs(o.X[:3] - ref["X"][:3]).max() < 1e-5 and np.abs(o.X[3:] - ref["X"][3:]).max() < 1e-6
        np.testing.assert_allclose(o.pred_stds, ref["pred_stds"], rtol=2e-3)
        assert np.abs(o.mu1[has] - ref["mu1"][has]).max() < 1e-5
        sg = np.abs(o.sigma1[has] - ref["sigma1"][has]).reshape(-1, 9).max(1) / np.abs(ref["sigma1"][has]).reshape(-1, 9).max(1)
        assert sg.max() < 1e-5


@pytest.mark.parametrize("name", CASES)
def test_oracle_reproduces_reference_golden(po, name):
    g = np.load(os.path.join(GOLDEN, "ref_%s.npz" % name))
    s1, s2 = _inputs(name, g)
    rl, nphi, nth = (int(v) for v in g["params"])
    mode = int(g["order_mode"])
    ntb = g["n_thresh_buff"] if "n_thresh_buff" in g else (25, 0.1, 0.1)
    o = po.run(s1, s2, X0=g["x0"], dumps="small", order_mode=mode, runlen=rl, bins_phi=nphi, bins_theta=nth,
               n=int(ntb[0]), thresh=float(ntb[1]), buff=float(ntb[2]))
    _check(name, g, o, shipped=(mode == po.ORDER_REF_SHIPPED))


def test_reference_test_points(po):
    """public member testPoints (src/icet.cpp:214-232): rows 6*cell+2k, +1 = mu1 +- 2 sqrt(lambda_k) * U.row(k) for every
    axis k the reference found extended (L(k,k) = 0; `rotated = axislen * U^T` makes that V.row(k), SURVEY.md A.8) --
    reproduced from the oracle's mu1 / eigenpairs."""
    g = np.load(os.path.join(GOLDEN, "ref_frame_shipped.npz"))
    d = np.load(os.path.join(GOLDEN, "inputs_frame.npz"))
    o = po.run(d["scan1"], d["scan2"], dumps="small", order_mode=po.ORDER_REF_SHIPPED)
    tp = g["testPoints"].reshape(-1, 6, 3)
    n = 0
    for c in np.where(o.has1 > 0)[0]:
        for k in range(3):
            if o.lmask[c, k]:
                continue
            rot = np.float32(2.0) * np.sqrt(o.eval1[c, k]) * o.evec1[c][k, :]      # axislen * U^T = diag * V: ROW k of V
            np.testing.assert_allclose(tp[c, 2 * k], o.mu1[c] + rot, rtol=0, atol=1e-5)
            np.testing.assert_allclose(tp[c, 2 * k + 1], o.mu1[c] - rot, rtol=0, atol=1e-5)
            n += 1
    assert n > 20


def test_live_reference_build_matches_oracle(po):
    """Where the compiled reference is available, rerun it instead of trusting the stored vectors."""
    from oracle import pyref
    if not pyref.available():
        pytest.skip("neither /root/reference nor a prebuilt oracle/_ref/libicet_ref.so")
    d = np.load(os.path.join(GOLDEN, "inputs_frame.npz"))
    for x0 in (None, [1, 0, 0, 0, 0, 0], [-0.3, 0.2, 0.0, 0.01, 0.0, -0.02]):
        ref = pyref.run(d["scan1"], d["scan2"], X0=x0)
        o = po.run(d["scan1"], d["scan2"], X0=x0, dumps="small", order_mode=po.ORDER_REF_SHIPPED)
        _check("live", ref, o, shipped=True)
    s1 = po.presort_by_range(d["scan1"])
    for kw in (dict(), dict(n=40, thresh=0.3, buff=0.5), dict(runlen=3, bins_phi=12, bins_theta=40)):
        ref = pyref.run(s1, d["scan2"], **kw)
        o = po.run(s1, d["scan2"], dumps="small", **kw)
        _check("live_presorted", ref, o, shipped=False)
