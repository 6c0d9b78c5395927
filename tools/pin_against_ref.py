#!/usr/bin/env python
"""Pin the CPU oracle against the REFERENCE ITSELF (run in the build container, where /root/reference exists).

    python tools/pin_against_ref.py [--eigen-include /usr/include/eigen3] [--write]

1. builds oracle/_ref/libicet_ref.so from the reference's unmodified sources (`make -C oracle ref`; against
   oracle/eigen_shim unless a real Eigen tree is given);
2. runs it on the bundled pairs (as shipped: X0 = 0 and the demo's X0; and with scan 1 pre-sorted by range, which
   makes the reference's broken permutation loop a no-op and so exercises the order its comments intend), on a
   synthetic 64-channel pair and on edge cases;
3. diffs every public member against the oracle restatement (REF_SHIPPED mode / SORTED mode) -- bit for bit;
4. --write: stores the reference's outputs as tests/golden/ref_*.npz, which tests/test_ref_pin.py asserts against on
   any machine (the reference sources do not travel).
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po  # noqa: E402
from oracle import pyref  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
KEYS = ["X", "pred_stds", "clusterBounds", "cnt1", "cnt2", "has1", "mu1", "sigma1", "U", "L", "HTWH", "HTWdz", "testPoints"]


presort = po.presort_by_range


def cases():
    from tools import synth_host
    out = []
    for name in ("frame", "sample_pc"):
        d = np.load(os.path.join(GOLDEN, "inputs_%s.npz" % name))
        s1, s2 = d["scan1"], d["scan2"]
        out.append((name + "_shipped", s1, s2, None, po.ORDER_REF_SHIPPED, {}))
        out.append((name + "_presorted", presort(s1), s2, None, po.ORDER_SORTED, {}))
    d = np.load(os.path.join(GOLDEN, "inputs_frame.npz"))
    out.append(("frame_shipped_x0demo", d["scan1"], d["scan2"], [1, 0, 0, 0, 0, 0], po.ORDER_REF_SHIPPED, {}))
    # the other settings test_live_reference_build_matches_oracle reruns the reference with
    out.append(("frame_shipped_x0tilt", d["scan1"], d["scan2"], [-0.3, 0.2, 0.0, 0.01, 0.0, -0.02], po.ORDER_REF_SHIPPED,
                {}))
    out.append(("frame_presorted_loose", presort(d["scan1"]), d["scan2"], None, po.ORDER_SORTED,
                dict(n=40, thresh=0.3, buff=0.5)))
    out.append(("frame_presorted_coarse", presort(d["scan1"]), d["scan2"], None, po.ORDER_SORTED,
                dict(runlen=3, bins_phi=12, bins_theta=40)))
    sc = synth_host.scans(2, first_scan=100)
    out.append(("synth100_shipped", sc[0], sc[1], None, po.ORDER_REF_SHIPPED, {}))
    out.append(("synth100_presorted", presort(sc[0]), sc[1], None, po.ORDER_SORTED, {}))
    out.append(("synth100_presorted_fine", presort(sc[0]), sc[1], None, po.ORDER_SORTED,
                dict(runlen=10, bins_phi=48, bins_theta=150)))
    rng = np.random.default_rng(11)   # the corridor of test_truncated_solution_axis: checkCondition drops an axis
    n = 60000
    x = rng.uniform(-30, 30, n)
    side = rng.integers(0, 3, n)
    y = np.where(side == 0, -4.0, np.where(side == 1, 4.0, rng.uniform(-4, 4, n)))
    zc = np.where(side == 2, -1.5, rng.uniform(-1.5, 2.0, n))
    c1 = np.stack([x, y + 0.005 * rng.standard_normal(n), zc + 0.005 * rng.standard_normal(n)]).astype(np.float32)
    c2 = c1.copy()
    c2[1] += 0.05
    c2 += (0.005 * rng.standard_normal(c2.shape)).astype(np.float32)
    out.append(("corridor_presorted", presort(c1), c2, None, po.ORDER_SORTED, {}))
    z = np.zeros((3, 4096), np.float32)
    out.append(("all_zero", z, z, [0.1, 0, 0, 0, 0, 0.01], po.ORDER_REF_SHIPPED, {}))
    return out


def compare(name, ref, o, order_mode):
    """max deviations of the oracle from the reference build, member by member"""
    has = ref["has1"] > 0
    rep = {
        "X_bits_equal": bool(np.array_equal(ref["X"].view(np.int32), o.X.view(np.int32))),
        "dX": float(np.abs(ref["X"] - o.X).max()),
        "dstds": float(np.abs(ref["pred_stds"] - o.pred_stds).max()),
        "bounds_equal": bool(np.array_equal(ref["clusterBounds"], o.bounds)),
        "cnt1_equal": bool(np.array_equal(ref["cnt1"], o.cnt1)),
        "cnt2_last_equal": bool(np.array_equal(ref["cnt2"], o.cnt2[-1])),
        "has1_equal": bool(np.array_equal(ref["has1"], o.has1)),
        "gaussians": int(has.sum()),
        "dmu1": float(np.abs(ref["mu1"][has] - o.mu1[has]).max()) if has.any() else 0.0,
        "dsigma1_rel": float((np.abs(ref["sigma1"][has] - o.sigma1[has]).reshape(-1, 9).max(1) /
                              np.abs(ref["sigma1"][has]).reshape(-1, 9).max(1)).max()) if has.any() else 0.0,
        "U_equal": bool(np.array_equal(ref["U"][has], o.evec1[has].transpose(0, 2, 1))),
        "L_equal": bool(np.array_equal(np.diagonal(ref["L"][has], axis1=1, axis2=2), o.lmask[has].astype(np.float32))),
        "dHTWH_rel": float(np.abs(ref["HTWH"] - o.HTWH[-1]).max() / max(np.abs(ref["HTWH"]).max(), 1e-30)),
    }
    print("%-26s X bits equal %-5s |dX| %.1e  bounds/cnt1/cnt2/has1 equal %s  gaussians %d  U/L equal %s %s  |dmu1| %.1e "
          "|dS1| %.1e |dHTWH| %.1e" % (name, rep["X_bits_equal"], rep["dX"],
                                      (rep["bounds_equal"], rep["cnt1_equal"], rep["cnt2_last_equal"], rep["has1_equal"]),
                                      rep["gaussians"], rep["U_equal"], rep["L_equal"], rep["dmu1"], rep["dsigma1_rel"],
                                      rep["dHTWH_rel"]))
    return rep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--eigen-include", default=None, help="a real Eigen 3 include directory (default: oracle/eigen_shim)")
    ap.add_argument("--write", action="store_true", help="store the reference's outputs under tests/golden/ref_*.npz")
    a = ap.parse_args()
    pyref.build(eigen_include=a.eigen_include)
    ok = True
    for name, s1, s2, x0, mode, kw in cases():
        ref = pyref.run(s1, s2, X0=x0, **kw)
        o = po.run(s1, s2, X0=x0, dumps="small", order_mode=mode, **kw)
        rep = compare(name, ref, o, mode)
        ok &= rep["bounds_equal"] and rep["cnt1_equal"] and rep["has1_equal"] and rep["dX"] < 1e-6
        if a.write:
            extra = dict(scan1=s1, scan2=s2) if name.startswith(("corridor", "all_zero")) else {}
            np.savez_compressed(os.path.join(GOLDEN, "ref_%s.npz" % name),
                                x0=np.zeros(6, np.float32) if x0 is None else np.float32(x0), order_mode=mode,
                                eigen="shim" if a.eigen_include is None else a.eigen_include,
                                params=np.int32([kw.get("runlen", 7), kw.get("bins_phi", 24), kw.get("bins_theta", 75)]),
                                n_thresh_buff=np.float32([kw.get("n", 25), kw.get("thresh", 0.1), kw.get("buff", 0.1)]),
                                n_ellipsoids=ref["n_ellipsoids"], **{k: ref[k] for k in KEYS}, **extra)
    print("oracle == reference build:", "YES" if ok else "NO")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
