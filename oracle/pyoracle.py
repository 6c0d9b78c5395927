"""ctypes binding of the CPU oracle (oracle/icet_oracle.cpp).

TEST INFRASTRUCTURE ONLY: import this from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / reference arm -- never from the icet_b200 package.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORDER_SORTED, ORDER_REF_SHIPPED = 0, 1
EIGEN_337, EIGEN_340 = 0, 1


class _Params(C.Structure):
    _fields_ = [("runlen", C.c_int32), ("bins_phi", C.c_int32), ("bins_theta", C.c_int32),
                ("n", C.c_int32), ("thresh", C.c_float), ("buff", C.c_float),
                ("order_mode", C.c_int32), ("eigen_flavor", C.c_int32), ("precise", C.c_int32),
                ("stats2_mode", C.c_int32)]


_FP, _IP, _BP = C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_uint8)
# (name, ctype, numpy dtype, shape builder)
_DUMPS = [
    ("sph1", _FP, np.float32, lambda d: (3, d["n1"])),
    ("cell1", _IP, np.int32, lambda d: (d["n1"],)),
    ("cnt1", _IP, np.int32, lambda d: (d["ncell"],)),
    ("bounds", _FP, np.float32, lambda d: (d["ncell"], 6)),
    ("nin1", _IP, np.int32, lambda d: (d["ncell"],)),
    ("has1", _BP, np.uint8, lambda d: (d["ncell"],)),
    ("mu1", _FP, np.float32, lambda d: (d["ncell"], 3)),
    ("sigma1", _FP, np.float32, lambda d: (d["ncell"], 3, 3)),
    ("eval1", _FP, np.float32, lambda d: (d["ncell"], 3)),
    ("evec1", _FP, np.float32, lambda d: (d["ncell"], 3, 3)),
    ("lmask", _BP, np.uint8, lambda d: (d["ncell"], 3)),
    ("sph2", _FP, np.float32, lambda d: (d["rl"], 3, d["n2"])),
    ("cell2", _IP, np.int32, lambda d: (d["rl"], d["n2"])),
    ("cnt2", _IP, np.int32, lambda d: (d["rl"], d["ncell"])),
    ("nin2", _IP, np.int32, lambda d: (d["rl"], d["ncell"])),
    ("used2", _BP, np.uint8, lambda d: (d["rl"], d["ncell"])),
    ("mu2", _FP, np.float32, lambda d: (d["rl"], d["ncell"], 3)),
    ("sigma2", _FP, np.float32, lambda d: (d["rl"], d["ncell"], 3, 3)),
    ("HTWH", _FP, np.float32, lambda d: (d["rl"], 6, 6)),
    ("HTWdz", _FP, np.float32, lambda d: (d["rl"], 6)),
    ("dx", _FP, np.float32, lambda d: (d["rl"], 6)),
    ("Xit", _FP, np.float32, lambda d: (d["rl"], 6)),
    ("Qit", _FP, np.float32, lambda d: (d["rl"], 6, 6)),
    ("stds_it", _FP, np.float32, lambda d: (d["rl"], 6)),
    ("cond_it", _FP, np.float32, lambda d: (d["rl"],)),
    ("trunc_it", _IP, np.int32, lambda d: (d["rl"],)),
    ("in2", _BP, np.uint8, lambda d: (d["rl"], d["n2"])),
    ("points2_final", _FP, np.float32, lambda d: (3, d["n2"])),
    ("perm2", _IP, np.int32, lambda d: (d["n2"],)),
]
_BIG = {"sph1", "cell1", "sph2", "cell2", "in2", "points2_final", "perm2"}
STATS2_REFERENCE, STATS2_MOMENTS = 0, 1


class _Out(C.Structure):
    _fields_ = ([("X", C.c_float * 6), ("pred_stds", C.c_float * 6), ("Q", C.c_float * 36),
                 ("status", C.c_int32)] + [(n, t) for n, t, _, _ in _DUMPS] +
                [("evec1_in", _FP), ("evec1_in_mask", _BP), ("X_in", _FP)])


def _build() -> str:
    """Compile the oracle if the .so is missing or older than its sources."""
    out = os.path.join(_HERE, "_build")
    target = os.path.join(out, "libicet_oracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("icet_oracle.cpp", "icet_oracle.h", "eigen_algos.h", "Makefile")]
    if (not os.path.exists(target)) or os.path.getmtime(target) < max(map(os.path.getmtime, srcs)):
        subprocess.run(["make", "-C", _HERE, "all", "OUT=" + out], check=True,
                       stdout=subprocess.DEVNULL)
    return target


def _load_native() -> C.CDLL:
    """-march=native code must be built on the machine that runs it, so it is built at run time, once per process, in
    a private temporary directory: the source tree is never written (it may be read-only) and no other build is
    ever picked up.  The library stays mapped after the directory is removed."""
    with tempfile.TemporaryDirectory(prefix="icet_oracle_native-") as out:
        subprocess.run(["make", "-C", _HERE, "native", "OUT=" + out], check=True, stdout=subprocess.DEVNULL)
        return C.CDLL(os.path.join(out, "libicet_oracle_native.so"))


_LIBS: dict = {}


def lib(native: bool = False) -> C.CDLL:
    if native not in _LIBS:
        L = _load_native() if native else C.CDLL(_build())
        L.icet_oracle_run.restype = C.c_int
        L.icet_oracle_run.argtypes = [C.POINTER(_Params), _FP, C.c_int32, C.c_int32, _FP, C.c_int32,
                                      C.c_int32, _FP, C.POINTER(_Out)]
        L.icet_oracle_run_sequence.restype = C.c_double
        L.icet_oracle_run_sequence.argtypes = [C.POINTER(_Params), _FP, C.c_int32, C.c_int32,
                                               C.c_int32, _FP]
        L.icet_oracle_eig3.argtypes = [_FP, C.c_int32, _FP, _FP]
        L.icet_oracle_eigsym.argtypes = [_FP, C.c_int32, C.c_int32, _FP, _FP]
        L.icet_oracle_pinv.argtypes = [_FP, C.c_int32, C.c_int32, _FP, _IP]
        L.icet_oracle_c2s.argtypes = [_FP, C.c_int32, C.c_int32, _FP]
        L.icet_oracle_bins.argtypes = [_FP, C.c_int32, C.c_int32, C.c_int32, _IP]
        _LIBS[native] = L
    return _LIBS[native]


def _fp(a):
    return a.ctypes.data_as(_FP)


def as_planes(cloud) -> np.ndarray:
    """N x 3 (any dtype / order) -> float32 [3, N] planes (x | y | z), i.e. the memory of a
    column-major Eigen::MatrixXf(N, 3)."""
    a = np.asarray(cloud)
    if a.ndim != 2:
        raise ValueError("cloud must be 2-D")
    if a.shape[1] == 3 and a.shape[0] != 3:
        a = a.T
    elif a.shape[0] != 3:
        raise ValueError("cloud must be N x 3 or 3 x N")
    return np.ascontiguousarray(a, dtype=np.float32)


@dataclass
class OracleResult:
    X: np.ndarray
    pred_stds: np.ndarray
    Q: np.ndarray
    status: int
    dumps: dict = field(default_factory=dict)

    def __getattr__(self, k):
        d = self.__dict__.get("dumps", {})
        if k in d:
            return d[k]
        raise AttributeError(k)


def run(scan1, scan2, runlen=7, X0=None, bins_phi=24, bins_theta=75, n=25, thresh=0.1, buff=0.1,
        order_mode=ORDER_SORTED, eigen_flavor=EIGEN_337, precise=False, dumps="small",
        native=False, evec_override=None, stats2_mode=STATS2_REFERENCE, X_iterates=None) -> OracleResult:
    """Mirror of the reference constructor  ICET(scan1, scan2, runlen, X0, num_bins_phi,
    num_bins_theta, n, thresh, buff)  (include/icet.h:38-40).  dumps: None | "small" | "all"."""
    s1, s2 = as_planes(scan1), as_planes(scan2)
    n1, n2 = s1.shape[1], s2.shape[1]
    x0 = np.zeros(6, np.float32) if X0 is None else np.ascontiguousarray(X0, np.float32)
    p = _Params(runlen, bins_phi, bins_theta, n, thresh, buff, order_mode, eigen_flavor,
                1 if precise else 0, stats2_mode)
    o = _Out()
    dims = dict(n1=n1, n2=n2, ncell=bins_phi * bins_theta, rl=runlen)
    arrays = {}
    for name, ct, dt, shp in _DUMPS:
        if dumps is None or (dumps == "small" and name in _BIG):
            continue
        arrays[name] = np.zeros(shp(dims), dt)
        setattr(o, name, arrays[name].ctypes.data_as(ct))
    if evec_override is not None:  # (evec [ncell,3,3] float32, mask [ncell] uint8): see icet_oracle.h
        ev_in = np.ascontiguousarray(evec_override[0], np.float32)
        ev_mask = np.ascontiguousarray(evec_override[1], np.uint8)
        assert ev_in.size == 9 * dims["ncell"] and ev_mask.size == dims["ncell"]
        o.evec1_in = ev_in.ctypes.data_as(_FP)
        o.evec1_in_mask = ev_mask.ctypes.data_as(_BP)
    if X_iterates is not None:  # [runlen, 6]: the X every iteration starts from (iterate alignment, see icet_oracle.h)
        x_in = np.ascontiguousarray(X_iterates, np.float32)
        assert x_in.shape == (runlen, 6)
        o.X_in = x_in.ctypes.data_as(_FP)
    rc = lib(native).icet_oracle_run(C.byref(p), _fp(s1), n1, n1, _fp(s2), n2, n2, _fp(x0),
                                     C.byref(o))
    if rc != 0:
        raise RuntimeError("icet_oracle_run failed: %d" % rc)
    return OracleResult(np.array(o.X[:], np.float32), np.array(o.pred_stds[:], np.float32),
                        np.array(o.Q[:], np.float32).reshape(6, 6), int(o.status), arrays)


def run_sequence(scans: np.ndarray, nthreads=1, native=True, **kw):
    """scans: float32 [K+1, 3, N].  Registers the K consecutive pairs with X0 = 0 on `nthreads`
    host threads.  Returns (results [K, 48], elapsed seconds)."""
    scans = np.ascontiguousarray(scans, np.float32)
    k1, three, n = scans.shape
    assert three == 3 and k1 >= 2
    p = _Params(kw.get("runlen", 7), kw.get("bins_phi", 24), kw.get("bins_theta", 75),
                kw.get("n", 25), kw.get("thresh", 0.1), kw.get("buff", 0.1),
                kw.get("order_mode", ORDER_SORTED), kw.get("eigen_flavor", EIGEN_337), 0,
                kw.get("stats2_mode", STATS2_REFERENCE))
    res = np.zeros((k1 - 1, 48), np.float32)
    dt = lib(native).icet_oracle_run_sequence(C.byref(p), _fp(scans), n, k1 - 1, nthreads, _fp(res))
    return res, float(dt)


def eig3(a, flavor=EIGEN_337):
    a = np.ascontiguousarray(a, np.float32).reshape(9)
    ev, V = np.zeros(3, np.float32), np.zeros(9, np.float32)
    lib().icet_oracle_eig3(_fp(a), flavor, _fp(ev), _fp(V))
    return ev, V.reshape(3, 3)


def eigsym(a, flavor=EIGEN_337):
    a = np.ascontiguousarray(a, np.float32)
    n = a.shape[0]
    ev, V = np.zeros(n, np.float32), np.zeros(n * n, np.float32)
    lib().icet_oracle_eigsym(_fp(a.reshape(-1)), n, flavor, _fp(ev), _fp(V))
    return ev, V.reshape(n, n)


def pinv(a):
    a = np.ascontiguousarray(a, np.float32)
    r, c = a.shape
    out, rank = np.zeros(r * c, np.float32), C.c_int32(0)
    lib().icet_oracle_pinv(_fp(a.reshape(-1)), r, c, _fp(out), C.byref(rank))
    return out.reshape(c, r), rank.value


def c2s(planes):
    s = as_planes(planes)
    out = np.zeros_like(s)
    lib().icet_oracle_c2s(_fp(s), s.shape[1], s.shape[1], _fp(out))
    return out


def bins(sph, bins_phi=24, bins_theta=75):
    sph = np.ascontiguousarray(sph, np.float32)
    out = np.zeros(sph.shape[1], np.int32)
    lib().icet_oracle_bins(_fp(sph), sph.shape[1], bins_phi, bins_theta,
                           out.ctypes.data_as(_IP))
    return out


def presort_by_range(scan):
    """Rows of a [3, N] cloud in ascending fp32 range order (stable), the range computed like the reference does
    (src/utils.cpp:98).  On such a scan 1 the reference's radial permutation loop (src/icet.cpp:72-83) is a no-op up
    to rows of equal range, i.e. the reference itself runs in the order its comments intend."""
    s = as_planes(scan)
    return np.ascontiguousarray(s[:, np.argsort(c2s(s)[0], kind="stable")])
