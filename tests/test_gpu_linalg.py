"""The dense linear algebra of the Gauss-Newton loop against plain float64 references, at its branch edges.

tests/linalg_harness.cu includes the library's translation unit and adds test kernels around its own device routines:
  * icet::eig3f (the fp32 port of Eigen 3.3.7's 3x3 solver): bit for bit against the oracle's eig3;
  * W = pinv(M) of vox_algebra_core: the closed form masked_inv3, else the COD (icet::cod_pinv);
  * icet::cod_pinv for shapes up to 6x6, and icet::jacobi6;
  * the 6x6 solve as the split loop runs it (k_solve6) and as the cluster loop runs it (solve_pair_warp, then
    solve_pair on one lane when the warp form declines): against a float64 restatement of src/icet.cpp:410-492, and
    against each other byte for byte;
  * vox_algebra_core against a float64 restatement of src/icet.cpp:308-338.
The harness is compiled with the library's own nvcc flags (-fmad=false included) into a temporary directory.
"""
from __future__ import annotations

import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "tests", "linalg_harness.cu")
FLT_EPS = float(np.finfo(np.float32).eps)
FLT_MIN = float(np.finfo(np.float32).tiny)
FLAG_FULL_EIG = 1
COND_CUTOFF = 1e6        # checkCondition, src/icet.cpp:469
TRACE_BOUND = 0.999e6    # the fast 6x6 path: trace(A) * trace(A^-1) below this proves cond <= 1e6
_P = C.c_void_p


def compile_harness(out_dir: str) -> str:
    b = importlib.import_module("icet_b200.build")
    assert "-fmad=false" in b.NVCC_FLAGS  # the bit-identity checks below mean nothing with contraction
    so = os.path.join(out_dir, "liblinalg_harness.so")
    r = subprocess.run([b.nvcc_path()] + list(b.NVCC_FLAGS) + ["-o", so, HARNESS], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed on the linear-algebra harness:\n" + r.stdout + r.stderr)
    return so


def test_harness_compiles_for_sm100a(tmp_path):
    """The harness builds against the library's source with the library's flags (no GPU needed)."""
    so = compile_harness(str(tmp_path))
    cuobjdump = os.path.join(os.path.dirname(importlib.import_module("icet_b200.build").nvcc_path()), "cuobjdump")
    if os.path.exists(cuobjdump):
        out = subprocess.run([cuobjdump, "-lelf", so], capture_output=True, text=True).stdout
        assert "sm_100a" in out
    names = subprocess.run(["nm", "-D", so], capture_output=True, text=True).stdout
    for sym in ("lh_eig3", "lh_wpinv", "lh_cod", "lh_jacobi", "lh_solve_split", "lh_solve_cluster", "lh_vox"):
        assert sym in names


# ------------------------------------------------------------------------------------------------ harness binding
VOX1_DTYPE = np.dtype([("mu", np.float64, 3), ("S1n", np.float64, 6), ("LV", np.float64, 9), ("lmask", np.int32),
                       ("pad", np.int32)])


class Harness:
    def __init__(self, so: str):
        from icet_b200 import api
        self.L = L = C.CDLL(so)
        for name in ("lh_eig3", "lh_wpinv", "lh_cod", "lh_jacobi", "lh_solve_split", "lh_solve_cluster", "lh_vox"):
            getattr(L, name).restype = C.c_int
        L.lh_eig3.argtypes = [_P, C.c_int, _P, _P]
        L.lh_wpinv.argtypes = [_P, _P, C.c_int, _P, _P]
        L.lh_cod.argtypes = [_P, C.c_int, C.c_int, C.c_int, _P, _P]
        L.lh_jacobi.argtypes = [_P, C.c_int, _P, _P]
        L.lh_solve_split.argtypes = L.lh_solve_cluster.argtypes = [_P, _P, C.c_int, C.c_int, _P, _P, _P]
        L.lh_vox.argtypes = [_P, _P, _P, _P, _P, C.c_int, _P]
        assert L.lh_result_size() == api.RESULT_DTYPE.itemsize
        assert L.lh_vox1_size() == VOX1_DTYPE.itemsize
        self.result_dtype = api.RESULT_DTYPE

    @staticmethod
    def _ok(rc):
        assert rc == 0, "CUDA error %d in the harness" % rc

    def eig3(self, A):
        A = np.ascontiguousarray(A, np.float32).reshape(-1, 9)
        n = len(A)
        ev, V = np.zeros((n, 3), np.float32), np.zeros((n, 9), np.float32)
        self._ok(self.L.lh_eig3(A.ctypes.data, n, ev.ctypes.data, V.ctypes.data))
        return ev, V.reshape(n, 3, 3)

    def wpinv(self, M, masks):
        M = np.ascontiguousarray(M, np.float64).reshape(-1, 9)
        masks = np.ascontiguousarray(masks, np.int32)
        n = len(M)
        W, br = np.zeros((n, 9)), np.zeros(n, np.int32)
        self._ok(self.L.lh_wpinv(M.ctypes.data, masks.ctypes.data, n, W.ctypes.data, br.ctypes.data))
        return W.reshape(n, 3, 3), br

    def cod(self, A):
        A = np.asarray(A, np.float64)
        n, r, c = A.shape
        buf = np.zeros((n, 36))
        buf[:, : r * c] = A.reshape(n, r * c)
        P, rank = np.zeros((n, 36)), np.zeros(n, np.int32)
        self._ok(self.L.lh_cod(buf.ctypes.data, r, c, n, P.ctypes.data, rank.ctypes.data))
        return P[:, : r * c].reshape(n, c, r), rank

    def jacobi(self, A):
        A = np.ascontiguousarray(A, np.float64).reshape(-1, 36)
        n = len(A)
        ev, U = np.zeros((n, 6)), np.zeros((n, 36))
        self._ok(self.L.lh_jacobi(A.ctypes.data, n, ev.ctypes.data, U.ctypes.data))
        return ev, U.reshape(n, 6, 6)

    def solve(self, cluster: bool, tot, X, flags):
        tot = np.ascontiguousarray(tot, np.float64)
        X = np.ascontiguousarray(X, np.float32)
        n = len(tot)
        res = np.zeros(n, self.result_dtype)
        TR, J = np.zeros((n, 12), np.float32), np.zeros((n, 27), np.float32)
        f = self.L.lh_solve_cluster if cluster else self.L.lh_solve_split
        self._ok(f(tot.ctypes.data, X.ctypes.data, flags, n, res.ctypes.data, TR.ctypes.data, J.ctypes.data))
        return res, TR, J

    def vox(self, vox, mean, cov, nbin, Jm):
        vox = np.ascontiguousarray(vox, VOX1_DTYPE)
        mean, cov = np.ascontiguousarray(mean, np.float64), np.ascontiguousarray(cov, np.float64)
        nbin, Jm = np.ascontiguousarray(nbin, np.int64), np.ascontiguousarray(Jm, np.float32)
        n = len(vox)
        acc = np.zeros((n, 28))
        self._ok(self.L.lh_vox(vox.ctypes.data, mean.ctypes.data, cov.ctypes.data, nbin.ctypes.data, Jm.ctypes.data, n,
                               acc.ctypes.data))
        return acc


@pytest.fixture(scope="session")
def lh(tmp_path_factory):
    return Harness(compile_harness(str(tmp_path_factory.mktemp("linalg_harness"))))


# ------------------------------------------------------------------------------------------------ case generators
def rotation(rng, n):
    q, r = np.linalg.qr(rng.standard_normal((n, n)))
    return q * np.sign(np.diag(r))


def spd(rng, evals):
    Q = rotation(rng, len(evals))
    A = (Q * np.asarray(evals, np.float64)) @ Q.T
    return 0.5 * (A + A.T)


def geometric(kappa, n):
    return np.geomspace(1.0, 1.0 / kappa, n)


def trace_product_spectrum(target, n):
    """Eigenvalues [1]*(n-1) + [x] with (sum lam)(sum 1/lam) == target."""
    k = n - 1
    p = k * k + 1 - target
    x = (-p + np.sqrt(p * p - 4 * k * k)) / (2 * k)
    return np.array([1.0] * k + [x])


def near(values, rels=(1e-3, 1e-9)):
    out = []
    for v in values:
        for r in rels:
            out += [v * (1 - r), v * (1 + r)]
    return out


def bits_equal_nan(a, b):
    """Bit identity of float arrays; NaN only has to be NaN on both sides (payloads differ between CPU and GPU)."""
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    if not np.array_equal(na, nb):
        return False
    ia = a.view(np.uint32 if a.dtype == np.float32 else np.uint64)
    ib = b.view(np.uint32 if b.dtype == np.float32 else np.uint64)
    return bool(np.array_equal(ia[~na], ib[~nb]))


# ------------------------------------------------------------------------------------------------ eig3f
def eig3_cases(rng):
    cases, kinds = [], []

    def add(kind, A):
        A = np.asarray(A, np.float64)
        cases.append(np.tril(A) + np.tril(A, -1).T)  # eig3f reads the lower triangle
        kinds.append(kind)

    for kappa in 10.0 ** np.arange(0, 15):
        for _ in range(12):
            add("spd", spd(rng, geometric(kappa, 3) * 10 ** rng.uniform(-3, 3)))
    for _ in range(40):
        add("repeated2", spd(rng, [2.0, 2.0, 0.5]))
        add("repeated2", spd(rng, [3.0, 1e-3, 1e-3]))
        add("repeated3", spd(rng, [1.5, 1.5, 1.5]))
    for rank in range(3):
        for noise in (0.0, 1e-7):
            for _ in range(20):
                A = spd(rng, np.r_[rng.uniform(0.5, 2.0, rank), np.zeros(3 - rank)])
                add("rank%d" % rank, A + noise * rng.standard_normal((3, 3)))
    for _ in range(20):
        d = rng.uniform(-2, 2, 3)
        add("diagonal", np.diag(d))
        P = np.eye(3)[rng.permutation(3)]
        add("permuted_diagonal", P @ np.diag(d) @ P.T)
        add("indefinite", spd(rng, [rng.uniform(0.1, 2), -rng.uniform(0.1, 2), rng.uniform(-1, 1)]))
    # the v1norm2 <= FLT_MIN branch of the tridiagonalisation: |m20| / scale around sqrt(FLT_MIN)
    edge = np.sqrt(FLT_MIN)
    for m20 in [0.0, edge * 0.5, edge * (1 - 1e-6), edge, edge * (1 + 1e-6), edge * 2, 1e-19, 1e-25, 1e-30]:
        for sgn in (1, -1):
            A = spd(rng, [1.0, 0.6, 0.3])
            A[2, 0] = A[0, 2] = sgn * m20 * np.abs(A).max()
            add("flt_min_m20", A)
    # scales, FLT_MIN and subnormal entries
    for s in [1e-30, 1e-20, 1e-10, 1e10, 1e20, 1e30, 3e38]:
        for _ in range(6):
            add("scale", spd(rng, [1.0, 0.3, 0.01]) * s)
    for s in [FLT_MIN, FLT_MIN * 4, 1e-39, 1e-42, 1.4e-45]:
        for _ in range(6):
            add("subnormal", spd(rng, [1.0, 0.5, 0.25]) * s)
            A = spd(rng, [1.0, 0.5, 0.25])
            A[2, 0] = A[0, 2] = s
            A[1, 0] = A[0, 1] = s
            add("subnormal_offdiag", A)
    # non-finite entries at every position of the lower triangle
    for pos in [(0, 0), (1, 0), (1, 1), (2, 0), (2, 1), (2, 2)]:
        for v in (np.nan, np.inf, -np.inf):
            A = spd(rng, [1.0, 0.5, 0.2])
            A[pos] = A[pos[::-1]] = v
            add("nonfinite", A)
    add("nonfinite", np.full((3, 3), np.nan))
    add("zero", np.zeros((3, 3)))
    return np.array(cases, np.float32), kinds


@pytest.mark.gpu
def test_eig3f_bit_identical_to_oracle(lh, po):
    """eig3f is an operation-for-operation port of the oracle's Eigen 3.3.7 restatement (DESIGN.md 3.8): same
    eigenvalues and eigenvectors, bit for bit, on every branch -- including NaN / inf input, which must not hang."""
    rng = np.random.default_rng(3801)
    A, kinds = eig3_cases(rng)
    ev, V = lh.eig3(A)
    bad = []
    for i in range(len(A)):
        oev, oV = po.eig3(A[i])
        if not (bits_equal_nan(ev[i], oev) and bits_equal_nan(V[i], oV)):
            bad.append((kinds[i], A[i].tolist(), ev[i].tolist(), oev.tolist()))
    counts = {k: kinds.count(k) for k in sorted(set(kinds))}
    print("eig3f cases:", counts)
    assert not bad, "%d of %d cases differ from the oracle, first: %r" % (len(bad), len(A), bad[:3])


# ------------------------------------------------------------------------------------------------ W = pinv(M)
def svd_pinv(A, rank):
    U, s, Vt = np.linalg.svd(A)
    P = np.zeros((A.shape[1], A.shape[0]))
    for k in range(rank):
        P += np.outer(Vt[k], U[:, k]) / s[k]
    return P, s


def truncate(A, rank):
    U, s, Vt = np.linalg.svd(A)
    return (U[:, :rank] * s[:rank]) @ Vt[:rank]


def check_pinv(A, W, rank, what):
    """W against the pseudo-inverse with the cut at `rank`, and the four Penrose conditions of the truncated A.
    Tolerance: rounding amplified by the kept condition number, plus what a QR-based cut may leave of the dropped
    singular values."""
    P, s = svd_pinv(A, rank)
    if rank == 0:
        assert np.all(W == 0), what
        return
    kap = s[0] / s[rank - 1]
    tail = s[rank] / s[rank - 1] if rank < len(s) else 0.0
    tol = 1e-12 * kap + 10 * tail
    nW = np.abs(P).max()
    assert np.abs(W - P).max() <= tol * nW, "%s: |W - pinv| = %.3e of %.3e (tol %.1e)" % (
        what, np.abs(W - P).max(), nW, tol)
    Ar = truncate(A, rank)
    nA = np.abs(Ar).max()
    assert np.abs(Ar @ W @ Ar - Ar).max() <= tol * nA, what
    assert np.abs(W @ Ar @ W - W).max() <= tol * nW, what
    AW, WA = Ar @ W, W @ Ar
    assert np.abs(AW - AW.T).max() <= tol, what
    assert np.abs(WA - WA.T).max() <= tol, what


def embed(block, mask):
    idx = [i for i in range(3) if mask >> i & 1]
    M = np.zeros((3, 3))
    M[np.ix_(idx, idx)] = block
    return M


def wpinv_cases(rng):
    """(M, mask, kind): M = L U^T R L U^T^T has zero rows / columns outside the mask, as in vox_algebra_core."""
    out = []
    for mask in range(8):
        k = bin(mask).count("1")
        if k == 0:
            out.append((np.zeros((3, 3)), mask, "empty"))
            continue

        def add(kind, block):
            out.append((embed(block, mask), mask, kind))

        for kappa in 10.0 ** np.arange(0, 15):
            for _ in range(4):
                add("spd", spd(rng, geometric(kappa, k) * 10 ** rng.uniform(-6, 2)))
        if k >= 2:  # the closed form's own limits: trace(M) trace(M^-1) < 5e5 (2x2) / 1e5 (3x3)
            lim = 5e5 if k == 2 else 1e5
            for t in near([lim]):
                for _ in range(3):
                    add("trace_edge", spd(rng, trace_product_spectrum(t, k) * 10 ** rng.uniform(-4, 0)))
            for kappa in near([1.0 / (3 * FLT_EPS), 1e6, 1e7]):  # around the COD rank threshold
                add("cod_edge", spd(rng, geometric(kappa, k)))
            for _ in range(4):
                add("repeated", spd(rng, np.full(k, rng.uniform(0.1, 2))))
            for r in range(k):
                for noise in (0.0, 1e-12):
                    B = spd(rng, np.r_[rng.uniform(0.5, 2.0, r), np.zeros(k - r)])
                    E = rng.standard_normal((k, k)) * noise
                    add("rank%d" % r, B + 0.5 * (E + E.T))
            add("indefinite", spd(rng, np.r_[1.0, -0.5, 0.25][:k]))
        add("diagonal", np.diag(rng.uniform(0.1, 3, k)))
        for s in [1e-30, FLT_MIN, 1e-20, 1e20, 1e30]:
            add("scale", spd(rng, np.geomspace(1, 0.1, k)) * s)
        add("negative", -spd(rng, np.geomspace(1, 0.5, k)))
        add("nan", np.full((k, k), np.nan))
    return out


@pytest.mark.gpu
def test_voxel_weight_pinv_branches(lh, po):
    """W = pinv(M) of vox_algebra_core for all 8 masks.  Closed form taken => W is the float64 inverse of the kept
    block and the COD (device and oracle) finds rank popcount(mask): the shortcut never disagrees with the COD on
    rank.  COD taken => W is the pseudo-inverse with the cut at the COD's rank (Penrose conditions)."""
    rng = np.random.default_rng(3802)
    cases = wpinv_cases(rng)
    M = np.array([c[0] for c in cases])
    masks = np.array([c[1] for c in cases], np.int32)
    W, branch = lh.wpinv(M, masks)
    _, cod_rank = lh.cod(M)
    stats = {}
    for i, (Mi, mask, kind) in enumerate(cases):
        key = (mask, "closed" if branch[i] else "cod")
        stats[key] = stats.get(key, 0) + 1
        what = "mask %d %s case %d" % (mask, kind, i)
        if kind == "nan":
            assert branch[i] == 0, what
            continue
        k = bin(mask).count("1")
        if branch[i] and k == 0:
            assert np.all(W[i] == 0) and cod_rank[i] == 0, what
        elif branch[i]:
            idx = [j for j in range(3) if mask >> j & 1]
            B = Mi[np.ix_(idx, idx)]
            kap = np.linalg.cond(B)
            ref = embed(np.linalg.inv(B), mask)
            assert np.abs(W[i] - ref).max() <= 1e-12 * kap * np.abs(ref).max(), what
            assert cod_rank[i] == k, what + ": closed form taken but the device COD has rank %d" % cod_rank[i]
            if 1e-12 <= np.abs(Mi).max() <= 1e12:  # the oracle's COD is fp32 and squares the entries
                assert po.pinv(Mi.astype(np.float32))[1] == k, what + ": closed form taken, oracle COD rank differs"
        else:
            check_pinv(Mi, W[i], int(cod_rank[i]), what)
    print("W = pinv(M) branches (mask, branch): count", dict(sorted(stats.items())))


# ------------------------------------------------------------------------------------------------ cod_pinv
SHAPES = [(1, 1), (2, 2), (3, 3), (6, 6), (6, 3), (5, 2), (6, 1), (3, 6), (2, 5), (1, 6), (4, 6), (6, 4)]


def cod_cases(rng, r, c):
    n = min(r, c)
    out = []
    for kappa in 10.0 ** np.arange(0, 15, 2):
        for _ in range(3):
            s = geometric(kappa, n) * 10 ** rng.uniform(-3, 3)
            out.append(("spectrum", (rotation(rng, r)[:, :n] * s) @ rotation(rng, c)[:n]))
    for rank in range(n):
        for noise in (0.0, 1e-12):
            for _ in range(3):
                s = np.r_[rng.uniform(0.5, 2.0, rank), np.zeros(n - rank)]
                A = (rotation(rng, r)[:, :n] * s) @ rotation(rng, c)[:n]
                out.append(("rank%d" % rank, A + noise * rng.standard_normal((r, c))))
    D = np.zeros((r, c))
    D[np.arange(n), np.arange(n)] = rng.uniform(0.1, 3, n)
    out.append(("diagonal", D))
    out.append(("permuted_diagonal", D[rng.permutation(r)][:, rng.permutation(c)]))
    out.append(("zero", np.zeros((r, c))))
    for s in (1e-30, 1e30):
        out.append(("scale", rng.standard_normal((r, c)) * s))
    return out


@pytest.mark.gpu
def test_cod_pinv_rank_and_penrose(lh, po):
    """icet::cod_pinv, square / tall / wide up to 6x6: the oracle's rank wherever no singular value lies within a
    factor 10 of the rank threshold, and the Penrose conditions with the cut at its rank."""
    rng = np.random.default_rng(3803)
    total = compared = 0
    for r, c in SHAPES:
        cases = cod_cases(rng, r, c)
        # the same matrix on both sides: the oracle is fp32, so the device gets the fp32-rounded entries
        A = np.array([a for _, a in cases]).astype(np.float32).astype(np.float64)
        P, rank = lh.cod(A)
        for i, (kind, _) in enumerate(cases):
            what = "%dx%d %s case %d" % (r, c, kind, i)
            s = np.linalg.svd(A[i], compute_uv=False)
            thr = FLT_EPS * min(r, c) * s[0]
            clear = not np.any((s > thr / 10) & (s < thr * 10))
            if clear:
                assert rank[i] == int(np.sum(s > thr)), what
                if 1e-12 <= np.abs(A[i]).max() <= 1e12:
                    assert po.pinv(A[i].astype(np.float32))[1] == rank[i], what
                    compared += 1
            check_pinv(A[i], P[i], int(rank[i]), what)
            total += 1
    print("cod_pinv: %d cases, %d rank comparisons with the oracle" % (total, compared))


# ------------------------------------------------------------------------------------------------ jacobi6
def sym6_cases(rng):
    out = []
    for kappa in 10.0 ** np.arange(0, 15):
        for _ in range(6):
            out.append(("spd", spd(rng, geometric(kappa, 6) * 10 ** rng.uniform(-3, 6))))
    for t in near([TRACE_BOUND]):
        for _ in range(6):
            out.append(("trace_edge", spd(rng, trace_product_spectrum(t, 6) * 10 ** rng.uniform(-2, 5))))
    for kappa in near([COND_CUTOFF]):
        for _ in range(6):
            s = np.r_[1.0, rng.uniform(1.0 / kappa, 1.0, 4), 1.0 / kappa]
            out.append(("cond_edge", spd(rng, s * 10 ** rng.uniform(-2, 5))))
    for _ in range(6):
        out.append(("repeated2", spd(rng, [5.0, 5.0, 2.0, 1.0, 0.5, 0.1])))
        out.append(("repeated3", spd(rng, [4.0, 1.0, 1.0, 1.0, 0.3, 0.2])))
    for rank in range(6):
        for noise in (0.0, 1e-13):
            for _ in range(3):
                A = spd(rng, np.r_[rng.uniform(0.5, 2.0, rank), np.zeros(6 - rank)])
                E = rng.standard_normal((6, 6)) * noise
                out.append(("rank%d" % rank, A + 0.5 * (E + E.T)))
    d = rng.uniform(0.1, 10, 6)
    out.append(("diagonal", np.diag(d)))
    P = np.eye(6)[rng.permutation(6)]
    out.append(("permuted_diagonal", P @ np.diag(d) @ P.T))
    for _ in range(4):
        out.append(("indefinite", spd(rng, rng.uniform(-2, 2, 6))))
    return out


@pytest.fixture(scope="session")
def dump_systems(ctx, frame_pair, sample_pair):
    """H^T W H / H^T W dz of every iteration of the two bundled pairs and of the corridor of
    test_truncated_solution_axis, as recorded by the library (fp32 copies of the double sums)."""
    rng = np.random.default_rng(11)
    n = 60000
    x = rng.uniform(-30, 30, n)
    side = rng.integers(0, 3, n)
    y = np.where(side == 0, -4.0, np.where(side == 1, 4.0, rng.uniform(-4, 4, n)))
    zc = np.where(side == 2, -1.5, rng.uniform(-1.5, 2.0, n))
    s1 = np.stack([x, y + 0.005 * rng.standard_normal(n), zc + 0.005 * rng.standard_normal(n)]).astype(np.float32)
    s2 = s1.copy()
    s2[1] += 0.05
    s2 += (0.005 * rng.standard_normal(s2.shape)).astype(np.float32)
    out = []
    for name, (a, b) in (("frame", frame_pair), ("sample_pc", sample_pair), ("corridor", (s1, s2))):
        _, g = ctx.register(a, b, dump=True)
        for it in range(g["HTWH"].shape[0]):
            out.append(("%s it %d" % (name, it), g["HTWH"][it].astype(np.float64), g["HTWdz"][it].astype(np.float64)))
    return out


@pytest.mark.gpu
def test_jacobi6_against_eigh(lh, dump_systems):
    """icet::jacobi6: eigenvalues within 1e-13 max|lambda| of numpy's, orthonormal U, ascending order with the
    columns following, the largest component of every column positive."""
    rng = np.random.default_rng(3804)
    cases = sym6_cases(rng) + [("dump " + w, A) for w, A, _ in dump_systems]
    A = np.array([a for _, a in cases])
    ev, U = lh.jacobi(A)
    for i, (kind, Ai) in enumerate(cases):
        what = "%s case %d" % (kind, i)
        ref = np.linalg.eigvalsh(Ai)
        lm = np.abs(ref).max()
        assert np.all(np.diff(ev[i]) >= 0), what
        assert np.abs(ev[i] - ref).max() <= 1e-13 * lm + 1e-300, what
        assert np.abs(U[i].T @ U[i] - np.eye(6)).max() <= 1e-13, what
        assert np.abs(Ai @ U[i] - U[i] * ev[i]).max() <= 1e-13 * lm + 1e-300, what
        for c in range(6):
            col = U[i][:, c]
            assert col[np.argmax(np.abs(col))] > 0, what + " column %d" % c
    print("jacobi6: %d cases (%d from the dumps)" % (len(cases), len(dump_systems)))


# ------------------------------------------------------------------------------------------------ the 6x6 solve
def pack(A, b, n_used=100):
    tot = np.zeros(28)
    t = 0
    for a in range(6):
        for c in range(a, 6):
            tot[t] = A[a, c]
            t += 1
    tot[21:27] = b
    tot[27] = n_used
    return tot


def solve_reference(A, b, X0):
    """float64 restatement of src/icet.cpp:410-492 as the library documents it: noise_mat = pinv(H^T W H) with the
    COD rank rule on the spectrum, pred_stds, checkCondition (:469-486, eigenvectors in the sign convention "largest
    component positive" for the :479 inflation), dx from the kept spectrum, X += dx in fp32."""
    ev, U = np.linalg.eigh(A)
    for c in range(6):
        if U[np.argmax(np.abs(U[:, c])), c] < 0:
            U[:, c] = -U[:, c]
    lm = np.abs(ev).max()
    keep = np.abs(ev) > FLT_EPS * 6 * lm
    Q = (U[:, keep] / ev[keep]) @ U[:, keep].T
    stds = np.sqrt(np.abs(np.diag(Q)))
    with np.errstate(divide="ignore", invalid="ignore"):
        ratios = ev[5] / ev
    cond = ratios[0]
    dropped, status, eyecount, c = 0, 0, 1, cond
    while abs(c) > COND_CUTOFF:
        if eyecount > 5:
            status = 1
            break
        stds = stds + U[:, eyecount - 1]
        dropped += 1
        c = ratios[eyecount]
        eyecount += 1
    kept = ev[dropped:]
    lmax = np.abs(kept).max() if len(kept) else 0.0
    tiny = FLT_EPS * (6 - dropped) * lmax
    dx = np.zeros(6)
    for k in range(dropped, 6):
        if abs(ev[k]) > tiny:
            dx += U[:, k] * (U[:, k] @ b / ev[k])
    near_cut = bool(np.any(np.abs(np.abs(ratios) / COND_CUTOFF - 1) < 1e-9))
    # the :479 inflation is comparable where every dropped eigenvector is well defined (simple eigenvalue)
    gaps = [np.min(np.abs(np.delete(ev, k) - ev[k])) for k in range(6)]
    dropped_gap = min([gaps[k] for k in range(dropped)], default=np.inf)
    kq = lm / np.abs(ev[keep]).min() if keep.any() else 1.0
    kx = lmax / np.abs(ev[dropped:][np.abs(ev[dropped:]) > tiny]).min() if np.any(np.abs(kept) > tiny) else 1.0
    trA, trQinv = np.trace(A), (np.sum(1.0 / ev) if np.all(ev > 0) else np.inf)
    return dict(X=(X0.astype(np.float64) + dx).astype(np.float32), dx=dx, Q=Q, stds=stds, dropped=dropped,
                status=status, cond=cond, near_cut=near_cut, dropped_gap=dropped_gap, lm=lm, kq=kq, kx=kx,
                trprod=trA * trQinv, ev=ev)


def solve_cases(rng, dump_systems):
    out = []

    def add(kind, A, b=None):
        A = 0.5 * (A + A.T)
        if b is None:
            b = rng.standard_normal(6) * np.abs(A).max() * 1e-3
        out.append((kind, A, b, (rng.standard_normal(6) * 0.05).astype(np.float32)))

    for kappa in 10.0 ** np.arange(0, 15):
        for _ in range(8):
            add("spd k=1e%d" % round(np.log10(kappa)), spd(rng, geometric(kappa, 6) * 10 ** rng.uniform(-2, 6)))
    for t in near([TRACE_BOUND]):
        for _ in range(16):
            add("trace product 0.999e6(1%+.0e)" % (t / TRACE_BOUND - 1),
                spd(rng, trace_product_spectrum(t, 6) * 10 ** rng.uniform(-2, 6)))
    # the trace bound decided by the last bits of trace(A^-1), and well-conditioned systems below it: the two solve
    # forms round Q, dx and the bound differently unless they share one arithmetic
    for rel in (0.0, 1e-16, -1e-16, 1e-15, -1e-15, 1e-14, -1e-14, 1e-13, -1e-13, 1e-12, -1e-12):
        for _ in range(8):
            add("trace product 0.999e6(1%+.0e)" % rel,
                spd(rng, trace_product_spectrum(TRACE_BOUND * (1 + rel), 6) * 10 ** rng.uniform(-2, 6)))
    for _ in range(1500):
        add("below the trace bound", spd(rng, geometric(10 ** rng.uniform(4, 5.4), 6) * 10 ** rng.uniform(-2, 6)))
    for kappa in near([COND_CUTOFF]):
        for _ in range(16):
            s = np.r_[1.0, rng.uniform(1.0 / kappa, 1.0, 4), 1.0 / kappa]
            add("cond 1e6(1%+.0e)" % (kappa / COND_CUTOFF - 1), spd(rng, s * 10 ** rng.uniform(-2, 6)))
    for _ in range(8):
        add("repeated2", spd(rng, [5.0, 5.0, 2.0, 1.0, 0.5, 0.1]))
        add("repeated3", spd(rng, [4.0, 1.0, 1.0, 1.0, 0.3, 0.2]))
        add("repeated small", spd(rng, [4.0, 1.0, 0.5, 0.2, 1e-8, 1e-8]))
    for rank in range(1, 6):
        for noise in (0.0, 1e-13):
            for _ in range(4):
                A = spd(rng, np.r_[rng.uniform(0.5, 2.0, rank), np.zeros(6 - rank)])
                E = rng.standard_normal((6, 6)) * noise
                add("rank%d%s" % (rank, " noisy" if noise else ""), A + 0.5 * (E + E.T))
    add("zero", np.zeros((6, 6)), np.zeros(6))
    d = rng.uniform(0.1, 10, 6)
    add("diagonal", np.diag(d))
    P = np.eye(6)[rng.permutation(6)]
    add("permuted_diagonal", P @ np.diag(d) @ P.T)
    for _ in range(4):
        add("indefinite", spd(rng, rng.uniform(-2, 2, 6)))
    for w, A, b in dump_systems:
        add("dump " + w, A, b)
    return out


@pytest.fixture(scope="session")
def solve_runs(lh, dump_systems):
    rng = np.random.default_rng(3805)
    cases = solve_cases(rng, dump_systems)
    tot = np.array([pack(A, b) for _, A, b, _ in cases])
    X0 = np.array([x for _, _, _, x in cases])
    runs = {(form, flags): lh.solve(form == "cluster", tot, X0, flags)
            for form in ("split", "cluster") for flags in (0, FLAG_FULL_EIG)}
    return cases, runs


@pytest.mark.gpu
def test_split_and_cluster_solves_are_byte_identical(solve_runs):
    """The split loop (k_solve6) and the cluster loop run the same 6x6 arithmetic: result records, next transform and
    get_H matrices are byte-identical on every case, so a batch row equals its single call (DESIGN.md 3.6)."""
    cases, runs = solve_runs
    for flags in (0, FLAG_FULL_EIG):
        (rs, trs, js), (rc, trc, jc) = runs[("split", flags)], runs[("cluster", flags)]
        diff = {}
        for i in range(len(cases)):
            fields = [(f, rs[i][f].tobytes(), rc[i][f].tobytes()) for f in rs.dtype.names]
            for name, a, b in fields + [("TR", trs[i].tobytes(), trc[i].tobytes()), ("J", js[i].tobytes(), jc[i].tobytes())]:
                if a != b:
                    diff.setdefault(name, []).append(cases[i][0])
        if flags == 0:
            pd = np.array([np.linalg.eigvalsh(A)[0] > 1e-9 * np.abs(A).max() for _, A, _, _ in cases])
            fs, fc = int(np.sum((rs["cond"] < 0) & pd)), int(np.sum((rc["cond"] < 0) & pd))
            print("flags 0: fast path split %d / cluster %d of %d cases; Jacobi split %d / cluster %d"
                  % (fs, fc, len(cases), len(cases) - fs, len(cases) - fc))
        assert not diff, "flags %d: split and cluster solves differ: %s" % (
            flags, {k: (len(v), sorted(set(v))[:8]) for k, v in diff.items()})


@pytest.mark.gpu
def test_solve_against_float64_restatement(solve_runs):
    """Both solve forms against the float64 restatement of src/icet.cpp:410-492: n_dropped exactly (cases within
    1e-9 of the cutoff are listed), X, Q, pred_stds and cond within tolerances scaled by the condition number, status 0."""
    cases, runs = solve_runs
    listed, jac_dump = [], set()
    for (form, flags), (res, _, _) in runs.items():
        for i, (kind, A, b, X0) in enumerate(cases):
            r = res[i]
            ref = solve_reference(A, b, X0)
            what = "%s flags %d: %s case %d" % (form, flags, kind, i)
            if ref["near_cut"]:
                listed.append(what)
                continue
            assert r["status"] == 0 and ref["status"] == 0, what
            assert r["n_dropped"] == ref["dropped"], what + ": n_dropped %d, reference %d" % (r["n_dropped"], ref["dropped"])
            assert r["n_used"] == 100, what
            # the warp solve reports -(trace(A) trace(A^-1)); a negative ev[5] / ev[0] needs a clearly negative ev[0]
            fast = r["cond"] < 0 and ref["ev"][0] > 1e-9 * ref["lm"]
            if fast:
                assert flags == 0 and r["n_dropped"] == 0, what
                assert abs(-float(r["cond"]) / ref["trprod"] - 1) <= 1e-6, what
                assert ref["trprod"] < TRACE_BOUND * (1 + 1e-9), what
            else:
                if kind.startswith("dump"):
                    jac_dump.add(kind)
                if np.isnan(ref["cond"]):
                    assert np.isnan(r["cond"]), what
                elif abs(ref["cond"]) < 1e12:  # ev[5] / ev[0]: ev[0] carries an error of ~eps * ev[5]
                    assert abs(float(r["cond"]) / ref["cond"] - 1) <= 1e-6 + 1e-14 * abs(ref["cond"]), what
            # X += dx in fp32: the rounding of the sum plus the float64 error of dx
            tol_x = 2 * np.spacing(np.abs(ref["X"])) + (1e-6 + 1e-13 * ref["kx"]) * np.abs(ref["dx"]).max()
            assert np.all(np.abs(r["X"].astype(np.float64) - ref["X"]) <= tol_x), what
            nq = np.abs(ref["Q"]).max()
            assert np.abs(r["Q"] - ref["Q"]).max() <= (3e-7 + 1e-13 * ref["kq"]) * nq + 1e-300, what
            if ref["dropped_gap"] > 1e-6 * ref["lm"]:
                tol_s = 3e-7 * np.abs(ref["stds"]).max() + 1e-12 * ref["lm"] / ref["dropped_gap"] + \
                    (1e-13 * ref["kq"]) * np.sqrt(nq)
                assert np.abs(r["pred_stds"] - ref["stds"]).max() <= tol_s, what
    kinds = {}
    for kind, *_ in cases:
        key = kind.split(" it ")[0]
        kinds[key] = kinds.get(key, 0) + 1
    print("solve cases:", kinds)
    print("listed (within 1e-9 of the 1e6 cutoff):", listed)
    print("dump iterations that take the Jacobi path:", sorted(jac_dump))


# ------------------------------------------------------------------------------------------------ vox_algebra_core
def vox_reference(v, mean, cov, nbin, Jm):
    """float64 restatement of src/icet.cpp:308-338 on the library's voxel record."""
    def sym(c):
        return np.array([[c[0], c[1], c[2]], [c[1], c[3], c[4]], [c[2], c[4], c[5]]])
    Rn = sym(v["S1n"]) + sym(cov) / (nbin - 1)
    LV = v["LV"].reshape(3, 3)
    M = LV @ Rn @ LV.T
    U, s, Vt = np.linalg.svd(M)
    rank = int(np.sum(s > FLT_EPS * 3 * s[0])) if s[0] > 0 else 0
    W = (Vt[:rank].T / s[:rank]) @ U[:, :rank].T
    J = Jm.astype(np.float64).reshape(3, 3, 3)  # J[j] row-major
    H = np.zeros((3, 6))
    H[:, :3] = -np.eye(3)
    for j in range(3):
        H[:, 3 + j] = J[j] @ mean
    Hz = LV @ H
    dz = LV @ (mean - v["mu"])
    HtWH = Hz.T @ W @ Hz
    acc = np.zeros(28)
    acc[:21] = HtWH[np.triu_indices(6)]
    acc[21:27] = Hz.T @ W @ dz
    acc[27] = 1.0
    kap = s[0] / s[rank - 1] if rank else 1.0
    tail = s[rank] / s[rank - 1] if 0 < rank < 3 else 0.0
    scale = np.abs(Hz).max() ** 2 * np.abs(W).max() * max(1.0, np.abs(dz).max() / max(np.abs(Hz).max(), 1e-300))
    return acc, kap, tail, scale, M


def vox_cases(rng):
    """Voxel records and scan-2 statistics for every lmask.  flat / thin: both Gaussians lose one / two of the axes
    the mask keeps, so the kept block of M is singular (the COD fallback); near_flat: that axis keeps 1e-4 of the
    smallest other variance, a condition number between the closed form's limits and the COD rank threshold."""
    recs, means, covs, nbins, Jms, kinds = [], [], [], [], [], []
    for lmask in range(8):
        kept = [k for k in range(3) if lmask >> k & 1]
        for kind in ("ordinary", "ordinary", "ordinary", "flat", "thin", "near_flat"):
            V = rotation(rng, 3)
            S1 = spd(rng, rng.uniform(0.05, 0.5, 3) ** 2)
            S2 = spd(rng, rng.uniform(0.05, 0.5, 3) ** 2)
            gone = []
            if kind in ("flat", "near_flat") and len(kept) >= 2:
                gone = kept[:1]
            elif kind == "thin" and len(kept) == 3:
                gone = kept[:2]
            if gone:
                G = V[gone].T @ V[gone]
                P = np.eye(3) - G
                d = 1e-4 * min(np.linalg.eigvalsh(S1)[0], np.linalg.eigvalsh(S2)[0]) if kind == "near_flat" else 0.0
                S1 = P @ S1 @ P + d * G
                S2 = P @ S2 @ P + d * G
            nb = int(rng.integers(30, 2000))
            rec = np.zeros((), VOX1_DTYPE)
            rec["mu"] = rng.uniform(-20, 20, 3)
            rec["S1n"] = S1[np.triu_indices(3)]
            rec["LV"] = (V * np.array([(lmask >> k) & 1 for k in range(3)])[:, None]).reshape(9)
            rec["lmask"] = lmask
            recs.append(rec)
            means.append(rec["mu"] + rng.normal(0, 0.05, 3))
            covs.append((S2 * (nb - 1))[np.triu_indices(3)])
            nbins.append(nb)
            Jms.append(rng.uniform(-1, 1, 27).astype(np.float32))
            kinds.append((lmask, kind))
    return np.array(recs, VOX1_DTYPE), np.array(means), np.array(covs), np.array(nbins), np.array(Jms), kinds


@pytest.mark.gpu
def test_vox_algebra_against_float64_restatement(lh):
    """vox_algebra_core for every lmask, including voxels whose M sends masked_inv3 to the COD fallback."""
    rng = np.random.default_rng(3806)
    recs, means, covs, nbins, Jms, kinds = vox_cases(rng)
    acc = lh.vox(recs, means, covs, nbins, Jms)
    M_all = []
    for i in range(len(recs)):
        ref, kap, tail, scale, M = vox_reference(recs[i], means[i], covs[i], nbins[i], Jms[i])
        M_all.append(M)
        tol = (1e-12 * kap + 10 * tail) * scale + 1e-13 * np.abs(ref).max()
        assert np.abs(acc[i] - ref).max() <= tol, "lmask %d %s case %d: %.3e > %.3e" % (
            *kinds[i], i, np.abs(acc[i] - ref).max(), tol)
    _, branch = lh.wpinv(np.array(M_all), recs["lmask"])
    n_cod = {m: int(np.sum((branch == 0) & (recs["lmask"] == m))) for m in range(8)}
    print("vox_algebra_core: %d voxels; COD fallback per lmask %s" % (len(recs), n_cod))
    assert sum(n_cod.values()) >= 5  # the flat and thin voxels of the masks with two or three axes
