"""CPU tests of the host side: the C ABI library builds, loads and exports every symbol include/icet_b200.h
declares (no compute without a GPU), fails loudly without a device, the host-side layout helpers, the
synthetic generator, pair sharding over world_size-2 gloo, and the reference arm of bench.py."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_library_exports_every_declared_symbol():
    import icet_b200
    from icet_b200 import api
    icet_b200.build()
    hdr = open(os.path.join(ROOT, "include", "icet_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(icet_b200_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 18
    L = icet_b200.load_library()
    for name in declared:
        assert hasattr(L, name), "missing export " + name
    assert sorted(api.EXPORTS) == declared
    assert L.icet_b200_version() == 105
    assert C.sizeof(api.Result) == 224 and C.sizeof(api.Params) == 32
    m = re.search(r"#define ICET_B200_NKERNELS (\d+)", hdr)
    assert int(m.group(1)) == api.NKERNELS
    assert L.icet_b200_kernel_name(7).decode() == "k_pass<scan2>"


def test_library_links_no_cpu_fallback():
    """The product library contains device code for sm_100a only and does not link the oracle."""
    import icet_b200
    lib = icet_b200.lib_path()
    out = subprocess.run(["cuobjdump", "-lelf", lib], capture_output=True, text=True).stdout
    assert "sm_100a" in out and "sm_90" not in out and "sm_80" not in out
    ldd = subprocess.run(["ldd", lib], capture_output=True, text=True).stdout
    assert "oracle" not in ldd
    csrc = os.path.join(ROOT, "icet_b200", "csrc")
    src = "".join(open(os.path.join(csrc, f)).read() for f in sorted(os.listdir(csrc))) + \
        open(os.path.join(ROOT, "icet_b200", "api.py")).read() + open(os.path.join(ROOT, "icet_b200", "nodes.py")).read()
    assert "pyoracle" not in src and "icet_oracle" not in src  # the product never references the checker


def test_no_device_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    import icet_b200
    with pytest.raises(icet_b200.IcetError) as e:
        icet_b200.Context(0)
    assert "no CPU fallback" in str(e.value)
    L = icet_b200.load_library()
    assert L.icet_b200_register(None, None, None, 0, 0, None, 0, 0, None, None) < 0
    assert b"NULL" in L.icet_b200_last_error()


def test_as_planes_layouts():
    from icet_b200.api import as_planes
    rng = np.random.default_rng(0)
    a = rng.standard_normal((50, 3))
    p = as_planes(a)
    assert p.shape == (3, 50) and p.dtype == np.float32 and p.flags["C_CONTIGUOUS"]
    np.testing.assert_array_equal(p, a.T.astype(np.float32))
    np.testing.assert_array_equal(as_planes(np.asfortranarray(a)), p)     # Eigen's column-major N x 3
    np.testing.assert_array_equal(as_planes(a.T.copy()), p)               # already planes
    with pytest.raises(ValueError):
        as_planes(np.zeros((4, 5)))


def test_synth_host_generator_properties():
    from tools import synth_host
    S = synth_host.scans(2, rings=16, azim=256)
    assert S.shape == (2, 3, 4096) and S.dtype == np.float32
    S2 = synth_host.scans(2, rings=16, azim=256, nthreads=1)
    np.testing.assert_array_equal(S, S2)                      # pure function of (seed, scan, ring, azimuth)
    np.testing.assert_array_equal(synth_host.scans(1, first_scan=1, rings=16, azim=256)[0], S[1])
    r = np.linalg.norm(S[0], axis=0)
    zero = (r == 0)
    assert 0.08 < zero.mean() < 0.35                          # dropped / no-hit returns are stored as (0,0,0)
    assert r[~zero].min() > 0.25 and r.max() <= 120.5
    el = np.degrees(np.arcsin(S[0, 2, ~zero] / r[~zero]))
    assert el.min() > -22.6 and el.max() < 22.6
    assert not np.array_equal(S[0], S[1])


def test_shard_ranges_cover_all_pairs():
    from icet_b200.sharding import shard_range, shard_scans
    for total in (0, 1, 7, 4096):
        for world in (1, 2, 3, 8):
            got = []
            for r in range(world):
                lo, hi = shard_range(total, r, world)
                got += list(range(lo, hi))
                fs, ns = shard_scans(total, r, world)
                assert (ns == 0) if hi == lo else (fs == lo and ns == hi - lo + 1)
            assert got == list(range(total))
    with pytest.raises(ValueError):
        shard_range(4, 2, 2)


_GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, %r)
import torch, torch.distributed as dist
from icet_b200 import sharding
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
P = 6
lo, hi = sharding.shard_range(world * P, rank, world)
local = torch.zeros((P, 48))
local[:, 0] = torch.arange(lo, hi, dtype=torch.float32)      # stand-in for X[0] of pair k: its global index
local[:, 1] = float(rank)
out = sharding.gather_results(local, world)
assert out.shape == (world * P, 48)
assert torch.equal(out[:, 0], torch.arange(world * P, dtype=torch.float32)), out[:, 0]
assert torch.equal(out[:, 1], torch.arange(world).repeat_interleave(P).float())
dist.barrier()
if rank == 0:
    print("GLOO_OK", world)
dist.destroy_process_group()
"""


def test_pair_sharding_world2_gloo(tmp_path):
    """N > 1 host path on CPU: contiguous pair ranges + the final all_gather keep the global pair order."""
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29611", str(script)],
                       capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "GLOO_OK 2" in r.stdout


def test_bench_reference_arm_runs():
    """`bench.py --impl reference` times the reference's CPU path on the host cores and prints one JSON line."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "pairs/s" and line["value"] > 0
    from oracle import pyref
    # the reference's own sources when oracle/_ref exists (or can be built: /root/reference), else the oracle port
    assert line["cpu_baseline"]["kind"] == ("reference" if pyref.available(True) or pyref.available(False) else "port")
    assert line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["port_value"] > 0
    assert line["config"]["pairs_per_step"] == max(2, min(2 * (os.cpu_count() or 1), 256))   # what really ran
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["higher_is_better"] is True


def test_bench_dump_outputs_layout(tmp_path, monkeypatch):
    """bench.py --dump-outputs: one float32 / float64 .npy per field of the result records (integer fields exact);
    above the size cap, the same seeded sample of the pairs on every run, named by pair_index."""
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)   # importing bench.py sets it
    import bench
    n = 50
    rows = np.random.default_rng(1).standard_normal((n, 48)).astype(np.float32)
    recs = np.random.default_rng(2).standard_normal((n, 5)).astype(np.float32)
    ints = np.arange(4 * n, dtype=np.int32).reshape(n, 4)
    recs[:, :4] = ints.view(np.float32)

    def load(d):
        return {f[:-4]: np.load(d / f) for f in os.listdir(d)}

    bench.dump_outputs(str(tmp_path / "all"), rows, recs)
    d = load(tmp_path / "all")
    assert sorted(d) == sorted(["X", "pred_stds", "Q", "status", "n_gauss1", "n_used", "n_dropped", "cond", "pair_index"])
    assert all(a.dtype in (np.float32, np.float64) and a.shape[0] == n for a in d.values())
    np.testing.assert_array_equal(d["X"], rows[:, :6])
    np.testing.assert_array_equal(d["Q"].reshape(n, 36), rows[:, 12:])
    np.testing.assert_array_equal(d["n_used"], ints[:, 2])
    np.testing.assert_array_equal(d["cond"], recs[:, 4])
    per_pair = sum(a.nbytes for a in d.values()) // n
    limit = 20 * per_pair + bench.NPY_HEADER_MAX * len(d)
    monkeypatch.setattr(bench, "DUMP_LIMIT", limit)
    for k in ("a", "b"):
        bench.dump_outputs(str(tmp_path / k), rows, recs)
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    idx = a["pair_index"].astype(np.int64)
    assert len(idx) == 20 and np.all(np.diff(idx) > 0)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= limit
    for name in a:
        np.testing.assert_array_equal(a[name], b[name])
        np.testing.assert_array_equal(a[name], d[name][idx])


def test_bench_rejects_zero_steps():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert r.returncode != 0 and "--steps" in r.stderr


def _build_demo():
    r = subprocess.run(["make", "-C", os.path.join(ROOT, "examples")], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return os.path.join(ROOT, "examples", "_build", "icet_cpp_demo_headless")


def test_cpp_dropin_class_compiles_and_fails_loudly_without_gpu(tmp_path, frame_pair):
    """include/icet.h + icet_b200/host/*.cpp (the C++ host side over the C ABI) compile against the test-only Eigen
    stub; without a GPU the constructor throws (std::runtime_error) instead of falling back to a CPU path."""
    import icet_b200
    icet_b200.build()
    exe = _build_demo()
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present (the GPU test runs the demo)")
    s1, s2 = frame_pair
    a, b = tmp_path / "a.f32", tmp_path / "b.f32"
    s1[:, :4096].tofile(a)
    s2[:, :4096].tofile(b)
    r = subprocess.run([exe, str(a), str(b), "f32"], capture_output=True, text=True)
    assert r.returncode == 1
    assert "no CPU fallback" in r.stderr


def test_utils_loader_formats(tmp_path):
    """Ouster CSV (two header rows, integer mm in columns 8-10) and tab-separated xyz (reference src/utils.cpp:19-88),
    exercised through the C++ demo's loader path is GPU-only; here the parser is checked via a tiny C++ probe."""
    probe = tmp_path / "probe.cpp"
    probe.write_text('''
#include <cstdio>
#include "utils.h"
int main(int argc, char** argv) {
  Eigen::MatrixXf m = utils::loadPointCloudCSV(argv[1], argv[2]);
  std::printf("%ld %ld", (long)m.rows(), (long)m.cols());
  for (long i = 0; i < m.rows(); i++) std::printf(" %.4f %.4f %.4f", m(i,0), m(i,1), m(i,2));
  Eigen::Matrix3f R = utils::R(0.1f, 0.2f, 0.3f);
  std::printf(" R %.6f %.6f %.6f", R(0,0), R(0,1), R(2,2));
  return 0;
}''')
    exe = tmp_path / "probe"
    r = subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-I" + os.path.join(ROOT, "include"),
                        "-I" + os.path.join(ROOT, "tests", "stubs"), "-o", str(exe), str(probe),
                        os.path.join(ROOT, "icet_b200", "host", "utils.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    csv = tmp_path / "o.csv"
    hdr = ",".join("c%d" % i for i in range(12))
    # two header lines + 5 data rows: the reference drops the two header lines AND the first two data rows
    csv.write_text(hdr + "\n" + hdr + "\n" + "\n".join(
        ",".join(["0"] * 8 + [str(1000 * (i + 1)), str(-250 * i), str(3), "9"]) for i in range(5)) + "\n")
    out = subprocess.run([str(exe), str(csv), "ouster"], capture_output=True, text=True).stdout.split()
    assert out[:2] == ["3", "3"]
    np.testing.assert_allclose([float(v) for v in out[2:11]], [3, -0.5, 0.003, 4, -0.75, 0.003, 5, -1.0, 0.003], atol=1e-6)
    tsv = tmp_path / "t.txt"
    tsv.write_text("0\t0\t0\n1.5\t2.5\t-3\n4\t5\t6\n")   # line 0 is taken as the header
    out = subprocess.run([str(exe), str(tsv), "txt"], capture_output=True, text=True).stdout.split()
    assert out[:2] == ["2", "3"] and float(out[4]) == -3.0
    # the same files through the REFERENCE's own loader (src/utils.cpp + csv.hpp, compiled by `make -C oracle ref`)
    from oracle import pyref
    if pyref.available():
        import ctypes as C
        L = pyref.lib()
        L.icet_ref_load_csv.argtypes = [C.c_char_p, C.c_char_p, C.c_void_p, C.c_int32]
        buf = np.zeros((16, 3), np.float32)
        for path, kind in ((csv, "ouster"), (tsv, "txt")):
            n = L.icet_ref_load_csv(str(path).encode(), kind.encode(), buf.ctypes.data, 16)
            mine = subprocess.run([str(exe), str(path), kind], capture_output=True, text=True).stdout.split()
            assert int(mine[0]) == n
            np.testing.assert_allclose([float(v) for v in mine[2:2 + 3 * n]], buf[:n].reshape(-1), atol=1e-6)
    # utils::R (reference src/utils.cpp:144-152): R(0,0) = cos(theta) cos(psi), R(2,2) = cos(phi) cos(theta)
    i = out.index("R")
    np.testing.assert_allclose([float(v) for v in out[i + 1:i + 4]],
                               [np.cos(0.2) * np.cos(0.3), np.sin(0.3) * np.cos(0.1) + np.sin(0.1) * np.sin(0.2) * np.cos(0.3),
                                np.cos(0.1) * np.cos(0.2)], rtol=1e-5)
