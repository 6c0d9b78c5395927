"""Keyframe registration against the ordinary path (include/icet_b200.h "keyframes"): prints one JSON line.

Three workloads, each with a keyframe arm and the existing path with the keyframe's cloud as scan 1; in every workload
both arms must give identical result bytes.
  (a) throughput: 4096 registrations -- scans 1-8 of the seeded sequence, 512 seeded X0 perturbations each -- against
      scan 0 (register_keyframe_batch_device against register_batch_device with scan 0 repeated).  Scans 1-8 total
      12 MB and are L2-resident in both arms.
  (b) map latency: one 64-channel scan against the 2 M-point map of BASELINE.json configs[4], >= 200 calls per arm:
      device-resident (CUDA events around each call) and the blocking host-buffer call (host clock; it includes the
      upload of the map, 24 MB, in the ordinary arm).
  (c) single pair: one 64-channel pair, device-resident and host-buffer, as in (b).
Also the per-kernel device time of one keyframe batch of (a) and one keyframe map call of (b) in a separate profiled
pass (k_kf_attach is listed as k_cell_scan).  Needs a GPU; there is no CPU path.

    python tools/keyframe_bench.py [--reps 5] [--calls 200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

SEED = 20240


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # the measurement stands without it, but says so
        return {"name": None, "power_limit": None, "error": str(e)}


def results(t):
    from icet_b200 import api
    return t.cpu().numpy().view(api.RESULT_DTYPE).reshape(-1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5, help="timed repetitions of the 4096-pair batch per arm")
    ap.add_argument("--calls", type=int, default=200, help="timed calls per arm of the latency workloads")
    args = ap.parse_args()
    import torch
    import icet_b200
    from icet_b200 import api
    from tools import synth_host
    if not torch.cuda.is_available():
        raise SystemExit("keyframe_bench: no CUDA device (there is no CPU path)")
    dev = torch.device("cuda:0")
    ctx = icet_b200.Context(0)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    out = {"tool": "keyframe_bench", "gpu": gpu_info()}
    p = api.make_params()

    # ---- (a) throughput
    scans = torch.empty((9, 3, 131072), dtype=torch.float32, device=dev)
    ctx.synth_scans_device(scans.data_ptr(), 9, first_scan=0, seed=SEED)
    ctx.synchronize()
    P = 4096
    rng = np.random.default_rng(7)
    x0 = np.zeros((P, 6), np.float32)
    x0[:, :3] = rng.normal(0, 0.05, (P, 3))
    x0[:, 3:] = rng.normal(0, 0.01, (P, 3))
    x0d = torch.from_numpy(x0).to(dev)
    ptr2 = np.array([scans[1 + i // 512].data_ptr() for i in range(P)], np.uint64)
    n2 = np.full(P, 131072, np.int32)
    ptr1 = np.full(P, scans[0].data_ptr(), np.uint64)
    kf = icet_b200.Keyframe.from_device(scans[0].data_ptr(), 131072, ctx=ctx)
    out_k = torch.zeros((P, 56), dtype=torch.float32, device=dev)
    out_b = torch.zeros((P, 56), dtype=torch.float32, device=dev)

    def arm_k():
        kf.register_batch_device(ptr2, n2, out_k.data_ptr(), x0d.data_ptr())

    def arm_b():
        ctx.register_batch_ptrs(ptr1, n2, ptr2, n2, out_b.data_ptr(), x0d.data_ptr(), params=p, device=True)

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        return a.elapsed_time(b)

    for fn in (arm_k, arm_b):  # warm-up
        timed(fn)
    tk, tb = [], []
    for _ in range(args.reps):  # alternating arms
        tk.append(timed(arm_k))
        tb.append(timed(arm_b))
    same_a = results(out_k).tobytes() == results(out_b).tobytes()
    mk, mb = float(np.median(tk)), float(np.median(tb))
    out["throughput_4096"] = {
        "workload": "scans 1-8 x 512 seeded X0 against scan 0, 64-ch, 75x24, 7 it, one call of 4096 pairs",
        "keyframe_pairs_per_s": P / (mk * 1e-3), "batch_pairs_per_s": P / (mb * 1e-3), "ratio": mb / mk,
        "keyframe_ms": tk, "batch_ms": tb, "identical_bytes": same_a}

    # ---- (b) map latency, (c) single pair
    def latency(s1, n1, s2h, s2, n2_, calls):
        kfm = icet_b200.Keyframe.from_device(s1.data_ptr(), n1, ctx=ctx)
        s1h = s1.cpu().numpy()
        rk = torch.zeros((1, 56), dtype=torch.float32, device=dev)
        rb = torch.zeros((1, 56), dtype=torch.float32, device=dev)
        dk, db, hk, hb = [], [], [], []
        for i in range(calls + 20):  # device-resident, alternating, the first 20 of each untimed
            t1 = timed(lambda: kfm.register_batch_device([s2.data_ptr()], [n2_], rk.data_ptr()))
            t2 = timed(lambda: ctx.register_batch_ptrs([s1.data_ptr()], [n1], [s2.data_ptr()], [n2_], rb.data_ptr(),
                                                       params=p, device=True))
            if i >= 20:
                dk.append(t1)
                db.append(t2)
        same_dev = results(rk).tobytes() == results(rb).tobytes()
        for i in range(calls + 5):  # host buffers, blocking calls
            t0 = time.perf_counter()
            a = kfm.register(s2h)
            t1 = time.perf_counter()
            b = ctx.register(s1h, s2h)
            t2 = time.perf_counter()
            if i >= 5:
                hk.append((t1 - t0) * 1e3)
                hb.append((t2 - t1) * 1e3)
        same_host = a.tobytes() == b.tobytes() == results(rk)[0].tobytes()
        kfm.close()
        q = lambda v, x: float(np.percentile(v, x))
        return {"device_keyframe_p50_ms": q(dk, 50), "device_keyframe_p95_ms": q(dk, 95),
                "device_register_p50_ms": q(db, 50), "device_register_p95_ms": q(db, 95),
                "host_keyframe_p50_ms": q(hk, 50), "host_keyframe_p95_ms": q(hk, 95),
                "host_register_p50_ms": q(hb, 50), "host_register_p95_ms": q(hb, 95),
                "calls": calls, "identical_bytes": bool(same_dev and same_host), "gaussians": int(a["n_gauss1"])}

    mp_h, cur_h = synth_host.submap()
    mp = torch.from_numpy(mp_h).to(dev)
    cur = torch.from_numpy(cur_h).to(dev)
    out["map_2M"] = dict(workload="configs[4]: one 64-ch scan against the %d-point map, 75x24, 7 it" % mp.shape[1],
                         **latency(mp, mp.shape[1], cur_h, cur, cur.shape[1], args.calls))
    s1h = scans[1].cpu().numpy()
    out["single_64ch"] = dict(workload="configs[1]: one 64-ch pair (scan 0 as keyframe, scan 1), 75x24, 7 it",
                              **latency(scans[0], 131072, s1h, scans[1], 131072, args.calls))

    # ---- per-kernel device time (separate profiled pass)
    kfm = icet_b200.Keyframe.from_device(mp.data_ptr(), mp.shape[1], ctx=ctx)
    rk = torch.zeros((1, 56), dtype=torch.float32, device=dev)
    prof = {}
    for name, fn in (("throughput_4096_keyframe", arm_k), ("throughput_4096_batch", arm_b),
                     ("map_2M_keyframe", lambda: kfm.register_batch_device([cur.data_ptr()], [cur.shape[1]], rk.data_ptr())),
                     ("map_2M_register", lambda: ctx.register_batch_ptrs([mp.data_ptr()], [mp.shape[1]], [cur.data_ptr()],
                                                                         [cur.shape[1]], rk.data_ptr(), params=p,
                                                                         device=True))):
        ctx.set_profile(True)
        fn()
        k = ctx.get_profile()
        ctx.set_profile(False)
        tot = sum(v[0] for v in k.values())
        prof[name] = {"kernel_ms": {n: round(v[0], 4) for n, v in k.items() if v[1]},
                      "launches": {n: v[1] for n, v in k.items() if v[1]}, "sum_ms": round(tot, 4),
                      "k_cell_scan_share": round(k["k_cell_scan"][0] / tot, 4) if tot else None}
    out["profile"] = prof
    kfm.close()
    kf.close()
    out["all_identical"] = bool(same_a and out["map_2M"]["identical_bytes"] and out["single_64ch"]["identical_bytes"])
    ctx.close()
    print(json.dumps(out), flush=True)
    if not out["all_identical"]:
        raise SystemExit("keyframe_bench: the arms differ")


if __name__ == "__main__":
    main()
