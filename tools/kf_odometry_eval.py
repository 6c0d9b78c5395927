"""Keyframe odometry against frame-to-frame odometry on one synthetic sequence (DESIGN.md §13).

Both nodes (icet_b200.OdometryNode's device node and icet_b200.KeyframeOdometryNode) run the same 64 x 2048 synthetic
scans (tools/synth_host.scans, seed 20240).  The ground truth is the generator's motion of every step
(synth_host.motions) composed as the nodes compose their poses, X_homo_k = X_homo_{k-1} Hi(motion_{k-1}): the
mapping test_full_size_sequence_properties uses for single steps (checked first on the odometry node's per-step X).

Prints one JSON line: per node the end-point translation / rotation drift, the relative translation error per 100 m
of travel, keyframes promoted and why, scans/s of push_device in blocks of 64 and p50 / p95 of a blocking push; the
GPU's name and power limit; and, with --sweep, the drift of a few policies (how the defaults were chosen).

With --local-map the same for local-map nodes (map_keyframes = M, DESIGN.md §14) at M in --map-keyframes, plus the
map's rows (mean / max over promotions), the same M without the overlap test, a max_trans sweep at the M > 1 with the
lowest relative error, and a
torch.profiler run of one push_device block per M: device time per kernel, so that the map assembly and the candidate
fit of the promoted scans and the empty fit of the others can be told apart.

    python tools/kf_odometry_eval.py --scans 1000 [--sweep] [--local-map] [--seed 20240]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True


def homo(X):
    from oracle import kf_odometry_oracle as no
    return no.homogeneous(X).astype(np.float64)


def ground_truth(motions):
    G = [np.eye(4)]
    for m in motions:
        G.append(G[-1] @ homo(m))
    return np.array(G)


def drift(E, G):
    """E, G: [N, 4, 4] estimated / true poses of scans 0 .. N-1."""
    dt = float(np.linalg.norm(E[-1][:3, 3] - G[-1][:3, 3]))
    Rd = E[-1][:3, :3].T @ G[-1][:3, :3]
    dr = float(np.arccos(np.clip((np.trace(Rd) - 1) / 2, -1, 1)))
    seg = np.linalg.norm(np.diff(G[:, :3, 3], axis=0), axis=1)
    cum = np.concatenate([[0.0], np.cumsum(seg)])
    errs = []
    for i in range(0, len(G), 5):
        j = int(np.searchsorted(cum, cum[i] + 100.0))
        if j >= len(G):
            break
        rg = np.linalg.inv(G[i]) @ G[j]
        re = np.linalg.inv(E[i]) @ E[j]
        errs.append(np.linalg.norm(rg[:3, 3] - re[:3, 3]) * 100.0 / (cum[j] - cum[i]))
    return {"end_trans_m": dt, "end_rot_rad": dr, "rte_m_per_100m": float(np.mean(errs)) if errs else None,
            "path_m": float(cum[-1])}


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return name, pl


def run_device(make, dev, n, block):
    """push_device in blocks; returns results / poses / infos (numpy) and the elapsed seconds (synchronised)."""
    import torch
    from icet_b200 import api
    ns = dev.shape[0]
    node, kf = make()
    res = torch.zeros((ns, 56), dtype=torch.float32, device="cuda")
    pose = torch.zeros((ns, 45), dtype=torch.float32, device="cuda")
    info = torch.zeros((ns, 10), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    done = 0
    for c0 in range(0, ns, block):
        m = min(block, ns - c0)
        if kf:
            done += node.push_device(dev[c0].data_ptr(), m, n, res[done].data_ptr(), pose[done].data_ptr(),
                                     info[done].data_ptr())
        else:
            done += node.push_device(dev[c0].data_ptr(), m, n, res[done].data_ptr(), pose[done].data_ptr())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    node.close()
    r = res[:done].cpu().numpy().view(api.RESULT_DTYPE).reshape(-1)
    p = pose[:done].cpu().numpy().view(api.POSE_DTYPE).reshape(-1)
    i = info[:done].cpu().numpy().view(api.KF_INFO_DTYPE).reshape(-1)
    return r, p, i, dt


def map_rows(p, i, n0, M):
    """rows of every map a promotion built: the kept counts (pose.n_points) of the last M keyframes, keyframe 0 whole"""
    kept = [n0] + [int(x) for x in p["n_points"][i["promoted"] != 0]]
    return [sum(kept[max(0, j + 1 - M): j + 1]) for j in range(len(kept))]


def kernel_profile(make, dev, n, block):
    """device time per kernel (torch.profiler, CUDA activity) of one push_device block: {name: [launches, total us]}"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    node, _ = make()
    ns = min(block, dev.shape[0])
    res = torch.zeros((ns, 56), dtype=torch.float32, device="cuda")
    pose = torch.zeros((ns, 45), dtype=torch.float32, device="cuda")
    info = torch.zeros((ns, 10), dtype=torch.float32, device="cuda")
    node.push_device(dev[0].data_ptr(), ns, n, res.data_ptr(), pose.data_ptr(), info.data_ptr())   # warm-up
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        node.push_device(dev[ns].data_ptr(), ns, n, res.data_ptr(), pose.data_ptr(), info.data_ptr())
        torch.cuda.synchronize()
    promoted = int(info.cpu().numpy().view(np.int32).reshape(ns, 10)[:, 1].sum())
    node.close()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0 and "Memcpy" not in e.key and "Memset" not in e.key:
            name = e.key.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0]
            out[name] = [int(e.count), round(float(t), 1)]
    return {"scans": ns, "promoted": promoted, "kernels": out}


def local_map_rows(a, ctx, dev, n, G, kfn, poses, reasons, blocking):
    from icet_b200 import api
    ns = dev.shape[0]
    default = api.KeyframePolicy()
    rows = []
    for M in [int(x) for x in a.map_keyframes.split(",")]:
        run_device(kfn(default, M), dev[:65], n, a.block)   # warm-up: workspace of the M * cap fit
        r, p, i, dt = run_device(kfn(default, M), dev, n, a.block)
        d = drift(poses(p), G)
        mr = map_rows(p, i, n, M)
        d.update(map_keyframes=M, keyframes=int(i["promoted"].sum()), reasons=reasons(i),
                 status_nonzero=int((r["status"] != 0).sum()), scans_per_s=(ns - 1) / dt,
                 map_rows_mean=float(np.mean(mr)), map_rows_max=int(np.max(mr)),
                 n_gauss1_mean=float(np.mean(r["n_gauss1"])), n_used_mean=float(np.mean(r["n_used"])),
                 blocking_push=blocking(kfn(default, M)))
        rows.append(d)
    # the overlap test compares n_used with the map's Gaussian count, which grows with M: the same rows without it
    no_overlap = []
    for M in [int(x) for x in a.map_keyframes.split(",")]:
        pol = api.KeyframePolicy(max_trans=1.0, max_rot=0.1, min_overlap=0.0, max_interval=10)
        r, p, i, dt = run_device(kfn(pol, M), dev, n, a.block)
        d = drift(poses(p), G)
        d.update(map_keyframes=M, keyframes=int(i["promoted"].sum()), reasons=reasons(i))
        no_overlap.append(d)
    # the max_trans sweep at the M > 1 with the lowest relative error (M = 1 is the sweep of DESIGN.md §13)
    best = min([d for d in rows if d["map_keyframes"] > 1] or rows, key=lambda d: d["rte_m_per_100m"])["map_keyframes"]
    sweep = []
    for mt in (0.5, 0.75, 1.5, 2.0):
        pol = api.KeyframePolicy(max_trans=mt, max_rot=0.1, min_overlap=0.5, max_interval=10)
        r, p, i, dt = run_device(kfn(pol, best), dev, n, a.block)
        d = drift(poses(p), G)
        d.update(map_keyframes=best, max_trans=mt, keyframes=int(i["promoted"].sum()), reasons=reasons(i))
        sweep.append(d)
    prof = {}
    for M in [int(x) for x in a.map_keyframes.split(",")]:
        try:
            prof[str(M)] = kernel_profile(kfn(default, M), dev, n, a.block)
        except Exception as e:   # the profiler is a diagnostic: report, do not lose the measurements above
            prof[str(M)] = {"error": repr(e)}
    return {"rows": rows, "overlap_off": no_overlap, "sweep_map_keyframes": best, "max_trans_sweep": sweep,
            "profile": prof}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=1000)
    ap.add_argument("--block", type=int, default=64)
    ap.add_argument("--blocking", type=int, default=200, help="scans of the blocking-push latency measurement")
    ap.add_argument("--sweep", action="store_true", help="also measure the drift of a few policies")
    ap.add_argument("--local-map", action="store_true", help="also measure local-map nodes")
    ap.add_argument("--map-keyframes", default="1,2,3,4,6", help="M values of --local-map")
    ap.add_argument("--seed", type=int, default=20240, help="seed of the synthetic sequence")
    a = ap.parse_args()
    import torch
    from icet_b200 import KeyframeOdometryNode, Node, api
    from tools import synth_host
    ctx = api.Context(0)
    ns, n = a.scans, 64 * 2048
    dev = torch.empty((ns, 3, n), dtype=torch.float32, device="cuda")
    for c0 in range(0, ns, 64):
        m = min(64, ns - c0)
        dev[c0:c0 + m] = torch.from_numpy(synth_host.scans(m, first_scan=c0, seed=a.seed))
    torch.cuda.synchronize()
    G = ground_truth(synth_host.motions(0, ns - 1, seed=a.seed))

    def odo():
        return Node(ctx, api.make_params(), api.OdometryParams(2.0, 1, 10.0, 0.0, 0.0), n), False

    def kfn(pol, M=None):
        return lambda: (KeyframeOdometryNode(ctx, max_points=n, policy=pol, map_keyframes=M), True)

    def poses(p):
        return np.concatenate([np.eye(4)[None], p["X_homo"].astype(np.float64)])

    def reasons(i):
        names = {"trans": api.KF_TRANS, "rot": api.KF_ROT, "overlap": api.KF_OVERLAP, "interval": api.KF_INTERVAL,
                 "status": api.KF_STATUS}
        return {k: int(((i["reason"] & b) != 0).sum()) for k, b in names.items()}

    def blocking(make):
        node, kf = make()
        host = [dev[k].cpu().numpy() for k in range(min(a.blocking + 1, ns))]
        lat = []
        for k, s in enumerate(host):
            t0 = time.perf_counter()
            node.callback(s) if kf else node.push(s)
            if k > 0:
                lat.append(time.perf_counter() - t0)
        node.close()
        return {"p50_ms": 1e3 * float(np.percentile(lat, 50)), "p95_ms": 1e3 * float(np.percentile(lat, 95))}

    out = {"scans": ns, "points_per_scan": n, "seed": a.seed}
    out["gpu"], out["power_limit"] = gpu_info()
    default = api.KeyframePolicy()
    out["default_policy"] = {f: getattr(default, f) for f in ("max_trans", "max_rot", "min_overlap", "max_interval")}
    # warm-up of both nodes (module load, workspace growth), then the measured passes
    run_device(odo, dev[:65], n, a.block)
    run_device(kfn(default), dev[:65], n, a.block)
    for name, make in (("odometry", odo), ("keyframe", kfn(default))):
        r, p, i, dt = run_device(make, dev, n, a.block)
        d = drift(poses(p), G)
        d["scans_per_s"] = (ns - 1) / dt
        d["blocking_push"] = blocking(make)
        d["status_nonzero"] = int((r["status"] != 0).sum())
        if name == "keyframe":
            d["keyframes"] = int(i["promoted"].sum())
            d["reasons"] = reasons(i)
        else:
            et = np.abs(r["X"][:, :3] - synth_host.motions(0, ns - 1, seed=a.seed)[:, :3]).max(1)
            d["step_error_median_m"] = float(np.median(et))   # the ground-truth mapping, checked on single steps
        out[name] = d
    if a.sweep:
        sweep = []
        for mi in (5, 10, 20):
            for mt in (0.5, 0.75, 1.0, 1.5, 2.0, 4.0):
                pol = api.KeyframePolicy(max_trans=mt, max_rot=0.1, min_overlap=0.5, max_interval=mi)
                r, p, i, dt = run_device(kfn(pol), dev, n, a.block)
                d = drift(poses(p), G)
                d.update(max_interval=mi, max_trans=mt, keyframes=int(i["promoted"].sum()), reasons=reasons(i))
                sweep.append(d)
        out["sweep"] = sweep
    if a.local_map:
        out["local_map"] = local_map_rows(a, ctx, dev, n, G, kfn, poses, reasons, blocking)
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
