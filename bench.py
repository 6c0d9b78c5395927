#!/usr/bin/env python
"""bench.py -- registrations/s of the ICET hot path on synthetic 64-channel scans (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W             (N > 1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR

A "step" registers the BASELINE.json configs[2] batch: --pairs-total (default 4096) consecutive scan pairs (64 rings x
2048 azimuth steps = 131 072 points per scan, 75 x 24 spherical voxels, 7 iterations, X0 = 0), pair-sharded by contiguous
range over the N ranks (strong scaling: 4096 / N pairs per GPU; no data-path collective, one all_gather of 48 floats per
pair closes each step).  --pairs-per-gpu P selects the weak-scaling form instead (N * P pairs).  Scans are resident in
HBM when the timed region starts (`value`), or start in pinned host memory (`e2e`, with a copy-only control that
measures what the host->device link of this box sustains with all ranks copying at once).  `configs` holds the other
BASELINE.json configurations (latency of one 64-channel pair, the 128-channel pair, scan-to-submap at 2 M points).

Prints ONE JSON line on rank 0.  --dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (see
dump_outputs): the inputs are a pure function of the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: bench.py writes nothing into it

RINGS, AZIM = 64, 2048
NPTS = RINGS * AZIM
RUNLEN, BINS_PHI, BINS_THETA, NMIN, THRESH, BUFF = 7, 24, 75, 25, 0.1, 0.1
SEED = 20240
METRIC = "registrations/s (64-ch, 75x24 vox, 7 it)"
README_PAIRS_PER_S = 1000.0 / 35.0  # reference README.md:59: 35 ms / pair on a Ryzen 5800X (other hardware)
B_ALG_PER_PAIR = 12 * (NPTS + NPTS) + 192  # SURVEY.md 8(d)
DEFAULT_CHUNK = 512  # pairs per launch of the device-resident batch (the library's default, icet_b200_set_chunk)
DUMP_LIMIT = 64_000_000  # bytes of all --dump-outputs files together (64 MB)
NPY_HEADER_MAX = 4096  # allowance per .npy file for its header (numpy writes 128 bytes for these arrays)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc, self.thr = gpu_index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thr = threading.Thread(target=self._read, daemon=True)
        self.thr.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if r[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def oracle_params():
    return dict(runlen=RUNLEN, bins_phi=BINS_PHI, bins_theta=BINS_THETA, n=NMIN, thresh=THRESH, buff=BUFF)


def cpu_time_sequence(scans_host: np.ndarray, threads: int):
    """Time the CPU restatement of the reference path (oracle, -O3 -march=native like the reference's
    CMakeLists.txt:38) on the given consecutive scans.  Returns (pairs/s, results)."""
    from oracle import pyoracle as po
    try:
        res, dt = po.run_sequence(scans_host, nthreads=threads, native=True, **oracle_params())
    except Exception:
        res, dt = po.run_sequence(scans_host, nthreads=threads, native=False, **oracle_params())
    return (scans_host.shape[0] - 1) / dt, res


def ref_time_sequence(scans_host: np.ndarray, threads: int):
    """Time the REFERENCE's own code (oracle/_ref: its unmodified src/icet.cpp, utils.cpp, ThreadPool.cpp compiled in the
    build container against the Eigen-API shim, see oracle/Makefile), one `ICET` object per pair like its callers.
    Returns pairs/s, or None when the library did not travel to this box."""
    from oracle import pyref
    for native in (True, False):
        if not os.path.exists(pyref.so_path(native)) and not os.path.isdir(os.path.join(pyref.REFERENCE, "src")):
            continue
        try:
            _, dt = pyref.run_sequence(scans_host, nthreads=threads, native=native, **oracle_params())
            return (scans_host.shape[0] - 1) / dt
        except Exception:
            continue
    return None


def cpu_baseline_measure(scans_host: np.ndarray, cores: int, warmup: int = 1, steps: int = 2):
    """The CPU baseline both arms report: `warmup` + `steps` passes over the sample with all host threads, the
    reference's own code when oracle/_ref is present (kind "reference"), else the oracle port (kind "port").  The
    port is timed as well (it is also the parity checker of the GPU results)."""
    sample = scans_host.shape[0] - 1
    ref_t, port_t, ores = [], [], None
    for s in range(warmup + steps):
        v = ref_time_sequence(scans_host, cores)
        pps, ores = cpu_time_sequence(scans_host, cores)
        if s >= warmup:
            port_t.append(sample / pps)
            if v:
                ref_t.append(sample / v)
    port = sample / float(np.mean(port_t))
    one_core, _ = cpu_time_sequence(scans_host[:5], 1)  # SURVEY.md 8(d)(i): one instance on one core
    if ref_t:
        value, kind = sample / float(np.mean(ref_t)), "reference"
        one_ref = ref_time_sequence(scans_host[:3], 1)
        note = ("%d consecutive synthetic 64-ch pairs per pass, %d host threads (one ICET object per pair, one pair per "
                "thread at a time), %d warm-up + %d timed passes; the reference's own sources (src/icet.cpp, utils.cpp, "
                "ThreadPool.cpp) built -O3 -march=x86-64-v3 in the build container against oracle/eigen_shim -- Eigen "
                "itself is not in the image: the reference's logic, allocations and libm calls are its own, Eigen's dense "
                "kernels are plain loops" % (sample, cores, warmup, steps))
    else:
        value, kind, one_ref = port, "port", None
        note = ("%d consecutive synthetic 64-ch pairs per pass, %d host threads, %d warm-up + %d timed passes; oracle "
                "restatement built -O3 -march=native (oracle/_ref did not travel to this box)" % (sample, cores, warmup, steps))
    cb = {"value": value, "unit": "pairs/s", "cores": cores, "kind": kind, "sample": note,
          "one_core_value": one_ref if one_ref else one_core, "port_value": port, "port_one_core_value": one_core}
    return cb, ores


def run_reference(args, rank: int, world: int):
    """Reference arm: the reference's own CPU implementation of the path on the box's host cores (oracle/_ref when it
    travelled, else the oracle port), all host threads, bounded sample of the same workload."""
    if rank != 0:
        return
    from tools import synth_host
    cores = os.cpu_count() or 1
    # one step = `sample` pairs: 2 per host thread (bounded so that the whole run ends within minutes)
    sample = max(2, min(2 * cores, 256))
    scans = synth_host.scans(sample + 1, first_scan=0, seed=SEED, rings=RINGS, azim=AZIM)
    cb, _ = cpu_baseline_measure(scans, cores, warmup=max(1, args.warmup), steps=args.steps)
    value = cb["value"]
    t = sample / value
    total, per_gpu, scaling = resolve_pairs(args, world)
    cfg = workload_config(per_gpu, world, scaling)
    cfg["pairs_per_step"] = sample          # what this arm really registers per step (a bounded sample of the batch)
    cfg["pairs_per_step_note"] = "bounded CPU sample of the %d-pair batch the GPU arm registers per step" % total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": scaling, "vs_baseline": value / README_PAIRS_PER_S, "dtype": "f32", "data": "synthetic",
        "config": cfg, "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def resolve_pairs(args, world: int):
    """(total pairs per step, pairs per GPU, "strong" | "weak")"""
    if args.pairs_per_gpu:
        return args.pairs_per_gpu * world, args.pairs_per_gpu, "weak"
    per = max(1, args.pairs_total // world)
    return per * world, per, "strong"


def workload_config(pairs_per_gpu: int, n_gpus: int, scaling: str = "strong") -> dict:
    return {"workload": "BASELINE.json configs[2]: batched synthetic 64-channel odometry sequence, consecutive pairs "
                        "(k,k+1), X0=0, pair-sharded by contiguous range (%s scaling)" % scaling,
            "points_per_scan": NPTS, "rings": RINGS, "azimuth_steps": AZIM, "voxels": "75x24",
            "iterations": RUNLEN, "pairs_per_gpu_per_step": pairs_per_gpu, "pairs_per_step": pairs_per_gpu * n_gpus,
            "l2_policy": "inputs larger than L2 (%d scans x 1.5 MiB per GPU)" % (pairs_per_gpu + 1),
            "seed": SEED}


def bench_callers(ctx, scans, stream, M):
    """Secondary measurements (not the headline metric): the reference's two ROS callbacks with every step on the
    device (include/icet_b200.h "callers either side of the path").
      odometry_chained: OdometryNode semantics (odometry.cpp: min range 2 m, 7 iterations, X0 <- X): M consecutive
        scans per call, ONE persistent kernel walks the pairs in chain order -- latency-bound by construction.
      mapmaker_batched: MapMakerNode's registration (simpleMapMaker.cpp: min range 0.2 m, 12 iterations, X0 = 0):
        independent pairs, throughput shape.
      map_add_scan: EigenQueue::add_new_scan on a full 600 000-point map: 2000 rows in, every row re-expressed
        (HBM-shaped streaming kernel, 24 B per map point; the 14.4 MB ring is L2 resident)."""
    import torch
    from icet_b200 import Node, PointMap, api
    dev = scans.device
    out = {}
    res = torch.zeros((M + 1, 56), dtype=torch.float32, device=dev)
    pose = torch.zeros((M + 1, 45), dtype=torch.float32, device=dev)
    for name, op, runlen in (("odometry_chained", api.OdometryParams(2.0, 1, 10.0, 0.0, 0.0), 7),
                             ("mapmaker_batched", api.OdometryParams(0.2, 0, 10.0, 0.3, 0.3), 12)):
        nd = Node(ctx, api.make_params(runlen, BINS_PHI, BINS_THETA, NMIN, THRESH, BUFF), op, NPTS)
        nd.push_device(scans.data_ptr(), M + 1, NPTS, res.data_ptr(), pose.data_ptr())  # warm-up, initialises the node
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        e0.record(stream)
        for r in range(reps):  # the sequence simply continues: scans (r+1)*M+1 .. (r+2)*M
            k = nd.push_device(scans[(r + 1) * M + 1].data_ptr(), M, NPTS, res.data_ptr(), pose.data_ptr())
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out[name] = {"pairs_per_s": k / (ms * 1e-3), "ms_per_pair": ms / k, "pairs_per_call": k, "iterations": runlen,
                     "min_range_m": float(op.min_range)}
        nd.close()
    cap = 600_000
    pm = PointMap(ctx, cap)
    X = torch.tensor([0.5, 0.01, -0.01, 0.001, -0.002, 0.01], dtype=torch.float32, device=dev)
    for k in range(6):  # fill the ring: 6 x 131 072 rows
        pm.add_scan_device(scans[k].data_ptr(), NPTS, NPTS, X.data_ptr(), count=NPTS)
    idx = np.arange(0, NPTS, NPTS // 2000, dtype=np.int32)[:2000]
    for _ in range(3):
        pm.add_scan_device(scans[7].data_ptr(), NPTS, NPTS, X.data_ptr(), idx=idx)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 50
    e0.record(stream)
    for _ in range(reps):
        pm.add_scan_device(scans[7].data_ptr(), NPTS, NPTS, X.data_ptr(), idx=idx)
    e1.record(stream)
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    peak, _ = peaks()
    gbs = cap * 24 / (us * 1e-6) / 1e9
    out["map_add_scan"] = {"us_per_insertion": us, "map_points": cap, "rows_in": 2000,
                           "algorithmic_bytes": cap * 24, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak,
                           "note": "two launches (enqueue + re-expression) and one 8 KB index upload per insertion; "
                                   "the ring (14.4 MB) stays in L2"}
    pm.close()
    return out


def bench_configs(ctx, stream, dev, latency):
    """The BASELINE.json configurations that are not the headline batch, one device-resident pair each:
    p50 / p95 of the call (CUDA events), the algorithmic bytes of SURVEY.md 8(d) (12 B per input point + 192 B of
    results) and the fraction of the HBM roofline they amount to."""
    import torch
    from icet_b200 import api
    from tools import synth_host
    peak, _ = peaks()

    def p50(s1, n1, s2, n2, p, reps):
        res = torch.zeros((1, 56), dtype=torch.float32, device=dev)
        lat = []
        for i in range(reps + 20):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            ctx.register_batch_ptrs([s1.data_ptr()], [n1], [s2.data_ptr()], [n2], res.data_ptr(), params=p, device=True)
            b.record(stream)
            torch.cuda.synchronize()
            if i >= 20:
                lat.append(a.elapsed_time(b))
        r = res.cpu().numpy().view(api.RESULT_DTYPE).reshape(-1)[0]
        return float(np.median(lat)), float(np.percentile(lat, 95)), r

    def entry(workload, n1, n2, m, q, r):
        b_alg = 12 * (n1 + n2) + 192
        return {"workload": workload, "p50_ms": m, "p95_ms": q, "algorithmic_bytes": b_alg,
                "achieved_gbs": b_alg / (m * 1e-3) / 1e9, "frac_of_hbm_peak": b_alg / (m * 1e-3) / 1e9 / peak,
                "gaussians": int(r["n_gauss1"]), "voxels_used": int(r["n_used"]), "status": int(r["status"])}

    out = {}
    if latency:
        b_alg = 12 * 2 * NPTS + 192
        out["latency_64ch"] = {"workload": "configs[1]: one synthetic 64-ch pair (131 072 points per scan), 75x24, 7 it",
                               "p50_ms": latency["device_resident_p50_ms"], "p95_ms": latency["device_resident_p95_ms"],
                               "host_api_pinned_p50_ms": latency["host_api_pinned_p50_ms"], "algorithmic_bytes": b_alg,
                               "achieved_gbs": b_alg / (latency["device_resident_p50_ms"] * 1e-3) / 1e9,
                               "frac_of_hbm_peak": b_alg / (latency["device_resident_p50_ms"] * 1e-3) / 1e9 / peak}
    n128 = 128 * 2048
    b = torch.empty((2, 3, n128), dtype=torch.float32, device=dev)
    ctx.synth_scans_device(b.data_ptr(), 2, first_scan=10, seed=SEED, rings=128, azim=2048)
    m, q, r = p50(b[0], n128, b[1], n128, api.make_params(10, 48, 150, NMIN, THRESH, BUFF), 100)
    out["ouster_128ch"] = entry("configs[3]: synthetic 128-channel pair (262 144 points per scan), 150x48, 10 it",
                                n128, n128, m, q, r)
    del b
    mp_h, cur_h = synth_host.submap()
    mp = torch.from_numpy(mp_h).to(dev)
    cur = torch.from_numpy(cur_h).to(dev)
    m, q, r = p50(mp, mp.shape[1], cur, NPTS, api.make_params(RUNLEN, BINS_PHI, BINS_THETA, NMIN, THRESH, BUFF), 50)
    out["submap_2M"] = entry("configs[4]: scan-to-submap, %d-point accumulated map (1240 scans x 2000 rays, exact "
                             "generator poses) vs one 64-ch scan, 75x24, 7 it" % mp.shape[1], mp.shape[1], NPTS, m, q, r)
    ctx.set_profile(True)   # per-kernel device time of this configuration (events around every launch)
    res = torch.zeros((1, 56), dtype=torch.float32, device=dev)
    for _ in range(3):
        ctx.register_batch_ptrs([mp.data_ptr()], [mp.shape[1]], [cur.data_ptr()], [NPTS], res.data_ptr(),
                                params=api.make_params(RUNLEN, BINS_PHI, BINS_THETA, NMIN, THRESH, BUFF), device=True)
    prof = ctx.get_profile()
    ctx.set_profile(False)
    out["submap_2M"]["kernel_ms"] = {k: round(v[0] / 3, 4) for k, v in prof.items() if v[1]}
    return out


def dump_outputs(out_dir: str, rows: np.ndarray, recs: np.ndarray) -> None:
    """--dump-outputs: the results of every pair of the last timed step, one DIR/<name>.npy per field.
    rows: [N, 48] float32, what a step returns (X | pred_stds | Q, in global pair order); recs: [N, 5] float32 words,
    the remaining fields of the same result records (status, n_gauss1, n_used, n_dropped as int32 bits, cond).
    Integer fields are written as float64 (exact).  When the files would exceed DUMP_LIMIT bytes, a fixed seeded
    sample of the pairs is written; pair_index.npy always names the pairs that were."""
    n = rows.shape[0]
    ints = np.ascontiguousarray(recs[:, :4]).view(np.int32).astype(np.float64)
    arrays = {"X": rows[:, 0:6], "pred_stds": rows[:, 6:12], "Q": rows[:, 12:48].reshape(n, 6, 6),
              "status": ints[:, 0], "n_gauss1": ints[:, 1], "n_used": ints[:, 2], "n_dropped": ints[:, 3],
              "cond": recs[:, 4], "pair_index": np.arange(n, dtype=np.float64)}
    per_pair = sum(a.nbytes for a in arrays.values()) // max(1, n)
    budget = DUMP_LIMIT - NPY_HEADER_MAX * len(arrays)
    if per_pair * n > budget:
        keep = np.sort(np.random.default_rng(SEED).choice(n, budget // per_pair, replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs-total", type=int, default=4096,
                    help="pairs per step over ALL ranks (BASELINE.json configs[2]: 4096; strong scaling)")
    ap.add_argument("--pairs-per-gpu", type=int, default=0,
                    help="weak-scaling form: this many pairs per step on every rank (overrides --pairs-total)")
    ap.add_argument("--no-configs", action="store_true", help="skip the 128-channel / submap configuration lines")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-callers", action="store_true", help="skip the odometry / map-maker node measurements")
    ap.add_argument("--lanes", type=int, default=0, help="compute lanes (0 = default 2)")
    ap.add_argument("--chunk", type=int, default=0, help="pairs per chunk of the device-resident path (0 = default)")
    ap.add_argument("--host-chunk", type=int, default=0, help="pairs per chunk of the host-buffer pipeline (0 = default)")
    ap.add_argument("--unfused", action="store_true", help="diagnostic: 3 launches per iteration instead of k_loop")
    ap.add_argument("--persistent", action="store_true", help="diagnostic: the persistent loop kernel for every chunk")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (GPU path only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the GPU path (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import icet_b200
    from icet_b200 import api, sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- icet_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if world != args.gpus and rank == 0:
        print("bench.py: warning: --gpus %d but WORLD_SIZE=%d" % (args.gpus, world), file=sys.stderr)

    total_pairs, P, scaling = resolve_pairs(args, world)
    ctx = icet_b200.Context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    if args.host_chunk:
        ctx.set_host_chunk(args.host_chunk)
    ctx.set_chunk(args.chunk or DEFAULT_CHUNK)
    if args.lanes:
        ctx.set_lanes(args.lanes)
    params = api.make_params(RUNLEN, BINS_PHI, BINS_THETA, NMIN, THRESH, BUFF,
                             flags=api.FLAG_UNFUSED_LOOP if args.unfused else
                             (api.FLAG_PERSISTENT_LOOP if args.persistent else 0))

    # synthetic sequence shard of this rank (contiguous pair range of the world*P-pair sequence), generated
    # on the device
    first_scan, nscans = sharding.shard_scans(world * P, rank, world)
    assert nscans == P + 1
    scans = torch.empty((P + 1, 3, NPTS), dtype=torch.float32, device=dev)
    for c0 in range(0, P + 1, 512):   # 512-scan slabs keep the generator's pose table small
        ctx.synth_scans_device(scans[c0].data_ptr(), min(512, P + 1 - c0), first_scan=first_scan + c0, seed=SEED,
                               rings=RINGS, azim=AZIM)
    results = torch.zeros((P, 56), dtype=torch.float32, device=dev)
    torch.cuda.synchronize()

    def step():
        ctx.register_sequence_device(scans.data_ptr(), P + 1, NPTS, results.data_ptr(), params)
        # final gather of poses + covariances (X 6 | pred_stds 6 | Q 36); no-op on one GPU
        return sharding.gather_results(results[:, :48], world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ------------------------------------------------------------
    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = ctx.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        rows = step()
    ev1.record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:  # before anything below reuses `results`
        recs = sharding.gather_results(results[:, 48:53], world)
        if rank == 0:
            dump_outputs(args.dump_outputs, rows.cpu().numpy(), recs.cpu().numpy())
    launches = ctx.kernel_launches - l0
    t_ms = ev0.elapsed_time(ev1)
    tt = torch.tensor([t_ms, float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = tt.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = tt.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        t_ms, launches = float(tmax[0]), int(tsum[1])
    value = world * P * args.steps / (t_ms * 1e-3)

    # ---- per-kernel device time (separate pass, events around every launch) -------------------------
    # (one compute lane here: with two, kernels of different chunks overlap and per-launch times are not additive)
    ctx.set_lanes(1)
    ctx.set_profile(True)
    ctx.register_sequence_device(scans.data_ptr(), P + 1, NPTS, results.data_ptr(), params)
    prof = ctx.get_profile()
    ctx.set_profile(False)
    ctx.set_lanes(args.lanes)
    tot_ms = sum(v[0] for v in prof.values())
    dom = max(prof, key=lambda k: prof[k][0])
    dom_ms, dom_n = prof[dom]
    peak, peak_src = peaks()
    # algorithmic bytes of one k_pass<scan2> launch: every scan-2 coordinate of the chunk read once
    # (12 B / point) -- DESIGN.md "Kernels"; other kernels: see DESIGN.md
    chunk_pairs = min(P, args.chunk or DEFAULT_CHUNK)
    alg_bytes = {"k_pass<scan2>": 12.0 * NPTS * chunk_pairs, "k_pass<scan1>": 12.0 * NPTS * chunk_pairs,
                 "k_prep2": 24.0 * NPTS * chunk_pairs, "k_scan1_bin": 20.0 * NPTS * chunk_pairs}.get(dom)
    roofline = {"bound": "hbm", "kernel": dom, "unit": "GB/s", "peak": peak, "peak_source": peak_src,
                "traffic": None, "kernel_share_of_step": dom_ms / tot_ms if tot_ms else None,
                "avg_launch_ms": dom_ms / dom_n if dom_n else None}
    # DRAM bytes per launch of that kernel from the latest committed `ncu --set full` capture
    # (dram__bytes_read.sum + dram__bytes_write.sum; profiles/traffic.json, written by tools/profile_summary.py),
    # scaled to this run's pairs per launch
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f).get(dom)
        if tj:
            roofline["traffic"] = (tj["dram_bytes_read"] + tj["dram_bytes_write"]) * chunk_pairs / tj["pairs_per_launch"]
            roofline["traffic_source"] = "ncu --set full, visit %s (profiles/%s.md)" % (tj["visit"], tj["visit"])
    except Exception:
        pass
    if alg_bytes and dom_n:
        ach = alg_bytes / (dom_ms / dom_n * 1e-3) / 1e9
        roofline.update({"achieved": ach, "frac": ach / peak, "algorithmic_bytes_per_launch": alg_bytes})
    path_gbs = B_ALG_PER_PAIR * (value / world) / 1e9
    roofline_path = {"algorithmic_bytes_per_pair": B_ALG_PER_PAIR, "achieved_gbs_per_gpu": path_gbs,
                     "frac": path_gbs / peak}

    # ---- end to end through the C ABI with HOST buffers -----------------------------------------------
    e2e = None
    if not args.no_e2e:
        host_scans = torch.empty((P + 1, 3, NPTS), dtype=torch.float32, pin_memory=True)
        host_scans.copy_(scans)
        torch.cuda.synchronize()
        host_out = torch.zeros((P, 56), dtype=torch.float32, pin_memory=True)
        ptr0 = host_scans.data_ptr()
        stride = 3 * NPTS * 4
        p1 = np.array([ptr0 + i * stride for i in range(P)], np.uint64)        # the caller's pointer tables, built once
        p2 = np.array([ptr0 + (i + 1) * stride for i in range(P)], np.uint64)
        nn = np.full(P, NPTS, np.int32)

        def e2e_step():
            ctx.register_batch_ptrs(p1, nn, p2, nn, host_out.data_ptr(), params=params, device=False)

        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        nst = args.steps
        for _ in range(nst):
            e2e_step()
        barrier()
        wall = time.perf_counter() - t0
        # copy-only control: the very same host buffer -> device memory, no kernels, all ranks at once: what the
        # host->device path of THIS box sustains (PCIe link, host memory / NUMA placement, shared root ports)
        sink = torch.empty((min(P + 1, 512), 3, NPTS), dtype=torch.float32, device=dev)
        def copy_only():
            for c0 in range(0, P + 1, sink.shape[0]):
                m = min(sink.shape[0], P + 1 - c0)
                sink[:m].copy_(host_scans[c0:c0 + m], non_blocking=True)
        copy_only()
        barrier()
        c0t = time.perf_counter()
        ncp = 3
        for _ in range(ncp):
            copy_only()
        barrier()
        cwall = time.perf_counter() - c0t
        tw = torch.tensor([wall, cwall], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        del sink
        h2d = int((P + 1) * stride + P * 24)
        e2e_v = world * P * nst / float(tw[0])
        ceil_gbs = world * (P + 1) * stride * ncp / float(tw[1]) / 1e9
        ceil_pairs = world * P * ncp / float(tw[1])
        e2e = {"value": e2e_v, "unit": "pairs/s", "steps": nst,
               "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": int(P * 224) * world,
               "h2d_gbs_achieved": h2d * world * nst / float(tw[0]) / 1e9,
               "h2d_ceiling_gbs": ceil_gbs, "h2d_ceiling_pairs_per_s": ceil_pairs, "frac_of_h2d_ceiling": e2e_v / ceil_pairs,
               "note": "icet_b200_register_batch on pinned host scans (each scan uploaded once), results copied back; "
                       "host wall clock around blocking calls, max over ranks.  h2d_ceiling_*: copy-only control (the same "
                       "pinned buffers copied to the device by all ranks at once, no kernels): the limiter of e2e is the "
                       "host->device path, not the kernels (value) and not NCCL"}
        del host_scans
    # ---- single-pair latency (BASELINE.json configs[1]) -----------------------------------------------------
    latency = None
    if rank == 0 and not args.no_latency:
        res1 = torch.zeros((1, 56), dtype=torch.float32, device=dev)
        lat = []
        for i in range(230):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            ctx.register_sequence_device(scans.data_ptr(), 2, NPTS, res1.data_ptr(), params)
            b.record(stream)
            torch.cuda.synchronize()
            if i >= 30:
                lat.append(a.elapsed_time(b))
        h1 = scans[0].cpu().numpy()
        h2 = scans[1].cpu().numpy()
        hl = []
        for i in range(220):
            t0 = time.perf_counter()
            ctx.register(h1, h2, params=params)
            if i >= 20:
                hl.append((time.perf_counter() - t0) * 1e3)
        # the same blocking call from PINNED host buffers (what the e2e contract assumes; the 3 MB upload then runs at
        # link speed instead of through the driver's staging copies)
        pin = torch.empty((2, 3, NPTS), dtype=torch.float32, pin_memory=True)
        pin.copy_(scans[:2])
        torch.cuda.synchronize()
        p1n, p2n = pin[0].numpy(), pin[1].numpy()
        hp = []
        for i in range(220):
            t0 = time.perf_counter()
            ctx.register(p1n, p2n, params=params)
            if i >= 20:
                hp.append((time.perf_counter() - t0) * 1e3)
        latency = {"workload": "configs[1]: one synthetic 64-ch pair, 75x24, 7 it", "device_resident_p50_ms": float(np.median(lat)),
                   "device_resident_p95_ms": float(np.percentile(lat, 95)), "host_api_p50_ms": float(np.median(hl)),
                   "host_api_p95_ms": float(np.percentile(hl, 95)), "host_api_pinned_p50_ms": float(np.median(hp)),
                   "host_api_pinned_p95_ms": float(np.percentile(hp, 95)), "reps": len(lat)}

    # ---- callers either side of the path (SURVEY.md 8f N1 / N2): device-resident node callbacks ------------------
    callers = None
    if rank == 0 and not args.no_callers:
        callers = bench_callers(ctx, scans, stream, max(1, min(P // 4, 128)))

    # ---- the other BASELINE.json configurations (rank 0) ------------------------------------------------------------
    configs = None
    if rank == 0 and not args.no_configs:
        configs = bench_configs(ctx, stream, dev, latency)

    # ---- CPU baseline beside it (rank 0, N = 1 only): the reference's CPU path on the box's host cores ---------------
    cpu_baseline = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        sample = max(2, min(2 * cores, P, 256))
        hs = scans[: sample + 1].cpu().numpy()
        cpu_baseline, ores = cpu_baseline_measure(hs, cores)
        g = results[:sample].cpu().numpy()
        parity = {"pairs_checked": sample, "max_abs_dX_m": float(np.abs(g[:, :3] - ores[:, :3]).max()),
                  "max_abs_dX_rad": float(np.abs(g[:, 3:6] - ores[:, 3:6]).max()),
                  "note": "GPU results of the timed batch against the oracle port (sorted order, like the product's default)"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_ms / args.steps, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": value / README_PAIRS_PER_S,
            "baseline_note": "reference README.md:59: 35 ms/pair (28.6 pairs/s) on a Ryzen 5800X CPU",
            "dtype": "f32", "data": "synthetic", "config": workload_config(P, world, scaling), "clocks": clocks,
            "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "roofline_path": roofline_path,
            "cpu_baseline": cpu_baseline, "latency": latency, "configs": configs, "parity_vs_oracle": parity,
            "callers": callers,
            "kernel_ms_per_step": {k: round(v[0], 4) for k, v in prof.items()},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
