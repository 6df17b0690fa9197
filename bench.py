#!/usr/bin/env python
"""bench.py -- scans/sec of the FAST-LIO2 iEKF measurement update (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one whole update of one synthetic scan: every iEKF pass of
update_iterated_dyn_share_modified, kNN included -- ONE launch of the persistent kernel k_update.  Workload at any N: BASELINE.json
configs[1] ("velodyne.yaml synthetic: 30k pts/scan vs 1M-pt map, 4 iEKF iters").

  value   scans/s with the scan, the map and the prior state resident in HBM
          (CUDA events on the launching stream around each step; L2 flushed before every
          timed step with a 256 MB memset outside the events; max over ranks).
  e2e     scans/s through the public C-ABI call fl_filter_update() with HOST buffers:
          scan + state host->device and state device->host inside the timed region.
  roofline  the kNN phase of one searching pass (the dominant part of the step), launched alone -- the persistent kernel
          k_update in its search_only mode -- and timed with CUDA events: algorithmic bytes per launch
          (SURVEY.md 8d: 16 + 32*ceil(log2 N) + 32*k per point) / launch time, against MEASURED_PEAKS.json's HBM copy bandwidth.
  parity  the resident and the e2e state against the final state of the cpu_baseline leg (same scan, same prior);
          above the north-star tolerance (1e-4 m / 1e-4 rad) the run exits with status 3.
  cpu_baseline  the reference's CPU path (its unmodified ikd-Tree from oracle/_ref + the
          restated h_share_model / esekf update) on this box's host cores, bounded sample.

--impl reference times that CPU path as the arm itself (rank 0 only under torchrun).

--dump-outputs DIR writes what the timed path returned for its last step as DIR/<name>.npy (float64 / float32):
x (26) and P (23x23), the updated state and covariance, and with one process the per-point outputs of the last
search pass: nearest (Q x 5 x 4, the plane points), nearest_count (Q) and selected (Q, point_selected_surf).  The
workloads are generated from fixed seeds, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "scans/sec (30k-pt scan, 1M-pt map iEKF)"
UNIT = "scans/s"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None
        self.thread = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- helpers
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def algorithmic_bytes_search(n_map: int, k: int = 5) -> int:
    """SURVEY.md 8(d): B_s = 16 + 32*ceil(log2 N) + 16k + 16k per (point, search pass)."""
    return 16 + 32 * math.ceil(math.log2(max(2, n_map))) + 32 * k


import contextlib


@contextlib.contextmanager
def c_stdout_to_stderr():
    """The reference's ikd_Tree.cpp printf()s to stdout (ikd_Tree.cpp:202,365); bench.py's stdout must carry
    exactly one JSON line, so file descriptor 1 points at stderr while the CPU oracle runs."""
    sys.stdout.flush()
    saved = os.dup(1)
    try:
        os.dup2(2, 1)
        yield
    finally:
        try:
            import ctypes
            ctypes.CDLL(None).fflush(None)
        except Exception:
            pass
        os.dup2(saved, 1)
        os.close(saved)


_CPU_CAL = {}


def cpu_update_loop(pr, n_scans: int, nthreads: int, warm: int = 3):
    """Times the CPU reference path (the reference's unmodified ikd-Tree + the restated h_share_model / update).

    The reference's OpenMP loop (laserMapping.cpp:646-650) does not scale to every core count (allocation inside
    KD_TREE::Nearest_Search), so the thread count is calibrated ONCE per process -- 5 scans each at nproc, nproc/2, ...
    >= 4, the candidate with the best median wins -- with the OpenMP threads pinned (OMP_PROC_BIND / OMP_PLACES are set
    by main() before any OpenMP runtime starts).  Then `warm` untimed scans and n_scans timed ones; the figure
    reported is the MEDIAN.  The reference's own default of 3 threads (CMakeLists.txt:23-26: MP_PROC_NUM = 3 on hosts
    with more than 4 cores) is timed beside it.  Returns a dict."""
    from oracle import bind
    tree = bind.KdTree(pr.map_pts, "auto")
    kind = "reference" if tree.backend == "reference" else "port"
    last = {}

    def one(nt):
        t0 = time.perf_counter()
        last["r"] = bind.update_iterated(tree, pr.scan, pr.x_prior, pr.P_prior, pr.cfg.max_iter, pr.R, pr.limit,
                                         pr.extrinsic_est_en, nthreads=nt)
        return time.perf_counter() - t0

    one(nthreads)                                   # warm the tree / page cache
    key = (pr.cfg.name, nthreads)
    if key not in _CPU_CAL:
        cands, nt = [], nthreads
        while nt >= 4:
            cands.append(nt)
            nt //= 2
        if not cands:
            cands = [max(1, nthreads)]
        med = {c: float(np.median([one(c) for _ in range(5)])) for c in cands}
        _CPU_CAL[key] = (min(cands, key=lambda c: med[c]), med)
    best, med = _CPU_CAL[key]
    for _ in range(max(3, warm)):
        one(best)
    times = [one(best) for _ in range(n_scans)]
    t3 = [one(3) for _ in range(7)][2:]
    result = last["r"]
    tree.close()
    return {"times": times, "median_s": float(np.median(times)), "mean_s": float(np.mean(times)), "kind": kind, "threads": best,
            "calibration_ms": {str(c): round(1e3 * v, 2) for c, v in med.items()},
            "median_s_3_threads": float(np.median(t3)), "x": result.x, "P": result.P, "result": result}


def dump_outputs(out_dir, arrays):
    """One .npy per array; integer outputs are stored as float32 (exact for counts and flags)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float32)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def rot_angle(qa, qb):
    qa = np.asarray(qa) / np.linalg.norm(qa); qb = np.asarray(qb) / np.linalg.norm(qb)
    return 2.0 * math.acos(min(1.0, abs(float(np.dot(qa, qb)))))


def state_parity(x, P, xo, Po):
    """North-star tolerance: 1e-4 m / 1e-4 rad on the state, against the CPU reference path's result on the same input."""
    pos = float(np.abs(x[0:3] - xo[0:3]).max())
    rot = max(rot_angle(x[3:7], xo[3:7]), rot_angle(x[7:11], xo[7:11]))
    rest = float(np.abs(x[11:] - xo[11:]).max())
    scale = np.sqrt(np.outer(np.diag(Po), np.diag(Po)))
    cov = float((np.abs(P - Po) / scale).max())
    return {"pos_err": pos, "rot_err": rot, "other_err": rest, "cov_rel_err": cov, "tol": 1e-4,
            "ok": bool(pos <= 1e-4 and rot <= 1e-4 and rest <= 1e-4 and cov <= 1e-3),
            "against": "cpu_baseline leg's final state (reference ikd-Tree + restated update), same scan / prior"}


# ----------------------------------------------------------------------------- reference arm
def run_reference(args, rank: int):
    if rank != 0:
        return 0
    from fast_lio_b200 import synth
    pr = synth.make_problem(args.workload)
    cores = os.cpu_count() or 1
    with c_stdout_to_stderr():
        c = cpu_update_loop(pr, args.steps, cores, warm=args.warmup)
    times = c["times"]
    val = 1.0 / c["median_s"]
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": max(3, args.warmup), "ms_per_step": 1e3 * c["median_s"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32 geometry / f64 filter", "data": "synthetic",
        "config": {"workload": args.workload, "n_map": pr.cfg.n_map, "n_scan": pr.cfg.n_scan, "max_iteration": pr.cfg.max_iter},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": c["threads"], "kind": c["kind"],
                         "sample": f"median of {len(times)} full scan updates of the same workload (mean {1e3 * c['mean_s']:.2f} ms), OpenMP over scan points, "
                                   f"threads pinned, thread count calibrated once (5 scans per candidate: {c['calibration_ms']} ms)",
                         "host_cores": os.cpu_count(), "value_3_threads": 1.0 / c["median_s_3_threads"],
                         "note_3_threads": "the reference's compiled-in default MP_PROC_NUM = 3 (CMakeLists.txt:23-26)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if args.dump_outputs:
        r = c["result"]
        dump_outputs(args.dump_outputs, {"x": r.x, "P": r.P, "nearest": r.nearest, "nearest_count": r.nearest_cnt,
                                         "selected": r.selected})
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------- our arm
def run_ours(args, rank: int, world: int, local_rank: int):
    import torch
    import torch.distributed as dist
    from fast_lio_b200 import api, synth

    if api.device_count() <= local_rank:
        raise SystemExit("bench.py: no CUDA device for this rank (the product has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))

    pr = synth.make_problem(args.workload)
    Q = len(pr.scan)
    tree = api.KdTree(local_rank, 0.5)
    tree.Build(pr.map_pts)                       # map replicated on every rank
    filt = api.Esekf(tree, max_points=Q, max_iter=pr.cfg.max_iter, limit=pr.limit,
                     extrinsic_est_en=bool(pr.extrinsic_est_en), solver=args.solver, search=args.search)
    if world > 1:
        comm = args.comm
        if comm == "p2p":
            # fused all-reduce over NVLink peer memory (CUDA IPC mailboxes), no NCCL on the data path;
            # the choice is collective: if any rank cannot map its peers, every rank uses NCCL
            ok = 1
            try:
                handles = [None] * world
                dist.all_gather_object(handles, filt.p2p_handle())
                filt.p2p_connect(world, rank, b"".join(handles))
            except api.FastLioError as e:
                print(f"bench.py[rank {rank}]: peer-memory exchange unavailable ({e})", file=sys.stderr)
                ok = 0
            flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 0:
                comm = "nccl"
                filt = api.Esekf(tree, max_points=Q, max_iter=pr.cfg.max_iter, limit=pr.limit,
                                 extrinsic_est_en=bool(pr.extrinsic_est_en), solver=args.solver, search=args.search)
        if comm == "nccl":
            uid = [api.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            filt.comm_init(world, rank, uid[0])
        args.comm = comm
        lo, hi = api.shard_range(Q, world, rank)
        filt.set_shard(lo, hi)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident path ("value")
    filt.upload_scan(pr.scan)
    filt.upload_state(pr.x_prior, pr.P_prior, pr.R)
    filt.time_resident(max(3, args.warmup), flush_l2=True)          # warm-up (>= 3 steps)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t_wall0 = time.perf_counter()
    ms_total = filt.time_resident(args.steps, flush_l2=True)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = filt.gpu_launches() * args.steps
    x_res, P_res, n_pass = filt.download_state()
    if args.dump_outputs:
        outputs = {"x": x_res, "P": P_res}
        if world == 1:
            outputs["nearest"], outputs["nearest_count"] = filt.nearest(Q)
            outputs["selected"] = filt.selected(Q)
    ms_warm = filt.time_resident(args.steps, flush_l2=False)
    # ---- dominant kernel alone
    ms_search = filt.time_search_pass(max(5, args.steps), flush_l2=True) / max(5, args.steps)
    ms_search_warm = filt.time_search_pass(max(5, args.steps), flush_l2=False) / max(5, args.steps)

    # ---- end-to-end through the C ABI with host buffers ("e2e"); the scan buffer is page-locked once,
    #      as an application reusing its scan buffer would do (fl_host_register)
    api.host_register(pr.scan)
    for _ in range(max(3, args.warmup)):
        filt.update_iterated_dyn_share_modified(pr.scan, pr.x_prior, pr.P_prior, pr.R)
    barrier()
    # the K calls are issued from native code (fl_filter_time_e2e loops the public fl_filter_update), as the reference's
    # C++ caller would: the ctypes/numpy marshalling of this harness (~20 us per call) is not part of the library
    t0 = time.perf_counter()
    e2e_native_s, x_e2e, P_e2e = filt.time_e2e(pr.scan, pr.x_prior, pr.P_prior, pr.R, args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    n_py = min(args.steps, 300)                            # the same call through this harness's Python wrapper, for the record
    t0 = time.perf_counter()
    for _ in range(n_py):
        filt.update_iterated_dyn_share_modified(pr.scan, pr.x_prior, pr.P_prior, pr.R)
    e2e_py_s = (time.perf_counter() - t0) / n_py
    clocks = sampler.stop()

    if world > 1:
        tt = torch.tensor([ms_total, e2e_s, ms_warm, ms_search], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total, e2e_s, ms_warm, ms_search = [float(v) for v in tt.tolist()]

    if rank == 0:
        peak, peak_src = load_peaks()
        shard = api.shard_range(Q, world, rank)
        n_local = shard[1] - shard[0]
        bytes_launch = algorithmic_bytes_search(pr.cfg.n_map) * n_local
        achieved = bytes_launch / (ms_search * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("k_search_dram_bytes_per_launch")
            except Exception:
                traffic = None
        # CPU baseline on a bounded sample (about 10-30 s of CPU work)
        cpu = None
        parity = None
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            with c_stdout_to_stderr():
                c = cpu_update_loop(pr, max(20, args.cpu_scans), cores)
            cpu = {"value": 1.0 / c["median_s"], "unit": UNIT, "cores": c["threads"], "kind": c["kind"],
                   "sample": f"median of {len(c['times'])} full scan updates of the same workload ({1e3 * c['median_s']:.2f} ms/scan, mean {1e3 * c['mean_s']:.2f}), "
                             f"threads pinned, thread count calibrated once ({c['calibration_ms']} ms)",
                   "host_cores": os.cpu_count(), "value_3_threads": 1.0 / c["median_s_3_threads"]}
            parity = state_parity(x_res, P_res, c["x"], c["P"])
            parity["e2e_path"] = state_parity(x_e2e, P_e2e, c["x"], c["P"])["ok"]
        line = {
            "metric": METRIC, "value": args.steps / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32 geometry / f64 filter", "data": "synthetic",
            "config": {"workload": args.workload, "n_map": pr.cfg.n_map, "n_scan": pr.cfg.n_scan,
                       "max_iteration": pr.cfg.max_iter, "passes_per_scan": n_pass, "solver": args.solver,
                       "parallelism": (f"scan-shard x{world}, map replicated, 92 f64 summed per pass via " + ("peer-memory mailboxes inside the persistent k_update kernel (solver block)" if args.comm == "p2p" else "ncclAllReduce")) if world > 1 else "1 GPU",
                       "l2": "flushed (256 MB memset) before every timed step; map (~21 MB) would otherwise be L2-resident"},
            "e2e": {"value": args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(pr.scan.nbytes + (26 + 529 + 32) * 8),
                    "d2h_bytes_per_step": int((26 + 529 + 32) * 8), "ms_per_step": 1e3 * e2e_s / args.steps,
                    "caller": "native loop over the public fl_filter_update (fl_filter_time_e2e)",
                    "via_python_ctypes_wrapper": 1.0 / e2e_py_s},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k_update, search_only launch (the kNN phase of one searching pass: transform, cell-directory search + BVH walks, neighbours stored)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": bytes_launch, "launch_ms": ms_search, "launch_ms_l2_warm": ms_search_warm},
            "cpu_baseline": cpu,
            "parity": parity,
            "clocks": clocks,
            "extra": {"value_l2_warm": args.steps / (ms_warm * 1e-3), "wall_s_timed_region": t_wall,
                      "pos_err_vs_truth_m": float(np.abs(x_res[:3] - pr.x_true[:3]).max())},
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
        if parity is not None and not (parity["ok"] and parity["e2e_path"]):
            print("bench.py: the GPU state differs from the CPU reference path beyond 1e-4 -- this number is not valid", file=sys.stderr)
            return 3
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="velodyne_30k_1m")
    ap.add_argument("--solver", type=int, default=1)
    ap.add_argument("--search", type=int, default=-1, help="-1: library default; 0: BVH walk; 1: cell directory")
    ap.add_argument("--comm", default="p2p", choices=["p2p", "nccl"])
    ap.add_argument("--cpu-scans", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    # Pin the OpenMP threads of the CPU reference path (must be in the environment before any OpenMP runtime starts) -- ONLY in a
    # single-process run: under torchrun the binding would put the main thread of EVERY rank on the same core (place 0), and the
    # ranks' host loops would time-share it (measured: 11 ms / 33 ms of wall clock per step at 4 / 8 ranks, device time unchanged).
    if args.impl != "reference" and world != args.gpus and world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun (before the binding below enters the environment the ranks would inherit)
        port = 29500 + (os.getpid() % 1000)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    if world == 1 or args.impl == "reference":
        os.environ.setdefault("OMP_PROC_BIND", "close")
        os.environ.setdefault("OMP_PLACES", "cores")
    if args.impl == "reference":
        return run_reference(args, rank)
    return run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    sys.exit(main())
