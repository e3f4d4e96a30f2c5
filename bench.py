#!/usr/bin/env python
"""bench.py -- ADD-S pose evaluations per second on B200 (BASELINE.json metric).

A "step" is one pass of the hot path over one batch of synthetic pose hypotheses:
BASELINE config 2, i.e. 65,536 hypotheses against 2,048-point symmetric-object meshes
(ADD + ADD-S + ADD-0.1d decision per pose, one kernel launch) per GPU, followed at N > 1
by the NCCL all-reduce of the per-object hit counts.  Weak scaling: every rank evaluates
its own 65,536 hypotheses; `value` is the whole-job rate.

  python bench.py [--gpus N --steps K --warmup W]        our arm (one process per GPU)
  python bench.py [...] --dump-outputs DIR               also write the per-pose outputs of the last timed
                                                         step as DIR/<name>.npy (see dump_outputs)
  python bench.py --impl reference [...]                 CPU arm: the UNMODIFIED reference
        (baseline/_ref or P6D_REFERENCE: ADDLoss.eval_metrics in batches of 16 on
        all host cores) when it is reachable, else the oracle port of its algorithm; same metric,
        bounded sample per step

Beside the headline the line carries
  `sweep`      BASELINE config 5 (13 objects x 4 variants x 1 M hypotheses, 500- and 2,048-point
               meshes) as a STRONG-scaling record: fixed total work sliced over the ranks, seconds
               (max over ranks), per-variant integer hit totals (identical for every N) and an
               oracle check of the first poses of every block;
  `secondary`  the other kernels of the path against their own bounds;
  `cpu_baseline` the reference itself (when reachable) and the oracle port on the host cores,
               with the reference's per-pose decisions compared to the GPU's.

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the roofline arithmetic.
"""
from __future__ import annotations

import argparse
import hashlib
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from

N_POINTS = 2048
POSES_PER_GPU = 65536
FLOP_PER_POSE = 8 * N_POINTS * N_POINTS            # 3 sub + 3 mul + 2 add per pair (SURVEY 8d)
BYTES_PER_POSE = 64 + 10                            # 14 floats + int64 id in, 2 floats + 2 bytes out
METRIC = "ADD-S pose evals/sec (2k-pt mesh)"
UNIT = "poses/s"
SWEEP_SEED = 5000
REF_BATCH = 16                                      # compare_all_models.py:121,125


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--poses", type=int, default=POSES_PER_GPU, help="hypotheses per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=0,
                    help="poses timed on the CPU port baseline (0 = sized for ~10 s of CPU work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-microbench", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary kernels")
    ap.add_argument("--no-sweep", action="store_true", help="skip the config-5 sweep record")
    ap.add_argument("--no-pruned", action="store_true", help="skip the record of the opt-in exact-pruned ADD-S kernel")
    ap.add_argument("--sweep-per-block", type=int, default=1_000_000, help="hypotheses per (object, variant) block")
    ap.add_argument("--sweep-points", default="500,2048", help="mesh sizes of the sweep record")
    ap.add_argument("--sweep-check", type=int, default=256, help="poses per block checked against the oracle")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed on rank 0 to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def config_dict(args, extra=None):
    c = {"workload": f"BASELINE config 2: ADD-S symmetric eval, {N_POINTS}-point synthetic meshes (ids 9,10), "
                     f"{args.poses} pose hypotheses per GPU per step",
         "n_points": N_POINTS, "poses_per_gpu_per_step": args.poses,
         "l2": "inputs (4.8 MB) are smaller than L2; a 256 MiB buffer is written between timed steps to flush it "
               "(the kernel is FP32-issue-bound, DRAM traffic is ~0.1% of the time)",
         "parallelism": f"hypothesis-sharded x{args.gpus}, NCCL all-reduce of int64 hit counts only"}
    if extra:
        c.update(extra)
    return c


def profiled_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the ADD-S kernel, from the newest
    committed `ncu --set full` summary under profiles/ (same workload and launch shape as the bench)."""
    import glob, re
    best = None
    def capture_order(path):       # adds_r2l < adds_r2ag: round number, then the visit tag a..z, aa..az
        m = re.search(r"adds_r(\d+)([a-z]*)_", os.path.basename(path))
        return (int(m.group(1)), len(m.group(2)), m.group(2)) if m else (0, 0, "")
    for path in sorted(glob.glob(os.path.join(REPO, "profiles", "adds_*_summary.txt")), key=capture_order):
        txt = open(path).read()
        r = re.search(r"dram__bytes_read\.sum\s+([0-9.]+)\s+(\w+)", txt)
        w = re.search(r"dram__bytes_write\.sum\s+([0-9.]+)\s+(\w+)", txt)
        if not r or not w:
            continue
        unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        best = {"bytes": float(r.group(1)) * unit.get(r.group(2), 1.0) + float(w.group(1)) * unit.get(w.group(2), 1.0),
                "source": os.path.relpath(path, REPO)}
    return best


# ------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks and throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [l for (t, l) in self.lines if self.t0 is None or (self.t0 <= t <= (self.t1 or t) + 0.05)]
        if not inside:
            inside = [l for (_, l) in self.lines[-3:]]
        for l in inside:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons),
                "sm_mhz_min": min(sm) if sm else None}


# ------------------------------------------------------------------------- CPU arms
def cpu_rate(W, n_poses, threads=None):
    """Oracle port of the reference algorithm on the host cores (bounded sample)."""
    import oracle as O
    O.build()
    threads = threads or O.max_threads()
    pts, dia = W.config2_meshes(N_POINTS)
    pq, pt, gq, gt, obj = W.config2(n_poses)
    table = O.MeshTable(pts, dia)
    O.add_eval(table, pq[:threads], pt[:threads], gq[:threads], gt[:threads], obj[:threads], n_threads=threads)
    t0 = time.perf_counter()
    O.add_eval(table, pq, pt, gq, gt, obj, n_threads=threads)
    dt = time.perf_counter() - t0
    return n_poses / dt, threads, dt


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm is meant to use every host
    core it can (only rank 0 runs it), so the intra-op pool is sized to the CPUs this process may run on."""
    import torch
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    if torch.get_num_threads() != n:
        torch.set_num_threads(n)
    return torch.get_num_threads()


def real_reference():
    """(root, criterion of the UNMODIFIED reference on the CPU with the config-2 meshes) or (None, why)."""
    use_all_host_threads()
    try:
        from oracle import torch_eager as E
        root = E.find_reference()
        if root is None:
            return None, "no reference checkout (P6D_REFERENCE, baseline/_ref)"
        W = importlib.import_module("6d-pose-estimation_b200.workloads")
        pts, dia = W.config2_meshes(N_POINTS)
        return root, E.reference_criterion(root, pts, dia)
    except Exception as e:  # an import error of the reference must not take the bench line down
        return None, f"reference not importable: {e!r}"


def reference_eval_batches(crit, poses, lo, hi):
    """The reference's own call pattern (scripts/visualization/compare_all_models.py:95): eval_metrics on
    batches of 16.  Returns the list of result dicts."""
    import torch
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    pq, pt, gq, gt, obj = poses
    out = []
    for b in range(lo, hi, REF_BATCH):
        e = min(hi, b + REF_BATCH)
        out.append(crit.eval_metrics(T(pq[b:e]), T(pt[b:e]), T(gq[b:e]), T(gt[b:e]), T(obj[b:e])))
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores.
    kind "reference": the unmodified ADDLoss.eval_metrics (PyTorch eager, all intra-op threads) called the
    way compare_all_models.py calls it; kind "port" (only when no reference checkout is reachable): the C
    restatement oracle/pose_oracle.c on all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    W = importlib.import_module("6d-pose-estimation_b200.workloads")
    import oracle as O
    O.build()
    threads = O.max_threads()
    root, crit = real_reference()
    n_probe = max(256, 32 * threads)
    port_probe, _, port_dt = cpu_rate(W, n_probe, threads)
    port = {"value": port_probe, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n_probe} poses, {port_dt:.2f} s, oracle/pose_oracle.c on all host threads"}
    if root is None:
        pts, dia = W.config2_meshes(N_POINTS)
        table = O.MeshTable(pts, dia)
        sample = int(max(64, min(args.poses, port_probe * 3.0)))
        pq, pt, gq, gt, obj = W.config2(sample)
        for _ in range(args.warmup):
            O.add_eval(table, pq[:sample // 4], pt[:sample // 4], gq[:sample // 4], gt[:sample // 4],
                       obj[:sample // 4], n_threads=threads)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            O.add_eval(table, pq, pt, gq, gt, obj, n_threads=threads)
        dt = time.perf_counter() - t0
        kind, cores = "port", threads
        desc = (f"{sample} poses of config 2 per step x {args.steps} steps; oracle/pose_oracle.c on all host threads "
                f"(bit-exact restatement); real reference unavailable: {crit}")
    else:
        poses = W.config2(4096)
        t0 = time.perf_counter()
        reference_eval_batches(crit, poses, 0, REF_BATCH)              # probe (also first-call warm-up)
        probe = REF_BATCH / (time.perf_counter() - t0)
        sample = int(min(1024, max(2 * REF_BATCH, round(probe * 2.5 / REF_BATCH) * REF_BATCH)))   # ~2.5 s per step
        for k in range(args.warmup):
            reference_eval_batches(crit, poses, 0, max(REF_BATCH, sample // 4))
        t0 = time.perf_counter()
        for k in range(args.steps):
            lo = (k * sample) % (4096 - sample + 1)
            reference_eval_batches(crit, poses, lo, lo + sample)
        dt = time.perf_counter() - t0
        kind, cores = "reference", torch.get_num_threads()
        desc = (f"{sample} poses of config 2 per step x {args.steps} steps through the unmodified reference at "
                f"{os.path.relpath(root, REPO) if root.startswith(REPO) else root} (models/add_loss.py ADDLoss.eval_metrics, "
                f"batches of {REF_BATCH}, torch {torch.__version__} CPU eager, {cores} intra-op threads of "
                f"{os.cpu_count()} host CPUs)")
    value = sample * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_dict(args, {"sample_poses_per_step": sample}),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": desc, "port": port},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def cpu_baseline_record(args, W, gpu_rows):
    """The `cpu_baseline` object of our arm: the real reference (when reachable) timed on a bounded sample of
    the same workload and its per-pose values compared with the GPU's; the oracle port beside it."""
    import torch
    from oracle import torch_eager as E
    n_cpu = args.cpu_sample
    if n_cpu <= 0:
        probe, _, _ = cpu_rate(W, 256)
        n_cpu = int(min(args.poses, max(256, probe * 10.0)))
    v, cores, dt = cpu_rate(W, n_cpu)
    port = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"first {n_cpu} poses of the same config-2 workload, {dt:.1f} s, "
                      "oracle/pose_oracle.c (C restatement, bit-exact vs the reference)"}
    root, crit = real_reference()
    if root is None:
        port["reference_unavailable"] = crit
        return port
    poses = W.config2(4096)
    n_ref = min(192, args.poses)
    reference_eval_batches(crit, poses, 4096 - REF_BATCH, 4096)               # warm-up
    t0 = time.perf_counter()
    batches = reference_eval_batches(crit, poses, 0, n_ref)
    dt = time.perf_counter() - t0
    # per-pose values out of the reference (batch size 1: the aggregate of one pose is the pose) for the decision check
    n_chk = min(64, n_ref)
    r_add, r_adds, r_hit, r_valid = E.reference_eval_poses(crit, *(x[:n_chk] for x in poses))
    u32 = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32)
    g = gpu_rows
    hits_equal = bool(np.array_equal(r_hit, g["hit"][:n_chk]) and np.array_equal(r_valid, g["valid"][:n_chk]))
    rec = {"value": n_ref / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "reference",
           "sample": f"first {n_ref} poses of the same config-2 workload in batches of {REF_BATCH}, {dt:.1f} s, through the "
                     f"unmodified reference at {os.path.relpath(root, REPO) if root.startswith(REPO) else root} "
                     f"(ADDLoss.eval_metrics, torch {torch.__version__} CPU eager, {torch.get_num_threads()} intra-op "
                     f"threads of {os.cpu_count()} host CPUs)",
           "reference_add_01d_acc_first_batch": float(batches[0]["add_01d_acc"]),
           "decision_check": {"poses": n_chk, "hits_equal_gpu": hits_equal,
                              "add_bits_equal": int((u32(r_add) == u32(g["add"][:n_chk])).sum()),
                              "adds_bits_equal": int((u32(r_adds) == u32(g["adds"][:n_chk])).sum()),
                              "how": "reference eval_metrics at batch size 1 on THIS box vs p6d_add_eval_host outputs"},
           "port": port}
    if not hits_equal:
        raise AssertionError("ADD-0.1d decisions of the reference on this box differ from the GPU's: " + json.dumps(rec))
    return rec


# ------------------------------------------------------------------------- secondary kernels
def secondary_rooflines(pkg, dev, hbm_peak, fp32_peak):
    """The other kernels of the path at scaled batches, timed with CUDA events around the bare C-ABI
    call (no Python wrapper in the timed region).  Algorithmic bytes per row: DESIGN.md section 4."""
    import torch
    core, W = pkg.core, pkg.workloads
    L, st = core.lib(), core.stream_ptr(dev)

    def timed(fn, reps=10):
        """Best CUDA-event time of one call.  A ~100 us device-side spin is queued first, so that the start
        event, the kernel and the stop event are all in the queue before the GPU reaches them -- otherwise the
        10-15 us the host needs to get from `record` through ctypes to the launch are counted as kernel time
        (ncu: 55 us for a kernel that timed 71 us that way)."""
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        best = 1e30
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(200_000)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b) * 1e-3)
        return best

    res = []

    def hbm_row(kernel, rows, bpr, t, **extra):
        r = {"kernel": kernel, "bound": "hbm", "rows": rows, "bytes_per_row": bpr, "us": round(t * 1e6, 1),
             "achieved": rows * bpr / t / 1e9, "peak": hbm_peak, "unit": "GB/s",
             "frac": rows * bpr / t / 1e9 / hbm_peak if hbm_peak else None}
        r.update(extra)
        res.append(r)

    n = 1 << 24            # ~1.4 GB per kernel: the fixed cost of a launch + event pair (2-4 us) stays below 1-2 %
    g = torch.Generator(device=dev); g.manual_seed(7)
    rnd = lambda *shape: torch.randn(*shape, generator=g, device=dev)
    pq, gq, pt, gt = rnd(n, 4), rnd(n, 4), rnd(n, 3), rnd(n, 3)
    o3 = torch.empty(3, device=dev); g1 = torch.empty_like(pq); g2 = torch.empty_like(pt)
    ws = torch.zeros(64, dtype=torch.uint8, device=dev)
    t = timed(lambda: core.check(L.p6d_pose_loss_fwd_bwd(pq.data_ptr(), pt.data_ptr(), gq.data_ptr(), gt.data_ptr(), n, 1.0,
                                                         10.0, 0, o3.data_ptr(), g1.data_ptr(), g2.data_ptr(),
                                                         ws.data_ptr(), dev.index, st)))
    hbm_row("pose_loss_fwd_bwd (c), geodesic", n, 84, t)
    z, uv = torch.rand(n, device=dev) + 0.4, torch.rand(n, 2, device=dev) * 400
    K1 = torch.tensor(pkg.DEFAULT_K, dtype=torch.float32, device=dev).contiguous()
    K = K1.expand(n, 3, 3).contiguous()
    o = torch.empty(n, 3, device=dev)
    t = timed(lambda: core.check(L.p6d_pinhole_fwd(z.data_ptr(), uv.data_ptr(), K.data_ptr(), 1, n, o.data_ptr(), dev.index, st)))
    hbm_row("pinhole_fwd (d1), K [B,3,3]", n, 60, t)
    t = timed(lambda: core.check(L.p6d_pinhole_fwd(z.data_ptr(), uv.data_ptr(), K1.data_ptr(), 0, n, o.data_ptr(), dev.index, st)))
    hbm_row("pinhole_fwd (d1), shared K [3,3]", n, 24, t)
    del pq, gq, pt, gt, g1, g2
    m = 1 << 22
    d8 = torch.rand(m, 8, 8, device=dev) * 1.5
    uv8 = torch.rand(m, 2, device=dev) * 8
    o8 = torch.empty(m, 3, device=dev)
    t = timed(lambda: core.check(L.p6d_depth_backproject(d8.data_ptr(), 8, 8, uv8.data_ptr(), K.data_ptr(), 1, m, 7.0,
                                                         o8.data_ptr(), dev.index, st)))
    hbm_row("depth_backproject (d2), 8x8 crops, K [B,3,3] (one 32-B sector of each 256-B crop is read)", m, 32 + 8 + 36 + 12, t)
    t = timed(lambda: core.check(L.p6d_depth_backproject(d8.data_ptr(), 8, 8, uv8.data_ptr(), K1.data_ptr(), 0, m, 7.0,
                                                         o8.data_ptr(), dev.index, st)))
    hbm_row("depth_backproject (d2), 8x8 crops, shared K [3,3]", m, 32 + 8 + 12, t)
    # N1 / config 4 (ii): one 480x640 uint16 frame, 256 boxes (latency), and 2^20 boxes of the same frame (rate)
    depth, boxes = W.config4_frame(40, 256)
    dfr = torch.from_numpy(depth.view(np.int16)).to(dev).contiguous()        # uint16 bits
    bx = torch.from_numpy(boxes).to(dev)
    xyz = torch.empty(256, 3, device=dev)
    t = timed(lambda: core.check(L.p6d_depth_crop_backproject(dfr.data_ptr(), 480, 640, bx.data_ptr(), 256, K1.data_ptr(), 224, 0,
                                                              xyz.data_ptr(), None, None, None, dev.index, st)), 20)
    res.append({"kernel": "depth_crop_backproject (N1, config 4 ii): 480x640 uint16 frame, 256 boxes", "bound": "latency",
                "boxes": 256, "us": round(t * 1e6, 2), "boxes_per_s": 256 / t})
    big = bx.repeat(4096, 1).contiguous()
    xyzb = torch.empty(big.shape[0], 3, device=dev)
    t = timed(lambda: core.check(L.p6d_depth_crop_backproject(dfr.data_ptr(), 480, 640, big.data_ptr(), big.shape[0], K1.data_ptr(),
                                                              224, 0, xyzb.data_ptr(), None, None, None, dev.index, st)))
    # ~330 warp instructions per box (the reference's float64 crop geometry, two float64 divisions per axis) on a
    # frame that stays in L2: issue / latency bound (ncu: issue slots 46 %, DRAM 10 %), the GB/s is informational
    res.append({"kernel": "depth_crop_backproject (N1), 2^20 boxes of one frame (frame stays in L2: 16 B box + 12 B out per row)",
                "bound": "issue/latency", "rows": big.shape[0], "us": round(t * 1e6, 1), "boxes_per_s": big.shape[0] / t,
                "hbm_gbs": big.shape[0] * 28 / t / 1e9})
    # N1, inference form: integer xyxy detector boxes, float32 resize, float64 centre / K_crop
    xyxy = bx.clone()
    xyxy[:, 2:] += xyxy[:, :2]
    K64 = torch.tensor(pkg.DEFAULT_K, dtype=torch.float64, device=dev).contiguous()
    t = timed(lambda: core.check(L.p6d_detection_backproject(dfr.data_ptr(), 480, 640, xyxy.data_ptr(), 256, K64.data_ptr(), 224,
                                                             xyz.data_ptr(), None, None, None, dev.index, st)), 20)
    res.append({"kernel": "detection_backproject (N1, inference-script form): 480x640 uint16 frame, 256 xyxy boxes",
                "bound": "latency", "boxes": 256, "us": round(t * 1e6, 2), "boxes_per_s": 256 / t})

    # FP32-issue-bound rows: (a) ADD only, (b) ADD-S at the reference's mesh sizes
    def fp32_row(kernel, poses, flop_per_pose, t, **extra):
        r = {"kernel": kernel, "bound": "fp32-issue", "poses": poses, "us": round(t * 1e6, 1), "poses_per_s": poses / t,
             "achieved": poses * flop_per_pose / t / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
             "frac": poses * flop_per_pose / t / 1e12 / fp32_peak if fp32_peak else None,
             "flop_per_pose": flop_per_pose}
        r.update(extra)
        res.append(r)

    del d8, uv8, o8, K, z, uv, o
    m = 1 << 20
    obj = torch.zeros(m, dtype=torch.int64, device=dev)
    qa, ta = torch.nn.functional.normalize(rnd(m, 4), dim=1), rnd(m, 3)
    qb, tb = torch.nn.functional.normalize(qa + 0.05 * rnd(m, 4), dim=1), ta + 0.005 * rnd(m, 3)
    for npts in (1000, 500):            # 500 points = the reference loader's own mesh size
        pts = {0: W.sphere_mesh(npts, 0.102, 100)}
        table = core.MeshTable(pts, {0: 0.102}, pkg.SYMMETRIC_OBJECT_IDS, dev)
        t = timed(lambda: table.evaluate_packed(qb, tb, qa, ta, obj, want_adds=False), 5)
        fp32_row(f"add_pose_kernel (a), ADD only, N={npts}", m, 46 * npts, t, hbm_gbs=m * 73 / t / 1e9)
    # the several-mesh form of kernel (a): the 13 LineMOD-sized meshes of the sweep, poses sorted by object
    pts13, dia13 = W.sweep_meshes(500)
    t13 = core.MeshTable(pts13, dia13, pkg.SYMMETRIC_OBJECT_IDS, dev)
    ids13 = torch.tensor(sorted(pts13), dtype=torch.int64, device=dev)
    obj13 = ids13[torch.arange(m, device=dev) % len(pts13)]
    ord13 = torch.argsort(obj13, stable=True).to(torch.int32)
    t = timed(lambda: t13.evaluate_packed(qb, tb, qa, ta, obj13, want_adds=False, order=ord13), 5)
    fp32_row("add_pose_kernel (a), ADD only, table of 13 meshes x 500 points, poses ordered by object", m, 46 * 500, t,
             hbm_gbs=m * 77 / t / 1e9)
    for npts, Bn in ((500, 1 << 20), (1000, 1 << 18)):
        pts = {9: W.box_mesh(npts, (0.1, 0.12, 0.05), 200 + npts)}
        tb_ = core.MeshTable(pts, {9: 0.1646}, pkg.SYMMETRIC_OBJECT_IDS, dev)
        ob = torch.full((Bn,), 9, dtype=torch.int64, device=dev)
        t = timed(lambda: tb_.evaluate(qb[:Bn], tb[:Bn], qa[:Bn], ta[:Bn], ob, want_adds=True), 5)
        fp32_row(f"adds_cta_kernel (b), ADD + ADD-S, N={npts}", Bn, 8 * npts * npts, t, schedule=tb_.schedule_state())
    # the B = 32 training step through the public PoseLoss module (config 3): host latency, not a roofline
    c = W.config3(32, 6)
    Tn = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    crit = pkg.PoseLoss(1.0, 10.0, "geodesic")
    rot, tr = Tn(c["rot_raw"]).requires_grad_(True), Tn(c["gt_trans"] + 0.01).requires_grad_(True)
    gr, gtr = Tn(c["gt_rot"]), Tn(c["gt_trans"])

    def train_step():
        rot.grad = None; tr.grad = None
        crit(rot, tr, gr, gtr).backward()
    for _ in range(20):
        train_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(200):
        train_step()
    torch.cuda.synchronize()
    res.append({"kernel": "PoseLoss forward+backward through autograd, B=32 (config 3)", "bound": "latency",
                "us_per_step": (time.perf_counter() - t0) / 200 * 1e6})
    # the same step captured in a CUDA graph (PoseLoss.capture): one cudaGraphLaunch per step
    cap = crit.capture(rot, tr, gr, gtr)
    for _ in range(20):
        cap.replay()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(1000):
        cap.replay()
    torch.cuda.synchronize()
    us_replay = (time.perf_counter() - t0) / 1000 * 1e6
    t0 = time.perf_counter()
    for _ in range(200):
        cap.copy_and_replay(rot, tr, gr, gtr)
    torch.cuda.synchronize()
    us_copies = (time.perf_counter() - t0) / 200 * 1e6
    for _ in range(20):
        cap(rot, tr, gr, gtr)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(1000):
        cap(rot, tr, gr, gtr)
    torch.cuda.synchronize()
    res.append({"kernel": "PoseLoss.capture: the same step replayed from a CUDA graph, B=32", "bound": "latency",
                "us_per_step": us_replay, "us_per_step_with_input_copies": us_copies,
                "us_per_step_called_on_the_callers_tensors": (time.perf_counter() - t0) / 1000 * 1e6,
                "loss_equals_eager": bool(cap.loss.item() == crit(rot, tr, gr, gtr).item())})
    return res


# ------------------------------------------------------------------------- config 5
def sweep_record(pkg, dev, rank, world, n_points, n_per_block, check_total, barrier, exact_pruning=False):
    """BASELINE config 5 for one mesh size: 13 objects x 4 variants x n_per_block hypotheses, the hypothesis
    axis of every block sliced over the ranks (strong scaling), one native call per rank
    (p6d_sweep_run) + one all-reduce of the accumulators.  The first poses of every block of every rank's
    slice are re-evaluated by the oracle after the timed region."""
    import torch
    import torch.distributed as dist
    import oracle as O
    W = pkg.workloads
    variants = pkg.sweep.VARIANTS
    pts, dia = W.sweep_meshes(n_points)
    ev = pkg.PoseEvaluator(pts, dia, dev, n_rows=len(variants), exact_pruning=exact_pruning)
    # warm-up through the same code path (also runs the one-time self-check of a re-laid kernel)
    pkg.evaluate_sweep(pts, dia, dev, 4096 * world, seed=SWEEP_SEED, rank=rank, world=world, evaluator=ev)
    cn = max(8, check_total // world)
    # a sweep of a second or two is ONE shot of ~180 launches per rank: a single host or box hiccup shows up whole
    # (r2as, 2 GPUs: 1.92 s once against 1.21 s on three repeats), so the short sweeps are timed twice, the
    # faster run is reported, both are listed and their integer hit tables must be identical
    runs, first_hits, run_clocks = [], None, []
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for _ in range(2 if n_points <= 1024 else 1):
        ev.acc.zero_()
        sampler = ClockSampler(dev.index)        # every rank watches its own GPU: a slow run should name its cause
        sampler.start()
        barrier()
        sampler.mark_begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        acc, launches, check = pkg.evaluate_sweep(pts, dia, dev, n_per_block, seed=SWEEP_SEED, rank=rank, world=world,
                                                  evaluator=ev, check_n=cn)
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        sampler.mark_end()
        ck = sampler.stop()
        # max over ranks of [wall, device time, -min SM clock, power, one flag per throttle reason]
        tm = torch.tensor([wall, e0.elapsed_time(e1) * 1e-3, -(ck.get("sm_mhz_min") or 0.0), ck.get("power_w_max") or 0.0]
                          + [float(n in ck["reasons"]) for n in names], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        tm = tm.tolist()
        runs.append((float(tm[0]), float(tm[1])))
        run_clocks.append({"sm_mhz_min_over_ranks": -tm[2] or None, "power_w_max_over_ranks": tm[3] or None,
                           "reasons_any_rank": [n for n, f in zip(names, tm[4:]) if f > 0]})
        if first_hits is None:
            first_hits = acc.hits.clone()
        elif not torch.equal(first_hits, acc.hits):
            raise SystemExit("bench: two runs of the same sweep gave different hit tables")
    wall_s, dev_s = min(runs)
    # oracle check of what was evaluated (outside the timed region)
    nb, k = check["pq"].shape[0], check["pq"].shape[1]
    rows = lambda name, w: np.ascontiguousarray(check[name].reshape(nb * k, w))
    ref = O.add_eval(O.MeshTable(pts, dia), rows("pq", 4), rows("pt", 3), rows("gq", 4), rows("gt", 3),
                     np.ascontiguousarray(check["obj"].reshape(-1)), n_threads=max(1, O.max_threads() // world))
    u32 = lambda a: np.ascontiguousarray(a, np.float32).reshape(-1).view(np.uint32)
    bad = int((u32(check["add"]) != u32(ref[0])).sum() + (u32(check["adds"]) != u32(ref[1])).sum()
              + (check["hit"].reshape(-1) != ref[2]).sum())
    chk = torch.tensor([bad, nb * k], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(chk)
    hits, valid = acc.hits.cpu().numpy(), acc.valid.cpu().numpy()
    total = int(valid.sum())
    ids = sorted(pts)
    table = [[int(hits[v, o]) for o in ids] for v in range(len(variants))]
    return {"workload": f"BASELINE config 5: {len(ids)} objects x {len(variants)} variants x {n_per_block} hypotheses, "
                        f"{n_points}-point meshes, ADD + ADD-S + ADD-0.1d for every pose; hypotheses generated on the device "
                        "(p6d_synth_poses), translations of the geometric variants by kernels (d1) / (d2)",
            "n_points": n_points, "hypotheses": total, "scaling": "strong", "n_gpus": world,
            "adds_kernel": "exact-pruned (opt-in)" if exact_pruning else "all-pairs",
            "seconds": wall_s, "device_seconds": dev_s, "seconds_of_every_run": [r[0] for r in runs],
            "clocks_of_every_run": run_clocks,
            "poses_per_s": total / wall_s,
            "tflops": total * (8 * n_points * n_points + 46 * n_points) / wall_s / 1e12,
            "launches_per_rank": launches,
            "hits_per_variant": {v: int(hits[i].sum()) for i, v in enumerate(variants)},
            "valid_per_variant": {v: int(valid[i].sum()) for i, v in enumerate(variants)},
            "hits_table_objects": ids, "hits_table": table,
            "hits_table_sha256": hashlib.sha256(json.dumps(table).encode()).hexdigest()[:16],
            "oracle_check": {"poses": int(chk[1]), "mismatches": int(chk[0]),
                             "what": f"first {k} hypotheses of every (object, variant) block of every rank's slice: ADD, ADD-S "
                                     "bits and decisions vs oracle/pose_oracle.c"}}


# ------------------------------------------------------------------------- outputs
DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, last, acc, counts=None):
    """What a caller of MeshTable.evaluate received from the last timed step, one DIR/<name>.npy per array:
    per-pose add, adds (metres), hit, valid and the per-object accumulators obj_hits, obj_valid, obj_add_sum,
    obj_adds_sum (at N > 1 also the all-reduced obj_hits_all_ranks, obj_valid_all_ranks).  Integers are
    stored as float64, hit / valid as float32.  The inputs are seeded, so two builds run with the same
    arguments can be compared file by file.  When the per-pose arrays would exceed 64 MB, a fixed seeded
    sample of poses is written instead, with its row numbers in pose_index."""
    import torch
    add, adds, hit, valid, _ = last
    per_pose = {"add": add.float(), "adds": adds.float(), "hit": hit.float(), "valid": valid.float()}
    per_object = {"obj_hits": acc[0], "obj_valid": acc[1], "obj_add_sum": acc[2], "obj_adds_sum": acc[3]}
    if counts is not None:
        per_object.update(obj_hits_all_ranks=counts[0], obj_valid_all_ranks=counts[1])
    arrays = {k: v.double().cpu().numpy() for k, v in per_object.items()}
    n = add.shape[0]
    room = DUMP_BYTES - sum(a.nbytes for a in arrays.values()) - 4096       # 4 KB for the .npy headers
    if 16 * n > room:                  # 4 float32 per pose; a sample also stores its float64 row numbers
        idx = np.sort(np.random.default_rng(0).choice(n, room // 24, replace=False))
        arrays["pose_index"] = idx.astype(np.float64)
        sel = torch.from_numpy(idx).to(add.device)
        per_pose = {k: v[sel] for k, v in per_pose.items()}
    arrays.update({k: v.cpu().numpy() for k, v in per_pose.items()})
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------- GPU arm
def run_b200(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    pkg = importlib.import_module("6d-pose-estimation_b200")
    core, W = pkg.core, pkg.workloads
    info = core.device_info(local)

    B = args.poses
    pts, dia = W.config2_meshes(N_POINTS)
    table = core.MeshTable(pts, dia, pkg.SYMMETRIC_OBJECT_IDS, dev)
    # each rank gets its own seeded hypotheses (weak scaling)
    host = W.config2(B, base_seed=2000 + 1000 * rank)
    pinned = [torch.from_numpy(x).pin_memory() for x in host]
    d_in = [t.to(dev) for t in pinned]
    order = torch.argsort(d_in[4], stable=True).to(torch.int32)
    acc = [torch.zeros(table.n_slots, dtype=torch.int64, device=dev) for _ in range(2)] + \
          [torch.zeros(table.n_slots, dtype=torch.float64, device=dev) for _ in range(2)]
    counts = torch.zeros(2, table.n_slots, dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    launches = 0
    last = None

    def step():
        nonlocal launches, last
        for a in acc:
            a.zero_()
        last = table.evaluate(*d_in, want_adds=True, order=order, acc=acc)
        launches += 1
        if world > 1:
            counts[0].copy_(acc[0]); counts[1].copy_(acc[1])
            dist.all_reduce(counts)          # per-object ADD-0.1d hit / valid counts: the only exchange

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches = 0
    barrier()
    sampler.mark_begin()
    t0 = time.perf_counter()
    for k in range(args.steps):
        flush.fill_(k & 0xFF)                # L2 flush between timed steps (outside the event pair)
        ev[k][0].record()
        step()
        ev[k][1].record()
    barrier()
    wall = time.perf_counter() - t0
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    step_ms = [a.elapsed_time(b) for a, b in ev]
    dev_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dev_ms, op=dist.ReduceOp.MAX)
    total_ms = float(dev_ms.item())
    value = world * B * args.steps / (total_ms * 1e-3)
    timed_launches = launches
    sched = table.schedule_state()

    # result sanity on the numbers just computed (accuracy is counts / totals, integer-exact)
    hits = int(acc[0].sum().item()); valid = int(acc[1].sum().item())
    assert valid == B, (valid, B)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, acc, counts if world > 1 else None)

    # ---------------- end-to-end: host buffers in, host results out, through the C ABI
    def e2e(bufs):
        for _ in range(2):
            table.evaluate_host(*bufs, want_adds=True, per_pose=True)
        barrier()
        t0 = time.perf_counter()
        steps = max(3, min(args.steps, 10))
        for _ in range(steps):
            r = table.evaluate_host(*bufs, want_adds=True, per_pose=True)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return world * B * steps / float(dt.item()), steps, r

    e2e_value, e2e_steps, r = e2e([t.numpy() for t in pinned])
    assert int(r["obj_hits"].sum()) == hits, "host-entry decisions differ from the device entry"
    e2e_pageable, _, r2 = e2e([np.array(x, copy=True) for x in host])        # a caller's ordinary NumPy arrays
    assert int(r2["obj_hits"].sum()) == hits

    # ---------------- BASELINE config 5, strong scaling (every rank takes part)
    sweeps = {}
    if not args.no_sweep and B == POSES_PER_GPU:
        for npts in [int(x) for x in args.sweep_points.split(",") if x]:
            sweeps[f"n{npts}"] = sweep_record(pkg, dev, rank, world, npts, args.sweep_per_block, args.sweep_check, barrier)

    # ---------------- opt-in exact-pruned ADD-S kernel (b'): the SAME outputs from less work.  Reported on its own:
    # `value`, `roofline` and `sweep` above are the all-pairs kernel the north-star names.
    pruned = None
    if not args.no_pruned and B == POSES_PER_GPU:
        ptable = core.MeshTable(pts, dia, pkg.SYMMETRIC_OBJECT_IDS, dev).set_pruning(True)
        ref_out = table.evaluate_packed(*d_in, want_adds=True, order=order)
        pr_out = ptable.evaluate_packed(*d_in, want_adds=True, order=order)
        equal = bool(torch.equal(ref_out[:10 * B], pr_out[:10 * B]))     # add, adds, hit, valid: every byte
        for _ in range(3):
            ptable.evaluate_packed(*d_in, want_adds=True, order=order)
        barrier()
        pe = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for k in range(args.steps):
            flush.fill_(k & 0xFF)
            pe[k][0].record()
            ptable.evaluate_packed(*d_in, want_adds=True, order=order)
            pe[k][1].record()
        barrier()
        pms = torch.tensor([sum(a.elapsed_time(b) for a, b in pe)], dtype=torch.float64, device=dev)
        eq = torch.tensor([1 if equal else 0], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(pms, op=dist.ReduceOp.MAX)
            dist.all_reduce(eq, op=dist.ReduceOp.MIN)
        pruned = {"what": "opt-in exact block pruning in the ADD-S kernel (p6d_mesh_table_set_pruning / ADDLoss.exact_pruning): "
                          "gt blocks that provably hold no nearest neighbour are skipped; every output byte equals the "
                          "all-pairs kernel's. Not a roofline number: it does less work",
                  "value": world * B * args.steps / (float(pms.item()) * 1e-3), "unit": UNIT, "workload": "the config-2 step above",
                  "ms_per_step": float(pms.item()) / args.steps, "outputs_equal_all_pairs": bool(eq.item()),
                  "speedup_vs_all_pairs": (world * B * args.steps / (float(pms.item()) * 1e-3)) / value}
        for key, full_rec in sweeps.items():       # the config-5 sweeps again, with the switch on
            ps = sweep_record(pkg, dev, rank, world, full_rec["n_points"], args.sweep_per_block, args.sweep_check, barrier,
                              exact_pruning=True)
            pruned[f"sweep_{key}"] = {k: ps[k] for k in ("seconds", "device_seconds", "poses_per_s", "hits_per_variant",
                                                         "hits_table_sha256", "oracle_check", "adds_kernel")}
            pruned[f"sweep_{key}"]["hits_table_equals_all_pairs"] = ps["hits_table_sha256"] == full_rec["hits_table_sha256"]
            pruned[f"sweep_{key}"]["speedup_vs_all_pairs"] = full_rec["seconds"] / ps["seconds"]
        del ptable

    if rank == 0:
        kernel_ms = float(np.mean(step_ms))            # rank 0's kernel; at N = 1 the step is the kernel
        achieved = B * FLOP_PER_POSE / (kernel_ms * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        sm_max = float(peaks.get("sm_max_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0)
        nominal = info["sm_count"] * 128 * 2 * sm_max * 1e6 / 1e12
        tr = profiled_traffic() if B == POSES_PER_GPU else None
        relaid = sched["built_relaid"] == 1 and sched["runtime_state"] == 1
        mb = {}
        if not args.no_microbench:
            for kind, name in ((0, "ffma"), (1, "ffma2"), (2, "adds_mix")):
                mb[name] = round(max(core.fp32_microbench(kind, local, 4000)[0] for _ in range(3)), 2)
        peak = mb.get("ffma2") or nominal
        roof = {"bound": "fp32", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "kernel": ("adds_cta_kernel<256,8,2,deferred minima>, scan loop re-laid after linking by "
                           "csrc/sass_sched.py, verified against the ptxas-scheduled kernel on this device before use")
                if relaid else "adds_cta_kernel<512,4,2,2> (ptxas schedule)",
                "schedule_state": sched,
                "frac": achieved / peak, "traffic": tr["bytes"] if tr else None,
                "traffic_source": tr["source"] if tr else None,
                "algorithmic_bytes_per_launch": B * BYTES_PER_POSE,
                "peak_source": ("FFMA2 issue-rate microbenchmark measured in this run (p6d_fp32_microbench kind 1); "
                                "MEASURED_PEAKS.json has no FP32 entry -- the kernel is neither HBM- nor tensor-bound "
                                "(SURVEY 7.3.2)") if mb.get("ffma2") else "nominal (microbenchmark skipped)",
                "peak_nominal": nominal, "frac_of_nominal": achieved / nominal,
                "peak_nominal_source": f"{info['sm_count']} SM x 128 lanes x 2 FLOP x {sm_max:.0f} MHz",
                "algorithmic_flop_per_pose": FLOP_PER_POSE,
                "hbm": {"achieved_gbs": B * BYTES_PER_POSE / (kernel_ms * 1e-3) / 1e9,
                        "peak_gbs": peaks.get("hbm_gbs"), "note": "of measured; informational"}}
        if mb:
            roof["measured_fp32_tflops"] = mb
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_dict(args), "roofline": roof, "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": r["h2d_bytes"],
                        "d2h_bytes_per_step": r["d2h_bytes"], "steps": e2e_steps,
                        "api": "p6d_add_eval_host via MeshTable.evaluate_host (pinned host buffers)",
                        "pageable_value": e2e_pageable,
                        "pageable_note": "same call with ordinary (pageable) NumPy arrays as a caller would pass them"},
                "gpu_launches": timed_launches, "wall_ms_per_step_incl_flush": wall / args.steps * 1e3,
                "add_01d_acc": 100.0 * hits / valid}
        if sweeps:
            line["sweep"] = sweeps
        if pruned:
            line["pruned"] = pruned
        if not args.no_secondary and B == POSES_PER_GPU:
            try:
                line["secondary"] = secondary_rooflines(pkg, dev, peaks.get("hbm_gbs"), peak)
            except Exception as e:  # never lose the headline line over the side measurements
                line["secondary"] = {"error": repr(e)}
        if not args.no_cpu_baseline and world == 1:        # the CPU leg belongs to the N = 1 line only
            line["cpu_baseline"] = cpu_baseline_record(args, W, r)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line of the contract goes to the real stdout; everything else any library
    prints during the run (e.g. NCCL's version banner) has been routed to stderr."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    args = parse()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                      # fd 1 -> stderr for the duration of the run
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
