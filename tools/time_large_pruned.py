"""Throughput of the streamed exact-pruned ADD-S kernel (b''', csrc/p6d_adds_pruned.cu) against the streamed
all-pairs kernel (b'', csrc/p6d_adds_streamed.cu) on meshes beyond shared memory.

Reports, with the card's name, power limit and maximum SM clock read in the same run:
  * sphere and box meshes at N = 8,192 / 16,384 / 32,768 points, rotation error sigma 0.02 / 0.1 / 0.5 rad, B = 2,048
    and B = 16 poses per call: poses/s of the forced new entry (prune_streamed=True) and of the forced streamed
    kernel (streamed=True), alternated, with a byte comparison of their outputs, and the speed-up over b'';
  * N = 4,096, where the resident pruned kernel b' still runs: b''' against b' (prune=True) and b'', to show what
    streaming the per-pose state through global memory costs;
  * torch.profiler kernel times of b''''s two passes in one call at 32,768 points.
Pruning does less work, not the same work faster, so no number here is a share of peak.  Every shape is warmed up;
every number is CUDA events around a window of >= --window seconds of back-to-back calls.
Usage: python tools/time_large_pruned.py [--out profiles/large_pruned_b200.json] [--window 0.3]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def timed(fn, window):
    """Seconds per call: calls doubled until one window of back-to-back calls lasts >= `window` seconds."""
    fn()
    torch.cuda.synchronize()
    k = 1
    while True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        e1.synchronize()
        s = e0.elapsed_time(e1) / 1e3
        if s >= window:
            return s / k
        k *= 2


def alternated(fns, window, rounds=2):
    """Median seconds per call of every entry of fns, the entries alternated `rounds` times."""
    t = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            t[k].append(timed(fn, window))
    return {k: float(np.median(v)) for k, v in t.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "large_pruned_b200.json"))
    ap.add_argument("--window", type=float, default=0.3)
    a = ap.parse_args()
    pkg = importlib.import_module("6d-pose-estimation_b200")
    core, W = pkg.core, pkg.workloads
    dev = torch.device("cuda", 0)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": smi,
           "window_s": a.window, "rows": []}
    print(json.dumps({"gpu": res["gpu"], "smi": smi}), flush=True)

    def mesh(kind, n):
        return W.sphere_mesh(n, 0.15, n) if kind == "sphere" else W.box_mesh(n, (0.1, 0.12, 0.05), n)

    def inputs(B, sigma, seed):
        pq, pt, gq, gt = W.random_poses(B, seed, rot_sigma=sigma)
        return [T(x) for x in (pq, pt, gq, gt, np.full(B, 9, np.int64))]

    for n in (8192, 16384, 32768):
        for kind in ("sphere", "box"):
            table = core.MeshTable({9: mesh(kind, n)}, {9: 0.16}, {9}, dev)
            for sigma in (0.02, 0.1, 0.5):
                for B in (2048, 16):
                    d = inputs(B, sigma, n + B)
                    new = table.evaluate_packed(*d, prune_streamed=True)[:11 * B].clone()
                    ref = table.evaluate_packed(*d, streamed=True)[:11 * B].clone()
                    t = alternated({"pruned_streamed": lambda: table.evaluate_packed(*d, prune_streamed=True),
                                    "streamed": lambda: table.evaluate_packed(*d, streamed=True)}, a.window)
                    row = {"points": n, "mesh": kind, "sigma": sigma, "batch": B,
                           "outputs_equal": bool(torch.equal(new, ref)),
                           "pruned_streamed_poses_per_s": round(B / t["pruned_streamed"], 1),
                           "streamed_poses_per_s": round(B / t["streamed"], 1),
                           "speedup_over_streamed": round(t["streamed"] / t["pruned_streamed"], 3)}
                    res["rows"].append(row)
                    print(json.dumps(row), flush=True)

    # N = 4,096: the resident pruned kernel still runs
    n, B = 4096, 8192
    res["n4096"] = []
    for kind in ("sphere", "box"):
        table = core.MeshTable({9: mesh(kind, n)}, {9: 0.16}, {9}, dev)
        for sigma in (0.02, 0.1, 0.5):
            d = inputs(B, sigma, 7)
            outs = [table.evaluate_packed(*d, **kw)[:11 * B].clone()
                    for kw in ({"prune_streamed": True}, {"prune": True}, {"streamed": True})]
            t = alternated({"pruned_streamed": lambda: table.evaluate_packed(*d, prune_streamed=True),
                            "pruned": lambda: table.evaluate_packed(*d, prune=True),
                            "streamed": lambda: table.evaluate_packed(*d, streamed=True)}, a.window)
            row = {"points": n, "mesh": kind, "sigma": sigma, "batch": B,
                   "outputs_equal": bool(torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])),
                   **{f"{k}_poses_per_s": round(B / v, 1) for k, v in t.items()},
                   "pruned_streamed_over_pruned_time": round(t["pruned_streamed"] / t["pruned"], 3)}
            res["n4096"].append(row)
            print(json.dumps(row), flush=True)

    # where the time goes: the two passes of one call
    from torch.profiler import ProfilerActivity, profile
    n, B = 32768, 2048
    table = core.MeshTable({9: mesh("sphere", n)}, {9: 0.16}, {9}, dev)
    res["passes_n32768_b2048"] = {}
    for sigma in (0.02, 0.1, 0.5):
        d = inputs(B, sigma, 11)
        table.evaluate_packed(*d, prune_streamed=True)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            table.evaluate_packed(*d, prune_streamed=True)
            torch.cuda.synchronize()
        us = {}
        for e in prof.key_averages():
            if "pruned_streamed" in e.key:
                name = "xform" if "xform" in e.key else "scan"
                us[name] = us.get(name, 0.0) + e.device_time_total
        res["passes_n32768_b2048"][str(sigma)] = {k: round(v / 1e3, 3) for k, v in us.items()} | {"unit": "ms"}
        print(json.dumps({"sigma": sigma, **res["passes_n32768_b2048"][str(sigma)]}), flush=True)

    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
