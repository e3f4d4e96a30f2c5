"""Throughput of the streamed ADD / ADD-S kernel (csrc/p6d_adds_streamed.cu) on meshes beyond shared memory.

Reports, with the card's name, power limit and maximum SM clock read in the same run:
  * poses/s and TFLOP/s at N = 8,192, 16,384 and 32,768 points (B = 2,048 poses per call), counting 8 N^2 FLOP per
    pose (SURVEY 8d), and their share of the FFMA2 rate measured by p6d_fp32_microbench in the same run;
  * the forced-streamed kernel against the resident ADD-S kernel at N = 4,096 on the same table and poses,
    alternated in one run, with a byte comparison of their outputs;
  * B = 16 poses (the reference's evaluation batch) at N = 16,384: time per call, against 16 x the per-pose time
    of the large-B run.
Every shape is warmed up; every number is CUDA events around a window of >= --window seconds of back-to-back calls.
The mesh (3 x 4 x N bytes) is L2-resident, as it is in use: the kernel is compute-bound.
Usage: python tools/time_large_meshes.py [--out profiles/large_meshes_b200.json] [--window 0.5]
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
            return s / k, k
        k *= 2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "large_meshes_b200.json"))
    ap.add_argument("--window", type=float, default=0.5)
    ap.add_argument("--batch", type=int, default=2048)
    a = ap.parse_args()
    pkg = importlib.import_module("6d-pose-estimation_b200")
    core, W = pkg.core, pkg.workloads
    dev = torch.device("cuda", 0)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    ffma2 = max(core.fp32_microbench(1, 0)[0] for _ in range(3))
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": smi,
           "ffma2_tflops_measured": round(ffma2, 2), "flop_per_pose": "8 N^2", "window_s": a.window}

    def inputs(B, seed):
        pq, pt, gq, gt = W.random_poses(B, seed, rot_sigma=0.05)
        return [T(x) for x in (pq, pt, gq, gt, np.full(B, 9, np.int64))]

    rows = []
    for n in (8192, 16384, 32768):
        table = core.MeshTable({9: W.box_mesh(n, (0.1, 0.12, 0.05), 9)}, {9: 0.16}, {9}, dev).set_large_meshes(True)
        d = inputs(a.batch, n)
        s, k = timed(lambda: table.evaluate_packed(*d), a.window)
        tf = 8.0 * n * n * a.batch / s / 1e12
        rows.append({"points": n, "batch": a.batch, "ms_per_call": round(s * 1e3, 3), "calls": k,
                     "poses_per_s": round(a.batch / s, 1), "tflops": round(tf, 2), "share_of_ffma2": round(tf / ffma2, 4)})
        print(json.dumps(rows[-1]), flush=True)
    res["large_batch"] = rows

    # forced-streamed vs resident on the same table, alternated
    n, B = 4096, 8192
    table = core.MeshTable({9: W.box_mesh(n, (0.1, 0.12, 0.05), 9)}, {9: 0.16}, {9}, dev)
    d = inputs(B, 4)
    ref = table.evaluate_packed(*d)[:11 * B].clone()
    st = table.evaluate_packed(*d, streamed=True)[:11 * B].clone()
    times = {"resident": [], "streamed": []}
    for _ in range(5):
        times["resident"].append(timed(lambda: table.evaluate_packed(*d), a.window)[0])
        times["streamed"].append(timed(lambda: table.evaluate_packed(*d, streamed=True), a.window)[0])
    r, s = float(np.median(times["resident"])), float(np.median(times["streamed"]))
    res["n4096_streamed_vs_resident"] = {
        "points": n, "batch": B, "outputs_equal": bool(torch.equal(ref, st)),
        "resident_ms_all": [round(x * 1e3, 3) for x in times["resident"]],
        "streamed_ms_all": [round(x * 1e3, 3) for x in times["streamed"]],
        "resident_share_of_ffma2": round(8.0 * n * n * B / r / 1e12 / ffma2, 4),
        "streamed_share_of_ffma2": round(8.0 * n * n * B / s / 1e12 / ffma2, 4),
        "streamed_over_resident_time": round(s / r, 4)}
    print(json.dumps(res["n4096_streamed_vs_resident"]), flush=True)

    # the reference's evaluation batch
    n, B = 16384, 16
    table = core.MeshTable({9: W.box_mesh(n, (0.1, 0.12, 0.05), 9)}, {9: 0.16}, {9}, dev).set_large_meshes(True)
    d = inputs(B, 16)
    s, k = timed(lambda: table.evaluate_packed(*d), a.window)
    per_pose_large = next(x for x in rows if x["points"] == n)["ms_per_call"] / a.batch
    res["b16_n16384"] = {"ms_per_call": round(s * 1e3, 4), "calls": k,
                         "sixteen_times_large_batch_per_pose_ms": round(16 * per_pose_large, 4),
                         "ratio": round(s * 1e3 / (16 * per_pose_large), 3)}
    print(json.dumps(res["b16_n16384"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
