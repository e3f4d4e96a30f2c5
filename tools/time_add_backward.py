"""Kernel time of the ADDLoss backward (p6d_add_backward) at the training size: B = 32 poses of one
symmetric 500-point object (ADD-S: every pred point scans all gt points for its nearest).

CUDA events around replays of a CUDA graph of --launches back-to-back launches of the raw entry point,
so the host's ctypes call is not in the number.  Prints one JSON line with the GPU's name and power limit.
Usage: python tools/time_add_backward.py [--repeats 7] [--launches 200]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--points", type=int, default=500)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=7)
    a = ap.parse_args()
    pkg = importlib.import_module("6d-pose-estimation_b200")
    core, W = pkg.core, pkg.workloads
    dev = torch.device("cuda", 0)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    crit = pkg.ADDLoss(tempfile.mkdtemp(), dev)
    crit.points[9] = T(W.box_mesh(a.points, (0.05, 0.12, 0.06), 1))
    crit.diameters[9] = 0.14
    pq, pt, gq, gt = (T(x) for x in W.random_poses(a.batch, 2, rot_sigma=0.1, trans_sigma=0.01))
    obj = T(np.full(a.batch, 9, np.int64))
    table = crit._mesh_table(dev)
    _, count = table.forward_loss(pq, pt, gq, gt, obj)
    go = torch.ones(1, device=dev)
    g1, g2 = torch.empty_like(pq), torch.empty_like(pt)
    L, p = core.lib(), core.ptr

    def launch():
        core.check(L.p6d_add_backward(table.handle, p(pq), p(pt), p(gq), p(gt), p(obj), a.batch, p(go), p(count), 0.0,
                                      p(g1), p(g2), core.stream_ptr(dev)))

    for _ in range(20):
        launch()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(a.launches):
            launch()
    graph.replay()
    torch.cuda.synchronize()
    us = []
    for _ in range(a.repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record()
        e1.synchronize()
        us.append(e0.elapsed_time(e1) * 1e3 / a.launches)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    print(json.dumps({"kernel": "p6d_add_backward", "batch": a.batch, "points": a.points, "symmetric": True,
                      "us_per_launch_median": round(float(np.median(us)), 3), "us_per_launch_all": [round(u, 3) for u in us],
                      "gpu": torch.cuda.get_device_name(0), "power_limit": q,
                      "grad_t_checksum": float(g2.double().abs().sum())}))


if __name__ == "__main__":
    main()
