"""Time of ADDLoss.forward and its backward on meshes beyond shared memory (large_mesh_loss, csrc/p6d_adds_streamed.cu
loss form and csrc/p6d_add_bwd.cu add_backward_streamed_kernel).

Reports, with the card's name, power limit and maximum SM clock read in the same run:
  * forward (forward_loss), backward (add_backward) and the whole ADDLoss step (forward + loss.backward()) at
    N = 8,192, 16,384 and 32,768 points, one symmetric or one asymmetric object, B = 32 and 2,048 samples; for
    symmetric samples the forward and backward count 8 N^2 FLOP per sample (SURVEY 8d), reported as a share of the
    FFMA2 rate measured by p6d_fp32_microbench in the same run;
  * the forced streamed kernels against the resident ones on the same table and inputs, alternated: the forward at
    N = 4,096 and the backward at N = 16,384 (symmetric, B = 32 and 2,048), with a comparison of their outputs.
Every shape is warmed up; every number is CUDA events around a window of >= --window seconds of back-to-back calls.
Usage: python tools/time_large_loss.py [--out profiles/large_loss_b200.json] [--window 0.3]
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
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "large_loss_b200.json"))
    ap.add_argument("--window", type=float, default=0.3)
    a = ap.parse_args()
    pkg = importlib.import_module("6d-pose-estimation_b200")
    core, W = pkg.core, pkg.workloads
    dev = torch.device("cuda", 0)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    ffma2 = max(core.fp32_microbench(1, 0)[0] for _ in range(3))
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": smi,
           "ffma2_tflops_measured": round(ffma2, 2), "flop_per_symmetric_sample": "8 N^2", "window_s": a.window}

    def inputs(B, oid, seed):
        pq, pt, gq, gt = W.random_poses(B, seed, rot_sigma=0.05, trans_sigma=0.01)
        return [T(x) for x in (pq, pt, gq, gt, np.full(B, oid, np.int64))]

    def backward_fn(table, d, streamed=False):
        _, count = table.forward_loss(*d)
        saved = (*d, count, table, dev)
        go = torch.ones((), device=dev)
        return lambda: core.add_backward(saved, go, streamed=streamed)

    rows = []
    for n in (8192, 16384, 32768):
        for oid in (9, 3):            # 9: symmetric (ADD-S), 3: asymmetric (ADD)
            mesh = W.box_mesh(n, (0.1, 0.12, 0.05), 9)
            crit = pkg.ADDLoss(tempfile.mkdtemp(), dev)
            crit.points[oid] = T(mesh)
            crit.large_mesh_loss = True
            table = crit._mesh_table(dev)
            for B in (32, 2048):
                d = inputs(B, oid, n + B)
                fwd, _ = timed(lambda: table.forward_loss(*d), a.window)
                bwd, _ = timed(backward_fn(table, d), a.window)

                def step():
                    x = d[0].clone().requires_grad_(True)
                    crit(x, d[1], d[2], d[3], d[4]).backward()
                st, _ = timed(step, a.window)
                r = {"points": n, "symmetric": oid == 9, "batch": B, "forward_ms": round(fwd * 1e3, 4),
                     "backward_ms": round(bwd * 1e3, 4), "step_ms": round(st * 1e3, 4)}
                if oid == 9:
                    flop = 8.0 * n * n * B
                    r["forward_share_of_ffma2"] = round(flop / fwd / 1e12 / ffma2, 4)
                    r["backward_share_of_ffma2"] = round(flop / bwd / 1e12 / ffma2, 4)
                rows.append(r)
                print(json.dumps(r), flush=True)
    res["large_meshes"] = rows

    # forced streamed vs resident, alternated on the same table and inputs
    ab = []
    for what, n in (("forward", 4096), ("backward", 16384)):
        table = core.MeshTable({9: W.box_mesh(n, (0.1, 0.12, 0.05), 9)}, {9: 0.16}, {9}, dev).set_large_mesh_loss(True)
        for B in (32, 2048):
            d = inputs(B, 9, 7 * n + B)
            if what == "forward":
                fns = {"resident": lambda: table.forward_loss(*d), "streamed": lambda: table.forward_loss(*d, streamed=True)}
                outs = {k: torch.cat([x.view(torch.int32) for x in (f()[0], f()[1])]) for k, f in fns.items()}
                same = bool(torch.equal(outs["resident"], outs["streamed"]))
                agree = {"loss_and_count_bits_equal": same}
            else:
                fns = {"resident": backward_fn(table, d), "streamed": backward_fn(table, d, True)}
                r_, s_ = fns["resident"](), fns["streamed"]()
                err = max(float(((x - y).abs().max(dim=1)[0] / x.abs().max(dim=1)[0].clamp_min(1e-30)).max())
                          for x, y in zip(r_, s_))
                agree = {"max_rel_row_difference": err}
            times = {"resident": [], "streamed": []}
            for _ in range(5):
                for k in ("resident", "streamed"):
                    times[k].append(timed(fns[k], a.window)[0])
            r, s = float(np.median(times["resident"])), float(np.median(times["streamed"]))
            e = {"what": what, "points": n, "batch": B, **agree,
                 "resident_ms_all": [round(x * 1e3, 4) for x in times["resident"]],
                 "streamed_ms_all": [round(x * 1e3, 4) for x in times["streamed"]],
                 "streamed_over_resident_time": round(s / r, 4)}
            ab.append(e)
            print(json.dumps(e), flush=True)
    res["streamed_vs_resident"] = ab
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
