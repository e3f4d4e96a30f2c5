"""Batched, device-resident evaluation sweeps (SURVEY.md section 8e and "next" row N2).

The reference evaluates pose hypotheses in a Python loop inside
``ADDLoss.eval_metrics`` and aggregates on the host (``scripts/visualization/
compare_all_models.py:65-104``: batches of 16, mean of per-batch means).  This module is
the caller-side counterpart of the kernels:

* ``PoseEvaluator`` keeps per-object accumulators (ADD-0.1d hits, valid poses, float64
  ADD / ADD-S sums) on the device; every ``evaluate`` call is one kernel launch and no
  host synchronisation;
* hypotheses are independent, so N GPUs shard the hypothesis axis (``shard_range``) with
  no exchange during compute; the only collective is one all-reduce of the integer
  accumulators (plus the float64 sums) at the end (``PoseEvaluator.all_reduce``) --
  accuracy = hits / valid is computed from integers and is therefore identical for any
  number of GPUs;
* ``reference_batch_means`` reproduces the reference's reporting convention (mean of
  per-batch means) from per-pose outputs, for scripts that must print the same numbers.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as core
from .models.add_loss import SYMMETRIC_OBJECT_IDS

VARIANTS = ("rgb", "rgb_geometric", "rgbd", "rgbd_geometric")


def shard_range(total: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous, balanced slice [lo, hi) of `total` items for `rank` of `world`."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    base, extra = divmod(total, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def reference_batch_means(add, add_s, hit, valid, batch_size: int) -> dict:
    """The numbers ``compare_all_models.py`` prints (:95-104): per batch the reference
    takes ``eval_metrics`` (float64 means over the valid poses of the batch, 0 for an
    empty batch) and then averages the per-batch values over the number of batches --
    the last, shorter batch is over-weighted.  Inputs are per-pose host arrays."""
    add, add_s = np.asarray(add, np.float32), np.asarray(add_s, np.float32)
    hit, valid = np.asarray(hit).astype(bool), np.asarray(valid).astype(bool)
    n = add.shape[0]
    sums = np.zeros(3, np.float64)
    batches = 0
    for lo in range(0, n, batch_size):
        v = valid[lo:lo + batch_size]
        batches += 1
        if not v.any():
            continue
        sums[0] += np.mean(add[lo:lo + batch_size][v].astype(np.float64)) * 1000
        sums[1] += np.mean(add_s[lo:lo + batch_size][v].astype(np.float64)) * 1000
        sums[2] += np.mean(hit[lo:lo + batch_size][v].astype(np.float64)) * 100
    if batches == 0:
        return {"add_mean": 0.0, "add_s_mean": 0.0, "add_01d_acc": 0.0}
    return {"add_mean": sums[0] / batches, "add_s_mean": sums[1] / batches, "add_01d_acc": sums[2] / batches}


class Accumulators:
    """[n_rows, n_slots] device accumulators; one row per model variant (or just one)."""

    def __init__(self, n_rows: int, n_slots: int, device):
        self.hits = torch.zeros(n_rows, n_slots, dtype=torch.int64, device=device)
        self.valid = torch.zeros(n_rows, n_slots, dtype=torch.int64, device=device)
        self.add_sum = torch.zeros(n_rows, n_slots, dtype=torch.float64, device=device)
        self.adds_sum = torch.zeros(n_rows, n_slots, dtype=torch.float64, device=device)

    def row(self, r: int):
        return [self.hits[r], self.valid[r], self.add_sum[r], self.adds_sum[r]]

    def zero_(self):
        for t in (self.hits, self.valid, self.add_sum, self.adds_sum):
            t.zero_()

    def all_reduce(self, group=None):
        """Sum over ranks.  Integers first (exact, order-independent), then the float64
        sums.  Works with NCCL (CUDA tensors) and, for the CPU tests, gloo."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return self
        counts = torch.stack([self.hits, self.valid])
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
        self.hits.copy_(counts[0]); self.valid.copy_(counts[1])
        sums = torch.stack([self.add_sum, self.adds_sum])
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
        self.add_sum.copy_(sums[0]); self.adds_sum.copy_(sums[1])
        return self

    def table(self, row_names=None) -> dict:
        """Host summary: per row and object id -> accuracy %, mean ADD / ADD-S in mm, counts."""
        hits, valid = self.hits.cpu().numpy(), self.valid.cpu().numpy()
        a, s = self.add_sum.cpu().numpy(), self.adds_sum.cpu().numpy()
        out = {}
        for r in range(hits.shape[0]):
            name = row_names[r] if row_names else r
            rows = {}
            for o in np.nonzero(valid[r])[0]:
                n = int(valid[r, o])
                rows[int(o)] = {"n": n, "hits": int(hits[r, o]), "add_01d_acc": 100.0 * int(hits[r, o]) / n,
                                "add_mean": a[r, o] / n * 1000, "add_s_mean": s[r, o] / n * 1000}
            tot = int(valid[r].sum())
            rows["all"] = {"n": tot, "hits": int(hits[r].sum()),
                           "add_01d_acc": 100.0 * int(hits[r].sum()) / tot if tot else 0.0}
            out[name] = rows
        return out


class PoseEvaluator:
    """Device-resident ADD / ADD-S / ADD-0.1d evaluation over large hypothesis sets."""

    def __init__(self, points: dict, diameters: dict, device, symmetric_ids=SYMMETRIC_OBJECT_IDS,
                 n_rows: int = 1, exact_pruning: bool = False, large_meshes: bool = False,
                 large_mesh_pruning: bool = False):
        self.device = core.require_cuda(device)
        self.table = core.MeshTable(points, diameters, symmetric_ids, self.device)
        if exact_pruning:       # opt-in: same bits from the pruned ADD-S kernel where the table qualifies
            self.table.set_pruning(True)
        if large_meshes:        # opt-in: meshes beyond shared memory (up to 32,768 points) through the streamed kernel
            self.table.set_large_meshes(True)
        if large_mesh_pruning:  # opt-in: exact pruning beyond the pruned kernel's shared memory (up to 32,768 points)
            self.table.set_large_mesh_pruning(True)
        self.acc = Accumulators(n_rows, self.table.n_slots, self.device)
        self.launches = 0

    def evaluate(self, pred_q, pred_t, gt_q, gt_t, obj_ids, row: int = 0, want_adds: bool = True,
                 sort: bool = True, per_pose: bool = False):
        """One launch over B poses; accumulates into row `row`.  No host sync unless
        per_pose outputs are converted by the caller."""
        dev = self.device
        pq = core.as_cuda_f32(pred_q, dev, (4,)); pt = core.as_cuda_f32(pred_t, dev, (3,))
        gq = core.as_cuda_f32(gt_q, dev, (4,)); gt = core.as_cuda_f32(gt_t, dev, (3,))
        obj = obj_ids.to(dev, torch.int64).reshape(-1).contiguous()
        order = torch.argsort(obj, stable=True).to(torch.int32) if sort else None
        add, adds, hit, valid, _ = self.table.evaluate(pq, pt, gq, gt, obj, want_adds, order, self.acc.row(row))
        self.launches += 1
        return (add, adds, hit, valid) if per_pose else None

    def all_reduce(self, group=None):
        return self.acc.all_reduce(group)


VARIANT_KINDS = {"rgb": 0, "rgbd": 0, "rgb_geometric": 1, "rgbd_geometric": 2}


def synth_block(n: int, first: int, seed: int, obj_index: int, variant_index: int, variant: str, oid: int, device,
                K=None, rot_sigma=0.05, trans_sigma=0.005) -> dict:
    """Hypotheses [first, first + n) of block (obj_index, variant_index) as the native sweep generates
    them (p6d_synth_poses: counter-based, a pure function of seed / block / hypothesis index), plus
    the variant's raw translation inputs: ``pt`` (kind 0), ``z``/``uv`` (kind 1) or
    ``uv``/``kc``/``depth`` (kind 2).  For tests and for callers that want the data itself."""
    dev = core.require_cuda(device)
    kind = VARIANT_KINDS[variant]
    if K is None:
        from .utils.camera import DEFAULT_K
        K = DEFAULT_K
    Kh = np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
    f32 = lambda *shape: torch.empty(*shape, dtype=torch.float32, device=dev)
    out = {"pq": f32(n, 4), "gq": f32(n, 4), "gt": f32(n, 3), "obj": torch.empty(n, dtype=torch.int64, device=dev)}
    if kind == 0:
        out["pt"] = f32(n, 3)
    elif kind == 1:
        out["z"], out["uv"] = f32(n), f32(n, 2)
    else:
        out["uv"], out["kc"], out["depth"] = f32(n, 2), f32(n, 3, 3), f32(n, 8, 8)
    g = lambda k: core.ptr(out.get(k))
    core.check(core.lib().p6d_synth_poses(int(seed), int(obj_index), int(variant_index), int(first), int(n),
                                          float(rot_sigma), float(trans_sigma), kind, core.ptr(Kh), int(oid),
                                          g("pq"), g("pt"), g("gq"), g("gt"), g("obj"), g("z"), g("uv"), g("kc"),
                                          g("depth"), dev.index, core.stream_ptr(dev)))
    return out


def variant_translation(variant: str, block: dict, K):
    """How each model family produces its translation (SURVEY.md section 8d, config 5), from the
    raw inputs of ``synth_block``: rgb / rgbd regress xyz directly; rgb_geometric predicts Z and
    back-projects the bbox centre (kernel d1, reference models/pose_net_rgb_geometric.py:93-109);
    rgbd_geometric reads Z from a depth crop under the crop-space centre (kernel d2, reference
    models/pose_net_rgbd_geometric.py:56-85)."""
    from .utils.camera import depth_backproject, pinhole_translation
    kind = VARIANT_KINDS[variant]
    if kind == 0:
        return block["pt"]
    if kind == 1:
        return pinhole_translation(block["z"].reshape(-1, 1), block["uv"], K)
    return depth_backproject(block["depth"], block["uv"], block["kc"], clamp_hi=7.0)


def evaluate_sweep(points: dict, diameters: dict, device, n_per_block: int, variants=VARIANTS, chunk: int = 1 << 20,
                   seed: int = 5000, rank: int = 0, world: int = 1, group=None, K=None, check_n: int = 0,
                   rot_sigma: float = 0.05, trans_sigma: float = 0.005, evaluator: "PoseEvaluator | None" = None,
                   exact_pruning: bool = False, large_meshes: bool = False, large_mesh_pruning: bool = False):
    """compare_all_models-style sweep (reference scripts/visualization/compare_all_models.py:65-104 at the
    scale of BASELINE config 5): for every (object, variant) block, `n_per_block` seeded hypotheses, the
    hypothesis axis of each block sliced across `world` ranks (`shard_range`).  The whole sweep of this
    rank is ONE native call (p6d_sweep_run: generation, the variant's translation kernel and the
    evaluation overlap on two streams); the only collective is the all-reduce of the accumulators at
    the end.  Returns (Accumulators after the all-reduce, kernel launches on this rank, check) where
    `check` holds the first `check_n` hypotheses of every block of this rank's slice exactly as they
    were evaluated (inputs and outputs, host arrays) for an independent re-evaluation, or None."""
    dev = core.require_cuda(device)
    ev = evaluator or PoseEvaluator(points, diameters, dev, n_rows=len(variants), exact_pruning=exact_pruning,
                                    large_meshes=large_meshes, large_mesh_pruning=large_mesh_pruning)
    if K is None:
        from .utils.camera import DEFAULT_K
        K = DEFAULT_K
    Kh = np.ascontiguousarray((K.detach().cpu().numpy() if isinstance(K, torch.Tensor) else np.asarray(K))
                              .astype(np.float32).reshape(9))
    objs = np.ascontiguousarray(sorted(int(o) for o in points), dtype=np.int32)
    kinds = np.ascontiguousarray([VARIANT_KINDS[v] for v in variants], dtype=np.int32)
    lo, hi = shard_range(n_per_block, rank, world)
    cn = min(int(check_n), hi - lo)
    nb = len(objs) * len(variants)
    check = None
    if cn > 0:
        check = {"pq": np.empty((nb, cn, 4), np.float32), "pt": np.empty((nb, cn, 3), np.float32),
                 "gq": np.empty((nb, cn, 4), np.float32), "gt": np.empty((nb, cn, 3), np.float32),
                 "add": np.empty((nb, cn), np.float32), "adds": np.empty((nb, cn), np.float32),
                 "hit": np.empty((nb, cn), np.uint8),
                 "obj": np.repeat(objs.astype(np.int64), len(variants))[:, None].repeat(cn, 1),
                 "variant": np.tile(np.arange(len(variants)), len(objs)), "first": lo}
    launches = C.c_int(0)
    cp = lambda k: core.ptr(check[k]) if check is not None else None
    acc = ev.acc
    core.check(core.lib().p6d_sweep_run(ev.table.handle, core.ptr(objs), len(objs), core.ptr(kinds), len(variants),
                                        int(n_per_block), int(lo), int(hi), int(chunk), int(seed), core.ptr(Kh),
                                        float(rot_sigma), float(trans_sigma), core.ptr(acc.hits), core.ptr(acc.valid),
                                        core.ptr(acc.add_sum), core.ptr(acc.adds_sum), cn, cp("pq"), cp("pt"), cp("gq"),
                                        cp("gt"), cp("add"), cp("adds"), cp("hit"), C.byref(launches),
                                        core.stream_ptr(dev)))
    ev.launches += launches.value
    ev.all_reduce(group)
    return ev.acc, launches.value, check
