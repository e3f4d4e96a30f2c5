"""Second checker -- TEST INFRASTRUCTURE, NOT PRODUCT: the reference's op sequence executed by the
PyTorch build of THIS machine (CPU eager), and a locator for the real reference.

Why a second checker next to the C restatement (oracle/pose_oracle.c): the C code states how
torch 2.11 / MKL round (``torch.mm`` per mesh size, ``torch.norm``, ATen's cascade sum); that was
probed in the build container.  The kernels reproduce those bits, so the bit-exactness claim is
only as good as the assumption that the box the numbers come from rounds the same way.  The
functions below make that a live test on every box: they run the very torch ops the reference
calls, in its order, on the local CPU, with no knowledge of any rounding rule.

    eval_pose / eval_poses   models/add_loss.py:168-195 (loop body of ADDLoss.eval_metrics)
    forward_value            models/add_loss.py:101-150 (ADDLoss.forward)
    quat_to_mat              models/add_loss.py:203-215
    resolve_borderline       decisions for poses the kernels flag as within 4 ulp of the threshold
    find_reference / load_reference   the unmodified reference, when reachable
                             (P6D_REFERENCE, baseline/_ref)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs use this
module.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import tempfile

import numpy as np
import torch

SYMMETRIC = frozenset({9, 10})     # models/add_loss.py:10
_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def quat_to_mat(q: torch.Tensor) -> torch.Tensor:
    """[B,4] scalar-last quaternion -> [B,3,3], no normalisation (models/add_loss.py:203-215)."""
    x, y, z, w = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    xx, yy, zz = x * x, y * y, z * z
    xy, xz, yz = x * y, x * z, y * z
    wx, wy, wz = w * x, w * y, w * z
    rows = [torch.stack([1 - 2 * yy - 2 * zz, 2 * xy - 2 * wz, 2 * xz + 2 * wy], dim=1),
            torch.stack([2 * xy + 2 * wz, 1 - 2 * xx - 2 * zz, 2 * yz - 2 * wx], dim=1),
            torch.stack([2 * xz - 2 * wy, 2 * yz + 2 * wx, 1 - 2 * xx - 2 * yy], dim=1)]
    return torch.stack(rows, dim=1)


@torch.no_grad()
def eval_pose(mesh: torch.Tensor, Rp, tp, Rg, tg, want_adds: bool = True):
    """(ADD, ADD-S) of one pose as Python floats (models/add_loss.py:178-190)."""
    cloud_gt = torch.mm(mesh, Rg.T) + tg
    cloud_pred = torch.mm(mesh, Rp.T) + tp
    add = torch.norm(cloud_pred - cloud_gt, dim=1, p=2).mean().item()
    if not want_adds:
        return add, 0.0
    pair = torch.norm(cloud_pred.unsqueeze(1) - cloud_gt.unsqueeze(0), dim=2)
    return add, pair.min(dim=1)[0].mean().item()


@torch.no_grad()
def eval_poses(points: dict, diameters: dict, pq, pt, gq, gt, obj, want_adds: bool = True):
    """Per-pose float32 ADD, ADD-S, uint8 hit / valid for a batch (models/add_loss.py:156-195)."""
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float32))
    pq, pt, gq, gt = T(pq).reshape(-1, 4), T(pt).reshape(-1, 3), T(gq).reshape(-1, 4), T(gt).reshape(-1, 3)
    obj = np.asarray(obj, np.int64).ravel()
    meshes = {int(k): T(v).reshape(-1, 3) for k, v in points.items()}
    Rp_all, Rg_all = quat_to_mat(pq), quat_to_mat(gq)
    B = obj.shape[0]
    add, adds = np.zeros(B, np.float32), np.zeros(B, np.float32)
    hit, valid = np.zeros(B, np.uint8), np.zeros(B, np.uint8)
    for i in range(B):
        oid = int(obj[i])
        if oid not in meshes:
            continue
        a, s = eval_pose(meshes[oid], Rp_all[i], pt[i], Rg_all[i], gt[i], want_adds)
        thr = 0.1 * diameters.get(oid, 0.1)
        decide = s if (oid in SYMMETRIC and want_adds) else a
        add[i], adds[i], valid[i] = a, s, 1
        hit[i] = 1 if decide < thr else 0
    return add, adds, hit, valid


@torch.no_grad()
def forward_value(points: dict, pq, pt, gq, gt, obj) -> np.float32:
    """Value of ADDLoss.forward (models/add_loss.py:101-150): grouping by object in order of first
    appearance, batched matmul per group, per-group sum, total / count."""
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float32))
    pq, pt, gq, gt = T(pq).reshape(-1, 4), T(pt).reshape(-1, 3), T(gq).reshape(-1, 4), T(gt).reshape(-1, 3)
    obj = np.asarray(obj, np.int64).ravel()
    meshes = {int(k): T(v).reshape(-1, 3) for k, v in points.items()}
    Rp, Rg = quat_to_mat(pq), quat_to_mat(gq)
    groups: dict[int, list[int]] = {}
    for i, o in enumerate(obj):
        if int(o) in meshes:
            groups.setdefault(int(o), []).append(i)
    total, count = torch.tensor(0.0), 0
    for oid, idx in groups.items():
        idx_t = torch.tensor(idx, dtype=torch.long)
        m = meshes[oid].unsqueeze(0)
        cg = torch.matmul(m, Rg[idx_t].transpose(-1, -2)) + gt[idx_t].unsqueeze(1)
        cp = torch.matmul(m, Rp[idx_t].transpose(-1, -2)) + pt[idx_t].unsqueeze(1)
        if oid in SYMMETRIC:
            per = torch.norm(cp.unsqueeze(2) - cg.unsqueeze(1), dim=3).min(dim=2)[0].mean(dim=1)
        else:
            per = torch.norm(cp - cg, dim=2).mean(dim=1)
        total = total + per.sum()
        count += len(idx)
    return np.float32(0.0) if count == 0 else np.float32((total / count).item())


def resolve_borderline(points: dict, diameters: dict):
    """A ``borderline_resolver`` for ``ADDLoss`` (6d-pose-estimation_b200/models/add_loss.py): re-decides
    the flagged poses with this machine's own torch CPU ops."""
    def resolver(indices, pred_r, pred_t, gt_r, gt_t, obj_ids):
        to = lambda t: (t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t))
        idx = np.asarray(indices, np.int64)
        _, _, hit, _ = eval_poses(points, diameters, to(pred_r)[idx], to(pred_t)[idx], to(gt_r)[idx], to(gt_t)[idx],
                                  to(obj_ids)[idx])
        return hit
    return resolver


# --------------------------------------------------------------------------- the real reference
def find_reference() -> str | None:
    """Directory of the unmodified reference if this machine has one (P6D_REFERENCE, or baseline/_ref)."""
    for cand in (os.environ.get("P6D_REFERENCE"), os.path.join(_REPO, "baseline", "_ref")):
        if cand and os.path.isfile(os.path.join(cand, "models", "add_loss.py")):
            return cand
    return None


def load_reference(root: str):
    """The reference's own ``ADDLoss`` class, imported from its file without touching sys.modules'
    ``models`` package (the product's drop-in layout may own that name)."""
    spec = importlib.util.spec_from_file_location("_p6d_reference_add_loss", os.path.join(root, "models", "add_loss.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[spec.name] = mod
    spec.loader.exec_module(mod)
    return mod.ADDLoss


def reference_criterion(root: str, points: dict, diameters: dict):
    """ADDLoss of the real reference on the CPU with the given meshes (SURVEY.md section 0.5: an empty
    model directory, then the public ``points`` / ``diameters`` dicts)."""
    crit = load_reference(root)(tempfile.mkdtemp(), "cpu")
    for k, v in points.items():
        crit.points[int(k)] = torch.from_numpy(np.ascontiguousarray(v, np.float32))
    for k, v in diameters.items():
        crit.diameters[int(k)] = float(v)
    return crit


@torch.no_grad()
def reference_eval_poses(crit, pq, pt, gq, gt, obj):
    """Per-pose values out of the real reference: ``eval_metrics`` at batch size 1 (SURVEY.md 8c)."""
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    B = len(obj)
    add, adds = np.zeros(B, np.float32), np.zeros(B, np.float32)
    hit, valid = np.zeros(B, np.uint8), np.zeros(B, np.uint8)
    for i in range(B):
        if int(obj[i]) not in crit.points:
            continue
        m = crit.eval_metrics(T(pq[i:i + 1]), T(pt[i:i + 1]), T(gq[i:i + 1]), T(gt[i:i + 1]), T(obj[i:i + 1]))
        add[i], adds[i] = np.float32(m["add_mean"] / 1000.0), np.float32(m["add_s_mean"] / 1000.0)
        hit[i], valid[i] = (1 if m["add_01d_acc"] == 100.0 else 0), 1
    return add, adds, hit, valid
