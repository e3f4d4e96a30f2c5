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
    add_loss_grad, pose_loss_grad, geometric_loss_grad, pinhole_translation
                             the gradients of ADDLoss.forward, PoseLoss.forward and the RGB-Geometric
                             step under autograd, in float32 and in float64 (tests/test_gradients.py)
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


# --------------------------------------------------------------------------- autograd references
# Each gradient reference runs in two forms.  float32 (decisions=None) is the reference's own op
# sequence under autograd: it rounds like the reference, so it takes the reference's discrete decisions,
# and it returns them.  float64 (dtype=torch.float64, decisions=<those>) repeats the computation on the
# same inputs with every discrete decision taken from the float32 run -- nearest-point indices, the
# dot < 0 flip, the L1 branch, the 1e-12 clamp, zero distances and sign(0) -- because float64 takes
# other branches on degenerate rows (an antipodal prediction scaled by 3 has a gradient of exactly 0 in
# float32, not in float64).  Within those decisions the float64 form is the exact gradient up to 1e-15.
def _const(a, dtype, shape):
    return torch.from_numpy(np.array(a)).reshape(shape).to(dtype)


def _leaf(a, dtype, shape):
    return _const(a, dtype, shape).requires_grad_(True)


def add_loss_grad(points: dict, pq, pt, gq, gt, obj, grad_out=1.0, dtype=torch.float32, decisions=None):
    """(grad_q [B,4], grad_t [B,3], decisions) of ADDLoss.forward (models/add_loss.py:101-150) under
    autograd.  The clouds are transformed per object group with the reference's batched matmul; the
    nearest gt point of a symmetric object is found per sample with the reference's own
    ``torch.norm(...).min(dim=2)`` (no [n,N,N,3] graph for all n at once), and the gradient flows through
    the chosen points, which is what min's backward does.  decisions: per sample, the chosen gt index of
    every pred point and the mask of zero distances."""
    B = np.asarray(obj).size
    a, b = _leaf(pq, dtype, (B, 4)), _leaf(pt, dtype, (B, 3))
    gqt, gtt = _const(gq, dtype, (B, 4)), _const(gt, dtype, (B, 3))
    objs = np.asarray(obj, np.int64).ravel()
    meshes = {int(k): _const(v, dtype, (-1, 3)) for k, v in points.items()}
    Rp, Rg = quat_to_mat(a), quat_to_mat(gqt)
    groups: dict[int, list[int]] = {}
    for i, o in enumerate(objs):
        if int(o) in meshes:
            groups.setdefault(int(o), []).append(i)
    count = sum(len(v) for v in groups.values())
    out_dec = {}
    total = None
    for oid, idx in groups.items():
        idx_t = torch.tensor(idx, dtype=torch.long)
        m = meshes[oid].unsqueeze(0)
        cg = torch.matmul(m, Rg[idx_t].transpose(-1, -2)) + gtt[idx_t].unsqueeze(1)
        cp = torch.matmul(m, Rp[idx_t].transpose(-1, -2)) + b[idx_t].unsqueeze(1)
        for k, s in enumerate(idx):
            if decisions is None:
                if oid in SYMMETRIC:
                    with torch.no_grad():
                        near = torch.norm(cp[k].unsqueeze(1) - cg[k].unsqueeze(0), dim=2).min(dim=1)[1]
                else:
                    near = torch.arange(m.shape[1])
                diff = cp[k] - cg[k][near]
                d = torch.norm(diff, dim=1)
                out_dec[s] = (near, (d == 0).detach())
            else:
                near, zero = decisions[s]
                diff = (cp[k] - cg[k][near]) * (~zero).to(dtype).unsqueeze(1)
                d = torch.norm(diff, dim=1)
            term = d.mean()
            total = term if total is None else total + term
    if total is None:
        z = np.zeros((B, 4), np.float64 if dtype == torch.float64 else np.float32)
        return z, z[:, :3].copy(), out_dec
    loss = total / count
    loss.backward(torch.tensor(grad_out, dtype=dtype))
    ga = a.grad if a.grad is not None else torch.zeros_like(a)
    gb = b.grad if b.grad is not None else torch.zeros_like(b)
    return ga.numpy(), gb.numpy(), (out_dec if decisions is None else decisions)


def pose_loss_grad(pq, pt, gq, gt, rot_weight=1.0, trans_weight=1.0, mode="geodesic", grad_out=1.0,
                   dtype=torch.float32, decisions=None):
    """(loss, grad_q [B,4], grad_t [B,3], decisions) of PoseLoss.forward (models/pose_loss.py:19-61) under
    autograd: F.normalize, where(dot < 0), 2*atan2(|q1-q2|, |q1+q2|) or the torch.min of the two L1 sums,
    F.l1_loss, the weights.  Anything but 'geodesic' selects the L1 distance, as in the reference."""
    import torch.nn.functional as F
    B = np.asarray(pq).size // 4
    a, b = _leaf(pq, dtype, (B, 4)), _leaf(pt, dtype, (B, 3))
    c, g = _const(gq, dtype, (B, 4)), _const(gt, dtype, (B, 3))
    if decisions is None:
        q1, q2 = F.normalize(a, dim=1), F.normalize(c, dim=1)
        dec = {"clamp": (torch.norm(a.detach(), dim=1) < 1e-12)}
        if mode == "geodesic":
            dot = torch.sum(q1 * q2, dim=1, keepdim=True)
            q2 = torch.where(dot < 0, -q2, q2)
            dn, sn = torch.norm(q1 - q2, dim=1), torch.norm(q1 + q2, dim=1)
            rot = (2 * torch.atan2(dn, sn)).mean()
            dec.update(flip=(dot < 0).detach(), dn0=(dn == 0).detach(), sn0=(sn == 0).detach())
        else:
            dp, dm = torch.sum(torch.abs(q1 - q2), dim=1), torch.sum(torch.abs(q1 + q2), dim=1)
            rot = torch.min(dp, dm).mean()
            dec.update(wp=torch.where(dp < dm, 1.0, torch.where(dp == dm, 0.5, 0.0)).detach(),
                       ap0=(q1 - q2 == 0).detach(), am0=(q1 + q2 == 0).detach())
        dec["t0"] = (b - g == 0).detach()
        trans = F.l1_loss(b, g)
    else:
        dec = decisions
        keep = lambda x, zero: x * (~zero).to(dtype)
        na = torch.where(dec["clamp"], torch.full((B,), 1e-12, dtype=dtype), torch.norm(a, dim=1))
        q1 = a / na.unsqueeze(1)
        q2 = c / torch.norm(c, dim=1).clamp_min(1e-12).unsqueeze(1)
        if mode == "geodesic":
            q2 = torch.where(dec["flip"], -q2, q2)
            dn = torch.norm(keep(q1 - q2, dec["dn0"].unsqueeze(1)), dim=1)
            sn = torch.norm(keep(q1 + q2, dec["sn0"].unsqueeze(1)), dim=1)
            rot = (2 * torch.atan2(dn, sn)).mean()
        else:
            wp = dec["wp"].to(dtype)
            dp = torch.sum(torch.abs(keep(q1 - q2, dec["ap0"])), dim=1)
            dm = torch.sum(torch.abs(keep(q1 + q2, dec["am0"])), dim=1)
            rot = (wp * dp + (1 - wp) * dm).mean()
        trans = torch.abs(keep(b - g, dec["t0"])).mean()
    loss = rot_weight * rot + trans_weight * trans
    loss.backward(torch.tensor(grad_out, dtype=dtype))
    return loss.item(), a.grad.numpy(), b.grad.numpy(), dec


def pinhole_translation(z, uv, K):
    """PoseNetRGBGeometric._compute_pinhole_translation (models/pose_net_rgb_geometric.py:93-109) on
    tensors: [(u - cx) * z / fx, (v - cy) * z / fy, z], K [3,3] or [B,3,3]; differentiable in z."""
    K = K.reshape(-1, 3, 3)
    fx, fy, cx, cy = K[:, 0, 0:1], K[:, 1, 1:2], K[:, 0, 2:3], K[:, 1, 2:3]
    z = z.reshape(-1, 1)
    return torch.cat([(uv[:, 0:1] - cx) * z / fx, (uv[:, 1:2] - cy) * z / fy, z], dim=1)


def geometric_loss_grad(pq, z, uv, K, gq, gt, rot_weight=1.0, trans_weight=1.0, mode="geodesic", grad_out=1.0,
                        dtype=torch.float32, decisions=None):
    """(loss, grad_q [B,4], grad_z [B,1], decisions): PoseLoss on the pinhole translation, autograd through
    both (the RGB-Geometric training step, train_rgb_geometric.py:104-108)."""
    B = np.asarray(pq).size // 4
    zz = _leaf(z, dtype, (B, 1))
    tr = pinhole_translation(zz, _const(uv, dtype, (B, 2)), _const(K, dtype, (-1, 3, 3)))
    t32 = tr.detach().to(torch.float32).numpy() if dtype == torch.float32 else None
    if decisions is None:
        loss, gq_, gt_, dec = pose_loss_grad(pq, t32, gq, gt, rot_weight, trans_weight, mode, grad_out)
    else:
        dec = decisions
        loss, gq_, gt_, _ = pose_loss_grad(pq, tr.detach().numpy(), gq, gt, rot_weight, trans_weight, mode,
                                           grad_out, torch.float64, dec)
    tr.backward(torch.from_numpy(gt_).to(dtype))
    return loss, gq_, zz.grad.numpy(), dec


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
