"""ADD / ADD-S / ADD-0.1d on B200 -- drop-in for the reference's ``models/add_loss.py``.

Same names, argument order, defaults and return types as the reference
(SFR-Vision/6d-pose-estimation ``models/add_loss.py``); the arithmetic runs in
``libp6d.so`` (hand-written sm_100a kernels) instead of a per-pose Python loop of eager
ops.  One kernel launch and one device->host copy per ``eval_metrics`` call replace
~12 launches and 4 host syncs per pose (reference ``add_loss.py:168-195``).

There is no CPU path: the device must be CUDA.
"""
import os

import numpy as np
import torch
import torch.nn as nn


try:                                    # imported as part of the package ...
    from .._p6d_bootstrap import core as _core
except ImportError:                     # ... or as top-level `models` / `utils` (drop-in layout: this
    from _p6d_bootstrap import core as _core   # directory is at the front of sys.path, see dropin.py)


# eggbox and glue (reference add_loss.py:10)
SYMMETRIC_OBJECT_IDS = {9, 10}

_SORT_THRESHOLD = 256  # batches at least this large are processed in object order


def _read_ascii_ply(path):
    """Vertex block of an ASCII PLY, with the reference's permissive rule
    (add_loss.py:83-99): after the header every line with >= 3 whitespace-separated
    tokens contributes its first three as a vertex -- face lines ``3 i j k`` included."""
    rows = []
    with open(path, "r") as fh:
        in_body = False
        for raw in fh:
            if not in_body:
                in_body = "end_header" in raw
                continue
            tok = raw.split()
            if len(tok) >= 3:
                rows.append((float(tok[0]), float(tok[1]), float(tok[2])))
    return np.array(rows)


class _AddForward(torch.autograd.Function):
    """ADDLoss.forward as one launch (p6d_add_forward) with the fused backward
    (p6d_add_backward) attached; nothing is read back to the host on either side."""

    @staticmethod
    def forward(ctx, pred_r, pred_t, crit, prepared):
        dev, pq, pt, gq, gt, obj, table = prepared
        loss, count = table.forward_loss(pq, pt, gq, gt, obj)
        ctx.saved = (pq, pt, gq, gt, obj, count, table, dev)
        ctx.shapes = (pred_r.shape, pred_t.shape, pred_r.dtype, pred_t.dtype)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_out):
        gq, gt = _core().add_backward(ctx.saved, grad_out)
        rs, ts, rd, td = ctx.shapes
        return gq.reshape(rs).to(rd), gt.reshape(ts).to(td), None, None


class ADDLoss(nn.Module):
    """ADD, ADD-S and ADD-0.1d for 6-D pose estimation (reference add_loss.py:13-215)."""

    def __init__(self, model_dir, device, rot_weight=0.0, trans_weight=0.0):
        super().__init__()
        self.points = {}       # object id -> float32 [N,3] tensor on `device`
        self.diameters = {}    # object id -> metres
        self.device = device
        self.rot_weight = rot_weight      # stored, unused -- as in the reference (:24-25)
        self.trans_weight = trans_weight
        self._table = None
        self._table_key = None
        self._table_pruning = False
        self._table_large = False
        self._table_large_loss = False
        self._table_large_pruning = False
        # optional callable(indices, pred_r, pred_t, gt_r, gt_t, obj_ids) -> 0/1 per index, consulted by
        # eval_metrics for decisions flagged `borderline`; None (default): the kernel's decision stands
        self.borderline_resolver = None
        # opt-in: exact block pruning in the ADD-S kernel (same bits; pays for meshes of >= 128 points, the
        # all-pairs kernel is kept below that) -- not part of the reference surface, default off
        self.exact_pruning = False
        # opt-in: meshes beyond shared memory (up to 32,768 points) through the streamed kernel in eval_metrics /
        # eval_poses (same bits; evaluation only) -- not part of the reference surface, default off
        self.large_meshes = False
        # opt-in: meshes beyond shared memory (up to 32,768 points) through the streamed loss-form and gradient
        # kernels in forward / train_loss and loss.backward() (same loss bits; the resident kernels wherever they
        # run) -- not part of the reference surface, default off
        self.large_mesh_loss = False
        # opt-in: exact block pruning for meshes beyond the pruned kernel's shared memory (up to 32,768 points) in
        # eval_metrics / eval_poses (same bits; evaluation only) -- not part of the reference surface, default off
        self.large_mesh_pruning = False
        self._load_models(model_dir)

    # ------------------------------------------------------------------ loading
    def _load_ply(self, path):
        return _read_ascii_ply(path)

    def _load_models(self, model_dir, num_points=500):
        """PLY meshes + diameters.  Consumes the global NumPy RNG exactly like the
        reference (diameter-fallback ``choice`` first, then the down-sampling ``choice``,
        per PLY in sorted order; add_loss.py:29-81) so a fixed ``np.random.seed`` gives
        the same 500-point subsets."""
        known = {}
        info_file = os.path.join(model_dir, "models_info.yml")
        if os.path.exists(info_file):
            import yaml
            with open(info_file, "r") as fh:
                info = yaml.safe_load(fh)
            for key, entry in info.items():
                try:
                    if "diameter" in entry:
                        known[int(key) - 1] = entry["diameter"] / 1000.0
                except Exception:
                    continue
        for name in sorted(n for n in os.listdir(model_dir) if n.endswith(".ply")):
            try:
                oid = int(name.split("_")[1].split(".")[0]) - 1
            except Exception:
                continue
            cloud = self._load_ply(os.path.join(model_dir, name)) / 1000.0
            cloud = cloud[np.linalg.norm(cloud, axis=1) < 0.5]      # outlier filter (:61-62)
            if oid in known:
                self.diameters[oid] = known[oid]
            elif cloud.shape[0] > 10:
                pick = np.random.choice(cloud.shape[0], min(100, cloud.shape[0]), replace=False)
                sub = cloud[pick]
                self.diameters[oid] = np.max(np.linalg.norm(sub[:, None] - sub[None, :], axis=2))
            else:
                self.diameters[oid] = 0.1
            if cloud.shape[0] > num_points:
                cloud = cloud[np.random.choice(cloud.shape[0], num_points, replace=False)]
            self.points[oid] = torch.from_numpy(cloud.astype(np.float32)).to(self.device)

    # ------------------------------------------------------------------ device table
    def _cuda_device(self, like=None):
        core = _core()
        dev = torch.device(self.device) if not isinstance(self.device, torch.device) else self.device
        if dev.type != "cuda" and like is not None and like.is_cuda:
            dev = like.device
        return core.require_cuda(dev)

    def _mesh_table(self, device):
        """(Re)build the device mesh table when points / diameters were mutated."""
        key = (str(device),) + tuple(
            (k, v.data_ptr(), v._version, tuple(v.shape)) if isinstance(v, torch.Tensor)
            else (k, id(v)) for k, v in sorted(self.points.items())
        ) + tuple(sorted((k, float(v)) for k, v in self.diameters.items()))
        if self._table is None or key != self._table_key:
            if self._table is not None:
                self._table.close()
            self._table = _core().MeshTable(self.points, self.diameters, SYMMETRIC_OBJECT_IDS, device)
            self._table_key = key
            self._table_pruning = False
            self._table_large = False
            self._table_large_loss = False
            self._table_large_pruning = False
        if bool(self.exact_pruning) != self._table_pruning:
            self._table.set_pruning(bool(self.exact_pruning))
            self._table_pruning = bool(self.exact_pruning)
        if bool(self.large_meshes) != self._table_large:
            self._table.set_large_meshes(bool(self.large_meshes))
            self._table_large = bool(self.large_meshes)
        if bool(self.large_mesh_loss) != self._table_large_loss:
            self._table.set_large_mesh_loss(bool(self.large_mesh_loss))
            self._table_large_loss = bool(self.large_mesh_loss)
        if bool(self.large_mesh_pruning) != self._table_large_pruning:
            self._table.set_large_mesh_pruning(bool(self.large_mesh_pruning))
            self._table_large_pruning = bool(self.large_mesh_pruning)
        return self._table

    def _prepare(self, pred_r, pred_t, gt_r, gt_t, obj_ids, sort=True):
        core = _core()
        dev = self._cuda_device(pred_r if isinstance(pred_r, torch.Tensor) else None)
        pq = core.as_cuda_f32(pred_r, dev, (4,))
        pt = core.as_cuda_f32(pred_t, dev, (3,))
        gq = core.as_cuda_f32(gt_r, dev, (4,))
        gt = core.as_cuda_f32(gt_t, dev, (3,))
        obj = obj_ids if isinstance(obj_ids, torch.Tensor) else torch.as_tensor(np.asarray(obj_ids))
        obj = obj.detach().to(dev, torch.int64, non_blocking=True).reshape(-1).contiguous()
        B = obj.shape[0]
        if not (pq.shape[0] == pt.shape[0] == gq.shape[0] == gt.shape[0] == B):
            raise ValueError("pred_r, pred_t, gt_r, gt_t and obj_ids must share the batch dimension")
        order = None
        if sort and B >= _SORT_THRESHOLD:
            order = torch.argsort(obj, stable=True).to(torch.int32)
        return dev, pq, pt, gq, gt, obj, order

    # ------------------------------------------------------------------ evaluation
    @torch.no_grad()
    def eval_metrics(self, pred_r, pred_t, gt_r, gt_t, obj_ids):
        """{'add_mean' [mm], 'add_s_mean' [mm], 'add_01d_acc' [%]} over the poses whose
        object has a mesh; int 0 entries when there is none (reference :156-201)."""
        per_pose = self.eval_poses(pred_r, pred_t, gt_r, gt_t, obj_ids)
        keep = per_pose["valid"].view(np.bool_)
        n_keep = int(np.count_nonzero(keep))
        if n_keep == 0:
            return {"add_mean": 0, "add_s_mean": 0, "add_01d_acc": 0}
        hit = per_pose["hit"]
        if self.borderline_resolver is not None and per_pose["borderline"].any():
            # decisions within 4 ulp of the threshold: let the caller's own reference decide
            # (see INTEGRATION.md; tests/ use the torch-eager restatement on the host)
            idx = np.nonzero(per_pose["borderline"] & per_pose["valid"])[0]
            if idx.size:
                hit = hit.copy()
                hit[idx] = np.asarray(self.borderline_resolver(idx, pred_r, pred_t, gt_r, gt_t, obj_ids), np.uint8)
        add, add_s = per_pose["add"], per_pose["add_s"]
        if n_keep != keep.shape[0]:
            add, add_s, hit = add[keep], add_s[keep], hit[keep]
        # the reference averages lists of Python floats on the host: np.mean over a float64 ARRAY
        # (np.mean(x32, dtype=float64) casts in 8192-element buffers and sums in another pairwise order:
        # it differs in the last bit from 65,536 elements on)
        return {
            "add_mean": np.mean(add.astype(np.float64)) * 1000,
            "add_s_mean": np.mean(add_s.astype(np.float64)) * 1000,
            "add_01d_acc": np.mean(hit.astype(np.float64)) * 100,
        }

    @torch.no_grad()
    def eval_poses(self, pred_r, pred_t, gt_r, gt_t, obj_ids):
        """Per-pose float32 ADD, ADD-S, uint8 hit / valid / borderline as NumPy arrays (one
        launch, one device->host copy).  Addition to the reference surface.  ``borderline`` marks
        decisions whose distance lies within 4 float32 ulp of 0.1*diameter (SURVEY.md 7.3.1)."""
        dev, pq, pt, gq, gt, obj, order = self._prepare(pred_r, pred_t, gt_r, gt_t, obj_ids)
        B = obj.shape[0]
        if B == 0 or not self.points:
            z = np.zeros(B, np.float32)
            zb = np.zeros(B, np.uint8)
            return {"add": z, "add_s": z.copy(), "hit": zb, "valid": zb.copy(), "borderline": zb.copy()}
        table = self._mesh_table(dev)
        host = table.packed_to_host(table.evaluate_packed(pq, pt, gq, gt, obj, True, order)).copy()
        return {"add": host[:4 * B].view(np.float32), "add_s": host[4 * B:8 * B].view(np.float32),
                "hit": host[8 * B:9 * B], "valid": host[9 * B:10 * B], "borderline": host[10 * B:11 * B]}

    # ------------------------------------------------------------------ differentiable loss
    def forward(self, pred_r, pred_t, gt_r, gt_t, obj_ids):
        """Mean over valid samples of ADD (asymmetric ids) or ADD-S (symmetric ids); 0-d tensor
        (reference :101-150).  ONE kernel launch, no host synchronisation: the reference's grouping
        (objects in order of first appearance, float32 sum per group, total / count) happens on the
        device.  When no sample has a mesh the value is 0 and, like the reference's fresh
        ``tensor(0.0, requires_grad=True)``, carries no gradient to the inputs."""
        dev, pq, pt, gq, gt, obj, _ = self._prepare(pred_r, pred_t, gt_r, gt_t, obj_ids, sort=False)
        if obj.shape[0] == 0 or not self.points:
            return torch.tensor(0.0, device=dev).requires_grad_(True)
        prepared = (dev, pq, pt, gq, gt, obj, self._mesh_table(dev))
        wants_grad = torch.is_grad_enabled() and any(
            isinstance(t, torch.Tensor) and t.requires_grad for t in (pred_r, pred_t))
        if not wants_grad:
            loss, _ = prepared[-1].forward_loss(pq, pt, gq, gt, obj)
            loss = loss.reshape(())
            # No input asks for a gradient.  The reference then returns a plain tensor -- except when no
            # sample has a mesh, where it returns a fresh leaf with requires_grad=True so that a training
            # loop's .backward() does not raise.  Which case applies is only known on the device, so the
            # result is a leaf that accepts .backward() in both (deviation: also in the non-empty case).
            return loss.requires_grad_(True) if torch.is_grad_enabled() else loss
        pr = pred_r if isinstance(pred_r, torch.Tensor) else torch.as_tensor(pred_r)
        pt_in = pred_t if isinstance(pred_t, torch.Tensor) else torch.as_tensor(pred_t)
        return _AddForward.apply(pr, pt_in, self, prepared)

    def train_loss(self, pred_r, pred_t, gt_r, gt_t, obj_ids):
        return self.forward(pred_r, pred_t, gt_r, gt_t, obj_ids)

    # ------------------------------------------------------------------ quaternion -> matrix
    def _quat_to_mat(self, q):
        """[B,4] scalar-last quaternions -> [B,3,3]; no normalisation (reference :203-215)."""
        core = _core()
        dev = self._cuda_device(q if isinstance(q, torch.Tensor) else None)
        qq = core.as_cuda_f32(q, dev, (4,))
        out = torch.empty(qq.shape[0], 3, 3, dtype=torch.float32, device=dev)
        core.check(core.lib().p6d_quat_to_mat(core.ptr(qq), qq.shape[0], core.ptr(out), dev.index,
                                              core.stream_ptr(dev)))
        return out
