"""ctypes binding of ``csrc/libp6d.so`` (the C ABI declared in ``include/p6d.h``).

This is the only module that talks to native code.  It is registered in
``sys.modules`` as ``p6d_b200_core`` so that the reference-shaped modules
(``models/add_loss.py``, ``models/pose_loss.py``, ``utils/camera.py``) find the same
instance whether they are imported as part of this package or as top-level ``models`` /
``utils`` (the drop-in layout, see INTEGRATION.md).

There is no fallback of any kind: if the shared object is missing or was built for
another architecture, importing the compute entry points raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
SO_PATH = os.path.join(CSRC, "libp6d.so")

P6D_OK, P6D_EINVAL, P6D_ECUDA, P6D_ENOMEM, P6D_ETOOBIG = 0, -1, -2, -3, -4

P6D_VERSION = 4

EXPORTS = (
    "p6d_version", "p6d_last_error", "p6d_device_info", "p6d_mesh_table_create",
    "p6d_mesh_table_destroy", "p6d_adds_max_points", "p6d_adds_schedule", "p6d_adds_schedule_state",
    "p6d_adds_selfcheck", "p6d_selftest_sqrt2", "p6d_add_eval", "p6d_add_eval_pruned", "p6d_mesh_table_set_pruning", "p6d_add_eval_streamed",
    "p6d_mesh_table_set_large_meshes", "p6d_add_eval_host",
    "p6d_add_forward_workspace_bytes", "p6d_add_forward", "p6d_add_backward",
    "p6d_mesh_table_set_large_mesh_loss", "p6d_add_forward_streamed", "p6d_add_backward_streamed",
    "p6d_mesh_table_set_large_mesh_pruning", "p6d_add_eval_pruned_streamed",
    "p6d_quat_to_mat", "p6d_pose_loss_workspace_bytes", "p6d_pose_loss_fwd_bwd",
    "p6d_pose_loss_pinhole_fwd_bwd", "p6d_pinhole_fwd", "p6d_pinhole_bwd", "p6d_depth_backproject",
    "p6d_depth_crop_backproject", "p6d_detection_backproject", "p6d_project_points", "p6d_synth_poses", "p6d_sweep_run",
    "p6d_adds_tf32_eval", "p6d_fp32_microbench",
)


class P6DError(RuntimeError):
    """A libp6d entry point returned a non-zero status."""


class Accumulators(C.Structure):
    _fields_ = [("hits", C.c_void_p), ("valid", C.c_void_p), ("add_sum", C.c_void_p),
                ("adds_sum", C.c_void_p)]


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a with the committed Makefile (nvcc cross-compiles
    without a GPU)."""
    r = subprocess.run(["make", "-C", CSRC, "-j4"], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout[-4000:] + r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("building libp6d.so failed")
    return SO_PATH


_lib = None


def lib() -> C.CDLL:
    """Load libp6d.so (loudly: a missing library is an error, never a fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise P6DError(
            f"{SO_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C 6d-pose-estimation_b200/csrc`. There is no CPU/PyTorch fallback.")
    L = C.CDLL(SO_PATH)
    vp, i32, i64, f32, f64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double
    L.p6d_version.restype = i32
    L.p6d_last_error.restype = C.c_char_p
    L.p6d_device_info.argtypes = [i32] + [C.POINTER(i32)] * 4 + [C.POINTER(i64)]
    L.p6d_mesh_table_create.argtypes = [vp, vp, vp, vp, vp, i32, i32, C.POINTER(vp)]
    L.p6d_mesh_table_destroy.argtypes = [vp]
    L.p6d_adds_max_points.argtypes = [i32, C.POINTER(i32)]
    L.p6d_adds_schedule_state.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    L.p6d_adds_selfcheck.argtypes = [vp, i64, C.POINTER(i64)]
    L.p6d_selftest_sqrt2.argtypes = [i32, C.POINTER(i64)]
    L.p6d_add_eval.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp, C.POINTER(Accumulators), vp]
    L.p6d_add_eval_pruned.argtypes = L.p6d_add_eval.argtypes
    L.p6d_mesh_table_set_pruning.argtypes = [vp, i32]
    L.p6d_add_eval_streamed.argtypes = L.p6d_add_eval.argtypes
    L.p6d_mesh_table_set_large_meshes.argtypes = [vp, i32]
    L.p6d_add_eval_pruned_streamed.argtypes = L.p6d_add_eval.argtypes
    L.p6d_mesh_table_set_large_mesh_pruning.argtypes = [vp, i32]
    L.p6d_add_eval_host.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                    C.POINTER(i32)]
    L.p6d_add_forward_workspace_bytes.argtypes = [vp, i64]
    L.p6d_add_forward_workspace_bytes.restype = i64
    L.p6d_add_forward.argtypes = [vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp]
    L.p6d_add_forward_streamed.argtypes = L.p6d_add_forward.argtypes
    L.p6d_mesh_table_set_large_mesh_loss.argtypes = [vp, i32]
    u64 = C.c_uint64
    L.p6d_synth_poses.argtypes = [u64, i32, i32, i64, i64, f32, f32, i32, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                  i32, vp]
    L.p6d_sweep_run.argtypes = [vp, vp, i32, vp, i32, i64, i64, i64, i64, u64, vp, f32, f32, vp, vp, vp, vp, i64,
                                vp, vp, vp, vp, vp, vp, vp, C.POINTER(i32), vp]
    L.p6d_adds_tf32_eval.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, vp, i32, vp]
    L.p6d_quat_to_mat.argtypes = [vp, i64, vp, i32, vp]
    L.p6d_pose_loss_workspace_bytes.restype = i64
    L.p6d_pose_loss_fwd_bwd.argtypes = [vp, vp, vp, vp, i64, f32, f32, i32, vp, vp, vp, vp, i32, vp]
    L.p6d_pose_loss_pinhole_fwd_bwd.argtypes = [vp, vp, vp, vp, i32, vp, vp, i64, f32, f32, i32, vp, vp, vp, vp, vp,
                                                i32, vp]
    L.p6d_pinhole_fwd.argtypes = [vp, vp, vp, i32, i64, vp, i32, vp]
    L.p6d_pinhole_bwd.argtypes = [vp, vp, vp, i32, i64, vp, i32, vp]
    L.p6d_depth_backproject.argtypes = [vp, i32, i32, vp, vp, i32, i64, f32, vp, i32, vp]
    L.p6d_fp32_microbench.argtypes = [i32, i32, i32, C.POINTER(f64), C.POINTER(f64)]
    L.p6d_depth_crop_backproject.argtypes = [vp, i32, i32, vp, i64, vp, i32, i32, vp, vp, vp, vp, i32, vp]
    L.p6d_detection_backproject.argtypes = [vp, i32, i32, vp, i64, vp, i32, vp, vp, vp, vp, i32, vp]
    L.p6d_project_points.argtypes = [vp, i32, vp, i32, vp, vp, i64, vp, i32, vp]
    L.p6d_add_backward.argtypes = [vp, vp, vp, vp, vp, vp, i64, vp, vp, f32, vp, vp, vp]
    L.p6d_add_backward_streamed.argtypes = L.p6d_add_backward.argtypes
    missing = [n for n in EXPORTS if not hasattr(L, n)]
    if missing:
        raise P6DError(f"{SO_PATH} is stale: missing symbols {missing}; rebuild it")
    if L.p6d_version() != P6D_VERSION:
        raise P6DError(f"{SO_PATH} implements ABI version {L.p6d_version()}, this package needs {P6D_VERSION}; rebuild it")
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != P6D_OK:
        msg = lib().p6d_last_error().decode("utf-8", "replace")
        raise P6DError(f"libp6d error {rc}: {msg}")


def ptr(t) -> int | None:
    """Raw pointer of a torch tensor / numpy array (None -> NULL)."""
    if t is None:
        return None
    if isinstance(t, torch.Tensor):
        return t.data_ptr()
    return t.ctypes.data


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr(device: torch.device) -> int:
    """cudaStream_t of torch's current stream on `device` (the raw accessor costs ~0.3 us, building a
    torch.cuda.Stream object ~2 us -- it matters at the reference's batch sizes)."""
    if _raw_stream is not None and device.index is not None:
        return _raw_stream(device.index)
    return torch.cuda.current_stream(device).cuda_stream


def as_cuda_f32(t: torch.Tensor, device: torch.device, shape_tail) -> torch.Tensor:
    """Contiguous float32 view of `t` on `device` with trailing shape `shape_tail`.
    Host tensors are copied to the device (compute never runs on the CPU)."""
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(np.asarray(t))
    elif (t.dtype is torch.float32 and t.device == device and t.dim() == 1 + len(shape_tail)
          and tuple(t.shape[1:]) == tuple(shape_tail) and t.is_contiguous() and t.data_ptr() % 16 == 0):
        return t.detach() if t.requires_grad else t      # already what the kernels read: no torch op at all
    t = t.detach()
    if t.device != device:
        t = t.to(device, non_blocking=True)
    if t.dtype != torch.float32:
        t = t.float()
    t = t.reshape(-1, *shape_tail) if shape_tail else t.reshape(-1)
    t = t.contiguous()
    if t.data_ptr() % 16:          # a view with a storage offset: the kernels use float4 / float2 loads
        t = t.clone()
    return t


def require_cuda(device) -> torch.device:
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError(
            "6d-pose-estimation_b200 runs on CUDA (sm_100a) only; there is no CPU fallback. "
            f"Got device={device}.")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


class MeshTable:
    """Device-resident mesh table built from ``ADDLoss.points`` / ``.diameters``."""

    def __init__(self, points: dict, diameters: dict, symmetric_ids, device: torch.device):
        self.device = require_cuda(device)
        ids = sorted(int(k) for k in points)
        if any(i < 0 for i in ids):
            raise ValueError("object ids must be >= 0")
        self.n_slots = (ids[-1] + 1) if ids else 1
        offsets = np.zeros(self.n_slots, np.int32)
        counts = np.zeros(self.n_slots, np.int32)
        dia = np.full(self.n_slots, 0.1, np.float64)  # self.diameters.get(oid, 0.1)
        sym = np.zeros(self.n_slots, np.uint8)
        chunks, off = [], 0
        for oid in ids:
            p = points[oid]
            m = (p.detach().to("cpu", torch.float32).numpy() if isinstance(p, torch.Tensor)
                 else np.asarray(p, np.float32)).reshape(-1, 3)
            offsets[oid], counts[oid] = off, m.shape[0]
            off += m.shape[0]
            chunks.append(np.ascontiguousarray(m))
            if oid in diameters:
                dia[oid] = float(diameters[oid])
            sym[oid] = 1 if oid in symmetric_ids else 0
        xyz = np.concatenate(chunks, 0) if chunks else np.zeros((1, 3), np.float32)
        self.counts = counts
        self.symmetric = sym
        self.thresholds = 0.1 * dia
        self.max_count = int(counts.max()) if ids else 0
        h = C.c_void_p()
        check(lib().p6d_mesh_table_create(ptr(xyz), ptr(offsets), ptr(counts), ptr(dia), ptr(sym),
                                          self.n_slots, self.device.index, C.byref(h)))
        self.handle = h

    def close(self):
        if getattr(self, "handle", None):
            lib().p6d_mesh_table_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_pruning(self, enable=True):
        """Opt in to (or out of) the exact-pruned ADD-S kernel for this table: same bits as the all-pairs
        kernel, taken where it pays (largest mesh >= 128 points); see include/p6d.h."""
        check(lib().p6d_mesh_table_set_pruning(self.handle, 1 if enable else 0))
        return self

    def set_large_meshes(self, enable=True):
        """Opt in to (or out of) the streamed ADD / ADD-S kernel for this table: same bits as the resident
        kernels, taken only when the largest mesh is beyond their shared-memory limit (up to 32,768 points);
        see include/p6d.h."""
        check(lib().p6d_mesh_table_set_large_meshes(self.handle, 1 if enable else 0))
        return self

    def set_large_mesh_loss(self, enable=True):
        """Opt in to (or out of) the streamed loss-form and gradient kernels for this table: the same loss bits
        as the resident loss form, taken by forward_loss / add_backward only when the largest mesh is beyond the
        resident kernels' shared-memory limit (up to 32,768 points); independent of set_large_meshes; see
        include/p6d.h."""
        check(lib().p6d_mesh_table_set_large_mesh_loss(self.handle, 1 if enable else 0))
        return self

    def set_large_mesh_pruning(self, enable=True):
        """Opt in to (or out of) the streamed exact-pruned ADD-S kernel for this table: same bits as the other
        evaluation kernels, taken for ADD-S evaluation only when the largest mesh is beyond the pruned kernel's
        shared-memory limit (up to 32,768 points); independent of the other switches; refused for a table
        without a block structure; see include/p6d.h."""
        check(lib().p6d_mesh_table_set_large_mesh_pruning(self.handle, 1 if enable else 0))
        return self

    # -- device-buffer evaluation ---------------------------------------------------
    def evaluate_packed(self, pq, pt, gq, gt, obj, want_adds=True, order=None, acc=None, prune=False, streamed=False,
                        prune_streamed=False):
        """Launch the evaluation kernels on the current stream and return the ONE buffer behind the
        per-pose outputs: add f32 [B] | adds f32 [B] | hit u8 [B] | valid u8 [B] | borderline u8 [B]
        (adds is left unwritten when want_adds is False).  All inputs must already be contiguous CUDA
        tensors on this table's device.  No views are created: at the reference's batch sizes every
        torch op is 2-3 us of a ~100 us call.  prune / streamed: always the exact-pruned (ADD-S only) or the
        streamed kernel (p6d_add_eval_pruned / p6d_add_eval_streamed) instead of the table's choice.
        prune_streamed: always the streamed exact-pruned kernel (p6d_add_eval_pruned_streamed, ADD-S only); it
        takes precedence over prune / streamed."""
        B = obj.shape[0]
        out = torch.empty(11 * B + 16, dtype=torch.uint8, device=self.device)
        base = out.data_ptr()
        acc_struct = None
        if acc is not None:
            acc_struct = Accumulators(*(ptr(a) for a in acc))
        if prune_streamed and want_adds:
            entry = lib().p6d_add_eval_pruned_streamed
        elif streamed:
            entry = lib().p6d_add_eval_streamed
        else:
            entry = lib().p6d_add_eval_pruned if (prune and want_adds) else lib().p6d_add_eval
        check(entry(self.handle, pq.data_ptr(), pt.data_ptr(), gq.data_ptr(), gt.data_ptr(), obj.data_ptr(),
                    ptr(order), B, base, (base + 4 * B) if want_adds else None, base + 8 * B, base + 9 * B,
                    base + 10 * B, C.byref(acc_struct) if acc_struct is not None else None,
                    stream_ptr(self.device)))
        return out

    def evaluate(self, pq, pt, gq, gt, obj, want_adds=True, order=None, acc=None, prune=False, streamed=False,
                 prune_streamed=False):
        """evaluate_packed + views: returns (add, adds, hit, valid, packed) device tensors (adds is
        None when want_adds is False)."""
        B = obj.shape[0]
        out = self.evaluate_packed(pq, pt, gq, gt, obj, want_adds, order, acc, prune, streamed, prune_streamed)
        add = out[: 4 * B].view(torch.float32)
        adds = out[4 * B: 8 * B].view(torch.float32)
        return add, (adds if want_adds else None), out[8 * B: 9 * B], out[9 * B: 10 * B], out

    def packed_to_host(self, packed):
        """The packed per-pose buffer as a NumPy array: one async copy into a cached pinned buffer and one
        stream synchronisation (the only synchronisation of an eval_metrics call).  The array is a view of
        the cached buffer: consume it before the next call."""
        n = packed.numel()
        buf = getattr(self, "_pinned", None)
        if buf is None or buf.numel() < n:
            buf = torch.empty(max(n, 4096), dtype=torch.uint8).pin_memory()
            self._pinned = buf
        host = buf[:n]
        host.copy_(packed, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return host.numpy()

    def forward_loss(self, pq, pt, gq, gt, obj, streamed=False):
        """ADDLoss.forward value: one launch, no host synchronisation.  Returns (loss [1] f32,
        count [1] i32) device tensors.  streamed: always the streamed loss form (p6d_add_forward_streamed)
        instead of the table's choice."""
        B = obj.shape[0]
        dev = self.device
        L = lib()
        ws = torch.empty(int(L.p6d_add_forward_workspace_bytes(self.handle, B)) + 16, dtype=torch.uint8, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        count = torch.empty(1, dtype=torch.int32, device=dev)
        entry = L.p6d_add_forward_streamed if streamed else L.p6d_add_forward
        check(entry(self.handle, ptr(pq), ptr(pt), ptr(gq), ptr(gt), ptr(obj), B, ptr(loss), ptr(count), ptr(ws),
                    stream_ptr(dev)))
        return loss, count

    def schedule_state(self) -> dict:
        """{'built_relaid': 0/1, 'runtime_state': 0 unchecked / 1 verified / 2 rejected} for this table's
        mesh-size class (see include/p6d.h, p6d_adds_schedule_state)."""
        a, b = C.c_int(0), C.c_int(0)
        check(lib().p6d_adds_schedule_state(self.handle, C.byref(a), C.byref(b)))
        return {"built_relaid": a.value, "runtime_state": b.value}

    def selfcheck(self, n_poses: int = 592) -> int:
        """Re-laid vs ptxas-scheduled ADD-S kernel on n_poses seeded poses: differing output bytes."""
        bad = C.c_int64(0)
        check(lib().p6d_adds_selfcheck(self.handle, int(n_poses), C.byref(bad)))
        return bad.value

    # -- host-buffer evaluation (end-to-end path) -------------------------------------
    def evaluate_host(self, pq, pt, gq, gt, obj, want_adds=True, per_pose=True):
        """numpy / CPU-tensor inputs -> numpy outputs through p6d_add_eval_host."""
        def arr(x, dt, tail):
            a = x.numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
            return np.ascontiguousarray(a, dtype=dt).reshape((-1,) + tail)
        pq, gq = arr(pq, np.float32, (4,)), arr(gq, np.float32, (4,))
        pt, gt = arr(pt, np.float32, (3,)), arr(gt, np.float32, (3,))
        obj = arr(obj, np.int64, ())
        B = obj.shape[0]
        add = np.empty(B, np.float32) if per_pose else None
        adds = np.empty(B, np.float32) if (per_pose and want_adds) else None
        hit = np.empty(B, np.uint8) if per_pose else None
        valid = np.empty(B, np.uint8) if per_pose else None
        border = np.empty(B, np.uint8) if per_pose else None
        ns = self.n_slots
        a_hits, a_valid = np.zeros(ns, np.int64), np.zeros(ns, np.int64)
        a_add, a_adds = np.zeros(ns, np.float64), np.zeros(ns, np.float64)
        launches = C.c_int(0)
        check(lib().p6d_add_eval_host(self.handle, ptr(pq), ptr(pt), ptr(gq), ptr(gt), ptr(obj), B,
                                      1 if want_adds else 0, ptr(add), ptr(adds), ptr(hit), ptr(valid), ptr(border),
                                      ptr(a_hits), ptr(a_valid), ptr(a_add), ptr(a_adds), C.byref(launches)))
        return {"add": add, "adds": adds, "hit": hit, "valid": valid, "borderline": border, "obj_hits": a_hits,
                "obj_valid": a_valid, "obj_add_sum": a_add, "obj_adds_sum": a_adds,
                "gpu_launches": launches.value,
                "h2d_bytes": B * (16 + 16 + 12 + 12 + 8),
                "d2h_bytes": (B * (4 + (4 if want_adds else 0) + 3) if per_pose else 0) + 32 * ns}


def add_backward(saved, grad_out, streamed=False):
    """Gradients of ADDLoss.forward w.r.t. (pred_r, pred_t) through p6d_add_backward; the number of
    valid samples stays on the device (written by p6d_add_forward).  streamed: always the streamed
    backward (p6d_add_backward_streamed) instead of the table's choice."""
    pq, pt, gq, gt, obj, count, table, dev = saved
    go = grad_out.detach().to(dev, torch.float32).reshape(1).contiguous()
    gq_out = torch.empty_like(pq)
    gt_out = torch.empty_like(pt)
    entry = lib().p6d_add_backward_streamed if streamed else lib().p6d_add_backward
    check(entry(table.handle, ptr(pq), ptr(pt), ptr(gq), ptr(gt), ptr(obj), obj.shape[0], ptr(go), ptr(count), 0.0,
                ptr(gq_out), ptr(gt_out), stream_ptr(dev)))
    return gq_out, gt_out


def selftest_sqrt2(device=0) -> int:
    bad = C.c_int64(0)
    check(lib().p6d_selftest_sqrt2(int(device), C.byref(bad)))
    return bad.value


def device_info(device=0) -> dict:
    sm, maj, mnr, clk = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    smem = C.c_int64()
    check(lib().p6d_device_info(int(device), C.byref(sm), C.byref(maj), C.byref(mnr), C.byref(clk), C.byref(smem)))
    return {"sm_count": sm.value, "cc": (maj.value, mnr.value), "sm_clock_khz": clk.value,
            "smem_optin": smem.value}


def fp32_microbench(kind: int, device=0, iters=2000):
    t, ms = C.c_double(), C.c_double()
    check(lib().p6d_fp32_microbench(int(kind), int(device), int(iters), C.byref(t), C.byref(ms)))
    return t.value, ms.value


sys.modules.setdefault("p6d_b200_core", sys.modules[__name__])
