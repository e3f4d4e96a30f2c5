"""Gradients against autograd of the reference's op sequence (oracle/torch_eager.py: add_loss_grad,
pose_loss_grad, geometric_loss_grad), not against the C oracle's hand-derived backward, which makes the
same discrete decisions as the kernels and so shares their derivation mistakes.

Bar, per row: |g - ref| <= 1e-5 * max|ref row| against both reference forms -- float32 autograd (the
reference's rounding and decisions) and float64 autograd that takes its decisions from the float32 run.
Where the float32 reference row is exactly zero the kernel's row is exactly zero; where it is NaN the
kernel's is NaN in the same places.

CPU part: the C oracle against the same references.  GPU part (-m gpu): ADDLoss, PoseLoss (small,
streamed and grid-stride kernels, exact and FAST rows), the fused geometric step and the pinhole backward.
"""
import tempfile

import numpy as np
import pytest
import torch

from conftest import same_bits
from oracle import torch_eager as E

F32 = np.float32


def check_rows(got, ref32, ref64, what, scale=None):
    """The bar above.  Where the two references disagree by more than the bar, the kernel may be as far
    from either as they are from each other: the float32 forward rounds each cloud point and quaternion
    component, and on ill-conditioned rows (nearest-point distances of a few mm on a 2,048-point mesh, a
    projection or a sum whose terms cancel) that moves the reference's gradient by ~1e-5 of the row as much
    as the kernels'.  scale (per row) replaces max|ref row| for a row that is one such sum."""
    got = np.asarray(got, np.float64).reshape(ref32.shape[0], -1)
    r32 = np.asarray(ref32, np.float64).reshape(got.shape)
    r64 = np.asarray(ref64, np.float64).reshape(got.shape)
    nan = np.isnan(r32)
    assert np.array_equal(np.isnan(got), nan), f"{what}: NaN in other places, rows {np.nonzero((np.isnan(got) != nan).any(1))[0][:8]}"
    zero = (r32 == 0).all(1)
    assert not got[zero].any(), f"{what}: rows {np.nonzero(zero & (got != 0).any(1))[0][:8]} are not exactly 0"
    fin = ~nan.any(1)
    slack = np.abs(r32 - r64).max(1)
    for name, r in (("float32", r32), ("float64", r64)):
        s = np.abs(r).max(1) if scale is None else np.asarray(scale, np.float64).reshape(-1)
        err = np.abs(got - r).max(1)
        bad = np.nonzero(fin & (err > 1e-5 * s + slack))[0]
        assert bad.size == 0, f"{what} vs {name} autograd: rows {bad[:8]}, rel err {(err[bad] / np.maximum(s[bad], 1e-300))[:4]}"


def refs_add(pts, pq, pt, gq, gt, obj, grad_out=1.0):
    q32, t32, dec = E.add_loss_grad(pts, pq, pt, gq, gt, obj, grad_out)
    q64, t64, _ = E.add_loss_grad(pts, pq, pt, gq, gt, obj, grad_out, torch.float64, dec)
    return q32, t32, q64, t64


def refs_pose(pq, pt, gq, gt, wr, wt, mode, grad_out=1.0):
    _, q32, t32, dec = E.pose_loss_grad(pq, pt, gq, gt, wr, wt, mode, grad_out)
    _, q64, t64, _ = E.pose_loss_grad(pq, pt, gq, gt, wr, wt, mode, grad_out, torch.float64, dec)
    return q32, t32, q64, t64


# ------------------------------------------------------------------ fixtures
def f32_bits(*words):
    return np.array(words, np.uint32).view(F32)


def tie_fixture():
    """Two symmetric samples whose nearest-point choice is a tie.
    Object 9: pred point 0 lands at (0.01, 0, 0); gt points 1 and 2 have different float32 squared
    distances from it but the same correctly rounded root -- torch.norm(...).min takes point 1, a min over
    the squares takes point 2.  Object 10: pred point 2 lands at the origin, exactly between gt points 0 and
    1 (equal squares): the first index wins."""
    r = np.random.RandomState(1)
    fill = lambda n: (r.standard_normal((n, 3)) * 0.05 + 0.3).astype(F32)
    m9 = np.concatenate([np.zeros((1, 3), F32), f32_bits(0x3C541A59, 0xB9F609CF, 0xB9A7C982)[None],
                         f32_bits(0x3C31229A, 0x39954080, 0x3B3C5B73)[None], fill(60)])
    m10 = np.concatenate([np.array([[0.01, 0, 0], [-0.01, 0, 0], [0, 0, 0.1]], F32), fill(60)])
    pq = np.tile(np.array([0, 0, 0, 1], F32), (2, 1))
    pt = np.array([[f32_bits(0x3C23D70A)[0], 0, 0], [0, 0, -0.1]], F32)
    return {9: m9, 10: m10}, pq, pt, pq.copy(), np.zeros((2, 3), F32), np.array([9, 10], np.int64)


def rotations(B, seed, lo=0.3, hi=2.8):
    """gt unit quaternions, and predictions rotated away from them by an angle in [lo, hi] about a random
    axis, scaled by [0.5, 2] and with a random sign: small angles are avoided because there the gradient's
    direction is set by rounding (a 1-ulp change of u moves it by ~1e-7 / |u - v|)."""
    r = np.random.RandomState(seed)
    gq = r.standard_normal((B, 4)); gq /= np.linalg.norm(gq, axis=1, keepdims=True)
    ax = r.standard_normal((B, 3)); ax /= np.linalg.norm(ax, axis=1, keepdims=True)
    ang = r.uniform(lo, hi, B)
    dq = np.concatenate([ax * np.sin(ang / 2)[:, None], np.cos(ang / 2)[:, None]], 1)
    x1, y1, z1, w1 = dq.T
    x2, y2, z2, w2 = gq.T
    pq = np.stack([w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2, w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2,
                   w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2, w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2], 1)
    pq *= (r.uniform(0.5, 2.0, B) * np.where(r.rand(B) < 0.5, -1, 1))[:, None]
    return pq.astype(F32), gq.astype(F32)


EDGE_KINDS = ("identical", "antipodal", "antipodal_x3", "zero", "tiny", "dot0", "l1_tie", "t_equal")


def plant_edge_row(kind, pq, pt, gq, gt, i):
    if kind == "identical":
        pq[i] = gq[i]
    elif kind == "antipodal":
        pq[i] = -gq[i]
    elif kind == "antipodal_x3":
        # for this q, -3q normalises to exactly -q in float32 and the distance is exactly 0 (for most q
        # it is rounding noise, a direction no reference pins); a FAST row must see the 0 too
        gq[i] = (0.5, -0.5, 0.5, 0.5)
        pq[i] = F32(-3.0) * gq[i]
    elif kind == "zero":
        pq[i] = 0
    elif kind == "tiny":                          # |q| < 1e-12: clamped, no gradient through the norm
        pq[i] = F32(1e-13) * gq[i]
    elif kind == "dot0":                          # dot == 0 exactly; also an L1 tie
        pq[i], gq[i] = (1, 0, 0, 0), (0, 1, 0, 0)
    elif kind == "l1_tie":                        # |u - v|_1 == |u + v|_1 exactly, dot == 0
        pq[i], gq[i] = (0.6, 0.8, 0, 0), (0.8, -0.6, 0, 0)
    elif kind == "t_equal":                       # sign(0) of the translation term
        pt[i] = gt[i]


def pose_inputs(B, seed):
    """Random rows with every edge kind planted at rows 0, 255, 256 (first row of the second tile) and at
    the end of the batch (the ragged tail of the streamed kernel), clipped to the batch."""
    pq, gq = rotations(B, seed)
    r = np.random.RandomState(seed + 1)
    gt = r.uniform(-0.5, 0.5, (B, 3)).astype(F32)
    pt = (gt + r.standard_normal((B, 3)) * 0.02).astype(F32)
    for start in sorted({0, 255, 256, max(B - len(EDGE_KINDS), 0)}):
        for k, kind in enumerate(EDGE_KINDS):
            if start + k < B:
                plant_edge_row(kind, pq, pt, gq, gt, start + k)
    return pq, pt, gq, gt


# ------------------------------------------------------------------ CPU: the C oracle
def test_oracle_add_backward_breaks_root_ties_like_torch_min(oracle):
    pts, pq, pt, gq, gt, obj = tie_fixture()
    q32, t32, q64, t64 = refs_add(pts, pq, pt, gq, gt, obj)
    oq, ot = oracle.add_backward(oracle.MeshTable(pts, {9: 0.1, 10: 0.1}), pq, pt, gq, gt, obj)
    check_rows(ot, t32, t64, "grad_t")
    check_rows(oq, q32, q64, "grad_q")


def test_oracle_add_backward_matches_autograd_on_small_and_degenerate_meshes(oracle, W):
    """Meshes of 1-45 points (the loss form's matmul rounds unfused up to 44 points), symmetric and
    asymmetric ids, unknown ids, pred == gt, a zero and a non-unit pred quaternion, upstream gradient 2.5."""
    pts = {3: W.sphere_mesh(1, 0.1, 1), 9: W.sphere_mesh(11, 0.12, 2), 10: W.box_mesh(44, (0.04, 0.1, 0.05), 3),
           5: W.box_mesh(45, (0.1, 0.05, 0.05), 4), 1: W.sphere_mesh(2, 0.1, 5), 10 + 2: W.sphere_mesh(10, 0.1, 6)}
    B = 16
    pq, pt, gq, gt = W.random_poses(B, 7, rot_sigma=0.3, trans_sigma=0.01)
    obj = np.array([3, 9, 10, 5, 1, 12, -1, 2, 99, 9, 10, 3, 5, 9, 10, 12], np.int64)
    pq[9], pt[9] = gq[9], gt[9]                  # pred == gt on a symmetric object: all distances 0
    pq[10] = 0                                   # zero quaternion: R = I
    pq[11] *= 3                                  # non-unit
    q32, t32, q64, t64 = refs_add(pts, pq, pt, gq, gt, obj, 2.5)
    oq, ot = oracle.add_backward(oracle.MeshTable(pts), pq, pt, gq, gt, obj, 2.5)
    check_rows(ot, t32, t64, "grad_t")
    check_rows(oq, q32, q64, "grad_q")


def test_oracle_pose_loss_edge_rows_match_autograd(oracle):
    for mode in ("geodesic", "l1"):
        for wr, wt in ((1.0, 10.0), (0.5, 2.0)):
            pq, pt, gq, gt = pose_inputs(40, 11)
            q32, t32, q64, t64 = refs_pose(pq, pt, gq, gt, wr, wt, mode)
            o = oracle.pose_loss(pq, pt, gq, gt, wr, wt, mode)
            check_rows(o["grad_q"], q32, q64, f"{mode} grad_q")
            assert same_bits(o["grad_t"], t32), mode


def test_oracle_translation_gradient_bits_when_3b_exceeds_2_pow_24(oracle):
    """ATen divides float32(weight) by float32(3B); 3B = 18,000,003 is not a float32."""
    B = 6_000_001
    r = np.random.RandomState(5)
    pt = r.standard_normal((B, 3)).astype(F32)
    gt = r.standard_normal((B, 3)).astype(F32)
    pt[::7] = gt[::7]
    b = torch.from_numpy(pt).requires_grad_(True)
    (2.0 * torch.nn.functional.l1_loss(b, torch.from_numpy(gt))).backward()
    q = np.tile(np.array([0, 0, 0, 1], F32), (B, 1))
    o = oracle.pose_loss(q, pt, q, gt, 1.0, 2.0, "l1")
    assert same_bits(o["grad_t"], b.grad.numpy())


# ------------------------------------------------------------------ GPU
def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def make_crit(pkg, pts, dev):
    crit = pkg.ADDLoss(tempfile.mkdtemp(), dev)
    for k, v in pts.items():
        crit.points[k] = T(v, dev)
    crit.diameters.update({k: 0.1 for k in pts})
    return crit


def run_add(pkg, dev, pts, pq, pt, gq, gt, obj, grad_out=1.0):
    crit = make_crit(pkg, pts, dev)
    x, y = T(pq, dev).requires_grad_(True), T(pt, dev).requires_grad_(True)
    loss = crit(x, y, T(gq, dev), T(gt, dev), T(obj, dev))
    loss.backward(torch.tensor(grad_out, device=dev))
    return x.grad.cpu().numpy(), y.grad.cpu().numpy()


@pytest.mark.gpu
def test_add_backward_breaks_root_ties_like_torch_min(pkg, cuda_dev):
    pts, pq, pt, gq, gt, obj = tie_fixture()
    q32, t32, q64, t64 = refs_add(pts, pq, pt, gq, gt, obj)
    gq_, gt_ = run_add(pkg, cuda_dev, pts, pq, pt, gq, gt, obj)
    check_rows(gt_, t32, t64, "grad_t")
    check_rows(gq_, q32, q64, "grad_q")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 10, 11, 44, 45, 257, 500, 2048, 3000])
def test_add_backward_mesh_sizes(pkg, cuda_dev, W, n):
    """Both matmul roundings of the loss form (n <= 44 unfused), more points than threads (n > 256),
    symmetric and asymmetric ids mixed and repeated, unknown ids; B = 24 and B = 1."""
    pts = {3: W.sphere_mesh(n, 0.15, n), 9: W.box_mesh(n, (0.05, 0.12, 0.06), n + 1),
           10: W.sphere_mesh(n, 0.1, n + 2)}
    B = 24
    pq, pt, gq, gt = W.random_poses(B, n, rot_sigma=0.3, trans_sigma=0.01)
    obj = np.array([3, 9, 10, -1, 9, 3, 2, 10, 99] + [3, 9, 10] * 5, np.int64)
    for sl, go in ((slice(0, B), 2.5), (slice(1, 2), 1.0)):
        a = [x[sl] for x in (pq, pt, gq, gt, obj)]
        q32, t32, q64, t64 = refs_add(pts, *a, go)
        gq_, gt_ = run_add(pkg, cuda_dev, pts, *a, go)
        check_rows(gt_, t32, t64, f"n={n} B={len(a[4])} grad_t")
        check_rows(gq_, q32, q64, f"n={n} B={len(a[4])} grad_q")


@pytest.mark.gpu
def test_add_backward_planted_rows_and_grid_stride(pkg, cuda_dev, W):
    """B = 600 > 4 x 148 CTAs: the kernel loops over poses.  Planted: pred == gt; pt == gt with the
    rotation error about the z axis through mesh point 0 (its distance is exactly 0, the others' are not);
    duplicated gt vertices; the root-tie fixture; zero and non-unit quaternions; 50 m translations; one NaN
    sample (the other samples stay finite); an all-unknown batch."""
    m = W.sphere_mesh(500, 0.16, 8)
    m[0] = (0, 0, 0.05)
    sph = W.sphere_mesh(437, 0.16, 9)
    dup = sph.copy(); dup[1::2] = dup[0:-1:2]
    tie_pts, tq, tt, tgq, tgt, _ = tie_fixture()
    pts = {3: m, 9: np.concatenate([tie_pts[9], dup]), 10: np.concatenate([tie_pts[10], sph])}
    B = 600
    pq, pt, gq, gt = W.random_poses(B, 9, rot_sigma=0.3, trans_sigma=0.01)
    obj = np.array([3, 9, 10, 3, 9, 10, 2], np.int64)[np.random.RandomState(9).randint(0, 7, B)]
    pq[0], pt[0], obj[0] = gq[0], gt[0], 9
    pq[1], pt[1], obj[1] = gq[1], gt[1], 3
    for i in (2, 3):
        gq[i], gt[i], obj[i] = (0, 0, 0, 1), (0.1, 0.2, 0.7), 3
        pq[i], pt[i] = (0, 0, np.sin(0.1 * i), np.cos(0.1 * i)), gt[i]
    pq[4], pt[4], gq[4], gt[4], obj[4] = tq[0], tt[0], tgq[0], tgt[0], 9
    pq[5], pt[5], gq[5], gt[5], obj[5] = tq[1], tt[1], tgq[1], tgt[1], 10
    pq[6], obj[6] = 0, 10
    pq[7], obj[7] = 3 * pq[7], 9
    pt[8], obj[8] = gt[8] + 50, 3
    pt[9], obj[9] = gt[9] + (0, 0, 50), 10
    pt[B - 1], obj[B - 1] = (np.nan, 0, 0), 9
    q32, t32, q64, t64 = refs_add(pts, pq, pt, gq, gt, obj, 2.5)
    assert np.isnan(t32[B - 1]).all() and np.isfinite(t32[:B - 1]).all()
    assert (q32[2] != 0).any() and not q32[0].any()
    gq_, gt_ = run_add(pkg, cuda_dev, pts, pq, pt, gq, gt, obj, 2.5)
    check_rows(gt_, t32, t64, "grad_t")
    check_rows(gq_, q32, q64, "grad_q")
    gq_, gt_ = run_add(pkg, cuda_dev, pts, pq[:5], pt[:5], gq[:5], gt[:5], np.full(5, 7, np.int64))
    assert not gq_.any() and not gt_.any()


POSE_BATCHES = [1, 5, 32, 2048, 2049, 2303, 30_077, 6_000_001]


@pytest.mark.gpu
@pytest.mark.parametrize("B", POSE_BATCHES)
def test_pose_loss_backward_edge_rows(pkg, cuda_dev, B):
    """Single-CTA kernel (B <= 2048), streamed kernel with a ragged tail (2049, 2303, 30,077, 6,000,001;
    FAST rows in geodesic mode), both modes and both weight pairs; upstream gradient 1, so the
    translation gradient is compared bit for bit."""
    pq, pt, gq, gt = pose_inputs(B, B % 1000)
    for mode in ("geodesic", "l1"):
        for wr, wt in ((1.0, 10.0), (0.5, 2.0)):
            if B == 6_000_001 and (wr, wt) == (1.0, 10.0) and mode == "l1":
                continue        # the largest batch costs ~10 s of CPU autograd per reference pair
            q32, t32, q64, t64 = refs_pose(pq, pt, gq, gt, wr, wt, mode)
            x, y = T(pq, cuda_dev).requires_grad_(True), T(pt, cuda_dev).requires_grad_(True)
            pkg.PoseLoss(wr, wt, mode)(x, y, T(gq, cuda_dev), T(gt, cuda_dev)).backward()
            check_rows(x.grad.cpu().numpy(), q32, q64, f"{mode} ({wr}, {wt}) grad_q")
            assert same_bits(y.grad.cpu().numpy(), t32), f"{mode} ({wr}, {wt}) grad_t"


@pytest.mark.gpu
def test_pose_loss_backward_grid_stride_kernel(pkg, cuda_dev):
    """[B,3] rows that are only 4-byte aligned go through the grid-stride kernel (raw entry point)."""
    core, B = pkg.core, 30_077
    pq, pt, gq, gt = pose_inputs(B, 4)
    ws = torch.zeros(64, dtype=torch.uint8, device=cuda_dev)
    dpt = torch.zeros(3 * B + 1, device=cuda_dev)[1:].copy_(T(pt, cuda_dev).reshape(-1))
    dgt = torch.zeros(3 * B + 1, device=cuda_dev)[1:].copy_(T(gt, cuda_dev).reshape(-1))
    dq, dgq = T(pq, cuda_dev), T(gq, cuda_dev)
    for mode in ("geodesic", "l1"):
        q32, t32, q64, t64 = refs_pose(pq, pt, gq, gt, 1.0, 10.0, mode)
        out = torch.empty(3, device=cuda_dev)
        g1, g2 = torch.empty(B, 4, device=cuda_dev), torch.empty(3 * B, device=cuda_dev)
        core.check(core.lib().p6d_pose_loss_fwd_bwd(dq.data_ptr(), dpt.data_ptr(), dgq.data_ptr(), dgt.data_ptr(), B,
                                                    1.0, 10.0, 0 if mode == "geodesic" else 1, out.data_ptr(),
                                                    g1.data_ptr(), g2.data_ptr(), ws.data_ptr(), cuda_dev.index,
                                                    core.stream_ptr(cuda_dev)))
        torch.cuda.synchronize()
        check_rows(g1.cpu().numpy(), q32, q64, f"{mode} grad_q")
        assert same_bits(g2.cpu().numpy().reshape(B, 3), t32), mode


@pytest.mark.gpu
def test_pose_loss_backward_near_orthogonal_pairs(pkg, cuda_dev):
    """~1e5 rows with |dot| <= 1e-7 of both signs at B = 262,144 (FAST rows): the flip of q2 must be
    decided as the float32 reference decides it, or the row's gradient changes sign."""
    B = 262_144
    r = np.random.RandomState(12)
    gq = r.standard_normal((B, 4)); gq /= np.linalg.norm(gq, axis=1, keepdims=True)
    pq = r.standard_normal((B, 4))
    near = r.rand(B) < 0.4
    pq[near] -= (pq[near] * gq[near]).sum(1, keepdims=True) * gq[near]     # orthogonal in float64 ...
    pq[near] += gq[near] * r.uniform(-1e-7, 1e-7, (near.sum(), 1))          # ... then |dot| <= 1e-7
    pq, gq = pq.astype(F32), gq.astype(F32)
    pt = r.standard_normal((B, 3)).astype(F32); gt = r.standard_normal((B, 3)).astype(F32)
    q32, t32, q64, t64 = refs_pose(pq, pt, gq, gt, 1.0, 10.0, "geodesic")
    x = T(pq, cuda_dev).requires_grad_(True)
    pkg.PoseLoss(1.0, 10.0)(x, T(pt, cuda_dev), T(gq, cuda_dev), T(gt, cuda_dev)).backward()
    check_rows(x.grad.cpu().numpy(), q32, q64, "grad_q")


def grad_z_scale(g, uv, K):
    """Sum of |terms| of dL/dz = g_x (u - cx) / fx + g_y (v - cy) / fy + g_z: the bar for a sum whose terms
    can cancel (float32 rounds each term and the sums in autograd's order, the kernel in its own)."""
    K = np.broadcast_to(np.asarray(K, np.float64).reshape(-1, 3, 3), (len(uv), 3, 3))
    g = np.asarray(g, np.float64)
    return (np.abs(g[:, 0] * (uv[:, 0] - K[:, 0, 2]) / K[:, 0, 0]) + np.abs(g[:, 1] * (uv[:, 1] - K[:, 1, 2]) / K[:, 1, 1])
            + np.abs(g[:, 2]))


def geometric_inputs(W, B, seed):
    c = W.config3(B, seed)
    return c["rot_raw"], c["z_pred"], c["bbox_center"], c["K"], c["gt_rot"], c["gt_trans"]


@pytest.mark.gpu
@pytest.mark.parametrize("B", [32, 5000])
def test_fused_geometric_step_against_autograd(pkg, cuda_dev, W, B):
    rot, z, uv, K, gq, gt = geometric_inputs(W, B, 13)
    for mode in ("geodesic", "l1"):
        for Kin in (K, K[0]):
            _, q32, z32, dec = E.geometric_loss_grad(rot, z, uv, Kin, gq, gt, 1.0, 10.0, mode, 2.5)
            _, q64, z64, _ = E.geometric_loss_grad(rot, z, uv, Kin, gq, gt, 1.0, 10.0, mode, 2.5, torch.float64, dec)
            r, zz = T(rot, cuda_dev).requires_grad_(True), T(z, cuda_dev).requires_grad_(True)
            loss, _ = pkg.PoseLoss(1.0, 10.0, mode).forward_geometric(r, zz, T(uv, cuda_dev), T(Kin, cuda_dev),
                                                                     T(gq, cuda_dev), T(gt, cuda_dev))
            loss.backward(torch.tensor(2.5, device=cuda_dev))
            check_rows(r.grad.cpu().numpy(), q32, q64, f"{mode} K{Kin.ndim} grad_q")
            sc = grad_z_scale(np.full((B, 3), 2.5 * 10.0 / (3 * B)), uv, Kin)
            check_rows(zz.grad.cpu().numpy(), z32, z64, f"{mode} K{Kin.ndim} grad_z", scale=sc)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 4097, 65_539])
def test_pinhole_backward_against_autograd(pkg, cuda_dev, B):
    r = np.random.RandomState(B)
    z = (r.rand(B, 1) * 1.2 + 0.3).astype(F32)
    uv = (r.rand(B, 2) * np.array([640, 480])).astype(F32)
    go = r.standard_normal((B, 3)).astype(F32)
    K = pkg.DEFAULT_K.astype(F32)
    for Kin in (K, np.broadcast_to(K, (B, 3, 3)).copy()):
        refs = []
        for dt in (torch.float32, torch.float64):
            zz = torch.from_numpy(z).to(dt).requires_grad_(True)
            E.pinhole_translation(zz, torch.from_numpy(uv).to(dt), torch.from_numpy(Kin).to(dt)).backward(
                torch.from_numpy(go).to(dt))
            refs.append(zz.grad.numpy())
        zg = T(z, cuda_dev).requires_grad_(True)
        pkg.pinhole_translation(zg, T(uv, cuda_dev), T(Kin, cuda_dev)).backward(T(go, cuda_dev))
        check_rows(zg.grad.cpu().numpy(), refs[0], refs[1], f"K{Kin.ndim}", scale=grad_z_scale(go, uv, Kin))


@pytest.mark.gpu
def test_gradient_input_types(pkg, cuda_dev, W):
    """float64 predictions (gradients come back float64), pred_r / pred_t as column views of one [B,7]
    head tensor, and only one of the two requiring grad -- for ADDLoss and PoseLoss."""
    B = 24
    pts = {3: W.sphere_mesh(120, 0.15, 1), 9: W.box_mesh(120, (0.05, 0.12, 0.06), 2)}
    pq, pt, gq, gt = W.random_poses(B, 14, rot_sigma=0.3, trans_sigma=0.01)
    obj = np.array([3, 9] * 12, np.int64)
    aq32, at32, aq64, at64 = refs_add(pts, pq, pt, gq, gt, obj)
    pq2, pt2, gq2, gt2 = pose_inputs(B, 14)
    pq32, pt32, pq64, pt64 = refs_pose(pq2, pt2, gq2, gt2, 1.0, 10.0, "geodesic")
    crit, pl = make_crit(pkg, pts, cuda_dev), pkg.PoseLoss(1.0, 10.0)
    for case in ("float64", "head", "rot_only", "trans_only"):
        for name, fn, (a, b, c, d), (rq32, rt32, rq64, rt64) in (
                ("ADDLoss", lambda x, y, c, d: crit(x, y, c, d, T(obj, cuda_dev)), (pq, pt, gq, gt), (aq32, at32, aq64, at64)),
                ("PoseLoss", pl, (pq2, pt2, gq2, gt2), (pq32, pt32, pq64, pt64))):
            if case == "head":
                head = T(np.concatenate([a, b], 1), cuda_dev).requires_grad_(True)
                x, y = head[:, :4], head[:, 4:]
            else:
                x, y = T(a, cuda_dev), T(b, cuda_dev)
                if case == "float64":
                    x, y = x.double(), y.double()
                x.requires_grad_(case != "trans_only")
                y.requires_grad_(case != "rot_only")
            fn(x, y, T(c, cuda_dev), T(d, cuda_dev)).backward()
            if case == "head":
                gx, gy = head.grad[:, :4], head.grad[:, 4:]
            else:
                gx, gy = x.grad, y.grad
                assert (gx is None) == (case == "trans_only") and (gy is None) == (case == "rot_only")
                if case == "float64":
                    assert gx.dtype == torch.float64 and gy.dtype == torch.float64
            if gx is not None:
                check_rows(gx.float().cpu().numpy(), rq32, rq64, f"{name} {case} grad_q")
            if gy is not None:
                check_rows(gy.float().cpu().numpy(), rt32, rt64, f"{name} {case} grad_t")
