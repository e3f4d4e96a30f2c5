"""ADDLoss.forward and its gradient on meshes beyond shared memory: the streamed loss form and the streamed backward
(csrc/p6d_adds_streamed.cu, csrc/p6d_add_bwd.cu), opt-in per table (large_mesh_loss).

CPU part: the rounding rules the streamed loss form relies on, pinned live at the new sizes (the batched matmul of a
large group rounds like oracle.transform; oracle.add_forward's fold equals the reference's op sequence); a gradient
reference whose nearest-point decisions are taken over blocks of pred rows, so that it stays affordable at 32,768
points (the reference's [N,N,3] temporary is 12.9 GB per sample there), pinned to the unblocked one; the C oracle's
backward against it.
GPU part: the forced streamed kernels against the resident ones where both run, the switch beyond both resident
limits against the oracle and the references, and the ADDLoss surface.
"""
import re
import tempfile

import numpy as np
import pytest
import torch

from conftest import same_bits
from oracle import torch_eager as E
from test_gradients import check_rows, f32_bits
from test_large_meshes import edge_poses
from test_loss_form import GPU_N, forward_value_chunked

F32 = np.float32
PIN_N = [4096, 7157, 8192, 12345, 16384, 32768]
PIN_G = [1, 2, 3, 8, 32, 33]
SYMMETRIC = frozenset({9, 10})


def T32(a):
    return torch.from_numpy(np.ascontiguousarray(a, F32))


def oracle_loss(oracle, pts, pq, pt, gq, gt, obj, dia=None):
    """oracle.add_forward's fold (groups in first-appearance order, float32 ATen sum per group, total / count) on
    per-sample values from oracle.add_eval(bmm=True), with the all-pairs scan run for symmetric groups only: at
    32,768 points an asymmetric sample's ADD-S costs the C oracle 10^9 pairs it would not use."""
    obj = np.asarray(obj, np.int64).ravel()
    table = oracle.MeshTable(pts, dia or {})
    total, count = F32(0.0), 0
    ids, first = np.unique(obj, return_index=True)
    for o in ids[np.argsort(first)]:
        if int(o) not in pts:
            continue
        idx = np.nonzero(obj == o)[0]
        sym = int(o) in SYMMETRIC
        r = oracle.add_eval(table, pq[idx], pt[idx], gq[idx], gt[idx], obj[idx], want_adds=sym, bmm=True,
                            n_threads=oracle.max_threads())
        total = F32(total + oracle.aten_sum(r[1] if sym else r[0]))
        count += len(idx)
    return F32(0.0) if count == 0 else F32(total / F32(count))


@torch.no_grad()
def nearest_chunked(pts, pq, pt, gq, gt, obj, rows=256):
    """Decisions for E.add_loss_grad: per valid sample, the nearest gt index of every pred point and the mask of zero
    distances.  The clouds come from the reference's batched matmul over the whole group; the nearest index of a
    symmetric sample from the reference's torch.norm(...).min(dim=1), over blocks of pred rows (each row sees the same
    values as in the unblocked form, so it takes the same index)."""
    pq, pt, gq, gt = T32(pq).reshape(-1, 4), T32(pt).reshape(-1, 3), T32(gq).reshape(-1, 4), T32(gt).reshape(-1, 3)
    obj = np.asarray(obj, np.int64).ravel()
    Rp, Rg = E.quat_to_mat(pq), E.quat_to_mat(gq)
    dec = {}
    for o in np.unique(obj):
        if int(o) not in pts:
            continue
        idx = torch.from_numpy(np.nonzero(obj == o)[0])
        m = T32(pts[int(o)]).reshape(1, -1, 3)
        cg = torch.matmul(m, Rg[idx].transpose(-1, -2)) + gt[idx].unsqueeze(1)
        cp = torch.matmul(m, Rp[idx].transpose(-1, -2)) + pt[idx].unsqueeze(1)
        n = m.shape[1]
        for k, s in enumerate(idx.tolist()):
            if int(o) in SYMMETRIC:
                near = torch.cat([torch.norm(cp[k, i:i + rows].unsqueeze(1) - cg[k].unsqueeze(0), dim=2).min(dim=1)[1]
                                  for i in range(0, n, rows)])
            else:
                near = torch.arange(n)
            dec[s] = (near, torch.norm(cp[k] - cg[k][near], dim=1) == 0)
    return dec


def refs_chunked(pts, pq, pt, gq, gt, obj, grad_out=1.0):
    """(grad_q, grad_t) of float32 and float64 autograd of the reference's formulas with the blocked decisions."""
    dec = nearest_chunked(pts, pq, pt, gq, gt, obj)
    q32, t32, _ = E.add_loss_grad(pts, pq, pt, gq, gt, obj, grad_out, torch.float32, dec)
    q64, t64, _ = E.add_loss_grad(pts, pq, pt, gq, gt, obj, grad_out, torch.float64, dec)
    return q32, t32, q64, t64


def tie_mesh(W, n, a=500, b=1500, seed=3):
    """A symmetric mesh of n points whose pred point 0 (identity rotation, translation (0.01, 0, 0)) has two gt
    points at the same rooted distance but different squares: the first at index a, the second, with the smaller
    square, at index b (tests/test_gradients.py, tie_fixture).  With a < 1024 <= b they lie in different gt tiles.
    torch.norm(...).min takes index a; a minimum over the squares takes b."""
    r = np.random.RandomState(seed)
    m = (r.standard_normal((n, 3)) * 0.05 + 0.3).astype(F32)
    m[0] = 0
    m[a] = f32_bits(0x3C541A59, 0xB9F609CF, 0xB9A7C982)
    m[b] = f32_bits(0x3C31229A, 0x39954080, 0x3B3C5B73)
    return m


def tie_rows(W, B, seed):
    """B poses: row 0 is the tie pose (identity rotations, pred translation (0.01, 0, 0), gt at the origin); the
    others are random."""
    pq, pt, gq, gt = W.random_poses(B, seed, rot_sigma=0.3, trans_sigma=0.01)
    pq[0] = gq[0] = (0, 0, 0, 1)
    pt[0] = (f32_bits(0x3C23D70A)[0], 0, 0)
    gt[0] = 0
    return pq, pt, gq, gt


# ----------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("n", PIN_N)
def test_bmm_rounding_and_forward_value_at_large_sizes(oracle, W, n):
    """The batched torch.matmul([1,N,3], [g,3,3]) + t of ADDLoss.forward rounds every sample like oracle.transform
    (the FMA chain, SlotInfo::xform_bmm from 45 points on), and oracle.add_forward's fold equals the reference's
    op sequence (oracle/torch_eager.forward_value) for an asymmetric group, for every g."""
    mesh = W.sphere_mesh(n, 0.12, 60 + n)
    m = T32(mesh).unsqueeze(0)
    for g in PIN_G:
        pq, pt, gq, gt = W.random_poses(g, 7 * n + g, rot_sigma=np.geomspace(0.01, 0.5, g), trans_sigma=0.01)
        R = E.quat_to_mat(T32(pq))
        cloud = (torch.matmul(m, R.transpose(-1, -2)) + T32(pt).unsqueeze(1)).numpy()
        for i in range(g):
            assert same_bits(cloud[i], oracle.transform(mesh, pq[i], pt[i])), (n, g, i)
        obj = np.full(g, 3, np.int64)
        want = E.forward_value({3: mesh}, pq, pt, gq, gt, obj)
        assert same_bits(oracle_loss(oracle, {3: mesh}, pq, pt, gq, gt, obj), want), (n, g)
        if n <= 4096 and g <= 3:
            assert same_bits(oracle.add_forward(oracle.MeshTable({3: mesh}), pq, pt, gq, gt, obj), want), (n, g)


def test_oracle_loss_fold_equals_add_forward(oracle, W):
    """The test's fold (ADD-S only for symmetric groups) equals oracle.add_forward on mixed batches."""
    pts = {3: W.sphere_mesh(700, 0.12, 1), 9: W.box_mesh(500, (0.1, 0.12, 0.05), 2), 10: W.sphere_mesh(45, 0.1, 3)}
    pq, pt, gq, gt = edge_poses(W, 40, 4, 0.2)
    obj = np.array([9, 3, 10, 3, -1, 7] * 7, np.int64)[:40]
    for sl in (slice(0, 40), slice(4, 6), slice(0, 1)):
        a = [x[sl] for x in (pq, pt, gq, gt, obj)]
        assert same_bits(oracle_loss(oracle, pts, *a), oracle.add_forward(oracle.MeshTable(pts), *a))


def test_chunked_gradient_reference_equals_the_unchunked_one(W):
    """The blocked decisions are the reference's own (E.add_loss_grad without decisions), index for index, and give
    the same gradient bits; the tie across two gt tiles takes the first index."""
    pts = {9: tie_mesh(W, 1600), 3: W.sphere_mesh(1600, 0.12, 5), 10: W.box_mesh(700, (0.1, 0.12, 0.05), 6)}
    pq, pt, gq, gt = tie_rows(W, 6, 7)
    obj = np.array([9, 3, 10, 9, -1, 10], np.int64)
    q32, t32, dec = E.add_loss_grad(pts, pq, pt, gq, gt, obj, 2.5)
    mine = nearest_chunked(pts, pq, pt, gq, gt, obj, rows=96)
    assert sorted(mine) == sorted(dec)
    for s in dec:
        assert torch.equal(mine[s][0], dec[s][0]) and torch.equal(mine[s][1], dec[s][1]), s
    assert int(dec[0][0][0]) == 500
    c32, ct32, c64, ct64 = refs_chunked(pts, pq, pt, gq, gt, obj, 2.5)
    assert same_bits(c32, q32) and same_bits(ct32, t32)
    q64, t64, _ = E.add_loss_grad(pts, pq, pt, gq, gt, obj, 2.5, torch.float64, dec)
    assert np.array_equal(c64, q64) and np.array_equal(ct64, t64)


@pytest.mark.parametrize("n", [2048, 19286, 32768])
def test_oracle_backward_against_the_chunked_reference(oracle, W, n):
    """The C oracle's backward (the resident kernel's rule) against the blocked autograd references at 1e-5 of the
    row maximum, with one symmetric sample (the tie across tiles) and asymmetric ones."""
    pts = {9: tie_mesh(W, n), 3: W.sphere_mesh(n, 0.12, n)}
    pq, pt, gq, gt = tie_rows(W, 4, n)
    obj = np.array([9, 3, 3, -1], np.int64)
    q32, t32, q64, t64 = refs_chunked(pts, pq, pt, gq, gt, obj, 2.5)
    oq, ot = oracle.add_backward(oracle.MeshTable(pts), pq, pt, gq, gt, obj, 2.5)
    check_rows(ot, t32, t64, f"n={n} grad_t")
    check_rows(oq, q32, q64, f"n={n} grad_q")


# ----------------------------------------------------------------------------------------------- GPU
def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def adds_max_points(pkg, dev):
    n = pkg.core.C.c_int()
    pkg.core.check(pkg.core.lib().p6d_adds_max_points(dev.index, pkg.core.C.byref(n)))
    return n.value


def bwd_max_points(pkg, dev):
    """Largest mesh add_backward_kernel holds: 12 bytes per point plus 1 KB within the opt-in shared memory."""
    return (pkg.core.device_info(dev.index)["smem_optin"] - 1024) // 12


def batches(W, B, seed, ids):
    """(name, (pq, pt, gq, gt, obj)) of the forced-vs-resident comparisons: symmetric, asymmetric, mixed with
    unknown ids, all unknown, and the edge rows (identical poses, NaN, inf, zero and non-unit quaternions)."""
    r = np.random.RandomState(seed)
    rq, rt, rgq, rgt = W.random_poses(B, seed + 1, rot_sigma=np.geomspace(0.005, 1.0, B), trans_sigma=0.01)
    sym = [i for i in ids if i in SYMMETRIC]
    asym = [i for i in ids if i not in SYMMETRIC]
    out = []
    if sym:
        out.append(("symmetric", (rq, rt, rgq, rgt, np.array(sym, np.int64)[r.randint(0, len(sym), B)])))
    if asym:
        out.append(("asymmetric", (rq, rt, rgq, rgt, np.array(asym, np.int64)[r.randint(0, len(asym), B)])))
    mixed = np.array(list(ids) + [-1, 2, max(ids) + 5], np.int64)[r.randint(0, len(ids) + 3, B)]
    out.append(("unknown ids", (rq, rt, rgq, rgt, mixed)))
    out.append(("all unknown", (rq, rt, rgq, rgt, np.full(B, -3, np.int64))))
    if B >= 10:
        out.append(("edge rows", (*edge_poses(W, B, seed, np.geomspace(0.005, 1.0, B)), mixed)))
    return out


def table_for(pkg, W, sizes, dev):
    pts = {}
    for oid, n in sizes.items():
        pts[oid] = W.box_mesh(n, (0.1, 0.12, 0.05), 900 + n) if oid in SYMMETRIC else W.sphere_mesh(n, 0.1, 1000 + n)
    return pts, pkg.core.MeshTable(pts, {}, pkg.SYMMETRIC_OBJECT_IDS, dev)


def loss_pair(table, d, streamed):
    loss, count = table.forward_loss(*d, streamed=streamed)
    return loss.cpu().numpy(), count.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [n for n in GPU_N] + ["mixed"])
def test_forward_forced_equals_resident(pkg, cuda_dev, W, n):
    """p6d_add_forward_streamed against p6d_add_forward: equal loss and count bits for every batch layout, at every
    mesh size of the loss-form grid up to the resident limit, and on a table mixing 1- and 10-point slots (which
    keep the unfused rounding) with a large mesh."""
    nmax = adds_max_points(pkg, cuda_dev)
    if n == "mixed":
        sizes = {3: 1, 10: 10, 9: nmax, 1: 44}
    else:
        n = nmax if n == "nmax" else n
        sizes = {3: n, 9: n, 10: max(1, n // 2)}
    pts, table = table_for(pkg, W, sizes, cuda_dev)
    for B in (1, 37, 600):
        for name, arrs in batches(W, B, B + len(sizes), sorted(pts)):
            d = [T(x, cuda_dev) for x in arrs]
            want = loss_pair(table, d, False)
            got = loss_pair(table, d, True)
            assert same_bits(got[0], want[0]) and np.array_equal(got[1], want[1]), (sizes, B, name, got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("n", ["nmax+1", 8192, 12345, 16384, 32768])
def test_forward_beyond_the_limit(pkg, cuda_dev, W, oracle, n):
    """Switch on, tables the resident loss form refuses: the loss equals oracle.add_forward's fold and the reference's
    op sequence (blocked per-sample values), at B = 1, 32 and a batch above one 64 MB chunk of the workspace (the
    grouped sum then spans the per-sample values of several launches).  The count is the number of valid samples."""
    nmax = adds_max_points(pkg, cuda_dev)
    n = nmax + 1 if n == "nmax+1" else n
    pts = {9: W.box_mesh(n, (0.1, 0.12, 0.05), 900 + n), 3: W.sphere_mesh(n, 0.1, 1000 + n),
           1: W.sphere_mesh(n // 3 + 1, 0.1, 77)}
    table = pkg.core.MeshTable(pts, {}, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev)
    chunk = (64 << 20) // (8 * ((n + 3) // 4 * 4) + 4)
    for B in (1, 32, chunk + 45):
        pq, pt, gq, gt = W.random_poses(B, n + B, rot_sigma=np.geomspace(0.005, 0.5, B), trans_sigma=0.01)
        obj = np.where(np.arange(B) % 2 == 0, 3, 1).astype(np.int64)
        obj[np.arange(B) % 7 == 3] = -1
        sym = [0] if B == 1 else [1, B - 1]          # few symmetric samples: the references' CPU time
        obj[sym] = 9
        d = [T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)]
        with pytest.raises(pkg.core.P6DError, match="at most"):
            table.forward_loss(*d)
        table.set_large_mesh_loss(True)
        loss, count = loss_pair(table, d, False)
        table.set_large_mesh_loss(False)
        valid = int(np.isin(obj, list(pts)).sum())
        assert int(count[0]) == valid
        assert same_bits(loss[0], oracle_loss(oracle, pts, pq, pt, gq, gt, obj)), (n, B)
        assert same_bits(loss[0], forward_value_chunked(E, pts, pq, pt, gq, gt, obj)), (n, B)


def run_grads(pkg, table, d, go, streamed):
    """Loss through the table's forward (for the device count), then the backward, resident or forced streamed."""
    _, count = table.forward_loss(*d)
    q, t = pkg.core.add_backward((*d, count, table, d[0].device), torch.tensor(go, device=d[0].device),
                                 streamed=streamed)
    return q.cpu().numpy(), t.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["forced 2048", "forced bwd_max", "switch bwd_max+1", "switch 32768"])
def test_backward_forced_and_beyond(pkg, cuda_dev, W, where):
    """The streamed backward (forced at sizes the resident kernel takes, by the switch beyond it) against float32 and
    float64 autograd of the reference's formulas at 1e-5 of the row maximum, zero and NaN rows where the reference
    has them, upstream gradient 2.5.  Row 0 is a tie whose two gt points lie in different 1,024-point tiles, the
    later one with the smaller square: the first one is the nearest.  Rows 1-3: pred == gt (exact zeros), a NaN
    translation, an unknown id."""
    bmax = bwd_max_points(pkg, cuda_dev)
    kind, size = where.split()
    n = {"2048": 2048, "bwd_max": bmax, "bwd_max+1": bmax + 1, "32768": 32768}[size]
    pts = {9: tie_mesh(W, n), 3: W.sphere_mesh(n, 0.12, n)}
    table = pkg.core.MeshTable(pts, {}, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev)
    B = 12
    pq, pt, gq, gt = tie_rows(W, B, n)
    obj = np.array([9, 3, 9, -1] + [3] * (B - 5) + [9], np.int64)
    pq[1], pt[1] = gq[1], gt[1]
    pt[2, 1] = np.nan
    d = [T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)]
    q32, t32, q64, t64 = refs_chunked(pts, pq, pt, gq, gt, obj, 2.5)
    table.set_large_mesh_loss(True)       # the forward beyond the resident loss form's limit
    if kind == "forced":
        rq, rt = run_grads(pkg, table, d, 2.5, False)     # the resident backward takes this table
        check_rows(rt, t32, t64, f"{where} resident grad_t")
        check_rows(rq, q32, q64, f"{where} resident grad_q")
        gq_, gt_ = run_grads(pkg, table, d, 2.5, True)
    else:
        _, count = table.forward_loss(*d)
        table.set_large_mesh_loss(False)
        with pytest.raises(pkg.core.P6DError, match="does not fit shared memory"):
            pkg.core.add_backward((*d, count, table, cuda_dev), torch.tensor(2.5, device=cuda_dev))
        table.set_large_mesh_loss(True)
        gq_, gt_ = run_grads(pkg, table, d, 2.5, False)
    check_rows(gt_, t32, t64, f"{where} grad_t")
    check_rows(gq_, q32, q64, f"{where} grad_q")


@pytest.mark.gpu
def test_addloss_surface(pkg, cuda_dev, W, oracle):
    """ADDLoss with a 20,000-point symmetric mesh: large_meshes alone leaves forward refused ("at most");
    large_mesh_loss makes the loss equal the oracle's and loss.backward() give the reference's gradients with only
    pred_r (or only pred_t) requiring grad; 32,769
    points are refused with the thread-count reason; two streams at once and repeated calls give the sequential
    bytes; the profiler shows the streamed kernels beyond the limit and the resident ones within it."""
    n = 20000
    mesh9, mesh3 = tie_mesh(W, n), W.sphere_mesh(n, 0.12, 8)
    crit = pkg.ADDLoss(tempfile.mkdtemp(), cuda_dev)
    crit.points[9], crit.points[3] = T(mesh9, cuda_dev), T(mesh3, cuda_dev)
    crit.diameters.update({9: 0.1, 3: 0.1})
    B = 8
    pq, pt, gq, gt = tie_rows(W, B, 21)
    obj = np.array([9, 3, 3, 9, 3, -1, 3, 3], np.int64)
    pts = {9: mesh9, 3: mesh3}
    d = [T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)]
    crit.large_meshes = True
    with pytest.raises(pkg.core.P6DError, match="at most"):
        crit(*d)
    crit.large_mesh_loss = True

    def step():
        x = d[0].clone().requires_grad_(True)
        loss = crit(x, d[1], d[2], d[3], d[4])
        loss.backward(torch.tensor(2.5, device=cuda_dev))
        return loss.detach().clone(), x.grad.clone()

    def step_t():
        y = d[1].clone().requires_grad_(True)
        loss = crit(d[0], y, d[2], d[3], d[4])
        loss.backward(torch.tensor(2.5, device=cuda_dev))
        return y.grad.clone()

    loss, gx = step()
    gy = step_t()
    assert same_bits(loss.cpu().numpy(), oracle_loss(oracle, pts, pq, pt, gq, gt, obj))
    q32, t32, q64, t64 = refs_chunked(pts, pq, pt, gq, gt, obj, 2.5)
    check_rows(gx.cpu().numpy(), q32, q64, "ADDLoss grad_q")
    check_rows(gy.cpu().numpy(), t32, t64, "ADDLoss grad_t")
    for _ in range(3):
        l2, g2 = step()
        assert torch.equal(l2, loss) and torch.equal(g2, gx)
        assert torch.equal(step_t(), gy)
    torch.cuda.synchronize(cuda_dev)
    streams = [torch.cuda.Stream(cuda_dev), torch.cuda.Stream(cuda_dev)]
    outs = [None, None, None, None]
    for i, s in enumerate(streams):
        with torch.cuda.stream(s):
            outs[i] = step()
            outs[2 + i] = step_t()
    torch.cuda.synchronize(cuda_dev)
    for i in range(2):
        assert torch.equal(outs[i][0], loss) and torch.equal(outs[i][1], gx) and torch.equal(outs[2 + i], gy)

    # kernel names: beyond the limit the streamed kernels, within it the resident ones (switch on in both)
    def kernels(fn, expect):
        """libp6d kernels (names without template arguments) that calls of fn launch.  A CUDA trace can come back
        without some kernel records (seen: none at all, or one of three), never with records of kernels that did
        not run; so each profile covers three calls of fn (the route of a call does not depend on the calls before
        it), and profiles are taken until every name in `expect` has been seen, at most four times.  The union is
        returned, so a kernel that must not run is looked for in every record collected."""
        seen = set()
        for _ in range(4):
            torch.cuda.synchronize(cuda_dev)
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    fn()
                torch.cuda.synchronize(cuda_dev)
            for ev in prof.events():
                m = re.search(r"p6d::(\w+)[<(]", ev.name)
                if m:
                    seen.add(m.group(1))
            if expect <= seen:
                break
        return seen
    beyond_expect = {"adds_streamed_kernel", "loss_finalize_kernel", "add_backward_streamed_kernel"}
    beyond = kernels(step, beyond_expect)
    assert beyond_expect <= beyond, beyond
    assert not beyond & {"adds_cta_kernel", "add_backward_kernel"}, beyond
    small = pkg.ADDLoss(tempfile.mkdtemp(), cuda_dev)
    small.points[9] = T(W.box_mesh(500, (0.1, 0.12, 0.05), 9), cuda_dev)
    small.large_meshes = small.large_mesh_loss = True

    def small_step():
        x = d[0].clone().requires_grad_(True)
        small(x, d[1], d[2], d[3], torch.full((B,), 9, dtype=torch.int64, device=cuda_dev)).backward()
    within_expect = {"adds_cta_kernel", "add_backward_kernel"}
    within = kernels(small_step, within_expect)
    assert within_expect <= within, within
    assert not any("streamed" in k or k == "loss_finalize_kernel" for k in within), within

    # above 32,768 points: the thread-count reason, forward and forced entries
    huge = pkg.ADDLoss(tempfile.mkdtemp(), cuda_dev)
    huge.points[9] = T(W.sphere_mesh(32769, 0.1, 53), cuda_dev)
    huge.large_mesh_loss = True
    with pytest.raises(pkg.core.P6DError, match="at most 32768 points.*thread count"):
        huge(*d)
    table = huge._mesh_table(cuda_dev)
    with pytest.raises(pkg.core.P6DError, match="at most 32768 points.*thread count"):
        table.forward_loss(*d, streamed=True)
    count = torch.ones(1, dtype=torch.int32, device=cuda_dev)
    for streamed in (False, True):
        with pytest.raises(pkg.core.P6DError, match="at most 32768 points.*thread count"):
            pkg.core.add_backward((*d, count, table, cuda_dev), torch.tensor(1.0, device=cuda_dev), streamed=streamed)
