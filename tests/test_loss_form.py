"""ADDLoss.forward's value: p6d_add_forward (the loss-form instantiations of adds_cta_kernel, the batched-matmul
rounding xform_bmm and loss_finalize in csrc/p6d_add.cu) against the reference's op sequence, over mesh sizes,
group sizes, batch layouts and edge samples.

The reference (models/add_loss.py:101-150) groups the valid samples by object in order of first appearance,
transforms each group with ONE batched torch.matmul([1,n,3], [g,3,3]) -- the batch size g decides MKL's path,
so a group is never split there -- takes ADD (or ADD-S for ids 9, 10) per sample, adds each group's float32
``per.sum()`` to a float32 total and returns ``total / count``.  oracle/torch_eager.forward_value runs exactly
that, but builds a [g, n, n, 3] tensor for symmetric ids; ``forward_value_chunked`` below runs the same ops with
the pairwise norm / min taken over blocks of samples and pred rows, and is pinned to forward_value where both fit.

CPU part: the reference ops of this machine against the oracle (oracle.add_forward, the rules the kernels restate)
over an n x g grid; the (n, g) points where they disagree must be the documented MKL exception (two samples of a
97...106- or 200-point mesh).  Groups above 32,768 samples: torch's ``sum`` splits across threads there, so the
reference's own bits depend on the caller's thread count; the oracle and the kernel keep the 1-thread order.
GPU part: the kernel's loss bits against the oracle and against the reference ops run on the GPU box (1e-5 where
that box's grid found an exception), and ``count`` against the number of valid samples.
"""
import tempfile
import threading

import numpy as np
import pytest
import torch

from conftest import bits, same_bits

SYMMETRIC = frozenset({9, 10})
GRID_N = [1, 2, 3, 5, 10, 11, 12, 44, 45, 46, 64, 97, 100, 106, 107, 150, 200, 201, 256, 500, 777, 1000, 2048, 3000]
GRID_G = [1, 2, 3, 4, 5, 7, 8, 9, 16, 17, 31, 32, 33, 64, 65, 128, 257]
# MKL's batched sgemm takes another path for exactly two samples of these mesh sizes (include/p6d.h)
DOCUMENTED = frozenset({(n, 2) for n in range(97, 107)} | {(200, 2)})
SYM_PAIRS = 300_000_000          # symmetric grid points with g * n^2 above this are left out (CPU time)
GPU_N = [1, 2, 3, 10, 11, 44, 45, 97, 106, 200, 500, 512, 513, 1024, 1025, 2048, 2049, 4096, "nmax"]
GPU_G = [1, 2, 3, 7, 8, 31, 32, 33, 100, 257]
SYM_PAIRS_GPU = 200_000_000      # the GPU grid leaves out symmetric groups with g * n^2 above this at n >= 2048
ATEN_GRAIN = 32768               # torch's CPU sum splits a row across threads above this many elements


@pytest.fixture(scope="module")
def eager():
    from oracle import torch_eager
    return torch_eager


def T32(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32))


@torch.no_grad()
def _per_sample(cp, cg, symmetric, budget):
    """ADD (or ADD-S) of every sample of one group from its transformed clouds [g, n, 3], as the reference
    computes it (norm -> min(dim=2) -> mean(dim=1)), with at most ~budget floats in any temporary.  Norm and min
    are taken per (pred row, gt point) and per pred row, and mean(dim=1) reduces each sample's row of n values
    on its own, so the blocks see exactly the values the unblocked form sees."""
    g, n = cp.shape[0], cp.shape[1]
    if not symmetric:
        c = max(1, budget // (3 * n))
        return torch.cat([torch.norm(cp[i:i + c] - cg[i:i + c], dim=2).mean(dim=1) for i in range(0, g, c)])
    c = max(1, budget // (3 * n * n))
    r = max(1, min(n, budget // (3 * n)))
    out = []
    for i in range(0, g, c):
        p, q = cp[i:i + c], cg[i:i + c]
        mins = torch.cat([torch.norm(p[:, j:j + r].unsqueeze(2) - q.unsqueeze(1), dim=3).min(dim=2)[0]
                          for j in range(0, n, r)], dim=1)
        out.append(mins.mean(dim=1))
    return torch.cat(out)


@torch.no_grad()
def reference_groups(eager, points, pq, pt, gq, gt, obj, budget=1 << 24):
    """[(object id, sample indices, per-sample values)] in order of first appearance: the reference's grouping,
    one batched torch.matmul per whole group, then the blocked per-sample values."""
    pq, pt, gq, gt = T32(pq).reshape(-1, 4), T32(pt).reshape(-1, 3), T32(gq).reshape(-1, 4), T32(gt).reshape(-1, 3)
    obj = np.asarray(obj, np.int64).ravel()
    meshes = {int(k): T32(v).reshape(-1, 3) for k, v in points.items()}
    Rp, Rg = eager.quat_to_mat(pq), eager.quat_to_mat(gq)
    ids, first = np.unique(obj, return_index=True)
    out = []
    for oid in ids[np.argsort(first)]:
        if int(oid) not in meshes:
            continue
        idx = torch.from_numpy(np.nonzero(obj == oid)[0])
        m = meshes[int(oid)].unsqueeze(0)
        cg = torch.matmul(m, Rg[idx].transpose(-1, -2)) + gt[idx].unsqueeze(1)
        cp = torch.matmul(m, Rp[idx].transpose(-1, -2)) + pt[idx].unsqueeze(1)
        out.append((int(oid), idx.numpy(), _per_sample(cp, cg, int(oid) in SYMMETRIC, budget)))
    return out


@torch.no_grad()
def forward_value_chunked(eager, points, pq, pt, gq, gt, obj, budget=1 << 24):
    """Value of ADDLoss.forward: group sums, total and ``total / count`` exactly as oracle/torch_eager.forward_value
    does them, on the blocked per-sample values."""
    total, count = torch.tensor(0.0), 0
    for _, idx, per in reference_groups(eager, points, pq, pt, gq, gt, obj, budget):
        total = total + per.sum()
        count += len(idx)
    return np.float32(0.0) if count == 0 else np.float32((total / count).item())


def fits_unblocked(n, g, symmetric):
    return g * n * (n if symmetric else 1) * 3 <= 1 << 25


def grid_poses(W, n, g):
    return W.random_poses(g, 1000 * n + g, rot_sigma=np.geomspace(0.01, 0.3, g), trans_sigma=0.01)


def grid_meshes(W, n):
    return {3: W.sphere_mesh(n, 0.12, 40 + n), 9: W.box_mesh(n, (0.1, 0.12, 0.05), 41 + n)}


class OneThread:
    """torch.set_num_threads(1) for the block, the caller's thread count restored afterwards."""

    def __enter__(self):
        self.prev = torch.get_num_threads()
        torch.set_num_threads(1)

    def __exit__(self, *exc):
        torch.set_num_threads(self.prev)


@pytest.fixture(scope="module")
def grid_exceptions(oracle, eager, W):
    """{(n, g): [what differed]} over GRID_N x GRID_G, symmetric (id 9) and asymmetric (id 3) groups of g samples:
    the whole loss of the reference's op sequence on this machine against oracle.add_forward, and every
    per-sample value against oracle.add_eval(bmm=True)."""
    found = {}
    for n in GRID_N:
        pts = grid_meshes(W, n)
        table = oracle.MeshTable(pts, {3: 0.12, 9: 0.16})
        for g in GRID_G:
            pq, pt, gq, gt = grid_poses(W, n, g)
            for oid in (3, 9):
                sym = oid in SYMMETRIC
                if sym and g * n * n > SYM_PAIRS:
                    continue
                obj = np.full(g, oid, np.int64)
                if fits_unblocked(n, g, sym):
                    whole = eager.forward_value(pts, pq, pt, gq, gt, obj)
                else:
                    whole = forward_value_chunked(eager, pts, pq, pt, gq, gt, obj)
                if bits(whole) != bits(oracle.add_forward(table, pq, pt, gq, gt, obj)):
                    found.setdefault((n, g), []).append(f"loss id {oid}")
                (_, _, per), = reference_groups(eager, pts, pq, pt, gq, gt, obj)
                ref = oracle.add_eval(table, pq, pt, gq, gt, obj, bmm=True)[1 if sym else 0]
                if not same_bits(per.numpy(), ref):
                    found.setdefault((n, g), []).append(f"per-sample id {oid}")
    print(f"\nloss-form exceptions on this machine (torch {torch.__version__}, {torch.get_num_threads()} threads): "
          f"{sorted(found.items())}")
    return found


def exceptional(points, obj, exceptions):
    """True when some group of the batch has an (n, group size) at which this machine's reference ops and the
    oracle disagree."""
    ids, counts = np.unique(np.asarray(obj, np.int64), return_counts=True)
    return any((len(points[int(o)]), int(c)) in exceptions for o, c in zip(ids, counts) if int(o) in points)


# ----------------------------------------------------------------------------------------------- CPU
def test_chunked_reference_equals_forward_value(oracle, eager, W):
    """The blocked helper gives forward_value's bits where both fit: several groups in first-appearance order,
    unknown ids, symmetric and asymmetric meshes, blocks smaller than a sample and larger than a group."""
    pts = {3: W.sphere_mesh(200, 0.12, 1), 9: W.box_mesh(150, (0.1, 0.12, 0.05), 2),
           10: W.box_mesh(45, (0.04, 0.17, 0.04), 3), 0: W.sphere_mesh(7, 0.1, 4)}
    r = np.random.RandomState(5)
    for B in (1, 2, 37, 300):
        pq, pt, gq, gt = W.random_poses(B, 6 + B, rot_sigma=np.geomspace(0.01, 0.5, B), trans_sigma=0.01)
        obj = np.array([10, 3, -1, 0, 9, 4])[r.randint(0, 6, B)]
        want = eager.forward_value(pts, pq, pt, gq, gt, obj)
        for budget in (1000, 50_000, 1 << 24):
            assert bits(forward_value_chunked(eager, pts, pq, pt, gq, gt, obj, budget)) == bits(want), (B, budget)


def test_grid_disagreements_are_the_documented_exception(grid_exceptions):
    """Reference ops of this machine vs the oracle over the n x g grid: any (n, g) point where they disagree must be
    the documented MKL exception, so that a new exception on another box fails here and names itself."""
    new = {k: v for k, v in grid_exceptions.items() if k not in DOCUMENTED}
    assert not new, f"undocumented loss-form exceptions (n, group size): {sorted(new.items())}"


@pytest.mark.parametrize("g", [ATEN_GRAIN, ATEN_GRAIN + 1, 100_000])
@pytest.mark.parametrize("oid", [3, 9])
def test_large_groups_follow_the_one_thread_order(oracle, eager, W, g, oid):
    """One group of g samples on a 3-point mesh: with one torch thread the oracle equals the reference ops bit for
    bit; with the default thread count too up to 32,768 samples, and within 1e-5 above (where torch's sum splits
    the group across threads)."""
    pts = {oid: W.sphere_mesh(3, 0.12, 7)}
    pq, pt, gq, gt = W.random_poses(g, 8, rot_sigma=np.geomspace(0.01, 0.3, g), trans_sigma=0.01)
    obj = np.full(g, oid, np.int64)
    want = oracle.add_forward(oracle.MeshTable(pts, {oid: 0.12}), pq, pt, gq, gt, obj)
    with OneThread():
        assert bits(eager.forward_value(pts, pq, pt, gq, gt, obj)) == bits(want)
        assert bits(forward_value_chunked(eager, pts, pq, pt, gq, gt, obj, budget=20_000)) == bits(want)
    default = eager.forward_value(pts, pq, pt, gq, gt, obj)
    if g <= ATEN_GRAIN:
        assert bits(default) == bits(want)
    assert abs(float(default) - float(want)) <= 1e-5 * abs(float(want))


# ----------------------------------------------------------------------------------------------- GPU
def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def adds_max_points(pkg, dev):
    n = pkg.core.C.c_int()
    pkg.core.check(pkg.core.lib().p6d_adds_max_points(dev.index, pkg.core.C.byref(n)))
    return n.value


def make_crit(pkg, pts, dev, dia=None):
    crit = pkg.ADDLoss(tempfile.mkdtemp(), dev)
    for k, v in pts.items():
        crit.points[k] = torch.from_numpy(np.ascontiguousarray(v, np.float32)).to(dev)
    crit.diameters.update(dia or {k: 0.1 for k in pts})
    return crit


def kernel_loss(crit, dev, pq, pt, gq, gt, obj):
    """(loss, count) of one p6d_add_forward call through the ADDLoss's mesh table."""
    d = [T(x, dev) for x in (pq, pt, gq, gt)] + [T(np.asarray(obj, np.int64), dev)]
    loss, count = crit._mesh_table(dev).forward_loss(*d)
    return np.float32(loss.item()), int(count.item())


def n_valid(pts, obj):
    return int(np.isin(np.asarray(obj, np.int64), np.array(sorted(pts), np.int64)).sum())


def check(got, count, pts, obj, want_oracle, want_eager, exceptions, what):
    """The kernel's loss equals the oracle bit for bit, and the reference ops of this box bit for bit unless a group
    of the batch is at an exception point found by the grid (1e-5 there); count = valid samples."""
    assert count == n_valid(pts, obj), what
    assert same_bits(got, want_oracle), (what, float(got), float(want_oracle))
    if exceptional(pts, obj, exceptions):
        assert abs(float(got) - float(want_eager)) <= 1e-5 * abs(float(want_eager)), (what, got, want_eager)
    else:
        assert same_bits(got, want_eager), (what, float(got), float(want_eager))


def run_and_check(oracle, eager, crit, dev, pts, batch, exceptions, what):
    pq, pt, gq, gt, obj = batch
    got, count = kernel_loss(crit, dev, *batch)
    want_o = oracle.add_forward(oracle.MeshTable(pts), pq, pt, gq, gt, obj)
    want_e = forward_value_chunked(eager, pts, pq, pt, gq, gt, obj)
    check(got, count, pts, obj, want_o, want_e, exceptions, what)
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("n", GPU_N)
def test_shape_grid(pkg, cuda_dev, oracle, eager, W, grid_exceptions, n):
    """One group of g samples per call, asymmetric (id 3) and symmetric (id 9), n points: the loss-form kernel of
    every mesh-size class, both sides of the 44/45-point bmm edge and of the class edges, up to the forward's
    limit."""
    n = adds_max_points(pkg, cuda_dev) if n == "nmax" else n
    pts = grid_meshes(W, n)
    crit = make_crit(pkg, pts, cuda_dev)
    for g in GPU_G:
        pq, pt, gq, gt = grid_poses(W, n, g)
        for oid in (3, 9):
            if oid in SYMMETRIC and n >= 2048 and g * n * n > SYM_PAIRS_GPU:
                continue
            obj = np.full(g, oid, np.int64)
            run_and_check(oracle, eager, crit, cuda_dev, pts, (pq, pt, gq, gt, obj), grid_exceptions, (n, g, oid))


@pytest.mark.gpu
def test_small_meshes_in_the_large_class_kernel(pkg, cuda_dev, oracle, eager, W, grid_exceptions):
    """A 5-point and a 3,000-point mesh in one table: the 5-point groups run in the large-class loss kernel with
    the naive-bmm rounding, next to a symmetric 3,000-point group."""
    pts = {0: W.sphere_mesh(5, 0.1, 11), 9: W.box_mesh(3000, (0.1, 0.12, 0.05), 12)}
    crit = make_crit(pkg, pts, cuda_dev)
    for g in GPU_G:
        B = g + 3
        pq, pt, gq, gt = W.random_poses(B, 13 + g, rot_sigma=np.geomspace(0.01, 0.3, B), trans_sigma=0.01)
        obj = np.random.RandomState(g).permutation(np.r_[np.zeros(g, np.int64), np.full(3, 9)])
        run_and_check(oracle, eager, crit, cuda_dev, pts, (pq, pt, gq, gt, obj), grid_exceptions, g)
        pure = np.zeros(g, np.int64)
        run_and_check(oracle, eager, crit, cuda_dev, pts, (pq[:g], pt[:g], gq[:g], gt[:g], pure), grid_exceptions,
                      ("5 points alone", g))


LINEMOD_N = [5, 44, 45, 97, 150, 200, 300, 500, 512, 64, 250, 11, 3]     # ids 0..12; 9, 10 symmetric


@pytest.mark.gpu
@pytest.mark.parametrize("largest", [512, 1500])
def test_group_layouts(pkg, cuda_dev, oracle, eager, W, grid_exceptions, largest):
    """Group order, lone samples, all 13 LineMOD ids and ids without a mesh, in a table whose largest mesh selects
    the small (512) or the large (1,500) class of loss kernel.  Ids 13 and 14 are free slots (15 has a mesh)."""
    sizes = list(LINEMOD_N)
    sizes[12] = largest if largest > 512 else sizes[12]
    pts = {k: (W.box_mesh(n, (0.1, 0.12, 0.05), 20 + k) if k in SYMMETRIC else W.sphere_mesh(n, 0.12, 20 + k))
           for k, n in enumerate(sizes)}
    pts[15] = W.sphere_mesh(20, 0.1, 35)
    crit = make_crit(pkg, pts, cuda_dev)
    r = np.random.RandomState(largest)
    layouts = {
        "first appearance != id order": np.r_[[10, 3, 10, 0, 3], r.choice([0, 3, 7, 10], 95)],
        "lone last sample": np.r_[r.choice([1, 2, 9], 63), [5]],
        "all 13 ids interleaved": r.permutation(np.tile(np.arange(13), 40)),
        "ids without a mesh": r.choice([-1, 13, 10 ** 6, 4, 9, 12, 15], 200),
        "one sample each, descending": np.arange(15, -2, -1),
        "all unknown": r.choice([-1, 13, 14, 10 ** 6, -(10 ** 6)], 50),
    }
    for what, obj in layouts.items():
        obj = np.asarray(obj, np.int64)
        B = len(obj)
        pq, pt, gq, gt = W.random_poses(B, B + largest, rot_sigma=np.geomspace(0.01, 0.3, B), trans_sigma=0.01)
        got = run_and_check(oracle, eager, crit, cuda_dev, pts, (pq, pt, gq, gt, obj), grid_exceptions, what)
        # the module surface returns the same value, with and without autograd
        d = [T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)]
        assert same_bits(crit(*d).item(), got), what
        pr = d[0].clone().requires_grad_(True)
        assert same_bits(crit(pr, d[1], d[2], d[3], d[4]).item(), got), what
    assert bits(got) == bits(np.float32(0.0))


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 2, 4096, 65536])
def test_batch_sizes(pkg, cuda_dev, oracle, eager, W, grid_exceptions, B):
    """B = 1 ... 65,536 on meshes of 64 points or fewer: one CTA per pose up to many poses per CTA, where the
    last CTA's ticket decides who folds the groups."""
    pts = {3: W.sphere_mesh(64, 0.12, 50), 10: W.box_mesh(12, (0.04, 0.17, 0.04), 51), 1: W.sphere_mesh(45, 0.1, 52)}
    crit = make_crit(pkg, pts, cuda_dev)
    pq, pt, gq, gt = W.random_poses(B, 53 + B, rot_sigma=np.geomspace(0.01, 0.3, B), trans_sigma=0.01)
    obj = np.array([3, 10, 1, -1])[np.random.RandomState(B).randint(0, 4, B)]
    obj[0] = 10
    run_and_check(oracle, eager, crit, cuda_dev, pts, (pq, pt, gq, gt, obj), grid_exceptions, B)


@pytest.mark.gpu
@pytest.mark.parametrize("g", [7, 8, 31, 32, 33, 511, 512, 8192, ATEN_GRAIN])
def test_group_sums_across_the_cascade_edges(pkg, cuda_dev, oracle, eager, W, grid_exceptions, g):
    """Two interleaved groups of g samples each (a 64-point asymmetric and a 12-point symmetric mesh): group sizes
    on both sides of the edges of ATen's cascade sum (8-lane vectors, 32 accumulators, 16-step levels)."""
    pts = {3: W.sphere_mesh(64, 0.12, 60), 10: W.box_mesh(12, (0.04, 0.17, 0.04), 61)}
    crit = make_crit(pkg, pts, cuda_dev)
    B = 2 * g
    pq, pt, gq, gt = W.random_poses(B, 62 + g, rot_sigma=np.geomspace(0.01, 0.5, B), trans_sigma=0.02)
    obj = np.where(np.arange(B) % 2 == 0, 10, 3).astype(np.int64)
    run_and_check(oracle, eager, crit, cuda_dev, pts, (pq, pt, gq, gt, obj), grid_exceptions, g)


@pytest.mark.gpu
@pytest.mark.parametrize("g", [ATEN_GRAIN + 1, 100_000])
def test_groups_above_the_grain_keep_the_one_thread_order(pkg, cuda_dev, oracle, eager, W, g):
    """Groups of more than 32,768 samples: the kernel gives the oracle's bits, which are the reference's with one
    torch thread; with the default thread count the reference agrees within 1e-5."""
    pts = {3: W.sphere_mesh(64, 0.12, 70), 9: W.box_mesh(12, (0.1, 0.12, 0.05), 71)}
    crit = make_crit(pkg, pts, cuda_dev)
    B = g + 5
    pq, pt, gq, gt = W.random_poses(B, 72 + g, rot_sigma=np.geomspace(0.01, 0.5, B), trans_sigma=0.02)
    obj = np.full(B, 3, np.int64)
    obj[[0, 17, 1000, 5000, B - 1]] = 9
    got, count = kernel_loss(crit, cuda_dev, pq, pt, gq, gt, obj)
    assert count == B
    assert same_bits(got, oracle.add_forward(oracle.MeshTable(pts), pq, pt, gq, gt, obj))
    with OneThread():
        assert same_bits(got, forward_value_chunked(eager, pts, pq, pt, gq, gt, obj))
    default = forward_value_chunked(eager, pts, pq, pt, gq, gt, obj)
    assert abs(float(got) - float(default)) <= 1e-5 * abs(float(default))


@pytest.mark.gpu
def test_count_beyond_float32_integers(pkg, cuda_dev, oracle, eager):
    """B = 2^24 + 3 samples of a 1-point mesh: (float)count rounds to 2^24 + 4, as the reference's
    ``total / count`` does.  The inputs are such that dividing in float64 would give another float32."""
    B = (1 << 24) + 3
    pts = {0: np.array([[0.01, -0.02, 0.03]], np.float32)}
    crit = make_crit(pkg, pts, cuda_dev)
    q = np.zeros((B, 4), np.float32)
    q[:, 3] = 1.0
    gt = np.zeros((B, 3), np.float32)
    pt = np.zeros((B, 3), np.float32)
    pt[:, 0] = np.random.RandomState(80).rand(B).astype(np.float32) * np.float32(0.01)
    obj = np.zeros(B, np.int64)
    got, count = kernel_loss(crit, cuda_dev, q, pt, q, gt, obj)
    assert count == B
    table = oracle.MeshTable(pts)
    want = oracle.add_forward(table, q, pt, q, gt, obj)
    total = oracle.aten_sum(oracle.add_eval(table, q, pt, q, gt, obj, bmm=True)[0])
    assert bits(np.float32(np.float64(total) / B)) != bits(want)        # the case discriminates
    assert same_bits(got, want)
    with OneThread():
        assert same_bits(got, forward_value_chunked(eager, pts, q, pt, q, gt, obj))


@pytest.mark.gpu
def test_edge_samples(pkg, cuda_dev, oracle, eager, W, grid_exceptions):
    """NaN and inf samples propagate into the loss, a zero quaternion is the identity, identical poses give an
    exact +0, and a NaN sample under an id without a mesh changes nothing."""
    pts = {3: W.sphere_mesh(100, 0.12, 90), 10: W.box_mesh(64, (0.04, 0.17, 0.04), 91)}
    crit = make_crit(pkg, pts, cuda_dev)
    B = 64
    base = W.random_poses(B, 92, rot_sigma=np.geomspace(0.01, 0.3, B), trans_sigma=0.01)
    obj = np.where(np.arange(B) % 3 == 0, 10, 3).astype(np.int64)
    obj[7] = -1

    def case(edit):
        pq, pt, gq, gt = (a.copy() for a in base)
        o = obj.copy()
        edit(pq, pt, gq, gt)
        return run_and_check(oracle, eager, crit, cuda_dev, pts, (pq, pt, gq, gt, o), grid_exceptions, edit.__name__)

    def nan_pred_t(pq, pt, gq, gt): pt[5, 1] = np.nan
    def nan_symmetric(pq, pt, gq, gt): pq[6] = np.nan
    def inf_pred_t(pq, pt, gq, gt): pt[4, 2] = np.inf
    def zero_quaternion(pq, pt, gq, gt): pq[8] = 0.0
    def non_unit(pq, pt, gq, gt): pq[9] *= 3.0; gq[10] *= 1e-3
    def identical(pq, pt, gq, gt): pq[:] = gq; pt[:] = gt
    def nan_unknown(pq, pt, gq, gt): pt[7] = np.nan; pq[7] = np.nan
    def unchanged(pq, pt, gq, gt): pass

    assert np.isnan(case(nan_pred_t)) and np.isnan(case(nan_symmetric))
    assert case(inf_pred_t) == np.inf
    assert np.isfinite(case(zero_quaternion)) and np.isfinite(case(non_unit))
    assert bits(case(identical)) == bits(np.float32(0.0))
    assert bits(case(nan_unknown)) == bits(case(unchanged))


@pytest.mark.gpu
def test_repeat_and_two_streams(pkg, cuda_dev, oracle, eager, W, grid_exceptions):
    """The same call twice gives the same bits (the ticket is left zeroed), and two host threads calling on two
    streams with different batches on one table each get their own reference value."""
    pts = {3: W.sphere_mesh(300, 0.12, 100), 9: W.box_mesh(200, (0.1, 0.12, 0.05), 101), 0: W.sphere_mesh(30, 0.1, 102)}
    crit = make_crit(pkg, pts, cuda_dev)
    table = crit._mesh_table(cuda_dev)
    batches, wants = [], []
    for k, B in enumerate((3000, 517)):
        pq, pt, gq, gt = W.random_poses(B, 103 + k, rot_sigma=np.geomspace(0.01, 0.3, B), trans_sigma=0.01)
        obj = np.array([0, 3, 9, 5])[np.random.RandomState(104 + k).randint(0, 4, B)]
        got = run_and_check(oracle, eager, crit, cuda_dev, pts, (pq, pt, gq, gt, obj), grid_exceptions, B)
        assert bits(kernel_loss(crit, cuda_dev, pq, pt, gq, gt, obj)[0]) == bits(got)
        batches.append([T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)])
        wants.append((bits(got), n_valid(pts, obj)))
    torch.cuda.synchronize(cuda_dev)
    results, errors = [[], []], []

    def worker(i):
        try:
            s = torch.cuda.Stream(cuda_dev)
            with torch.cuda.stream(s):
                outs = [table.forward_loss(*batches[i]) for _ in range(20)]
            s.synchronize()
            results[i] = [(bits(np.float32(lo.item())), int(c.item())) for lo, c in outs]
        except Exception as e:              # reported by the main thread
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for i in range(2):
        assert results[i] == [wants[i]] * 20, i
