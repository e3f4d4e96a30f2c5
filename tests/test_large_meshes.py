"""Meshes beyond shared memory: the streamed ADD / ADD-S kernel (csrc/p6d_adds_streamed.cu), opt-in per table.

CPU part: the rounding rules the kernels reproduce, pinned live at the new sizes (tests/test_live_pins.py stops
at 2,048 points for torch.mm and 4,097 for Tensor.mean), and a pred-row-chunked restatement of the reference's
ADD-S op sequence that stays affordable at 32,768 points (the reference's [N,N,3] temporary is 12.9 GB there).
GPU part: the streamed kernel against the resident kernels byte for byte where both run, against the oracle and
the chunked restatement beyond the resident limit, and through every caller that takes it.
"""
import tempfile

import numpy as np
import pytest
import torch

from conftest import same_bits

SIZES_PIN = [4096, 7157, 8192, 16384, 20000, 32767, 32768]
BEYOND = ["nmax+1", 8192, 12345, 16384, 32768]


@pytest.fixture(scope="module")
def eager():
    from oracle import torch_eager
    return torch_eager


@torch.no_grad()
def eval_pose_chunked(mesh, Rp, tp, Rg, tg, rows=512):
    """(ADD, ADD-S) of one pose as Python floats: the reference's op sequence (models/add_loss.py:178-190) with
    the all-pairs norm / min taken over blocks of pred rows.  Every row's norm and min see exactly the values they
    see in the unchunked [N,N,3] form, so the per-point minima, and the mean over them, are the same."""
    cloud_gt = torch.mm(mesh, Rg.T) + tg
    cloud_pred = torch.mm(mesh, Rp.T) + tp
    add = torch.norm(cloud_pred - cloud_gt, dim=1, p=2).mean().item()
    mins = torch.cat([torch.norm(cloud_pred[i:i + rows].unsqueeze(1) - cloud_gt.unsqueeze(0), dim=2).min(dim=1)[0]
                      for i in range(0, mesh.shape[0], rows)])
    return add, mins.mean().item()


def chunked_poses(eager, mesh, pq, pt, gq, gt):
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float32))
    m = T(mesh).reshape(-1, 3)
    Rp, Rg = eager.quat_to_mat(T(pq).reshape(-1, 4)), eager.quat_to_mat(T(gq).reshape(-1, 4))
    out = [eval_pose_chunked(m, Rp[i], T(pt[i]), Rg[i], T(gt[i])) for i in range(len(pq))]
    return np.array([o[0] for o in out], np.float32), np.array([o[1] for o in out], np.float32)


# ----------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("n", SIZES_PIN)
def test_mm_mean_and_sum_rules_hold_at_large_sizes(oracle, eager, W, n):
    """torch.mm + t rounds as the FMA chain and Tensor.mean() / sum() sum in the oracle's cascade order up to
    32,768 elements, with torch's default thread count (above that ATen splits a row across threads)."""
    mesh = W.sphere_mesh(n, 0.15, 700 + n)
    pq, pt, _, _ = W.random_poses(2, 800 + n, rot_sigma=0.3, trans_sigma=0.01)
    for q, t in zip(pq, pt):
        R = eager.quat_to_mat(torch.from_numpy(q[None]))[0]
        got = (torch.mm(torch.from_numpy(mesh), R.T) + torch.from_numpy(t)).numpy()
        assert same_bits(got, oracle.transform(mesh, q, t)), f"torch.mm rounding rule changed for n = {n}"
    x = (np.random.RandomState(n).rand(n) * 0.02 + 1e-4).astype(np.float32)
    assert same_bits(oracle.aten_mean(x), np.float32(torch.from_numpy(x).mean().item()))
    assert same_bits(oracle.aten_sum(x), np.float32(torch.from_numpy(x).sum().item()))


def test_chunked_restatement_equals_the_reference_ops_and_the_oracle(oracle, eager, W):
    """The chunked form equals the unchunked op sequence (oracle/torch_eager.eval_pose) at 1,000 points and the
    oracle bit for bit at 8,192 points, where the unchunked form would need 805 MB per pose."""
    mesh = W.box_mesh(1000, (0.1, 0.12, 0.05), 31)
    pq, pt, gq, gt = W.random_poses(4, 32, rot_sigma=np.array([0.01, 0.1, 0.5, 1.0]))
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float32))
    Rp, Rg = eager.quat_to_mat(T(pq)), eager.quat_to_mat(T(gq))
    for i in range(4):
        a = eager.eval_pose(T(mesh), Rp[i], T(pt[i]), Rg[i], T(gt[i]))
        c = eval_pose_chunked(T(mesh), Rp[i], T(pt[i]), Rg[i], T(gt[i]), rows=96)
        assert same_bits(np.float32(a), np.float32(c))
    mesh = W.box_mesh(8192, (0.1, 0.12, 0.05), 33)
    pq, pt, gq, gt = W.random_poses(2, 34, rot_sigma=0.1)
    add, adds = chunked_poses(eager, mesh, pq, pt, gq, gt)
    ref = oracle.add_eval(oracle.MeshTable({9: mesh}, {9: 0.16}), pq, pt, gq, gt, np.full(2, 9, np.int64),
                          n_threads=oracle.max_threads())
    assert same_bits(add, ref[0]) and same_bits(adds, ref[1])


# ----------------------------------------------------------------------------------------------- GPU
def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def adds_max_points(pkg, dev):
    n = pkg.core.C.c_int()
    pkg.core.check(pkg.core.lib().p6d_adds_max_points(dev.index, pkg.core.C.byref(n)))
    return n.value


def make_crit(pkg, pts, dia, dev):
    crit = pkg.ADDLoss(tempfile.mkdtemp(), dev)
    for k, v in pts.items():
        crit.points[k] = torch.from_numpy(np.ascontiguousarray(v)).to(dev)
    crit.diameters.update(dia)
    return crit


def edge_poses(W, B, seed, sigma):
    pq, pt, gq, gt = W.random_poses(B, seed, rot_sigma=sigma)
    pq[3] = gq[3]; pt[3] = gt[3]                      # identical poses: every distance 0
    pt[4, 0] = np.nan                                 # NaN propagates through every minimum
    pq[5] = np.nan
    pt[6, 2] = np.inf
    pq[7] *= 3.0                                      # non-unit quaternion
    pq[8] = 0.0                                       # zero quaternion
    gq[9] *= 1e-3
    return pq, pt, gq, gt


def accumulators(n_slots, dev):
    return [torch.zeros(n_slots, dtype=torch.int64, device=dev), torch.zeros(n_slots, dtype=torch.int64, device=dev),
            torch.zeros(n_slots, dtype=torch.float64, device=dev), torch.zeros(n_slots, dtype=torch.float64, device=dev)]


def same_accumulators(a, b):
    # counts exactly; the float64 sums are atomics in launch order, equal to rounding (NaN where a NaN pose adds in)
    return (torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
            and torch.allclose(a[2], b[2], rtol=1e-12, atol=0, equal_nan=True)
            and torch.allclose(a[3], b[3], rtol=1e-12, atol=0, equal_nan=True))


def table_of(pkg, W, sizes, dev):
    pts = {}
    for k, n in enumerate(sizes):
        oid = (9, 1, 10)[k]
        pts[oid] = W.box_mesh(n, (0.1, 0.12, 0.05), 900 + n) if oid in (9, 10) else W.sphere_mesh(n, 0.1, 1000 + n)
    dia = {k: 0.1 + 0.01 * k for k in pts}
    return pts, dia, pkg.core.MeshTable(pts, dia, pkg.SYMMETRIC_OBJECT_IDS, dev)


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [(1, 2, 3), (10, 11, 37), (500, 1023, 1025), (2048, 4096), ("nmax",)])
def test_streamed_equals_resident_byte_for_byte(pkg, cuda_dev, W, sizes):
    """p6d_add_eval_streamed against p6d_add_eval where both run: all 11 B output bytes and the accumulators, for
    several objects per table, ids without a mesh (absent, negative), processing order None and argsort, rotation
    noise 0.01 / 0.1 / 1.0 with NaN / inf / zero / non-unit poses, and without ADD-S against the ADD-only kernel."""
    sizes = tuple(adds_max_points(pkg, cuda_dev) if s == "nmax" else s for s in sizes)
    pts, dia, table = table_of(pkg, W, sizes, cuda_dev)
    ids = np.array(sorted(pts) + [-1, 2, max(pts) + 5], np.int64)
    B = 2000
    r = np.random.RandomState(sum(sizes))
    for sigma in (0.01, 0.1, 1.0):
        pq, pt, gq, gt = edge_poses(W, B, int(100 * sigma) + sizes[0], sigma)
        obj = ids[r.randint(0, len(ids), B)]
        d = [T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)]
        order = torch.argsort(d[4], stable=True).to(torch.int32)
        for want_adds in (True, False):
            nbytes = 11 * B if want_adds else None
            for o in (None, order):
                acc_r, acc_s = accumulators(table.n_slots, cuda_dev), accumulators(table.n_slots, cuda_dev)
                res = table.evaluate_packed(*d, want_adds=want_adds, order=o, acc=acc_r)
                st = table.evaluate_packed(*d, want_adds=want_adds, order=o, acc=acc_s, streamed=True)
                if want_adds:
                    assert torch.equal(res[:nbytes], st[:nbytes]), (sizes, sigma, o is None)
                else:   # adds is not written without ADD-S
                    assert torch.equal(res[:4 * B], st[:4 * B]) and torch.equal(res[8 * B:11 * B], st[8 * B:11 * B])
                assert same_accumulators(acc_r, acc_s), (sizes, sigma, want_adds)
    # B = 0 and B = 1
    d1 = [x[:1] for x in d]
    assert torch.equal(table.evaluate_packed(*d1)[:11], table.evaluate_packed(*d1, streamed=True)[:11])
    d0 = [x[:0] for x in d]
    assert table.evaluate_packed(*d0, streamed=True).numel() == 16


@pytest.mark.gpu
@pytest.mark.parametrize("n", BEYOND)
def test_beyond_the_resident_limit_equals_the_oracle(pkg, cuda_dev, W, oracle, eager, n):
    """Tables the resident kernels refuse: with the switch on, a seeded sample of poses equals the oracle bit for
    bit (sphere and box meshes, one mesh with a NaN vertex), and two poses equal the chunked torch-eager
    restatement run on this machine."""
    nmax = adds_max_points(pkg, cuda_dev)
    n = nmax + 1 if n == "nmax+1" else n
    pts = {9: W.box_mesh(n, (0.1, 0.12, 0.05), 900 + n), 1: W.sphere_mesh(n, 0.1, 1000 + n),
           10: W.sphere_mesh(n // 3 + 1, 0.1, 77).copy()}
    pts[10][17, 1] = np.nan
    dia = {9: 0.16, 1: 0.1, 10: 0.17}
    table = pkg.core.MeshTable(pts, dia, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev)
    B = 300
    pq, pt, gq, gt = edge_poses(W, B, n, np.geomspace(0.005, 1.0, B))
    ids = np.array(sorted(pts) + [-1], np.int64)
    obj = ids[np.random.RandomState(n).randint(0, len(ids), B)]
    d = [T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)]
    with pytest.raises(pkg.core.P6DError, match="at most"):
        table.evaluate_packed(*d)
    table.set_large_meshes(True)
    out = table.evaluate_packed(*d).cpu().numpy()
    add, adds = out[:4 * B].view(np.float32), out[4 * B:8 * B].view(np.float32)
    hit, valid = out[8 * B:9 * B], out[9 * B:10 * B]
    sel = np.r_[np.arange(10), np.random.RandomState(n + 1).choice(np.arange(10, B), 22, replace=False)]
    ref = oracle.add_eval(oracle.MeshTable(pts, dia), pq[sel], pt[sel], gq[sel], gt[sel], obj[sel],
                          n_threads=oracle.max_threads())
    assert same_bits(add[sel], ref[0]) and same_bits(adds[sel], ref[1])
    assert np.array_equal(hit[sel], ref[2]) and np.array_equal(valid[sel], ref[3])
    two = np.nonzero(obj == 9)[0][10:12]
    e_add, e_adds = chunked_poses(eager, pts[9], pq[two], pt[two], gq[two], gt[two])
    assert same_bits(add[two], e_add) and same_bits(adds[two], e_adds)


@pytest.mark.gpu
def test_add_only_beyond_its_limit(pkg, cuda_dev, W, oracle):
    """Without ADD-S, the ADD-only kernel keeps its own larger limit; at 20,000 points the switch sends the call to
    the streamed kernel, and symmetric ids decide on ADD as before."""
    pts = {9: W.box_mesh(20000, (0.1, 0.12, 0.05), 5), 1: W.sphere_mesh(20000, 0.1, 6)}
    dia = {9: 0.16, 1: 0.1}
    table = pkg.core.MeshTable(pts, dia, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev)
    B = 256
    pq, pt, gq, gt = edge_poses(W, B, 7, np.geomspace(0.005, 0.5, B))
    obj = np.where(np.arange(B) % 3 == 0, 9, 1).astype(np.int64)
    obj[11] = -1
    d = [T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)]
    with pytest.raises(pkg.core.P6DError, match="at most"):
        table.evaluate_packed(*d, want_adds=False)
    table.set_large_meshes(True)
    out = table.evaluate_packed(*d, want_adds=False).cpu().numpy()
    ref = oracle.add_eval(oracle.MeshTable(pts, dia), pq, pt, gq, gt, obj, want_adds=False,
                          n_threads=oracle.max_threads())
    assert same_bits(out[:4 * B].view(np.float32), ref[0])
    assert np.array_equal(out[8 * B:9 * B], ref[2]) and np.array_equal(out[9 * B:10 * B], ref[3])


@pytest.mark.gpu
def test_addloss_surface_with_a_large_mesh(pkg, cuda_dev, W, oracle):
    """ADDLoss with a 10,000-point mesh: refused by default; with large_meshes = True eval_metrics equals the
    oracle's dict by repr and still consults borderline_resolver; forward keeps its limit; evaluate_host's
    per-object totals are the per-pose sums; 32,769 points are refused with the reason."""
    mesh = W.sphere_mesh(10000, 0.1, 50)
    pq, pt, gq, gt = W.random_poses(24, 51, rot_sigma=np.geomspace(0.005, 0.3, 24))
    obj = np.zeros(24, np.int64)
    obj[5] = 4
    d = [T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)]
    crit = make_crit(pkg, {0: mesh}, {0: 0.1}, cuda_dev)
    with pytest.raises(pkg.core.P6DError, match="at most"):
        crit.eval_metrics(*d)
    crit.large_meshes = True
    m = crit.eval_metrics(*d)
    ref = oracle.eval_metrics(oracle.MeshTable({0: mesh}, {0: 0.1}), pq, pt, gq, gt, obj,
                              n_threads=oracle.max_threads())
    assert {k: repr(v) for k, v in m.items()} == {k: repr(v) for k, v in ref.items()}
    # put pose 0 on its threshold: the kernel flags it and the hook decides
    add0 = crit.eval_poses(*d)["add"][0]
    crit.diameters[0] = float(add0) * 10.0
    calls = []
    crit.borderline_resolver = lambda idx, *a: (calls.append(list(idx)), [1] * len(idx))[1]
    crit.eval_metrics(*d)
    assert calls and 0 in calls[0]
    with pytest.raises(pkg.core.P6DError, match="at most"):
        crit(d[0], d[1], d[2], d[3], d[4])
    # host entry: per-object totals
    pts = {0: mesh, 9: W.box_mesh(9000, (0.1, 0.12, 0.05), 52)}
    table = pkg.core.MeshTable(pts, {0: 0.1, 9: 0.16}, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev).set_large_meshes(True)
    obj2 = np.where(np.arange(24) % 2 == 0, 0, 9).astype(np.int64)
    h = table.evaluate_host(pq, pt, gq, gt, obj2)
    for o in (0, 9):
        k = obj2 == o
        assert h["obj_valid"][o] == int(h["valid"][k].sum()) and h["obj_hits"][o] == int(h["hit"][k].sum())
        assert np.isclose(h["obj_add_sum"][o], h["add"][k].astype(np.float64).sum(), rtol=1e-12, atol=0)
        assert np.isclose(h["obj_adds_sum"][o], h["adds"][k].astype(np.float64).sum(), rtol=1e-12, atol=0)
    huge = pkg.core.MeshTable({0: W.sphere_mesh(32769, 0.1, 53)}, {0: 0.1}, pkg.SYMMETRIC_OBJECT_IDS,
                              cuda_dev).set_large_meshes(True)
    with pytest.raises(pkg.core.P6DError, match="at most 32768 points.*thread count"):
        huge.evaluate_packed(*d)
    with pytest.raises(pkg.core.P6DError, match="at most 32768 points"):
        huge.evaluate_packed(*d, streamed=True)


@pytest.mark.gpu
def test_switches_and_callers(pkg, cuda_dev, W, oracle):
    """Switch off, on, and with exact pruning: the same bytes wherever both run; PoseEvaluator and evaluate_sweep
    with large_meshes=True give hit tables equal to the oracle's per-pose decisions on the same hypotheses."""
    pts, dia, table = table_of(pkg, W, (3000, 700), cuda_dev)
    B = 2000
    pq, pt, gq, gt = edge_poses(W, B, 60, np.geomspace(0.005, 0.5, B))
    obj = np.array(sorted(pts) + [-1], np.int64)[np.random.RandomState(61).randint(0, 3, B)]
    d = [T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)]
    base = table.evaluate_packed(*d)[:11 * B].clone()
    table.set_large_meshes(True)
    assert torch.equal(base, table.evaluate_packed(*d)[:11 * B])
    table.set_pruning(True)
    assert torch.equal(base, table.evaluate_packed(*d)[:11 * B])
    table.set_large_meshes(False)
    assert torch.equal(base, table.evaluate_packed(*d)[:11 * B])
    # beyond the resident limit, both switches on: the streamed kernel
    big_pts, big_dia, big = table_of(pkg, W, (9000, 2000), cuda_dev)
    forced = big.evaluate_packed(*d, streamed=True)[:11 * B].clone()
    big.set_pruning(True)
    big.set_large_meshes(True)
    assert torch.equal(forced, big.evaluate_packed(*d)[:11 * B])

    # callers on one 8,192-point object
    mpts = {9: W.box_mesh(8192, (0.1, 0.12, 0.05), 62)}
    mdia = {9: 0.16}
    ot = oracle.MeshTable(mpts, mdia)
    ev = pkg.PoseEvaluator(mpts, mdia, cuda_dev, large_meshes=True)
    pq, pt, gq, gt = W.random_poses(96, 63, rot_sigma=np.geomspace(0.005, 0.3, 96))
    o9 = np.full(96, 9, np.int64)
    ev.evaluate(pq, pt, gq, gt, torch.from_numpy(o9))
    ref = oracle.add_eval(ot, pq, pt, gq, gt, o9, n_threads=oracle.max_threads())
    assert int(ev.acc.hits[0, 9]) == int(ref[2].sum()) and int(ev.acc.valid[0, 9]) == 96
    n = 24
    acc, _, check = pkg.evaluate_sweep(mpts, mdia, cuda_dev, n, seed=64, check_n=n, large_meshes=True)
    hits = acc.hits.cpu().numpy()
    for v in range(len(pkg.sweep.VARIANTS)):
        r = oracle.add_eval(ot, check["pq"][v], check["pt"][v], check["gq"][v], check["gt"][v], check["obj"][v],
                            n_threads=oracle.max_threads())
        assert np.array_equal(check["hit"][v], r[2]) and int(hits[v, 9]) == int(r[2].sum())


@pytest.mark.gpu
def test_two_streams_on_one_large_table(pkg, cuda_dev, W):
    """Re-entrant per device: the same large table evaluated on two streams at once gives the bytes of the
    sequential calls (each call has its own stream-ordered workspace)."""
    pts, dia, table = table_of(pkg, W, (8192, 12000), cuda_dev)
    table.set_large_meshes(True)
    batches = []
    for seed in (70, 71):
        pq, pt, gq, gt = W.random_poses(600, seed, rot_sigma=0.1)
        obj = np.array(sorted(pts), np.int64)[np.arange(600) % 2]
        batches.append([T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)])
    seq = [table.evaluate_packed(*b)[:6600].clone() for b in batches]
    torch.cuda.synchronize(cuda_dev)
    streams = [torch.cuda.Stream(cuda_dev), torch.cuda.Stream(cuda_dev)]
    outs = [None, None]
    for i, s in enumerate(streams):
        with torch.cuda.stream(s):
            outs[i] = table.evaluate_packed(*batches[i])
    torch.cuda.synchronize(cuda_dev)
    for i in range(2):
        assert torch.equal(seq[i], outs[i][:6600])
