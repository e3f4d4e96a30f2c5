"""Exact block pruning beyond shared memory: the streamed pruned ADD-S kernel (csrc/p6d_adds_pruned.cu, kernel
b'''), opt-in per table (MeshTable.set_large_mesh_pruning, ADDLoss.large_mesh_pruning).

It must return the bytes of every other evaluation kernel: against the streamed kernel at every size up to 32,768
points, against the resident all-pairs and pruned kernels where they run, and against the oracle beyond them.  The
route is checked with torch.profiler kernel names, as in tests/test_eval_routing.py.
"""
import re
import threading

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from conftest import same_bits

pytestmark = pytest.mark.gpu

SIGMAS = np.array([0.002, 0.02, 0.1, 0.5, 3.0])
NEW = {"adds_pruned_streamed_xform_kernel<256>", "adds_pruned_streamed_kernel<256,3>"}
STREAMED = r"adds_streamed_kernel<\d+,\d+,true>"
PRUNED = r"adds_pruned_kernel<\d+,\d+>"


def T(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def adds_max_points(pkg, dev):
    n = pkg.core.C.c_int()
    pkg.core.check(pkg.core.lib().p6d_adds_max_points(dev.index, pkg.core.C.byref(n)))
    return n.value


def mesh(W, kind, n, seed):
    q = np.random.RandomState(seed)
    if kind == "sphere": return W.sphere_mesh(n, 0.15, seed)
    if kind == "box": return W.box_mesh(n, (0.1, 0.12, 0.05), seed)
    if kind == "blob": return (q.standard_normal((n, 3)) * 0.03).astype(np.float32)
    if kind == "patch": return np.c_[q.uniform(-0.05, 0.05, (n, 2)), q.standard_normal(n) * 1e-4].astype(np.float32)
    if kind == "rod": return np.c_[q.uniform(-0.1, 0.1, n), q.standard_normal((n, 2)) * 1e-3].astype(np.float32)
    if kind == "clusters":
        c = (q.rand(n) < 0.5)[:, None] * np.array([[0.3, 0.0, 0.0]])
        return (c + q.standard_normal((n, 3)) * 0.01).astype(np.float32)
    if kind == "dups":
        base = q.standard_normal((max(n // 16, 1), 3)) * 0.04
        return base[q.randint(0, len(base), n)].astype(np.float32)
    if kind == "coincident": return np.tile(np.array([[0.01, -0.02, 0.03]], np.float32), (n, 1))
    if kind == "nan":
        m = W.sphere_mesh(n, 0.15, seed).copy()
        m[n // 2, 1] = np.nan
        return m
    raise ValueError(kind)


def edge_poses(W, B, seed):
    """Rotation errors cycling through SIGMAS, then NaN, inf, zero and non-unit quaternions, a NaN translation and
    pred == gt in the first rows."""
    pq, pt, gq, gt = W.random_poses(B, seed, rot_sigma=SIGMAS[np.arange(B) % len(SIGMAS)])
    if B >= 10:
        pq[3] = gq[3]; pt[3] = gt[3]
        pt[4, 0] = np.nan
        pq[5] = np.nan
        pt[6, 2] = np.inf
        pq[7] *= 3.0
        pq[8] = 0.0
        gq[9] *= 1e-3
    return pq, pt, gq, gt


def accumulators(n_slots, dev):
    return [torch.zeros(n_slots, dtype=torch.int64, device=dev), torch.zeros(n_slots, dtype=torch.int64, device=dev),
            torch.zeros(n_slots, dtype=torch.float64, device=dev), torch.zeros(n_slots, dtype=torch.float64, device=dev)]


def same_accumulators(a, b):
    return (torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
            and torch.allclose(a[2], b[2], rtol=1e-12, atol=0, equal_nan=True)
            and torch.allclose(a[3], b[3], rtol=1e-12, atol=0, equal_nan=True))


def compare(table, d, dev, other, both_orders=True):
    """The forced new entry against `other` (keyword arguments of evaluate_packed): all 11 bytes per pose and the
    accumulators, in index order and in object order."""
    B = d[4].shape[0]
    orders = [None, torch.argsort(d[4], stable=True).to(torch.int32)] if both_orders else [None]
    for o in orders:
        acc_n, acc_o = accumulators(table.n_slots, dev), accumulators(table.n_slots, dev)
        new = table.evaluate_packed(*d, order=o, acc=acc_n, prune_streamed=True)[:11 * B]
        ref = table.evaluate_packed(*d, order=o, acc=acc_o, **other)[:11 * B]
        assert torch.equal(new, ref), (table.max_count, o is None, other)
        assert same_accumulators(acc_n, acc_o), (table.max_count, o is None, other)


def batch(W, ids, B, seed, dev):
    pq, pt, gq, gt = edge_poses(W, B, seed)
    obj = np.asarray(ids, np.int64)[np.random.RandomState(seed).randint(0, len(ids), B)]
    return [T(x, dev) for x in (pq, pt, gq, gt, obj)]


# ----------------------------------------------------------------------------------------------- bytes
@pytest.mark.parametrize("n", [1, 5, 8, 31, 32, 33, 128, 500, 2048, "nmax-1", "nmax+1", 8192, 12345, 16384, 32767,
                               32768])
def test_equals_streamed_over_sizes(pkg, cuda_dev, W, n):
    """Sphere and box meshes of n points (and a smaller third object), ids without a mesh, every rotation error of
    SIGMAS with the degenerate poses, both processing orders."""
    nmax = adds_max_points(pkg, cuda_dev)
    n = {"nmax-1": nmax - 1, "nmax+1": nmax + 1}.get(n, n)
    pts = {9: mesh(W, "box", n, 900 + n), 1: mesh(W, "sphere", n, 1000 + n), 4: mesh(W, "sphere", n // 3 + 1, 7)}
    table = pkg.core.MeshTable(pts, {9: 0.16, 1: 0.1, 4: 0.17}, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev)
    d = batch(W, [9, 1, 4, -1, 2, 12], 60, n, cuda_dev)
    compare(table, d, cuda_dev, {"streamed": True})


@pytest.mark.parametrize("kind", ["sphere", "box", "blob", "patch", "rod", "clusters", "dups", "coincident", "nan"])
def test_equals_streamed_over_mesh_families(pkg, cuda_dev, W, kind):
    for n in (700, 8192, 32768):
        pts = {3: mesh(W, kind, n, 7 * n + len(kind)), 9: mesh(W, kind, max(n - 37, 1), 11 * n)}
        table = pkg.core.MeshTable(pts, {3: 0.1, 9: 0.1}, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev)
        d = batch(W, [3, 9], 40, n + len(kind), cuda_dev)
        compare(table, d, cuda_dev, {"streamed": True}, both_orders=n == 8192)


def test_mixed_table_and_batch_sizes(pkg, cuda_dev, W):
    """A table of 32,768 + 100 + 5 points; B = 0, 1, 16 and a batch that spans several 64 MB workspace chunks (about
    90 poses of 32,768 points each)."""
    pts = {2: mesh(W, "sphere", 32768, 1), 5: mesh(W, "box", 100, 2), 11: mesh(W, "blob", 5, 3)}
    table = pkg.core.MeshTable(pts, {2: 0.15, 5: 0.16, 11: 0.05}, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev)
    d = batch(W, [2, 5, 11, -3, 7], 16, 40, cuda_dev)
    compare(table, d, cuda_dev, {"streamed": True})
    d1 = [x[:1] for x in d]
    compare(table, d1, cuda_dev, {"streamed": True})
    d0 = [x[:0] for x in d]
    assert table.evaluate_packed(*d0, prune_streamed=True).numel() == 16
    big = batch(W, [2], 200, 41, cuda_dev)
    compare(table, big, cuda_dev, {"streamed": True}, both_orders=False)


@pytest.mark.parametrize("n", [500, 2048, 4096, 6000, "nmax"])
def test_equals_resident_kernels(pkg, cuda_dev, W, n):
    """Where the resident kernels run: the all-pairs kernel always, the pruned kernel up to its own limit (the band
    between the two limits included)."""
    n = adds_max_points(pkg, cuda_dev) if n == "nmax" else n
    pts = {9: mesh(W, "box", n, 300 + n), 1: mesh(W, "sphere", n - 17, 301 + n)}
    table = pkg.core.MeshTable(pts, {9: 0.16, 1: 0.1}, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev)
    d = batch(W, [9, 1, -1], 200, n, cuda_dev)
    compare(table, d, cuda_dev, {})
    try:
        table.evaluate_packed(*d, prune=True)
    except pkg.core.P6DError as e:
        assert n > 4096 and "at most" in str(e)
    else:
        compare(table, d, cuda_dev, {"prune": True})


@pytest.mark.parametrize("n", ["nmax+1", 16384, 32768])
def test_beyond_the_resident_limit_equals_the_oracle(pkg, cuda_dev, W, oracle, n):
    nmax = adds_max_points(pkg, cuda_dev)
    n = nmax + 1 if n == "nmax+1" else n
    pts = {9: mesh(W, "box", n, 900 + n), 1: mesh(W, "sphere", n, 1000 + n), 10: mesh(W, "nan", n // 3 + 1, 77)}
    dia = {9: 0.16, 1: 0.1, 10: 0.17}
    table = pkg.core.MeshTable(pts, dia, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev).set_large_mesh_pruning(True)
    B = 120
    pq, pt, gq, gt = edge_poses(W, B, n)
    obj = np.array([9, 1, 10, -1], np.int64)[np.random.RandomState(n).randint(0, 4, B)]
    d = [T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)]
    out = table.evaluate_packed(*d).cpu().numpy()
    sel = np.r_[np.arange(10), np.random.RandomState(n + 1).choice(np.arange(10, B), 8, replace=False)]
    ref = oracle.add_eval(oracle.MeshTable(pts, dia), pq[sel], pt[sel], gq[sel], gt[sel], obj[sel],
                          n_threads=oracle.max_threads())
    assert same_bits(out[:4 * B].view(np.float32)[sel], ref[0])
    assert same_bits(out[4 * B:8 * B].view(np.float32)[sel], ref[1])
    assert np.array_equal(out[8 * B:9 * B][sel], ref[2]) and np.array_equal(out[9 * B:10 * B][sel], ref[3])


# ----------------------------------------------------------------------------------------------- routing
def launched(fn, done=bool, tries=6):
    """libp6d evaluation kernels that calls of fn launch.  A CUDA trace can come back without some kernel records,
    never with records of kernels that did not run; so each profile covers three calls of fn, and profiles are taken
    until done(names seen so far) holds, at most `tries` times.  The union is returned, so a kernel that must not run
    is looked for in every record collected."""
    fn()
    torch.cuda.synchronize()
    names = set()
    for _ in range(tries):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
        for e in prof.events():
            m = re.search(r"p6d::(\w+<[^>]*>)", e.name)
            if m and m.group(1).startswith(("adds_", "add_pose_kernel")):
                names.add(re.sub(r"\s", "", m.group(1)))
        if done(names):
            break
    return names


def new_kernels(fn):
    return launched(fn, lambda names: NEW <= names)


def refused(pkg, fn, match):
    def call():
        with pytest.raises(pkg.core.P6DError, match=match):
            fn()
    return launched(call, tries=1)


def only(names, pattern):
    return len(names) == 1 and re.fullmatch(pattern, next(iter(names))) is not None


def table(pkg, W, n, dev):
    return pkg.core.MeshTable({9: W.box_mesh(n, (0.1, 0.12, 0.05), 300 + n)}, {9: 0.16}, pkg.SYMMETRIC_OBJECT_IDS, dev)


def poses(W, dev, B=64):
    pq, pt, gq, gt = W.random_poses(B, 7, rot_sigma=0.1)
    return [T(x, dev) for x in (pq, pt, gq, gt, np.full(B, 9, np.int64))]


def test_routing(pkg, cuda_dev, W):
    nmax = adds_max_points(pkg, cuda_dev)
    d = poses(W, cuda_dev)
    t500, t6000, tbig, t32k, t100 = (table(pkg, W, n, cuda_dev) for n in (500, 6000, nmax + 1, 32768, 100))
    # switch off, every other switch on: today's kernels
    for t in (t500, t6000, tbig):
        t.set_pruning(True).set_large_meshes(True)
    assert only(launched(lambda: t500.evaluate_packed(*d)), PRUNED)
    off6000 = launched(lambda: t6000.evaluate_packed(*d))
    assert len(off6000) == 1 and next(iter(off6000)).startswith("adds_cta_kernel<")
    assert only(launched(lambda: tbig.evaluate_packed(*d)), STREAMED)
    # switch on: the new kernel beyond the pruned kernel's shared memory
    for t in (t500, t6000, tbig, t32k, t100):
        t.set_large_mesh_pruning(True)
    assert new_kernels(lambda: t6000.evaluate_packed(*d)) == NEW
    assert new_kernels(lambda: tbig.evaluate_packed(*d)) == NEW
    assert new_kernels(lambda: t32k.evaluate_packed(*d)) == NEW
    # unchanged with the switch on: the pruned route, the resident route, ADD only and the loss form
    assert only(launched(lambda: t500.evaluate_packed(*d)), PRUNED)
    res100 = launched(lambda: t100.evaluate_packed(*d))
    assert len(res100) == 1 and next(iter(res100)).startswith("adds_cta_kernel<")
    assert launched(lambda: t6000.evaluate_packed(*d, want_adds=False)) == {"add_pose_kernel<true>"}
    loss = launched(lambda: t6000.forward_loss(*d))
    assert len(loss) == 1 and re.fullmatch(r"adds_cta_kernel<\d+,\d+,\d+,\d+,1>", next(iter(loss)))
    # the forced entry takes the new kernel at any size
    assert new_kernels(lambda: t100.evaluate_packed(*d, prune_streamed=True)) == NEW
    # 32,769 points: refused with the streamed kernel's reason, nothing launched
    t32769 = table(pkg, W, 32769, cuda_dev).set_large_mesh_pruning(True)
    assert refused(pkg, lambda: t32769.evaluate_packed(*d), "at most 32768 points.*thread count") == set()
    assert refused(pkg, lambda: t32769.evaluate_packed(*d, prune_streamed=True), "at most 32768") == set()
    # no block structure: the switch is refused, switching it off is fine
    huge = pkg.core.MeshTable({9: W.sphere_mesh(65535, 0.1, 5)}, {9: 0.16}, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev)
    assert refused(pkg, lambda: huge.set_large_mesh_pruning(True), "no block structure") == set()
    huge.set_large_mesh_pruning(False)
    with pytest.raises(pkg.core.P6DError, match="no block structure"):
        huge.evaluate_packed(*d, prune_streamed=True)


# ----------------------------------------------------------------------------------------------- surfaces
def test_addloss_evaluator_sweep_and_host_entry(pkg, cuda_dev, W):
    import tempfile
    m = mesh(W, "sphere", 16384, 50)
    pq, pt, gq, gt = edge_poses(W, 40, 51)
    obj = np.zeros(40, np.int64)
    obj[11] = 4
    d = [T(x, cuda_dev) for x in (pq, pt, gq, gt, obj)]
    crit = pkg.ADDLoss(tempfile.mkdtemp(), cuda_dev)
    crit.points[0] = T(m, cuda_dev)
    crit.diameters[0] = 0.15
    crit.large_meshes = True
    ref_m, ref_p = crit.eval_metrics(*d), crit.eval_poses(*d)
    crit.large_mesh_pruning = True
    assert new_kernels(lambda: crit.eval_metrics(*d)) == NEW
    got_m, got_p = crit.eval_metrics(*d), crit.eval_poses(*d)
    assert {k: repr(v) for k, v in got_m.items()} == {k: repr(v) for k, v in ref_m.items()}
    for k in ref_p:
        a, b = np.asarray(ref_p[k].cpu() if torch.is_tensor(ref_p[k]) else ref_p[k]), \
            np.asarray(got_p[k].cpu() if torch.is_tensor(got_p[k]) else got_p[k])
        assert a.tobytes() == b.tobytes(), k
    crit.large_meshes = False          # the new switch alone takes the call
    assert {k: repr(v) for k, v in crit.eval_metrics(*d).items()} == {k: repr(v) for k, v in ref_m.items()}

    pts, dia = {9: mesh(W, "box", 8192, 62)}, {9: 0.16}
    hq = W.random_poses(96, 63, rot_sigma=np.geomspace(0.005, 0.3, 96))
    o9 = torch.from_numpy(np.full(96, 9, np.int64))
    ev_s = pkg.PoseEvaluator(pts, dia, cuda_dev, large_meshes=True)
    ev_p = pkg.PoseEvaluator(pts, dia, cuda_dev, large_mesh_pruning=True)
    ev_s.evaluate(*hq, o9)
    ev_p.evaluate(*hq, o9)
    assert torch.equal(ev_s.acc.hits, ev_p.acc.hits) and torch.equal(ev_s.acc.valid, ev_p.acc.valid)
    acc_s = pkg.evaluate_sweep(pts, dia, cuda_dev, 32, seed=64, large_meshes=True)[0]
    acc_p = pkg.evaluate_sweep(pts, dia, cuda_dev, 32, seed=64, large_mesh_pruning=True)[0]
    assert torch.equal(acc_s.hits, acc_p.hits) and torch.equal(acc_s.valid, acc_p.valid)

    table = pkg.core.MeshTable({**pts, 1: mesh(W, "sphere", 6000, 64)}, {9: 0.16, 1: 0.1}, pkg.SYMMETRIC_OBJECT_IDS,
                               cuda_dev)
    o2 = np.where(np.arange(96) % 2 == 0, 9, 1).astype(np.int64)
    h_ref = table.set_large_meshes(True).evaluate_host(*hq, o2)
    h_new = table.set_large_mesh_pruning(True).evaluate_host(*hq, o2)
    for k in ("add", "adds", "hit", "valid", "borderline", "obj_hits", "obj_valid"):
        assert np.array_equal(h_ref[k], h_new[k]), k
    assert np.allclose(h_ref["obj_adds_sum"], h_new["obj_adds_sum"], rtol=1e-12, atol=0)


def test_two_threads_two_streams_and_repeated_calls(pkg, cuda_dev, W):
    pts = {9: mesh(W, "box", 12000, 70), 1: mesh(W, "sphere", 8192, 71)}
    table = pkg.core.MeshTable(pts, {9: 0.16, 1: 0.1}, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev).set_large_mesh_pruning(True)
    batches = [batch(W, [9, 1], 300, seed, cuda_dev) for seed in (72, 73)]
    seq = [table.evaluate_packed(*b, streamed=True)[:3300].clone() for b in batches]
    for _ in range(3):
        for i, b in enumerate(batches):
            assert torch.equal(seq[i], table.evaluate_packed(*b)[:3300])
    torch.cuda.synchronize(cuda_dev)
    outs = [None, None]

    def run(i):
        s = torch.cuda.Stream(cuda_dev)
        with torch.cuda.stream(s):
            for _ in range(3):
                outs[i] = table.evaluate_packed(*batches[i])
        s.synchronize()

    threads = [threading.Thread(target=run, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for i in range(2):
        assert torch.equal(seq[i], outs[i][:3300])
