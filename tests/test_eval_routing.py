"""Which kernel evaluates each call (csrc/p6d_add.cu, launch_eval).

Wherever two evaluation kernels can run a call they return the same bytes, so no output test can see the route: a
call that took another kernel than intended would only be slower.  Each case here runs its call once under
torch.profiler and names the libp6d kernels that ran.  Every call is made once before it is profiled, so the
one-time self-check of the re-laid ADD-S kernels (which launches both schedules) is not in the profile.
"""
import re

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

pytestmark = pytest.mark.gpu

# resident ADD-S kernel (b) per mesh-size class (N <= 512, <= 1024, larger): (ptxas schedule, re-laid schedule)
RESIDENT = [("adds_cta_kernel<128,4,8,2,0>", "adds_cta_kernel<128,4,8,0,0>"),
            ("adds_cta_kernel<256,4,4,2,0>", "adds_cta_kernel<256,4,4,0,0>"),
            ("adds_cta_kernel<512,4,2,2,0>", "adds_cta_kernel<256,8,2,0,0>")]
LOSS = ["adds_cta_kernel<128,4,8,2,1>", "adds_cta_kernel<256,4,4,2,1>", "adds_cta_kernel<512,4,2,2,1>"]
PRUNED = r"adds_pruned_kernel<\d+,\d+>"
STREAMED = r"adds_streamed_kernel<\d+,\d+,true>"
STREAMED_ADD_ONLY = r"adds_streamed_kernel<\d+,\d+,false>"


def launched(fn):
    """Evaluation kernels (template arguments without spaces) that one call of fn launches."""
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        m = re.search(r"p6d::(\w+<[^>]*>)", e.name)
        if m and m.group(1).startswith(("adds_", "add_pose_kernel")):
            names.add(re.sub(r"\s", "", m.group(1)))
    return sorted(names)


def routed(fn):
    fn()
    return launched(fn)


def refused(pkg, fn, match):
    def call():
        with pytest.raises(pkg.core.P6DError, match=match):
            fn()
    return launched(call)


def one_of(names, pattern):
    return len(names) == 1 and re.fullmatch(pattern, names[0]) is not None


def resident(table):
    """The resident variant this table's launches take, by its mesh-size class and schedule state."""
    cls = 0 if table.max_count <= 512 else (1 if table.max_count <= 1024 else 2)
    st = table.schedule_state()
    return [RESIDENT[cls][1 if st["built_relaid"] == 1 and st["runtime_state"] == 1 else 0]]


def adds_max_points(pkg, dev):
    n = pkg.core.C.c_int()
    pkg.core.check(pkg.core.lib().p6d_adds_max_points(dev.index, pkg.core.C.byref(n)))
    return n.value


def table(pkg, W, sizes, dev):
    pts = {oid: W.box_mesh(n, (0.1, 0.12, 0.05), 300 + n) for oid, n in sizes.items()}
    return pkg.core.MeshTable(pts, {oid: 0.16 for oid in sizes}, pkg.SYMMETRIC_OBJECT_IDS, dev), pts


def poses(W, ids, dev, B=256, seed=7):
    pq, pt, gq, gt = W.random_poses(B, seed, rot_sigma=0.1)
    obj = np.array(sorted(ids), np.int64)[np.arange(B) % len(ids)]
    return [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in (pq, pt, gq, gt, obj)]


def test_default_route_and_pruning_switch(pkg, cuda_dev, W):
    """Switches off: the resident kernel.  Pruning on: the pruned kernel from 128 points up to its own shared-memory
    limit, the resident kernel below and beyond that."""
    t500, _ = table(pkg, W, {9: 500}, cuda_dev)
    d = poses(W, {9}, cuda_dev)
    assert routed(lambda: t500.evaluate_packed(*d)) == resident(t500)
    t500.set_pruning(True)
    assert one_of(routed(lambda: t500.evaluate_packed(*d)), PRUNED)
    t100, _ = table(pkg, W, {9: 100}, cuda_dev)
    t100.set_pruning(True)
    assert routed(lambda: t100.evaluate_packed(*d)) == resident(t100)
    assert 6000 <= adds_max_points(pkg, cuda_dev)
    t6000, _ = table(pkg, W, {9: 6000}, cuda_dev)
    assert refused(pkg, lambda: t6000.evaluate_packed(*d, prune=True), "pruned ADD-S kernel.*at most") == []
    t6000.set_pruning(True)
    assert routed(lambda: t6000.evaluate_packed(*d)) == resident(t6000)


def test_large_meshes_switch(pkg, cuda_dev, W):
    """Large meshes on: the streamed kernel only beyond the resident kernel's limit, also with pruning on; the loss
    form never takes it."""
    d = poses(W, {9}, cuda_dev, B=64)
    t6000, _ = table(pkg, W, {9: 6000}, cuda_dev)
    t6000.set_large_meshes(True)
    assert routed(lambda: t6000.evaluate_packed(*d)) == resident(t6000)
    big, _ = table(pkg, W, {9: adds_max_points(pkg, cuda_dev) + 1}, cuda_dev)
    assert refused(pkg, lambda: big.evaluate_packed(*d), "at most") == []
    big.set_large_meshes(True)
    assert one_of(routed(lambda: big.evaluate_packed(*d)), STREAMED)
    big.set_pruning(True)
    assert one_of(routed(lambda: big.evaluate_packed(*d)), STREAMED)
    assert refused(pkg, lambda: big.forward_loss(*d), "at most") == []


def test_add_only_route(pkg, cuda_dev, W):
    """Without ADD-S: the ADD-only kernel (its one-mesh form for a table of one mesh); beyond its shared memory the
    streamed kernel without ADD-S when large meshes are on, the ADD-only kernel's refusal otherwise."""
    one, _ = table(pkg, W, {9: 500}, cuda_dev)
    one.set_pruning(True).set_large_meshes(True)
    d = poses(W, {9}, cuda_dev)
    assert routed(lambda: one.evaluate_packed(*d, want_adds=False)) == ["add_pose_kernel<true>"]
    two, _ = table(pkg, W, {1: 300, 9: 500}, cuda_dev)
    d2 = poses(W, {1, 9}, cuda_dev)
    assert routed(lambda: two.evaluate_packed(*d2, want_adds=False)) == ["add_pose_kernel<false>"]
    t20k, _ = table(pkg, W, {9: 20000}, cuda_dev)
    d = poses(W, {9}, cuda_dev, B=32)
    assert refused(pkg, lambda: t20k.evaluate_packed(*d, want_adds=False), "ADD kernel.*at most") == []
    t20k.set_large_meshes(True)
    assert one_of(routed(lambda: t20k.evaluate_packed(*d, want_adds=False)), STREAMED_ADD_ONLY)


def test_loss_form_and_explicit_entries(pkg, cuda_dev, W):
    """ADDLoss.forward's value takes the loss form of the resident kernel with both switches on; the explicit
    pruned and streamed entries take their kernel whatever the switches say."""
    t500, _ = table(pkg, W, {9: 500}, cuda_dev)
    d = poses(W, {9}, cuda_dev)
    assert one_of(routed(lambda: t500.evaluate_packed(*d, prune=True)), PRUNED)
    assert one_of(routed(lambda: t500.evaluate_packed(*d, streamed=True)), STREAMED)
    t500.set_pruning(True).set_large_meshes(True)
    assert routed(lambda: t500.forward_loss(*d)) == [LOSS[0]]


def test_host_entry_evaluator_and_sweep_take_the_pruned_kernel(pkg, cuda_dev, W):
    t500, pts = table(pkg, W, {9: 500}, cuda_dev)
    t500.set_pruning(True)
    h = [x.cpu().numpy() for x in poses(W, {9}, cuda_dev)]
    assert one_of(routed(lambda: t500.evaluate_host(*h)), PRUNED)
    ev = pkg.PoseEvaluator(pts, {9: 0.16}, cuda_dev, exact_pruning=True)
    assert one_of(routed(lambda: ev.evaluate(h[0], h[1], h[2], h[3], torch.from_numpy(h[4]))), PRUNED)
    assert one_of(routed(lambda: pkg.evaluate_sweep(pts, {9: 0.16}, cuda_dev, 64, exact_pruning=True)), PRUNED)


def test_pruning_refused_without_block_structure(pkg, cuda_dev, W):
    """A mesh of more than 65,534 points has no block structure: the switch is refused and nothing is launched."""
    huge = pkg.core.MeshTable({9: W.sphere_mesh(65535, 0.1, 5)}, {9: 0.16}, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev)
    assert refused(pkg, lambda: huge.set_pruning(True), "no block structure") == []
