"""Live pins: the rounding rules the kernels and the C oracle rely on, re-checked against the PyTorch
build of THE MACHINE THE TESTS RUN ON (build container for the CPU suite, the B200 box for -m gpu).

The golden vectors were produced in the build container (torch 2.11.0, MKL, AVX-512).  They pin the
oracle to the reference there -- not to the ATen / MKL of another box.  These tests run the
reference's own op sequence (oracle/torch_eager.py: torch.mm / matmul / norm / min / mean on the
local CPU, no rounding rule built in) next to the oracle and next to the GPU:

  * a rule that does not hold on this machine fails here, by name, instead of surfacing as a
    one-ulp difference somewhere in a sweep;
  * on the GPU box, the kernels are compared with what the reference's ops give ON THAT BOX.
"""
import numpy as np
import pytest
import torch

from conftest import bits, golden_meshes, load_golden, same_bits

SIZES_MM = [1, 2, 3, 5, 10, 11, 12, 31, 44, 45, 100, 500, 1000, 2048]
GOLDEN_EVAL_CASES = ["eval_cfg1", "eval_cfg1_mixed", "eval_cfg2_subset", "eval_ragged", "eval_default_diameter",
                     "eval_degenerate"]


@pytest.fixture(scope="module")
def eager():
    from oracle import torch_eager
    return torch_eager


def _poses(W, B, seed):
    pq, pt, gq, gt = W.random_poses(B, seed, rot_sigma=np.geomspace(0.01, 0.3, B), trans_sigma=0.01)
    return pq, pt, gq, gt


@pytest.mark.parametrize("n", SIZES_MM)
def test_torch_mm_rounds_as_the_oracle_says(oracle, eager, W, n):
    """torch.mm([n,3],[3,3]) + t: n = 1 and 2..10 take unfused small-matrix kernels, n >= 11 the FMA
    chain (oracle p6o_xform_point; kernels: xform_coord<MODE>)."""
    mesh = W.sphere_mesh(n, 0.15, 400 + n)
    pq, pt, _, _ = _poses(W, 4, 500 + n)
    for q, t in zip(pq, pt):
        R = eager.quat_to_mat(torch.from_numpy(q[None]))[0]
        got = (torch.mm(torch.from_numpy(mesh), R.T) + torch.from_numpy(t)).numpy()
        assert same_bits(got, oracle.transform(mesh, q, t)), f"torch.mm rounding rule changed for n = {n}"
        assert same_bits(R.numpy(), oracle.quat_to_mat(q[None])[0])


@pytest.mark.parametrize("n", [1, 7, 8, 31, 32, 33, 100, 500, 512, 1000, 2048, 4097])
def test_tensor_mean_sums_in_the_oracles_order(oracle, n):
    x = (np.random.RandomState(n).rand(n) * 0.02 + 1e-4).astype(np.float32)
    t = torch.from_numpy(x)
    assert bits(oracle.aten_mean(x)) == bits(np.float32(t.mean().item()))
    assert bits(oracle.aten_sum(x)) == bits(np.float32(t.sum().item()))
    # a row of a [k, n] tensor reduced along dim 1 sums in the same order (ADDLoss.forward's mean(dim=1))
    m = torch.from_numpy(np.stack([x, x[::-1].copy(), x * 0.5]))
    assert bits(oracle.aten_mean(x[::-1].copy())) == bits(np.float32(m.mean(dim=1)[1].item()))


@pytest.mark.parametrize("n", [3, 8, 64, 500, 1000])
def test_torch_norm_rounds_as_the_oracle_says(oracle, eager, W, n):
    """torch.norm(v, dim=-1) over 3 components = sqrt(fma(z,z,fma(y,y,x*x))); checked through the ADD of a
    pose whose mean has a single term per lane pattern: every per-point distance enters the comparison."""
    mesh = W.sphere_mesh(n, 0.1, 600 + n)
    pq, pt, gq, gt = _poses(W, 3, 700 + n)
    for i in range(3):
        cp = oracle.transform(mesh, pq[i], pt[i])
        cg = oracle.transform(mesh, gq[i], gt[i])
        d = torch.norm(torch.from_numpy(cp) - torch.from_numpy(cg), dim=1, p=2).numpy()
        dx = (cp - cg).astype(np.float64)
        # fma chain in exact arithmetic: float64 holds x*x + y*y exactly enough to emulate one rounding per fma
        s = np.float32(dx[:, 0] * dx[:, 0]).astype(np.float64)
        s = np.float32(dx[:, 1] * dx[:, 1] + s).astype(np.float64)
        s = np.float32(dx[:, 2] * dx[:, 2] + s)
        assert same_bits(d, np.sqrt(s.astype(np.float64)).astype(np.float32))


@pytest.mark.parametrize("n", [1, 2, 9, 10, 11, 37, 100, 500, 777, 1000])
def test_reference_op_sequence_equals_the_oracle_on_this_machine(oracle, eager, W, n):
    """The whole per-pose chain -- torch.mm, +, -, norm, min, mean, float64 threshold -- executed by
    the local PyTorch against the C restatement: ADD, ADD-S and the decision, bit for bit."""
    pts = {3: W.sphere_mesh(n, 0.12, 800 + n), 9: W.box_mesh(n, (0.1, 0.12, 0.05), 900 + n)}
    dia = {3: 0.12, 9: 0.16}
    B = 6 if n >= 500 else 12
    pq, pt, gq, gt = _poses(W, B, 1000 + n)
    obj = np.array([3, 9] * (B // 2), np.int64)
    obj[-1] = 5                                              # id without a mesh
    ref = eager.eval_poses(pts, dia, pq, pt, gq, gt, obj)
    got = oracle.add_eval(oracle.MeshTable(pts, dia), pq, pt, gq, gt, obj, n_threads=4)
    assert same_bits(got[0], ref[0]) and same_bits(got[1], ref[1])
    assert np.array_equal(got[2], ref[2]) and np.array_equal(got[3], ref[3])


def test_batched_matmul_rule_of_the_loss_form(oracle, eager, W):
    """ADDLoss.forward's torch.matmul([1,n,3],[B,3,3]): naive bmm kernel for n <= 44, FMA chain above
    (group sizes other than 2, where MKL's batched sgemm was seen to differ for some n)."""
    pts = {0: W.sphere_mesh(5, 0.1, 1), 1: W.sphere_mesh(44, 0.1, 2), 4: W.sphere_mesh(45, 0.1, 3),
           9: W.box_mesh(300, (0.1, 0.12, 0.05), 4), 10: W.box_mesh(640, (0.04, 0.17, 0.04), 5)}
    dia = {k: 0.15 for k in pts}
    B = 30
    pq, pt, gq, gt = _poses(W, B, 77)
    obj = np.array([0, 1, 4, 9, 10, 6] * 5, np.int64)
    assert bits(eager.forward_value(pts, pq, pt, gq, gt, obj)) == \
        bits(oracle.add_forward(oracle.MeshTable(pts, dia), pq, pt, gq, gt, obj))


def test_real_reference_when_reachable(oracle, eager):
    """The unmodified reference's per-pose values (its eval_metrics at batch size 1, stored in tests/golden by
    oracle/gen_golden.py) against the torch-eager restatement run on this machine and the oracle."""
    for name in GOLDEN_EVAL_CASES:
        g = load_golden(name)
        pts, dia = golden_meshes(g)
        poses = [g[k] for k in ("pq", "pt", "gq", "gt", "obj")]
        ref = [g[k] for k in ("add", "adds", "hit", "valid")]
        mine = eager.eval_poses(pts, dia, *poses)
        got = oracle.add_eval(oracle.MeshTable(pts, dia), *poses, n_threads=4)
        for a, b, c in zip(ref, mine, got):
            assert same_bits(a, b) and same_bits(a, c), name


@pytest.mark.parametrize("cs", [7, 36, 137, 224, 300, 447, 448, 449, 768])
def test_cv2_resize_u16_arithmetic_of_this_machine(oracle, cs):
    """cv2.resize on uint16 (data/dataset_rgbd.py:173) as THIS machine's OpenCV computes it: the
    wheel's default goes through IPP (one float32 fma per lerp, float64 coordinate), with IPP switched
    off through OpenCV's C++ code (separate roundings, INTER_AREA at exactly 2x).  Both restatements
    (oracle.resize_linear_u16) must reproduce the whole 224x224 output."""
    cv2 = pytest.importorskip("cv2")
    if not (hasattr(cv2, "ipp") and cv2.ipp.useIPP()):
        pytest.skip("this OpenCV build has no IPP: its default is the generic path")
    r = np.random.RandomState(cs)
    img = r.randint(0, 65535 if cs == 300 else 1500, (cs, cs)).astype(np.uint16)
    try:
        got = cv2.resize(img, (224, 224))
        cv2.ipp.setUseIPP(False)
        gen = cv2.resize(img, (224, 224))
    finally:
        cv2.ipp.setUseIPP(True)
    assert np.array_equal(oracle.resize_linear_u16(img, 224, "cv2"), got), "cv2's default 16-bit bilinear changed"
    assert np.array_equal(oracle.resize_linear_u16(img, 224, "generic"), gen), "cv2's generic 16-bit bilinear changed"


# ------------------------------------------------------------------------------------------- GPU box
@pytest.mark.gpu
@pytest.mark.parametrize("n", [500, 1000, 2048])
def test_gpu_equals_the_reference_ops_run_on_this_box(pkg, cuda_dev, eager, W, n):
    """Kernels (a)+(b) against torch CPU eager ON THE GPU BOX: distances bit for bit, decisions equal."""
    pts = {3: W.sphere_mesh(n, 0.12, 60 + n), 9: W.box_mesh(n, (0.1, 0.12, 0.05), 61 + n),
           10: W.box_mesh(n, (0.04, 0.17, 0.04), 62 + n)}
    dia = {3: 0.12, 9: 0.1646, 10: 0.1759}
    B = 96 if n <= 1000 else 48
    pq, pt, gq, gt = _poses(W, B, 63 + n)
    obj = np.array([3, 9, 10] * (B // 3), np.int64)
    ref = eager.eval_poses(pts, dia, pq, pt, gq, gt, obj)
    crit = pkg.ADDLoss(__import__("tempfile").mkdtemp(), cuda_dev)
    for k, v in pts.items():
        crit.points[k] = torch.from_numpy(v).to(cuda_dev)
    crit.diameters.update(dia)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(cuda_dev)
    got = crit.eval_poses(T(pq), T(pt), T(gq), T(gt), T(obj))
    assert same_bits(got["add"], ref[0]) and same_bits(got["add_s"], ref[1])
    assert np.array_equal(got["hit"], ref[2]) and np.array_equal(got["valid"], ref[3])
    # ADD-only kernel and the loss form on the same data
    add_only = crit._mesh_table(cuda_dev).evaluate(T(pq), T(pt), T(gq), T(gt), T(obj), want_adds=False)[0]
    assert same_bits(add_only.cpu().numpy(), ref[0])
    assert bits(np.float32(crit(T(pq), T(pt), T(gq), T(gt), T(obj)).item())) == \
        bits(eager.forward_value(pts, pq, pt, gq, gt, obj))


@pytest.mark.gpu
def test_borderline_flags_and_the_resolver_hook(pkg, cuda_dev, eager, W):
    """Decisions whose distance lies within 4 float32 ulp of 0.1*diameter are flagged; the hook lets a
    caller re-decide exactly those with the reference's ops (here: torch eager on the host).  The
    diameter is chosen so that pose 0 sits exactly on its threshold's float32 neighbour."""
    import tempfile
    mesh = W.sphere_mesh(400, 0.1, 5)
    pq, pt, gq, gt = _poses(W, 64, 6)
    obj = np.zeros(64, np.int64)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(cuda_dev)
    crit = pkg.ADDLoss(tempfile.mkdtemp(), cuda_dev)
    crit.points[0] = torch.from_numpy(mesh).to(cuda_dev)
    crit.diameters[0] = 0.1
    first = crit.eval_poses(T(pq), T(pt), T(gq), T(gt), T(obj))
    assert not first["borderline"].any()                      # generic poses are far from the threshold
    d0 = float(first["add"][0])
    crit.diameters[0] = float(np.nextafter(np.float32(d0), np.float32(1.0))) * 10.0   # thr = next float above d0
    second = crit.eval_poses(T(pq), T(pt), T(gq), T(gt), T(obj))
    assert second["borderline"][0] == 1 and second["borderline"].sum() == 1
    calls = []
    inner = eager.resolve_borderline({0: mesh}, {0: crit.diameters[0]})

    def hook(idx, *args):
        calls.append(list(idx))
        return inner(idx, *args)
    crit.borderline_resolver = hook
    m = crit.eval_metrics(T(pq), T(pt), T(gq), T(gt), T(obj))
    assert calls == [[0]]
    ref = eager.eval_poses({0: mesh}, {0: crit.diameters[0]}, pq, pt, gq, gt, obj)
    assert m["add_01d_acc"] == np.mean(ref[2].astype(np.float64)) * 100


def test_float32_resize_restatement_equals_the_local_cv2(oracle):
    """The inference script resizes the crop as float32 (scripts/inference/inference_rgbd_geometric.py:140): the
    local cv2's default INTER_LINEAR on CV_32F against oracle.resize_linear_f32, whole 224x224 outputs, bit for bit
    (skipped when the local OpenCV has no IPP: its own C++ float path is not restated)."""
    cv2 = pytest.importorskip("cv2")
    if not (hasattr(cv2, "ipp") and cv2.ipp.useIPP()):
        pytest.skip("OpenCV without IPP")
    r = np.random.RandomState(8)
    for cs in (3, 36, 97, 150, 223, 224, 225, 301, 448, 449, 576):
        img = r.randint(400, 1500, (cs, cs)).astype(np.uint16)
        img[r.rand(cs, cs) < 0.1] = 0
        out = cv2.resize(img.astype(np.float32), (224, 224))
        assert np.array_equal(out.view(np.uint32), oracle.resize_linear_f32(img, 224).view(np.uint32)), cs


@pytest.mark.gpu
def test_detection_kernel_equals_cv2_run_on_this_box(pkg, cuda_dev, W):
    """N1, inference form, against cv2 itself ON THE GPU BOX: for detector boxes whose crop lies inside the frame,
    the float32 depth the kernel returns equals the pixel of cv2.resize(crop.astype(float32)) / 1000 the
    reference's script would hand to the network."""
    cv2 = pytest.importorskip("cv2")
    if not (hasattr(cv2, "ipp") and cv2.ipp.useIPP()):
        pytest.skip("OpenCV without IPP")
    depth, _ = W.config4_frame(48, 8)
    r = np.random.RandomState(49)
    n = 400
    w = r.randint(30, 300, n); h = r.randint(30, 300, n)
    x = (r.rand(n) * (640 - 1.2 * np.maximum(w, h)) + 0.1 * np.maximum(w, h)).astype(np.int64)
    y = (r.rand(n) * (480 - 1.2 * np.maximum(w, h)) + 0.1 * np.maximum(w, h)).astype(np.int64)
    xyxy = np.stack([x, y, x + w, y + h], 1).astype(np.int32)
    _, center, _, zm = pkg.detection_backproject(torch.from_numpy(depth).to(cuda_dev), xyxy, return_aux=True)
    center, zm = center.cpu().numpy(), zm.cpu().numpy()
    checked = 0
    for b in range(n):
        x1, y1, x2, y2 = (int(v) for v in xyxy[b])
        size = max(x2 - x1, y2 - y1) * 1.2
        cx1, cy1, cs = int((x1 + x2) / 2 - size / 2), int((y1 + y2) / 2 - size / 2), int(size)
        if cx1 < 0 or cy1 < 0 or cx1 + cs > 640 or cy1 + cs > 480:
            continue                           # padded boxes are covered by the golden fixture
        crop = cv2.resize(depth[cy1:cy1 + cs, cx1:cx1 + cs].astype(np.float32), (224, 224)) / 1000.0
        u, v = int(min(max(center[b, 0], 0), 223)), int(min(max(center[b, 1], 0), 223))
        assert np.float32(crop[v, u]).view(np.uint32) == zm[b].view(np.uint32), (b, xyxy[b])
        checked += 1
    assert checked > 100


@pytest.mark.gpu
def test_fused_crop_kernel_equals_cv2_run_on_this_box(pkg, cuda_dev, W):
    """N1 against cv2 itself ON THE GPU BOX: for boxes inside the frame, the z_mm the kernel returns
    equals the pixel of cv2.resize(crop) the reference would read, in cv2's default setting and with
    IPP switched off."""
    cv2 = pytest.importorskip("cv2")
    depth, _ = W.config4_frame(46, 8)
    r = np.random.RandomState(47)
    n = 400
    w = r.randint(30, 300, n); h = r.randint(30, 300, n)
    x = (r.rand(n) * (640 - 1.2 * np.maximum(w, h)) + 0.1 * np.maximum(w, h)).astype(np.int64)
    y = (r.rand(n) * (480 - 1.2 * np.maximum(w, h)) + 0.1 * np.maximum(w, h)).astype(np.int64)
    boxes = np.stack([x, y, w, h], 1).astype(np.int32)
    K = torch.tensor(pkg.DEFAULT_K, dtype=torch.float32, device=cuda_dev)
    has_ipp = hasattr(cv2, "ipp") and cv2.ipp.useIPP()
    for mode in ("cv2", "generic"):
        if mode == "cv2" and not has_ipp:
            continue
        _, center, _, zmm = pkg.depth_crop_backproject(torch.from_numpy(depth).to(cuda_dev), torch.from_numpy(boxes), K,
                                                       return_aux=True, bilinear=mode)
        center, zmm = center.cpu().numpy(), zmm.cpu().numpy()
        try:
            if has_ipp:
                cv2.ipp.setUseIPP(mode == "cv2")
            for b in range(n):
                bx, by, bw, bh = (int(v) for v in boxes[b])
                size = max(bw, bh) * 1.2
                x1, y1, cs = int(bx + bw / 2 - size / 2), int(by + bh / 2 - size / 2), int(size)
                if x1 < 0 or y1 < 0 or x1 + cs > 640 or y1 + cs > 480:
                    continue                       # padded boxes are covered by the golden fixtures
                crop = cv2.resize(depth[y1:y1 + cs, x1:x1 + cs], (224, 224))
                u, v = int(min(max(center[b, 0], 0), 223)), int(min(max(center[b, 1], 0), 223))
                assert crop[v, u] == zmm[b], (mode, b, boxes[b])
        finally:
            if has_ipp:
                cv2.ipp.setUseIPP(True)


@pytest.mark.gpu
def test_eval_metrics_dict_equals_the_unmodified_reference_on_this_box(pkg, cuda_dev):
    """Drop-in check against the reference itself: the dict ``ADDLoss.eval_metrics`` returns -- float64
    means over the batch in mm / per cent -- is EQUAL, key by key and type by type, to the dict the
    unmodified reference returned for the same batch (stored in tests/golden by oracle/gen_golden.py),
    incl. ids without a mesh and a mesh without a diameter."""
    import tempfile
    Tc = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(cuda_dev)
    for name in GOLDEN_EVAL_CASES:
        g = load_golden(name)
        pts, dia = golden_meshes(g)
        crit = pkg.ADDLoss(tempfile.mkdtemp(), cuda_dev)
        for k, v in pts.items():
            crit.points[k] = Tc(v)
        crit.diameters.update(dia)
        got = crit.eval_metrics(*(Tc(g[k]) for k in ("pq", "pt", "gq", "gt", "obj")))
        want = dict(zip(("add_mean", "add_s_mean", "add_01d_acc"), g["agg"]))
        assert set(got) == set(want)
        for k in want:
            assert (got[k] == want[k] or (np.isnan(got[k]) and np.isnan(want[k]))) and type(got[k]) is type(want[k]), \
                (name, k, got[k], want[k])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["geodesic", "l1"])
def test_pose_loss_equals_the_unmodified_reference_on_this_box(pkg, cuda_dev, mode):
    """PoseLoss forward + backward against what the reference's own class (models/pose_loss.py) computed for
    the same B = 32 batch (stored in tests/golden by oracle/gen_golden.py): loss within 1e-5, rotation
    gradients within 1e-5 of the row maximum, translation gradients within 1e-6."""
    g = load_golden("pose_loss_cfg3")
    k = f"{mode}_b32_"
    Tc = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(cuda_dev)
    rot, tr = Tc(g[k + "rot_in"]).requires_grad_(True), Tc(g[k + "trans_in"]).requires_grad_(True)
    got = pkg.PoseLoss(1.0, 10.0, mode)(rot, tr, Tc(g["gt_rot"]), Tc(g["gt_trans"]))
    got.backward()
    ref = float(g[k + "loss"])
    assert abs(got.item() - ref) <= 1e-5 * abs(ref)
    g_ref = g[k + "grad_rot"]
    sc = np.maximum(np.abs(g_ref).max(1, keepdims=True), 1e-30)
    assert np.all(np.abs(rot.grad.cpu().numpy() - g_ref) <= 1e-5 * sc)
    assert np.allclose(tr.grad.cpu().numpy(), g[k + "grad_trans"], rtol=1e-6, atol=0)
