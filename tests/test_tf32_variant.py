"""The evidence behind "no tensor cores in kernel (b)".

BASELINE.json north_star: "tensor cores are excluded unless a 3xTF32 variant passes the stated
tolerance" (distances within 1e-5 relative, ADD-0.1d decisions bit-exact).  SURVEY.md 7.3.2 asks for
a negative test that demonstrates it.  The variant exists for real --
6d-pose-estimation_b200/csrc/p6d_tf32.cu: ADD-S (reference models/add_loss.py:185-190) in GEMM form on
tcgen05.mma kind::tf32 with error-compensated 3xTF32 operands re-centred on the gt translation,
FP32 accumulators in TMEM -- and is measured here against the oracle:

  * CPU (no GPU needed): a NumPy emulation of the same operand construction with the two
    bracketing accumulation models (oracle/tf32_form.py);
  * -m gpu: the tensor-core kernel itself on BASELINE config 2 poses.

What the measurements say (numbers in profiles/tf32_variant_r2.json and DESIGN.md section 4):
  * plain TF32 is off by 1e-3 ... 1e-2 everywhere;
  * 3xTF32 has an absolute error of ~eps * |g|^2 on every d^2 (|g| ~ 0.1 m after re-centring).  At the
    coarse poses of config 2 (ADD-S 3 ... 20 mm) that is below 1e-5 IF the accumulator rounds to
    nearest, and ~3e-5 (a bias the mean does not average out) if it truncates;
  * at the poses a trained network produces (ADD-S below 1 mm) the same absolute error is
    1e-4 ... 1e-2 relative for every accumulation model, ideal included.
So the variant does not pass the stated tolerance on the input range of the reference, and the
tests ASSERT THAT FAILURE on the fine poses: if a future variant passes there, these tests fail
and the exclusion has to be revisited -- which is the point.
"""
import json

import numpy as np
import pytest
import torch

TOL = 1e-5      # north_star: "distances and loss within 1e-5 relative in FP32"


def _clouds(oracle, mesh, pq, pt, gq, gt):
    return oracle.transform(mesh, pq, pt), oracle.transform(mesh, gq, gt)


def _fine_poses(W, B, seed=5):
    """Poses as accurate as a trained network's: ADD-S of 0.2 ... 0.9 mm."""
    pq, pt, gq, gt = W.random_poses(B, seed, rot_sigma=0.002, trans_sigma=0.0003)
    return pq, pt, gq, gt, np.where(np.arange(B) % 2 == 0, 9, 10).astype(np.int64)


def _emulate(oracle, F, pts, poses, models):
    pq, pt, gq, gt, obj = poses
    out = {m: [] for m in models}
    for i in range(len(obj)):
        cp, cg = _clouds(oracle, pts[int(obj[i])], pq[i], pt[i], gq[i], gt[i])
        for name, (terms, acc) in models.items():
            out[name].append(float(F.adds_gemm_form(cp, cg, gt[i], terms, acc)))
    return {m: np.array(v) for m, v in out.items()}


def test_emulated_gemm_form_misses_the_tolerance(oracle, W):
    from oracle import tf32_form as F
    pts, dia = W.config2_meshes(500)
    table = oracle.MeshTable(pts, dia)
    models = {"3x_exact": (3, "exact"), "3x_rn": (3, "f32_seq"), "3x_rz": (3, "f32_rz"), "1x_exact": (1, "exact")}
    # (1) fine poses: outside the tolerance for every accumulation model, the ideal one included
    fine = _fine_poses(W, 32)
    ref = oracle.add_eval(table, *fine, n_threads=oracle.max_threads())[1]
    assert ref.max() < 1.0e-3
    rel = {m: np.abs(v - ref) / ref for m, v in _emulate(oracle, F, pts, fine, models).items()}
    for m in ("3x_exact", "3x_rn", "3x_rz"):
        assert (rel[m] > TOL).mean() > 0.5 and rel[m].max() > 10 * TOL, (m, rel[m])
    assert np.median(rel["1x_exact"]) > 100 * TOL
    # (2) coarse poses of config 2: the verdict hangs on how the hardware accumulates
    pq, pt, gq, gt, obj = W.config2(4096)
    sel = np.linspace(0, 4095, 32).astype(int)
    coarse = tuple(x[sel] for x in (pq, pt, gq, gt, obj))
    ref = oracle.add_eval(table, *coarse, n_threads=oracle.max_threads())[1]
    assert ref.min() > 3.0e-3
    rel = {m: np.abs(v - ref) / ref for m, v in _emulate(oracle, F, pts, coarse, models).items()}
    assert rel["3x_exact"].max() < TOL and rel["3x_rn"].max() < TOL          # would pass with a rounding adder
    assert (rel["3x_rz"] > TOL).mean() > 0.5                                  # fails with a truncating one
    assert np.median(rel["1x_exact"]) > 100 * TOL                             # plain TF32: never close
    # sanity: the form is not broken, just imprecise
    assert rel["3x_rz"].max() < 1e-3


@pytest.mark.gpu
def test_tensor_core_3xtf32_kernel_misses_the_tolerance_and_flips_decisions(pkg, cuda_dev, oracle, W):
    """The real thing: tcgen05.mma kind::tf32 + TMEM on config 2 (2,048-point meshes).  Reports max /
    median relative ADD-S error and the number of ADD-0.1d flips against the oracle, prints them as one
    JSON line (profiles/tf32_variant_r2.json is such a record), and asserts the failure."""
    import ctypes as C
    core = pkg.core
    pts, dia = W.config2_meshes(2048)
    table = core.MeshTable(pts, dia, pkg.SYMMETRIC_OBJECT_IDS, cuda_dev)
    B = 2048
    pq, pt, gq, gt, obj = W.config2(B)
    T = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(cuda_dev)
    d = [T(x) for x in (pq, pt, gq, gt, obj)]
    exact = table.evaluate(*d)[1].cpu().numpy()                       # product kernel (bit-exact vs oracle)
    n_oracle = 256
    ref = oracle.add_eval(oracle.MeshTable(pts, dia), pq[:n_oracle], pt[:n_oracle], gq[:n_oracle], gt[:n_oracle],
                          obj[:n_oracle], n_threads=oracle.max_threads())[1]
    assert np.array_equal(exact[:n_oracle].view(np.uint32), ref.view(np.uint32))
    report = {"tolerance": TOL, "kernel": "adds_tf32_kernel (tcgen05.mma kind::tf32, M=128 N=256 K=8, TMEM accumulators)"}

    def run(tag, poses_dev, exact_vals, thr_vals):
        n = exact_vals.shape[0]
        for terms in (3, 1):
            out = torch.empty(n, dtype=torch.float32, device=cuda_dev)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            core.check(core.lib().p6d_adds_tf32_eval(table.handle, *(core.ptr(x) for x in poses_dev), n, terms,
                                                     core.ptr(out), 0, core.stream_ptr(cuda_dev)))
            ev1.record()
            torch.cuda.synchronize()
            got = out.cpu().numpy().astype(np.float64)
            rel = np.abs(got - exact_vals) / exact_vals
            signed = (got - exact_vals) / exact_vals
            flips = int(((got < thr_vals) != (exact_vals.astype(np.float64) < thr_vals)).sum())
            report[f"{tag}_{terms}xTF32"] = {
                "poses": n, "adds_mm_min": float(exact_vals.min() * 1e3), "adds_mm_max": float(exact_vals.max() * 1e3),
                "max_rel_err": float(rel.max()), "median_rel_err": float(np.median(rel)),
                "mean_signed_rel_err": float(signed.mean()), "share_outside_tolerance": float((rel > TOL).mean()),
                "add01d_flips": flips, "ms": ev0.elapsed_time(ev1), "poses_per_s": n / (ev0.elapsed_time(ev1) * 1e-3)}

    thr = np.array([0.1 * dia[int(o)] for o in obj])
    run("config2", d, exact, thr)
    fine = _fine_poses(W, 1024)
    fd = [T(x) for x in fine]
    fexact = table.evaluate(*fd)[1].cpu().numpy()
    run("fine", fd, fexact, np.array([0.1 * dia[int(o)] for o in fine[4]]))
    print(json.dumps(report))
    # the kernel computes ADD-S (it is not garbage) ...
    assert report["config2_3xTF32"]["median_rel_err"] < 1e-3 and report["config2_1xTF32"]["median_rel_err"] < 0.5
    # ... plain TF32 is nowhere near the tolerance, 3xTF32 much closer ...
    assert report["config2_1xTF32"]["median_rel_err"] > 100 * TOL
    assert report["config2_1xTF32"]["median_rel_err"] > 10 * report["config2_3xTF32"]["median_rel_err"]
    # ... and at the accuracy of a trained network the 3xTF32 form is outside the stated tolerance
    assert report["fine_3xTF32"]["share_outside_tolerance"] > 0.5 and report["fine_3xTF32"]["max_rel_err"] > 10 * TOL
