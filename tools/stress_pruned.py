#!/usr/bin/env python
"""Dev tool (GPU box): randomized byte-equality of the opt-in exact-pruned ADD-S kernel (b') with the all-pairs
kernel (b) over mesh families (sphere / box surface, Gaussian blob, flat patch, thin rod, two distant clusters,
duplicated points), sizes 384..4096, prediction errors from 0.002 to 3 rad, translations from 0 to the object
size, scaled / degenerate quaternions.   python tools/stress_pruned.py [poses_per_case] [--large]
--large: the same families at 8,192 / 16,384 / 32,768 points, the streamed pruned kernel (prune_streamed=True) against
the streamed all-pairs kernel (streamed=True) instead of the pruned kernel against the all-pairs kernel."""
import importlib, json, os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
pkg = importlib.import_module("6d-pose-estimation_b200")
core, W = pkg.core, pkg.workloads
dev = torch.device("cuda", 0)
args = [x for x in sys.argv[1:] if x != "--large"]
large = "--large" in sys.argv[1:]
per = int(args[0]) if args else 100_000
SIZES = (8192, 16384, 32768) if large else (384, 500, 1000, 1777, 2048, 4096)
NEW, REF = ({"prune_streamed": True}, {"streamed": True}) if large else ({"prune": True}, {})
r = np.random.RandomState(2024)


def mesh(kind, n, seed):
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
    raise ValueError(kind)


g = torch.Generator(device=dev); g.manual_seed(99)
rnd = lambda *s: torch.randn(*s, generator=g, device=dev)
t0 = time.time()
cases, bad, poses = [], 0, 0
for kind in ("sphere", "box", "blob", "patch", "rod", "clusters", "dups"):
    for n in SIZES:
        pts = {3: mesh(kind, n, 7 * n + len(kind)), 9: mesh(kind, max(n - 37, 1), 11 * n)}
        table = core.MeshTable(pts, {3: 0.1, 9: 0.1}, pkg.SYMMETRIC_OBJECT_IDS, dev)
        B = per if n <= 2048 else per // 4 if n <= 4096 else max(per * 1024 // n, 64)
        sig = torch.exp(torch.empty(B, 1, device=dev).uniform_(np.log(0.002), np.log(3.0), generator=g))
        tsig = torch.exp(torch.empty(B, 1, device=dev).uniform_(np.log(1e-4), np.log(0.1), generator=g))
        qa, ta = torch.nn.functional.normalize(rnd(B, 4), dim=1), rnd(B, 3) * 0.2 + torch.tensor([0.0, 0.0, 0.8], device=dev)
        qb, tb = torch.nn.functional.normalize(qa + sig * rnd(B, 4), dim=1), ta + tsig * rnd(B, 3)
        k = B // 50
        qb[:k] *= torch.exp(rnd(k, 1))                  # non-unit quaternions: R is not a rotation
        qb[k:k + 8] = 0.0; tb[k + 8:k + 16] = ta[k + 8:k + 16]; qb[k + 8:k + 16] = qa[k + 8:k + 16]
        tb[k + 16, 0] = float("nan"); qa[k + 17, 2] = float("inf")
        obj = torch.where(torch.rand(B, generator=g, device=dev) < 0.5, 3, 9).to(torch.int64)
        full = table.evaluate(qb, tb, qa, ta, obj, **REF)[4]
        prun = table.evaluate(qb, tb, qa, ta, obj, **NEW)[4]
        diff = int((full[:11 * B] != prun[:11 * B]).sum())
        bad += diff; poses += B
        cases.append({"mesh": kind, "n": n, "poses": B, "differing_bytes": diff})
print(json.dumps({"large": large, "sizes": SIZES, "poses": poses, "cases": len(cases), "differing_bytes": bad, "seconds": round(time.time() - t0, 1),
                  "bad_cases": [c for c in cases if c["differing_bytes"]]}))
