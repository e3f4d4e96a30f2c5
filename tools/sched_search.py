#!/usr/bin/env python
"""sched_search.py -- dev tool (runs on a GPU box): hill-climb the schedule of one re-laid scan loop
with live timings.  Starts from the recipe the Makefile applies (csrc/sass_sched.py), then tries
single changes -- flip one yield bit, move one minimum by one slot -- and keeps a change when the
kernel gets faster.  Every candidate goes through the same safety checks as the build pass and its
output hash is compared with the baseline's.

  python tools/sched_search.py UNPATCHED.so KERNEL CLASS N_POINTS POSES BUDGET_SECONDS [policy|plan.json] [yield]
UNPATCHED.so is the PRODUCT library as ptxas made it (make NOSCHED=1 TARGET=...): the plan is only valid
for the loop it was measured on (sass_sched.fingerprint).  CLASS = 0 / 1 / 2 (N <= 512, <= 1024, larger): the letter of p6d_sched_state the candidate sets,
which makes the library use the re-laid kernel of that class -- after its own run-time self-check
against the ptxas-scheduled kernel, so a candidate that computes anything else is rejected twice.
A plan.json measured on another instruction order of the loop is used as a starting point by slot
position (the minima keep their positions in the trip) when that order is legal here.
Prints the best schedule as a plan (order + yield mask + fingerprint) for csrc/sched_plan_*.json.
"""
import ctypes as C
import hashlib, importlib, json, os, random, struct, sys, time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "6d-pose-estimation_b200", "csrc"))
import sass_sched as S
import numpy as np
import torch

base_so, kernel, cls, npts, poses, budget = sys.argv[1], sys.argv[2], int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5]), float(sys.argv[6])
policy = sys.argv[7] if len(sys.argv) > 7 else "spaced=FADD2:2"
yspec = sys.argv[8] if len(sys.argv) > 8 else "8,0"

pkg = importlib.import_module("6d-pose-estimation_b200")
core, W = pkg.core, pkg.workloads
dev = torch.device("cuda", 0)
pts, dia = W.config2_meshes(npts)
d = [torch.from_numpy(x).to(dev) for x in W.config2(poses)]
order_t = torch.argsort(d[4], stable=True).to(torch.int32)

kernel_instrs = S.load(base_so, kernel)
body = S.pick_loop(kernel_instrs, "uniform")
data0 = bytearray(open(base_so, "rb").read())
whole = b"".join(struct.pack("<QQ", i.lo, i.hi) for i in kernel_instrs)
assert data0.count(whole) == 1
loop_at = data0.find(whole) + (body[0].addr - kernel_instrs[0].addr)
assert data0.count(S.STATE_TAG) == 1
mark_at = data0.find(S.STATE_TAG) + len(S.STATE_TAG) + cls
assert data0[mark_at:mark_at + 1] == b"p", "the library is already re-laid: build it with NOSCHED=1"
n = len(body)
counter = [0]


def evaluate(order, yields, packed_stall=1):
    S.check_order(body, order)
    stalls, _ = S.assign_stalls(body, order, packed_stall)
    blob = S.emit(body, order, stalls, yields)
    data = bytearray(data0)
    data[loop_at:loop_at + len(blob)] = blob
    data[mark_at:mark_at + 1] = b"t"
    counter[0] += 1
    path = f"/dev/shm/p6d_cand_{os.getpid()}_{counter[0]}.so"
    open(path, "wb").write(data)
    core._lib = None
    core.SO_PATH = path
    table = core.MeshTable(pts, dia, pkg.SYMMETRIC_OBJECT_IDS, dev)
    out = table.evaluate(*d, want_adds=True, order=order_t)
    torch.cuda.synchronize()
    if table.schedule_state() != {"built_relaid": 1, "runtime_state": 1}:
        table.close(); os.unlink(path)
        raise AssertionError("the library's self-check rejected this candidate")
    ts = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); out = table.evaluate(*d, want_adds=True, order=order_t); e1.record()
        torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    h = hashlib.md5(out[4].cpu().numpy()[:10 * poses].tobytes()).hexdigest()
    table.close()
    os.unlink(path)
    return min(ts), h


seed_plan = None
if policy.endswith(".json"):
    seed_plan = json.load(open(policy))
    policy = "spaced=FADD2:2"
if seed_plan is not None and seed_plan.get("loop_fingerprint") == S.fingerprint(body):   # continue from an earlier result
    order, yields = seed_plan["order"], [int(c) for c in seed_plan["yield_mask"]]
else:
    order = S.make_order(body, policy)
    per, ph = (int(x) for x in yspec.split(","))
    yields = [0 if (q % per) == ph else 1 for q in range(n)]
ident = list(range(n))
t_ptxas, h0 = evaluate(ident, [i.field()["y"] for i in body], 2)
best_t, h = evaluate(order, yields)
assert h == h0
print(f"ptxas schedule {t_ptxas:.3f} ms; start recipe {best_t:.3f} ms", flush=True)
if seed_plan is not None and seed_plan.get("loop_fingerprint") != S.fingerprint(body) and len(seed_plan["order"]) == n:
    # a plan for another instruction order of the same loop: keep WHERE in the trip the minima and the
    # non-movable non-packed instructions sit, fill the other positions with this loop's instructions in order
    mov = [k for k in range(n) if S.movable(body[k])]
    rest = [k for k in range(n) if not S.movable(body[k])]
    old_body_movable = None
    try:
        slots = [p for p, k in enumerate(seed_plan["order"]) if k in set(seed_plan.get("movable", mov))]
        if len(slots) == len(mov):
            cand, mi, ri = [], iter(mov), iter(rest)
            slot_set = set(slots)
            for p in range(n):
                cand.append(next(mi) if p in slot_set else next(ri))
            cy = [int(c) for c in seed_plan["yield_mask"]]
            t, h = evaluate(cand, cy)
            print(f"slot-transferred plan {t:.3f} ms", flush=True)
            if h == h0 and t < best_t:
                best_t, order, yields = t, cand, cy
    except (SystemExit, AssertionError, StopIteration) as e:
        print("slot transfer not legal here:", e, flush=True)
t_end = time.time() + budget
rng = random.Random(int(os.environ.get('SEARCH_SEED', '1')))
evals, accepted = 0, 0
def mutate(cand_o, cand_y):
    if rng.random() < 0.5:
        p = rng.randrange(n - 1)
        cand_y[p] ^= 1
        return f"yield[{p}]"
    mins = [p for p, k in enumerate(cand_o) if S.movable(body[k])]
    p = rng.choice(mins)
    q = p + rng.choice((-1, 1))
    if q < 0 or q >= n - 1:
        return None
    cand_o[p], cand_o[q] = cand_o[q], cand_o[p]
    cand_y[p], cand_y[q] = cand_y[q], cand_y[p]
    return f"min {p}->{q}"


while time.time() < t_end:
    cand_o, cand_y = list(order), list(yields)
    # single moves have converged once; 40 % of the candidates now combine two or three changes
    k_moves = 1 if rng.random() < 0.6 else rng.choice((2, 3))
    what = [mutate(cand_o, cand_y) for _ in range(k_moves)]
    if None in what:
        continue
    what = "+".join(what)
    try:
        t, h = evaluate(cand_o, cand_y)
    except (SystemExit, AssertionError):
        continue
    evals += 1
    if h != h0:
        print("HASH MISMATCH for", what, flush=True)
        continue
    if t < best_t - 0.015:
        best_t, order, yields = t, cand_o, cand_y
        accepted += 1
        print(f"{evals:4d} {what:28s} -> {best_t:.3f} ms", flush=True)
        if os.environ.get("SEARCH_CHECKPOINT"):     # survive a kill: the best plan so far, rewritten on every accepted move
            with open(os.environ["SEARCH_CHECKPOINT"], "w") as fh:
                json.dump({"kernel": kernel, "evals": evals, "accepted": accepted, "ptxas_ms": t_ptxas, "best_ms": best_t,
                           "packed_stall": 1, "order": order, "yield_mask": "".join(str(y) for y in yields),
                           "movable": [k for k in range(n) if S.movable(body[k])], "loop_fingerprint": S.fingerprint(body)}, fh)
print(json.dumps({"kernel": kernel, "found_by": f"tools/sched_search.py: {evals} timed candidates on B200 ({poses} poses, N={npts}), "
                                               "hill climbing over yield bits and slot moves of the minima",
                  "evals": evals, "accepted": accepted, "ptxas_ms": t_ptxas, "best_ms": best_t, "packed_stall": 1,
                  "order": order, "yield_mask": "".join(str(y) for y in yields),
                  "movable": [k for k in range(n) if S.movable(body[k])],
                  "loop_fingerprint": S.fingerprint(body)}))
