"""Worker of the sharded re-solve test (tests/test_gpu_resolve.py): one process per rank, launched like
tests/cones_rank_worker.py (ranks share GPU 0 when there is only one).  Every rank solves the typed problem, takes a cold
update_data with new b and C (every rank passes the same full arrays) and solves again; rank 0 does the same unsharded
and compares the trajectories after the update, X, S and A^T y."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np  # noqa: E402
import cuadmm_b200 as cu  # noqa: E402
import cones_util as cz  # noqa: E402
from test_gpu_resolve import new_data  # noqa: E402

rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"])
job = bytes.fromhex(os.environ["JOB_ID"])
ndev = cu.device_count()
dev = rank % max(ndev, 1)
BLOCKS = [("s", 30), ("l", 5000), ("s", 12), ("u", 700), ("s", 180), ("l", 3), ("s", 45), ("u", 1), ("s", 7),
          ("l", 2500), ("s", 60), ("u", 40)]
P = cz.typed_synthetic(BLOCKS, 3000, seed=1)
DATA = new_data(P, seed=21, drop=0.1)


def make(distributed):
    s = cu.Solver(verbose=False)
    s.set_device(dev)
    if distributed:
        s.set_distributed(rank, world, job)
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
           P["C_idx"], P["C_val"], P["blk"], blk_types=P["types"])
    return s


def run(s):
    s.solve(100, 1e-12, 20, 5, 10, 40, 1.05)          # sGS -> ADMM switch at 40: dirty state before the update
    s.update_data(*DATA, keep_iterate=False, sig=1.3)
    s.solve(60, 1e-12, 20, 5, 10, 40, 1.05)
    out = {"iters": s.info_iter_num, "X": s.X, "y": s.y, "S": s.S}
    for k in ["errRp", "errRd", "pobj", "dobj", "sig", "relgap"]:
        out[k] = s.history(k)
    return out


sd = make(True)
d = run(sd)
ok = True
if rank == 0:
    s1 = make(False)
    r = run(s1)
    # control: a second one-GPU run.  The dense sign path (the n = 180 block) sums |A|_F^2 with floating-point
    # atomicAdd, so two runs differ from each other; the sharded run may differ from r by up to 10x that.
    s1.close()
    c = run(make(False))
    print("world", world, "devices", ndev,
          "iters sharded", d["iters"], "single", r["iters"])
    ok = d["iters"] == r["iters"] == 60
    for k in ["errRp", "errRd", "pobj", "dobj", "sig", "relgap"]:
        if len(d[k]) != len(r[k]):
            ok = False
            continue
        # relative to the largest entry of the history, as in test_gpu_resolve.compare_to_fresh
        rel = lambda a: float(np.max(np.abs(a - r[k])) / max(np.max(np.abs(r[k])), 1e-300)) if len(r[k]) else 0.0
        err, ctrl = rel(d[k]), rel(c[k]) if len(c[k]) == len(r[k]) else np.inf
        print(" ", k, "rel diff vs 1 GPU %.2e (1 GPU vs 1 GPU %.2e)" % (err, ctrl))
        ok = ok and err < max(1e-9 if k == "relgap" else 1e-12, 10 * ctrl)
    A = P["A"]
    d["Aty"], r["Aty"], c["Aty"] = A.T @ d["y"], A.T @ r["y"], A.T @ c["y"]
    for k in ("X", "S", "Aty"):
        err = float(np.linalg.norm(d[k] - r[k]) / max(np.linalg.norm(r[k]), 1e-300))
        ctrl = float(np.linalg.norm(c[k] - r[k]) / max(np.linalg.norm(r[k]), 1e-300))
        print(" ", k, "rel diff %.2e (1 GPU vs 1 GPU %.2e)" % (err, ctrl))
        ok = ok and err < max(1e-10, 10 * ctrl)
    off = cz.svec_offsets(P["blk"], P["types"])
    for k, t in enumerate(P["types"]):
        if t == "u":
            ok = ok and bool(np.all(d["S"][off[k]:off[k + 1]] == 0.0))
    print("RESOLVE_RANK_OK" if ok else "RESOLVE_RANK_MISMATCH", flush=True)
sd.close()
sys.exit(0 if ok else 1)
