"""Worker of the typed multi-rank test (tests/test_gpu_cones.py): one process per rank, launched like
tests/multi_rank_worker.py (ranks share GPU 0 when there is only one).  The problem mixes PSD blocks (Jacobi and dense
sizes) with 'l' and 'u' blocks; rank 0 also solves it unsharded and compares trajectories, X, S and A^T y."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np  # noqa: E402
import cuadmm_b200 as cu  # noqa: E402
import cones_util as cz  # noqa: E402

rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"])
job = bytes.fromhex(os.environ["JOB_ID"])
ndev = cu.device_count()
dev = rank % max(ndev, 1)
BLOCKS = [("s", 30), ("l", 5000), ("s", 12), ("u", 700), ("s", 180), ("l", 3), ("s", 45), ("u", 1), ("s", 7),
          ("l", 2500), ("s", 60), ("u", 40)]
P = cz.typed_synthetic(BLOCKS, 3000, seed=1)


def make(distributed):
    s = cu.Solver(verbose=False)
    s.set_device(dev)
    if distributed:
        s.set_distributed(rank, world, job)
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
           P["C_idx"], P["C_val"], P["blk"], blk_types=P["types"])
    return s


def run(s):
    s.solve(60, 1e-12, 20, 5, 10, 40, 1.05)          # sGS -> ADMM switch at 40, sigma updates every 5 / 10
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
    print("world", world, "devices", ndev, "iters sharded", d["iters"], "single", r["iters"])
    ok = d["iters"] == r["iters"]
    for k in ["errRp", "errRd", "pobj", "dobj", "sig", "relgap"]:
        if len(d[k]) != len(r[k]):
            ok = False
            continue
        err = float(np.max(np.abs(d[k] - r[k]) / np.maximum(np.abs(r[k]), 1e-9))) if len(r[k]) else 0.0
        print(" ", k, "max rel diff vs 1 GPU %.2e" % err)
        # the sharded sums run in another order; observed on a B200 (2 and 3 ranks on one GPU): <= 4.4e-13 on
        # errRp / errRd / pobj / dobj, 0 on sig, and up to 2.0e-10 on relgap = |pobj - dobj| / (1 + |pobj| + |dobj|),
        # whose cancellation magnifies the rounding of pobj and dobj
        ok = ok and err < (1e-9 if k == "relgap" else 1e-12)
    A = P["A"]
    d["Aty"], r["Aty"] = A.T @ d["y"], A.T @ r["y"]
    for k in ("X", "S", "Aty"):
        err = float(np.linalg.norm(d[k] - r[k]) / max(np.linalg.norm(r[k]), 1e-300))
        print(" ", k, "rel diff %.2e" % err)
        ok = ok and err < 1e-7
    off = cz.svec_offsets(P["blk"], P["types"])
    for k, t in enumerate(P["types"]):
        if t == "u":
            ok = ok and bool(np.all(d["S"][off[k]:off[k + 1]] == 0.0))
    print("CONES_RANK_OK" if ok else "CONES_RANK_MISMATCH", flush=True)
sd.close()
sys.exit(0 if ok else 1)
