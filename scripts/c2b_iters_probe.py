"""Iterations to 1e-6 KKT on the bench problem under different projection stopping thresholds (CUADMM_JACOBI_THR)."""
import os, sys, time, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from util_problems import make_solver
from cuadmm_b200.synthetic import c2b_blocks, chain_sdp
P = chain_sdp(c2b_blocks(), 700000, seed=0, coeffs=os.environ.get("COEFFS", "gauss"))
s = make_solver(P)
t = time.time(); s.solve(20000, 1e-6, 0, 50, 100, 11000); dt = time.time() - t
h = {k: s.history(k) for k in ("errRp", "errRd", "relgap", "pobj")}
print(json.dumps({"thr": os.environ.get("CUADMM_JACOBI_THR", "default"),
                  "coeffs": os.environ.get("COEFFS", "gauss"), "iters": int(s.info_iter_num), "seconds": dt,
                  "kkt_at": {str(k): float(max(h["errRp"][k], h["errRd"][k], h["relgap"][k])) for k in (999, 2999, 4999, 6999) if k < s.info_iter_num},
                  "pobj_err": float(abs(h["pobj"][-1] - P["pstar"]) / (1 + abs(P["pstar"])))}), flush=True)
