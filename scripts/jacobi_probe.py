"""Projection-stage time and Jacobi sweep counts in the regime the solver runs in: a sequence of slowly drifting
inputs (successive ADMM iterates), C2b block mix, warm-started plan.  Environment selects the build / threshold under
test (CUADMM_LIB_PATH, CUADMM_JACOBI_THR).  One JSON line."""
import json, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import cuadmm_b200 as cu
from cuadmm_b200.synthetic import c2b_blocks, random_svec
import oracle_np as onp
blk = c2b_blocks(2000, 6, 60, 0)
x = random_svec(blk, seed=0); d = random_svec(blk, seed=1)
out = {"lib": os.environ.get("CUADMM_LIB_PATH", "default"),
       "thr": os.environ.get("CUADMM_JACOBI_THR", "default"), "drift": {}}
for drift in [1e-1, 1e-2, 1e-3, 1e-4, 1e-6, 0.0]:
    p = cu.Plan(blk, device=0); q = cu.Plan(blk, device=0)
    ms, sw, err = [], [], 0.0
    for t in range(6):
        xt = x + (t * drift) * d
        dx = torch.from_numpy(xt).cuda(); dy = torch.empty_like(dx)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(); p.project_device(dx.data_ptr(), dy.data_ptr()); e1.record(); torch.cuda.synchronize()
        o, eig, s = q.project_eig_host(xt)
        if t >= 1:
            ms.append(e0.elapsed_time(e1)); sw.append(float(s[blk > 32].mean()))
        if t == 5:
            ref = onp.project_svec_cpp(blk, xt, 8)
            err = float(np.linalg.norm(dy.cpu().numpy() - ref) / np.linalg.norm(ref))
    out["drift"][str(drift)] = {"ms": float(np.mean(ms)), "sweeps_n>32": float(np.mean(sw)), "rel_err": err}
    p.close(); q.close()
print(json.dumps(out), flush=True)
