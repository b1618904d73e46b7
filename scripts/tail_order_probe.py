#!/usr/bin/env python
"""tail_order_probe.py — what relabelling the y-solve's dense tail in etree postorder buys on the C2b bench workload
(2000 blocks n ~ U{6..60}, m = 700,000, one GPU); writes profiles/tail_order_probe_r03.json (or --out) with the GPU
name, power limit and SM clocks read in the same run.

Two solvers in one process: one initialised with CUADMM_YSOLVE_TAIL_POSTORDER=0 (the dense tail stays in the order of
the fill-reducing ordering), one with the default postorder.  Recorded for each:
  - the y-solve statistics (dense tail size, deficient pivots, launches per solve) and the device memory init took
    (cudaMemGetInfo before and after init);
  - REPS alternating rounds of STEPS sGS iterations: ms per iteration without profiling events (CUDA events around the
    whole window), then a profiled pass of the same length with CUDA events around every y-solve and around the dense-
    tail stage of each (its two GEMVs): ms per iteration of the two y-solves and of the four tail GEMVs;
  - the iterates after one identical run (same start, same iteration count): max |difference| of X, y and S between
    the two orders, next to the difference between two runs of the postorder solver.

    python scripts/tail_order_probe.py [--out PATH] [--reps 3] [--steps 1000]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        name, plim, sm, smax = [x.strip() for x in out[0].split(",")]
        return dict(name=name, power_limit=plim, sm_clock=sm, sm_max_clock=smax)
    except Exception as e:   # the record says so rather than guessing
        return dict(error=repr(e))


def stats(v):
    v = np.asarray(v, float)
    return dict(min=float(v.min()), median=float(np.median(v)), max=float(v.max()), n=int(len(v)), all=[float(x) for x in v])


def make_solver(cu, torch, P, postorder):
    os.environ["CUADMM_YSOLVE_TAIL_POSTORDER"] = "1" if postorder else "0"      # read at init
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    s = cu.Solver(verbose=False)
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
           P["C_idx"], P["C_val"], P["blk"], None, None, None, 1.0)
    torch.cuda.synchronize()
    used = free0 - torch.cuda.mem_get_info()[0]
    os.environ.pop("CUADMM_YSOLVE_TAIL_POSTORDER")
    s.solve(1, -1.0, 500, 50, 100, 1 << 30, 1.05)          # sets the run parameters (1 iteration), as bench.py does
    return s, used


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tail_order_probe_r03.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=1000)
    args = ap.parse_args()
    import torch
    import cuadmm_b200 as cu
    from cuadmm_b200.synthetic import c2b_blocks, chain_sdp
    if cu.device_count() == 0:
        raise SystemExit("tail_order_probe: no CUDA device")
    torch.cuda.init()
    P = chain_sdp(c2b_blocks(2000, 6, 60, 0), 700000, seed=0)
    rec = dict(gpu_before=gpu_info(), workload="C2b: 2000 blocks n ~ U{6..60}, m = 700,000, one GPU",
               steps=args.steps, reps=args.reps, orders={})
    names = ("tail_order", "postorder")
    solvers = {}
    for name in names:
        s, used = make_solver(cu, torch, P, name == "postorder")
        solvers[name] = s
        rec["orders"][name] = dict(ysolve=s.ysolve_stats(), init_device_bytes=int(used), ms_per_iter=[],
                                   ysolve_x2_ms_per_iter=[], tail_gemv_x4_ms_per_iter=[])
    for s in solvers.values():
        s.run_iterations(50, sgs=True)                     # warm-up
    for rep in range(args.reps):
        for name in names:
            s, o = solvers[name], rec["orders"][name]
            o["ms_per_iter"].append(s.run_iterations(args.steps, sgs=True)["total_ms"] / args.steps)
            p = s.run_iterations_ex(args.steps, sgs=True)
            o["ysolve_x2_ms_per_iter"].append(p["ysolve_ms"] / args.steps)
            o["tail_gemv_x4_ms_per_iter"].append(p["tail_gemv_ms"] / args.steps)
            print("rep %d %-10s %.4f ms/iter, y-solves %.4f ms/iter, tail GEMVs %.4f ms/iter" % (
                rep, name, o["ms_per_iter"][-1], o["ysolve_x2_ms_per_iter"][-1], o["tail_gemv_x4_ms_per_iter"][-1]), flush=True)
    for name in names:
        o = rec["orders"][name]
        for k in ("ms_per_iter", "ysolve_x2_ms_per_iter", "tail_gemv_x4_ms_per_iter"):
            o[k] = stats(o[k])
        solvers[name].close()
    # iterates after one identical run: both orders, and the postorder twice
    runs = []
    for name in ("tail_order", "postorder", "postorder"):
        s, _ = make_solver(cu, torch, P, name == "postorder")
        s.run_iterations(200, sgs=True)
        runs.append((s.X.copy(), s.y.copy(), s.S.copy()))
        s.close()
    diff = lambda a, b: {k: float(np.max(np.abs(u - v))) for k, u, v in zip("XyS", a, b)}
    rec["iterates_after_200"] = dict(tail_order_vs_postorder=diff(runs[0], runs[1]), postorder_vs_postorder=diff(runs[1], runs[2]),
                                     max_abs=dict(X=float(np.max(np.abs(runs[1][0]))), y=float(np.max(np.abs(runs[1][1]))),
                                                  S=float(np.max(np.abs(runs[1][2])))))
    a, b = rec["orders"]["tail_order"], rec["orders"]["postorder"]
    rec["summary"] = dict(
        ms_per_iter=(a["ms_per_iter"]["median"], b["ms_per_iter"]["median"]),
        tail_gemv_x4_ms_per_iter=(a["tail_gemv_x4_ms_per_iter"]["median"], b["tail_gemv_x4_ms_per_iter"]["median"]),
        ysolve_x2_ms_per_iter=(a["ysolve_x2_ms_per_iter"]["median"], b["ysolve_x2_ms_per_iter"]["median"]),
        init_device_bytes_saved=a["init_device_bytes"] - b["init_device_bytes"])
    rec["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec["summary"]))
    print(json.dumps(rec["iterates_after_200"]))


if __name__ == "__main__":
    main()
