#!/usr/bin/env python
"""resolve_probe.py — what a re-solve with new b and C costs (cuadmm_solver_update_data) against a fresh init; writes
profiles/resolve_probe_r03.json (or --out) with the GPU name, power limit and SM clocks read in the same run.

  1. Init versus update: wall time of Solver.init and of Solver.update_data (host clock around the call; both end in a
     stream synchronise) on the C2b bench workload (2000 blocks n ~ U{6..60}, m = 700,000) and on the PushT_N=10
     fixture, REPS repeats each, with min / median / max.  The updates alternate keep_iterate 0 and 1 on seeded b.
  2. A receding-horizon loop on PushT_N=10: LOOP successive re-solves (tol 1e-3, as the committed log), each with the
     b scaled by a seeded factor in [0.99, 1.01] (feasible: t X* solves A X = t b).  Every re-solve runs three ways: a fresh init,
     a cold update (keep_iterate=0) and a warm update (keep_iterate=1, sigma of the previous solve) on one long-lived
     solver each.  Recorded per re-solve: wall time (init or update + solve), iterations, time per iteration, final
     objectives, and each mode's objective difference to its own fresh init.

    python scripts/resolve_probe.py [--out PATH] [--reps 5] [--loop 10]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

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


def perturbed_b(P, seed, rel=1e-2):
    """b scaled by a seeded factor in [1 - rel, 1 + rel]: A (t X*) = t b keeps the problem feasible"""
    t = 1 + rel * np.random.default_rng(seed).uniform(-1.0, 1.0)
    return P["b_idx"], P["b_val"] * t


def init_solver(cu, P, b=None):
    bi, bv = b if b is not None else (P["b_idx"], P["b_val"])
    s = cu.Solver(verbose=False)
    t0 = time.perf_counter()
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], bi, bv, P["C_idx"], P["C_val"],
           P["blk"], None, None, None, 1.0)
    return s, time.perf_counter() - t0


def init_vs_update(cu, P, reps):
    t_init = []
    for _ in range(reps):
        s, t = init_solver(cu, P)
        t_init.append(t)
        s.close()
    s, _ = init_solver(cu, P)
    s.solve(5, -1.0, 500, 50, 100, 11000, 1.05)        # X, y, S of a solve for the warm updates
    t_upd = {0: [], 1: []}
    t_upd_lib = {0: [], 1: []}
    for k in range(2 * reps + 2):
        keep = k % 2
        bi, bv = perturbed_b(P, 100 + k)
        t0 = time.perf_counter()
        s.update_data(bi, bv, P["C_idx"], P["C_val"], keep_iterate=bool(keep), sig=1.0)
        t = time.perf_counter() - t0
        if k >= 2:                                        # the first update of each mode allocates its staging buffers
            t_upd[keep].append(t)
            t_upd_lib[keep].append(s.times()["update"])
    s.close()
    return dict(init_s=stats(t_init), update_cold_s=stats(t_upd[0]), update_warm_s=stats(t_upd[1]),
                update_cold_in_library_s=stats(t_upd_lib[0]), update_warm_in_library_s=stats(t_upd_lib[1]),
                init_over_update_cold_median=float(np.median(t_init) / np.median(t_upd[0])))


def receding_horizon(cu, P, loop):
    run = (20000, 1e-3, 0, 50, 100, 11000, 1.05)
    cold, _ = init_solver(cu, P)
    warm, _ = init_solver(cu, P)
    cold.solve(*run); warm.solve(*run)
    rows = []
    tot = dict(fresh=0.0, cold=0.0, warm=0.0)
    for k in range(loop):
        b = perturbed_b(P, 1000 + k)
        t0 = time.perf_counter()
        f, _ = init_solver(cu, P, b)
        f.solve(*run)
        t_f = time.perf_counter() - t0
        sig = float(warm.history("sig")[-1])
        t0 = time.perf_counter()
        cold.update_data(*b, P["C_idx"], P["C_val"], keep_iterate=False, sig=1.0)
        cold.solve(*run)
        t_c = time.perf_counter() - t0
        t0 = time.perf_counter()
        warm.update_data(*b, P["C_idx"], P["C_val"], keep_iterate=True, sig=sig)
        warm.solve(*run)
        t_w = time.perf_counter() - t0
        row = dict(k=k, seconds=dict(fresh=t_f, cold=t_c, warm=t_w))
        for name, s in (("fresh", f), ("cold", cold), ("warm", warm)):
            it = int(s.info_iter_num)
            row[name] = dict(iters=it, pobj=float(s.history("pobj")[-1]), dobj=float(s.history("dobj")[-1]),
                             solve_s=float(s.times()["solve"]), ms_per_iter=1e3 * float(s.times()["solve"]) / max(it, 1))
        for name in ("cold", "warm"):
            row[name]["pobj_rel_diff_vs_fresh"] = abs(row[name]["pobj"] - row["fresh"]["pobj"]) / abs(row["fresh"]["pobj"])
        for name in tot:
            tot[name] += row["seconds"][name]
        rows.append(row)
        f.close()
        print("re-solve %d: iterations fresh %d cold %d warm %d, seconds %.2f %.2f %.2f" % (
            k, row["fresh"]["iters"], row["cold"]["iters"], row["warm"]["iters"], t_f, t_c, t_w), flush=True)
    cold.close(); warm.close()
    summary = dict(total_seconds=tot)
    for name in ("fresh", "cold", "warm"):
        summary[name + "_iters"] = [r[name]["iters"] for r in rows]
    for name in ("cold", "warm"):
        summary[name + "_max_pobj_rel_diff_vs_fresh"] = max(r[name]["pobj_rel_diff_vs_fresh"] for r in rows)
    return dict(summary=summary, rows=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "resolve_probe_r03.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--loop", type=int, default=10)
    args = ap.parse_args()
    import cuadmm_b200 as cu
    from cuadmm_b200.synthetic import c2b_blocks, chain_sdp
    from util_problems import load_fixture
    if cu.device_count() == 0:
        raise SystemExit("resolve_probe: no CUDA device (nothing here runs without one)")
    rec = dict(gpu=gpu_info(), method="host wall clock (time.perf_counter) around Solver.init / Solver.update_data, "
                                      "which both end in a stream synchronise; update_in_library is "
                                      "cuadmm_solver_times out[6], the same interval inside the library")
    pusht = load_fixture("pusht_n10")
    rec["pusht_n10"] = dict(vec_len=pusht["vec_len"], con_num=pusht["con_num"], **init_vs_update(cu, pusht, args.reps))
    print("PushT_N=10", json.dumps({k: v["median"] for k, v in rec["pusht_n10"].items() if isinstance(v, dict)}), flush=True)
    blk = c2b_blocks(2000, 6, 60, 0)
    c2b = chain_sdp(blk, 700000, seed=0)
    rec["c2b"] = dict(vec_len=int(c2b["vec_len"]), con_num=int(c2b["con_num"]), **init_vs_update(cu, c2b, args.reps))
    print("C2b", json.dumps({k: v["median"] for k, v in rec["c2b"].items() if isinstance(v, dict)}), flush=True)
    rec["receding_horizon_pusht_n10"] = receding_horizon(cu, pusht, args.loop)
    rec["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
