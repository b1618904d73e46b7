"""Cost of the infeasibility check (INTEGRATION.md §10) on one GPU, written as JSON (default profiles/infeas_probe_r03.json).

  * C2b (the bench workload: 2,000 blocks n ~ U{6..60}, m = 700,000): solves of N iterations with the check off and on
    at intervals 50 and 100, alternated, timed by the solver's CUDA events (cuadmm_solver_times total); the overhead per
    iteration and per check is the difference to the run without the check.  The projection share of a check is the
    time of one cold projection of a C2b svec vector (a plan with warm start off, as the check's plan), by CUDA events.
  * the device memory the check adds on C2b (cudaMemGetInfo around the first solve with the check on);
  * PushT_N=10 with constraint 17146 (X[5168] = 1, a diagonal entry of a PSD block) set to -1: time and iterations to
    the primal infeasibility stop, against the run to max_iter without the check, and what the checks saw in the sGS phase;
  * cuadmm_solver_infeasibility_stats (checks, projections run, smallest ratios and guard values) on the feasible
    fixtures.
Usage: python scripts/infeas_probe.py [--iters N] [--out path]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import cuadmm_b200 as cu  # noqa: E402
from cuadmm_b200.synthetic import c2b_blocks, chain_sdp  # noqa: E402
from util_problems import load_fixture  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def solver(P, interval=0):
    s = cu.Solver(verbose=False)
    if interval:
        s.set_infeasibility_check(interval, 1e-7)
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
           P["C_idx"], P["C_val"], P["blk"])
    return s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "infeas_probe_r03.json"))
    a = ap.parse_args()
    res = {"gpu": gpu_info(), "iters": a.iters}
    P = chain_sdp(c2b_blocks(2000, 6, 60, 0), 700000, seed=0)
    run = (a.iters, 1e-12, 500, 50, 100, 11000, 1.05)
    # one solver; every solve follows a cold update_data with the same b and C, which restarts it as a fresh init
    # would (no block of C2b takes the dense sign path), so the runs differ only in the check
    s = solver(P)
    data = (P["b_idx"], P["b_val"], P["C_idx"], P["C_val"])

    def solve(interval, r):
        s.set_infeasibility_check(interval, 1e-7)
        s.update_data(*data, keep_iterate=False)
        s.solve(*r)

    solve(0, (1,) + run[1:])
    # memory: the check's buffers and second plan are allocated by the first solve with the check on
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    solve(50, (1,) + run[1:])
    free1, _ = torch.cuda.mem_get_info()
    res["c2b_check_bytes_mem_get_info"] = int(free0 - free1)
    res["c2b_check_bytes_buffers"] = int(8 * (3 * P["con_num"] + 5 * P["vec_len"]))
    # timing, alternated (total device time of the solve from the update, by the solver's CUDA events)
    times = {0: [], 50: [], 100: []}
    stops = {}
    for _ in range(a.reps):
        for interval in (0, 50, 100):
            solve(interval, run)
            times[interval].append(s.times()["total"] * 1e3)
            stops[interval] = (int(s.info_iter_num), int(s.stop_reason))
            res.setdefault("c2b_check_stats", {})[str(interval)] = s.infeasibility_stats()
    base = min(times[0])
    res["c2b_solve_ms"] = {str(k): v for k, v in times.items()}
    res["c2b_stop"] = {str(k): v for k, v in stops.items()}
    for interval in (50, 100):
        d = min(times[interval]) - base
        res["c2b_interval_%d" % interval] = {"overhead_ms_per_iter": d / a.iters, "ms_per_check": d / (a.iters // interval),
                                             "overhead_share": d / base}
    # one cold projection of a C2b-size vector (the check's plan: warm start off)
    blk = P["blk"]
    p = cu.Plan(blk, device=0)
    p.set_warm_start(0)
    rng = np.random.default_rng(0)
    x = torch.from_numpy(rng.standard_normal(P["vec_len"])).cuda()
    out = torch.empty_like(x)
    for _ in range(3):
        p.project_device(x.data_ptr(), out.data_ptr())
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 20
    e0.record()
    for _ in range(n):
        p.project_device(x.data_ptr(), out.data_ptr())
    e1.record()
    torch.cuda.synchronize()
    res["c2b_cold_projection_ms_random_input"] = e0.elapsed_time(e1) / n
    # time to detect on PushT_N=10 made infeasible
    Q = load_fixture("pusht_n10")
    b = np.zeros(Q["con_num"]); b[Q["b_idx"]] = Q["b_val"]
    b[17146] = -1.0
    nz = np.nonzero(b)[0].astype(np.int32)
    prun = (20000, 1e-3, 0, 50, 100, 11000, 1.05)
    det = {}
    for interval in (0, 50):
        s = solver(Q, interval)
        s.update_data(nz, b[nz], Q["C_idx"], Q["C_val"], keep_iterate=False)
        t0 = time.perf_counter()
        s.solve(*prun)
        det[str(interval)] = {"wall_s": time.perf_counter() - t0, "iters": int(s.info_iter_num),
                              "stop_reason": int(s.stop_reason)}
        del s
    # the same instance stopped at the sGS -> ADMM switch (iteration 11000): what the checks saw during the sGS phase
    s = solver(Q, 50)
    s.update_data(nz, b[nz], Q["C_idx"], Q["C_val"], keep_iterate=False)
    s.solve(11000, *prun[1:])
    det["50_sgs_phase_only"] = {"iters": int(s.info_iter_num), "stop_reason": int(s.stop_reason), "stats": s.infeasibility_stats()}
    del s
    res["pusht_infeasible"] = det
    # guard values and ratios the check sees on the feasible fixtures (interval 50; none of them fires)
    fx = {"planarhand_n1": ("planarhand_n1", (5000, 1e-3, 0, 50, 100, 11000, 1.05)),
          "ros_2000": ("ros_2000", (20000, 1e-3, 0, 50, 100, 11000, 1.05)),
          "pusht_n10": ("pusht_n10", (20000, 1e-3, 0, 50, 100, 11000, 1.05)),
          "pendulum_n80": ("pendulum_n80", (3000, 1e-12, 0, 50, 100, 11000, 1.05))}
    feas = {}
    for name, (fix, args) in fx.items():
        s = solver(load_fixture(fix), 50)
        s.solve(*args)
        feas[name] = {"iters": int(s.info_iter_num), "stop_reason": int(s.stop_reason), "stats": s.infeasibility_stats()}
        del s
    feas["c2b_1000"] = {"iters": a.iters, "stop_reason": stops[50][1], "stats": res["c2b_check_stats"]["50"]}
    res["feasible_fixtures"] = feas
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
