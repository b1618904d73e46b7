#!/usr/bin/env python
"""cones_probe.py — measurements of the linear-cone ('l' / 'u') path on the GPU; writes profiles/cones_probe_r03.json
(or --out) with the GPU name and power limit read in the same run.

  1. proj_linear_kernel device time for N = 1e6, 1e7, 1e8 nonnegative entries as one 'l' block, without the epilogue
     (B_alg = 16 B per entry: read Xb, write Xproj) and with the solver's fused epilogue (56 B: also read X, Rd1, C,
     write S, S - C); the same N as N 1x1 PSD blocks while such a plan fits (host plan ~100 B per block).  CUDA events
     around REPS back-to-back calls; the buffers rotate over sets whose total exceeds 3x the 126 MB L2, so every call
     reads from HBM.  GB/s against B_alg and against the measured HBM peak of DESIGN.md section 3 (6,555.8 GB/s).
  2. sGS iterations per second of a typed synthetic problem (PSD blocks plus a large 'l' part and a 'u' part), split
     by cuadmm_solver_run_iterations_ex, next to the same PSD blocks without the linear part.

    python scripts/cones_probe.py [--out PATH] [--reps 50]
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

HBM_PEAK_GBS = 6555.8          # DESIGN.md section 3, measured on a B200
L2_BYTES = 126 * 2**20


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()
        name, plim, smax = [x.strip() for x in out[0].split(",")]
        return dict(name=name, power_limit=plim, sm_max_clock=smax)
    except Exception as e:   # the record says so rather than guessing
        return dict(error=repr(e))


def time_projection(plan, N, bytes_per_entry, epilogue, reps):
    import torch
    nvec = 7 if epilogue else 2
    nsets = max(1, int(np.ceil(3 * L2_BYTES / (N * 8 * nvec))))
    g = torch.Generator(device="cuda").manual_seed(0)
    sets = []
    for _ in range(nsets):
        v = [torch.randn(N, dtype=torch.float64, device="cuda", generator=g) for _ in range(nvec)]
        sets.append(v)
    sig = torch.tensor([1.3], dtype=torch.float64, device="cuda")

    def call(i):
        v = sets[i % nsets]
        if epilogue:
            plan.project_epilogue_device(v[0].data_ptr(), v[1].data_ptr(), v[2].data_ptr(), v[3].data_ptr(),
                                         v[4].data_ptr(), v[5].data_ptr(), v[6].data_ptr(), sig.data_ptr())
        else:
            plan.project_device(v[0].data_ptr(), v[1].data_ptr())

    for i in range(max(3, nsets)):
        call(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        call(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    gbs = bytes_per_entry * N / (ms * 1e-3) / 1e9
    del sets
    torch.cuda.empty_cache()
    return dict(ms=ms, gb_per_s_vs_b_alg=gbs, frac_of_hbm_peak=gbs / HBM_PEAK_GBS, buffer_sets=nsets,
                working_set_mb=nsets * N * 8 * nvec / 2**20, launches=int(plan.last_launches))


def part1(reps):
    import cuadmm_b200 as cu
    rows = []
    for N in (10**6, 10**7, 10**8):
        p = cu.Plan([N], device=0, types="l")
        for epi, B in ((False, 16), (True, 56)):
            r = time_projection(p, N, B, epi, reps)
            r.update(N=N, layout="one 'l' block", epilogue=epi, b_alg_bytes_per_entry=B)
            rows.append(r)
            print(json.dumps(r), flush=True)
        p.close()
        if N <= 10**7:
            t0 = time.time()
            q = cu.Plan(np.ones(N, np.int32), device=0)
            build_s = time.time() - t0
            for epi, B in ((False, 16), (True, 56)):
                r = time_projection(q, N, B, epi, max(5, reps // 5))
                r.update(N=N, layout="N 1x1 's' blocks", epilogue=epi, b_alg_bytes_per_entry=B, plan_build_s=build_s)
                rows.append(r)
                print(json.dumps(r), flush=True)
            q.close()
        else:
            rows.append(dict(N=N, layout="N 1x1 's' blocks", skipped="a host plan of 1e8 blocks needs ~10 GB of "
                                                                     "host memory (descriptors, offsets, pooled layout)"))
    return rows


def part2():
    import cuadmm_b200 as cu
    import cones_util as cz
    from cuadmm_b200.synthetic import c2b_blocks
    rng_blk = c2b_blocks(300, 6, 60, 0)
    psd = [("s", int(n)) for n in rng_blk]
    out = []
    for name, blocks in (("psd only", psd), ("psd + l 2e6 + u 2e5", psd + [("l", 2_000_000), ("u", 200_000)])):
        P = cz.typed_synthetic(blocks, 60000, seed=0)
        s = cu.Solver(verbose=False)
        s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
               P["C_idx"], P["C_val"], P["blk"], blk_types=P["types"])
        s.solve(1, 1e-12, 500, 50, 100, 11000, 1.05)
        s.run_iterations(20, sgs=True)
        t = s.run_iterations(200, sgs=True)
        ex = s.run_iterations_ex(200, sgs=True)
        r = dict(problem=name, vec_len=P["vec_len"], con_num=P["con_num"], nblk=len(blocks),
                 sgs_iter_per_s=200 / (t["total_ms"] * 1e-3), ms_per_iter=t["total_ms"] / 200,
                 split_ms_per_iter={k: v / 200 for k, v in ex.items()}, launches=int(s.launches))
        out.append(r)
        print(json.dumps(r), flush=True)
        s.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cones_probe_r03.json"))
    ap.add_argument("--reps", type=int, default=50)
    a = ap.parse_args()
    import cuadmm_b200 as cu
    if cu.device_count() == 0:
        raise SystemExit("cones_probe: no CUDA device (there is no CPU measurement path)")
    rec = dict(gpu=gpu_info(), hbm_peak_gb_per_s=HBM_PEAK_GBS, projection=part1(a.reps), solver=part2())
    rec["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(rec, open(a.out, "w"), indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
