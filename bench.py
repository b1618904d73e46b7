#!/usr/bin/env python
"""bench.py — ADMM iterations/s of the cuADMM hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write X, y, S after the timed steps as DIR/*.npy

A "step" is one sGS-ADMM iteration (src/solver.cu:469-799 of the reference): two A A^T y-solves, three
SpMV with A, two with A^T, the PSD projection of every block and the residual / sigma update.  Workload
of `value`: BASELINE.json configs[1], "~2,000 PSD blocks of size 6-60" = 2,000 blocks, n_k ~ U{6..60}
(numpy default_rng(0)), m = 700,000 chain-structured sparse constraints (cuadmm_b200/synthetic.py),
FP64, synthetic data — the same at every N (strong scaling: the SDP is fixed, the ranks split its blocks).
The line also carries `scale_c4`: the same measurement on BASELINE.json configs[3] (10,000 blocks
{10,50,200,800}, m = 1e6), the configuration north_star names for 1 -> 8 GPU scaling.
One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")

import numpy as np  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nblk", type=int, default=2000)
    ap.add_argument("--con", type=int, default=700000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-scale-c4", action="store_true", help="skip the C4 sub-record (scale_c4)")
    ap.add_argument("--workload", default="c2b", choices=["c2b", "c3", "c4", "c5"],
                    help="c2b (default, BASELINE.json configs[1]); c3 = max-cut n=4000 (configs[2]); c4 = 10k mixed "
                         "blocks {10,50,200,800}, m=1e6 (configs[3], the multi-GPU scaling configuration); "
                         "c5 = 4 x 8000 + 500 small blocks (configs[4])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the iterate X, y, S the timed steps end on as DIR/<name>.npy (float64; a fixed seeded sample "
                         "of each when they exceed 64 MB together), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed; it does not apply to --impl reference")
    return args


def workload(name, args):
    from cuadmm_b200.synthetic import c2b_blocks, chain_sdp, maxcut_sdp, c4_blocks, c5_blocks, random_sdp
    if name == "c3":
        P = maxcut_sdp(4000, p=0.01, seed=0)
        return P, {"workload": "C3 max-cut SDP: one dense PSD block n=4000, G(n, 0.01) seed 0, m=n diagonal constraints, "
                               "sGS-ADMM iteration", "nblk": 1, "vec_len": int(P["vec_len"]), "con_num": int(P["con_num"]),
                   "nnz_A": int(len(P["vals"])), "l2": "one 128 MB dense block per n x n operand: exceeds the 126 MB L2"}
    if name == "c4":
        blk = c4_blocks(seed=0)
        m = args.con if args.con != 700000 else 1000000
        P = random_sdp(blk, m, seed=0)
        return P, {"workload": "C4 synthetic multi-block SDP: 10,000 blocks {10: 6000, 50: 3000, 200: 900, 800: 100} shuffled "
                               "(seed 0), m=%d constraints with 1+Poisson(4) non-zeros at random svec positions of <= 2 blocks, sGS-ADMM iteration" % m, "nblk": int(len(blk)),
                   "vec_len": int(P["vec_len"]), "con_num": int(P["con_num"]), "nnz_A": int(len(P["vals"])),
                   "l2": "svec vectors of 434 MB each: far beyond the 126 MB L2"}
    if name == "c5":
        blk = c5_blocks(seed=0)
        m = args.con if args.con != 700000 else 100000
        P = random_sdp(blk, m, seed=0, cheap_factors=True)
        return P, {"workload": "C5 DIMACS-style SDP: 4 blocks n=8000 + 500 blocks n~U{6..32} (seed 0), m=%d constraints built as C4, "
                               "sGS-ADMM iteration" % m, "nblk": int(len(blk)), "vec_len": int(P["vec_len"]),
                   "con_num": int(P["con_num"]), "nnz_A": int(len(P["vals"])), "l2": "svec vectors of 1 GB each: far beyond the 126 MB L2"}
    blk = c2b_blocks(args.nblk, 6, 60, 0)
    P = chain_sdp(blk, args.con, seed=0)
    cfg = {"workload": "C2b synthetic moment-relaxation SDP: %d PSD blocks n~U{6..60} (seed 0), m=%d chain-structured "
                       "constraints, sGS-ADMM iteration" % (args.nblk, args.con),
           "nblk": int(args.nblk), "vec_len": int(P["vec_len"]), "con_num": int(P["con_num"]), "nnz_A": int(len(P["vals"])),
           "l2": "per-iteration working set (8 svec vectors + A + At + L ~ 190 MB) exceeds the 126 MB L2; no flush, "
                 "iterations run back to back exactly as in the solver"}
    return P, cfg


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the GPU runs the benchmark's iterations
    (B200_PROFILING.md recipe).  Started before the warm-up and stopped after the timed region and the profiled
    pass, so that even a 30 ms timed region is covered by samples taken under the same load."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def count(self):
        return len(self.rows)

    def stop(self, t_load0=None, t_load1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if (t_load0 is None or t >= t_load0) and (t_load1 is None or t <= t_load1 + 0.05)]
        if not rows:
            rows = [r for (_, r) in self.rows]
        sm = [float(r[1]) for r in rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons),
                "window": "samples taken while the GPU ran this workload's iterations (warm-up, timed region, profiled pass)"}


def ncu_traffic(name, args):
    """dram__bytes_read.sum + dram__bytes_write.sum of the projection stage from the committed ncu --set full
    capture; only valid for the workload it was taken on, else None"""
    for fn in ("ncu_traffic_r02.json", "ncu_traffic_r01.json"):
        p = os.path.join(ROOT, "profiles", fn)
        try:
            d = json.load(open(p))
            if name == "c2b" and d["workload"]["nblk"] == args.nblk and d["workload"]["con"] == args.con and args.gpus == 1:
                st = d["projection_stage"]
                return int(st["dram_bytes_read"] + st["dram_bytes_write"]), "profiles/" + fn
        except Exception:
            pass
    return None, None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def fp64_peak_tflops(torch):
    """FP64 peak the projection is held against: cuBLAS DGEMM 8192^3 timed here with CUDA events (best of 4);
    MEASURED_PEAKS.json holds no FP64 figure, so the denominator is measured in the run that uses it"""
    try:
        n = 8192
        a = torch.randn(n, n, dtype=torch.float64, device="cuda"); b = torch.randn(n, n, dtype=torch.float64, device="cuda")
        torch.matmul(a, b)
        best = 0.0
        for _ in range(4):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
            best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        del a, b
        torch.cuda.empty_cache()
        return best, "cuBLAS DGEMM 8192^3 (torch.matmul f64) timed in this run, best of 4"
    except Exception as ex:
        return 35.5, "fallback: 35.5 TFLOP/s (cuBLAS DGEMM 8192^3 measured on this pool in round 1); live probe failed: %s" % ex


# ---------------------------------------------------------------------------------------------
# CPU legs: the port of the reference's CPU path — LAPACK dsyevd on a std::thread pool in C++
# (oracle/cpu_baseline.cpp) inside the oracle's ADMM iteration, sparse solves by SuperLU
# (CHOLMOD-substitute).  The only places bench.py may execute oracle/ (cpu_baseline and --impl reference).
# ---------------------------------------------------------------------------------------------
def cpu_reference_iterations(P, n_iters, threads, budget_s=None):
    """n_iters timed iterations; with budget_s, fewer when they would run longer than budget_s seconds (at least one)"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_np as onp
    blk = np.ascontiguousarray(P["blk"], np.int32)
    proj = lambda v: onp.project_svec_cpp(blk, v, threads)
    t0 = time.time()
    o = onp.ADMMOracle(P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
                       P["C_idx"], P["C_val"], blk, project=proj)
    t_init = time.time() - t0
    o.solve(1, -1.0, 500, 50, 100, 1 << 30, 1.05)          # one untimed iteration
    done, t0 = 0, time.time()
    while done < n_iters and (budget_s is None or done == 0 or time.time() - t0 < budget_s):
        o.solve(1, -1.0, 500, 50, 100, 1 << 30, 1.05)
        done += 1
    dt = time.time() - t0
    return done / dt, dt, t_init, done


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    P, cfg = workload(args.workload, args)
    cores = os.cpu_count() or 1
    threads = min(30, cores)          # the reference's default cpu_eig_thread_num (src/main.cu:11)
    val, dt, t_init, steps = cpu_reference_iterations(P, max(1, args.steps), threads)     # exactly --steps timed iterations
    line = {"impl": "reference", "metric": "ADMM iterations/s", "value": val, "unit": "iter/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": 1, "ms_per_step": 1e3 / val, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": val, "unit": "iter/s", "cores": threads, "kind": "port",
                             "sample": "%d sGS-ADMM iterations of the same workload after 1 untimed (%.1f s): projection = LAPACK "
                                       "dsyevd + dgemm (OpenBLAS, 1 thread per call) on a %d-thread std::thread pool in C++ "
                                       "(oracle/cpu_baseline.cpp, restating src/duo_solver.cu:346-371,578-619), SpMV by scipy "
                                       "CSR kernels, A A^T solves by SuperLU (CHOLMOD-substitute); init %.1f s not counted"
                                       % (steps, dt, threads, t_init)},
            "e2e": {"value": val, "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "host_cores": cores}
    # Baseline A (informational): the reference's own cuSOLVER projection stage (src/solver.cu:531-647,
    # unmodified reference sources in oracle/_ref) on GPU 0 of this box, same blocks, same input
    try:
        import ctypes as C
        ref = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libcuadmm_ref.so"))
        ref.ref_proj_create.restype = C.c_void_p
        ref.ref_proj_run.restype = C.c_double
        from cuadmm_b200.synthetic import random_svec
        blk = np.ascontiguousarray(P["blk"], np.int32)
        x = random_svec(blk, seed=0)
        h = ref.ref_proj_create(blk.ctypes.data_as(C.POINTER(C.c_int)), len(blk), 15)
        ms = ref.ref_proj_run(C.c_void_p(h), x.ctypes.data_as(C.POINTER(C.c_double)), None, 2)
        ref.ref_proj_destroy(C.c_void_p(h))
        line["baseline_A_cusolver_projection_ms"] = ms
    except Exception as ex:
        line["baseline_A_cusolver_projection_ms"] = None
        line["baseline_A_note"] = "oracle/_ref not usable here: %s" % ex
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
class Job:
    """rank / world plumbing: torch.distributed (NCCL) for barriers and max-over-ranks, the solver's own peer-memory
    transport for the data path"""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, v):
        if self.dist is None:
            return float(v)
        t = self.torch.tensor([v], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def job_id(self, cu):
        """128-byte id of one sharded solver, created on rank 0 and broadcast"""
        torch = self.torch
        nccl = os.environ.get("CUADMM_COMM", "peer") == "nccl"
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if self.rank == 0:
            raw = cu.nccl_unique_id() if nccl else cu.unique_id()
            idt.copy_(torch.frombuffer(bytearray(raw), dtype=torch.uint8))
        self.dist.broadcast(idt, 0)
        return bytes(idt.cpu().numpy().tolist())


DUMP_BYTES = 60_000_000     # data of all dumped arrays; with the .npy headers under 64 MB


def dump_outputs(out_dir, arrays):
    """arrays (name -> float64 vector) as out_dir/<name>.npy.  Beyond DUMP_BYTES in all, every array keeps the same
    fraction k of its entries: one per stratum [i n // k, (i+1) n // k), at an offset drawn by default_rng(0), so the
    indices are sorted and distinct.  They depend only on the array's length: runs with the same arguments sample the
    same entries."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            k = len(a) * DUMP_BYTES // total
            lo = np.arange(k + 1, dtype=np.int64) * len(a) // k
            a = a[lo[:-1] + (np.random.default_rng(0).random(k) * np.diff(lo)).astype(np.int64)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure(job, cu, P, steps, warmup, e2e_steps, sampler=None, keep_outputs=False):
    """init + K timed iterations (+ the iterate they end on, read back to the host) + profiled pass (+ e2e) of one
    workload on job.world GPUs"""
    torch = job.torch
    s = cu.Solver(verbose=False)
    s.set_device(job.local)
    if job.world > 1:
        s.set_distributed(job.rank, job.world, job.job_id(cu))
    t0 = time.time()
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
           P["C_idx"], P["C_val"], P["blk"], None, None, None, 1.0)
    t_init = time.time() - t0
    s.solve(1, -1.0, 500, 50, 100, 1 << 30, 1.05)          # sets the run parameters (1 iteration)
    t_load0 = time.time()
    s.run_iterations(max(warmup, 3), sgs=True)              # untimed warm-up
    launches0 = s.launches
    job.barrier()
    r = s.run_iterations(steps, sgs=True)                   # EXACTLY K timed steps, CUDA events on the solver stream
    job.barrier()
    ms_total = job.max(r["total_ms"])
    launches = s.launches - launches0
    # read before the profiled pass moves the iterate on; X and S are gathered over the ranks, so all of them read
    outputs = {"X": s.X, "y": s.y, "S": s.S} if keep_outputs else None
    # stage breakdown (separate profiled pass: events around every y-solve and projection)
    nprof = min(steps, 50)
    prof = s.run_iterations(nprof, sgs=True, profile=True)
    if sampler is not None:
        # keep the GPU under the same load for ~0.6 s more so that nvidia-smi (50 ms period) delivers samples even when
        # the timed region is a few tens of ms; the count is derived from the max-reduced time: identical on all ranks
        extra = int(max(0, min(5000, 600.0 / max(ms_total / steps, 1e-3))))
        if extra:
            s.run_iterations(extra, sgs=True)
    t_load1 = time.time()
    out = {"ms_total": ms_total, "launches": int(launches), "init_s": t_init,
           "stage": {"projection": prof["projection_ms"] / nprof, "ysolve_x2": prof["ysolve_ms"] / nprof,
                     "spmv_and_rest": prof["other_ms"] / nprof},
           "t_load": (t_load0, t_load1), "ysolve": s.ysolve_stats(), "outputs": outputs}
    if e2e_steps > 0:
        # e2e: the same iteration through the public C ABI with HOST buffers — every step uploads the iterate
        # (X, y, S) from pinned host memory, runs one iteration (solve(max_iter=1, if_first=False), the
        # reference's warm-restart path src/solver.cu:385-409) and downloads X, y, S.
        n, m = P["vec_len"], P["con_num"]
        hX = torch.zeros(n, dtype=torch.float64).pin_memory(); hy = torch.zeros(m, dtype=torch.float64).pin_memory()
        hS = torch.zeros(n, dtype=torch.float64).pin_memory()
        aX, ay, aS = hX.numpy(), hy.numpy(), hS.numpy()
        s.get_into(aX, ay, aS)
        for _ in range(2):
            s.set_XyS(aX, ay, aS, 1.0); s.solve(1, -1.0, 500, 50, 100, 1 << 30, 1.05, if_first=False); s.get_into(aX, ay, aS)
        job.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            s.set_XyS(aX, ay, aS, 1.0)
            s.solve(1, -1.0, 500, 50, 100, 1 << 30, 1.05, if_first=False)
            s.get_into(aX, ay, aS)
        torch.cuda.synchronize()
        out["e2e_dt"] = job.max(time.perf_counter() - t0)
        out["e2e_steps"] = e2e_steps
        del hX, hy, hS
    if job.dist is not None:
        job.dist.barrier()
    s.close()
    return out


def run_ours(args):
    import cuadmm_b200 as cu
    if cu.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device — the CUDA extension has no CPU fallback")
    job = Job()
    torch = job.torch
    rank, world = job.rank, job.world
    fp64_peak, fp64_src = fp64_peak_tflops(torch)
    P, cfg = workload(args.workload, args)
    if world > 1:
        cfg["parallelism"] = ("blocks sharded over %d GPUs (LPT on eig cost); partial A x rows stored into the reducing rank's "
                              "staging area by the SpMV kernel and summed by a fused slice-reduction kernel over peer memory "
                              "(CUDA IPC / NVLink), dense-tail GEMV rows of the y-solve split over the ranks, sparse part of "
                              "the y-solve replicated" % world)
        if os.environ.get("CUADMM_COMM", "peer") == "nccl":
            cfg["parallelism"] = "blocks sharded over %d GPUs (LPT on eig cost), y-solve replicated, 2 NCCL all-reduces of m doubles per iteration" % world
    sampler = ClockSampler(job.local)
    if rank == 0:
        sampler.start()
    big = args.workload in ("c4", "c5")
    R = measure(job, cu, P, args.steps, args.warmup, max(3, min(args.steps, 10 if big else 30)), sampler,
                keep_outputs=args.dump_outputs is not None)
    clocks = sampler.stop(*R["t_load"]) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, R.pop("outputs"))     # after the clock window: files are written with the GPU idle

    # C4 sub-record: the configuration north_star names for multi-GPU scaling, measured the same way
    scale_c4 = None
    if args.workload == "c2b" and not args.no_scale_c4 and args.nblk == 2000 and args.con == 700000:
        P4, cfg4 = workload("c4", args)
        k4 = max(3, min(args.steps, 10))
        R4 = measure(job, cu, P4, k4, 3, 0)
        f4 = float(sum((20.0 / 3.0) * float(b) ** 3 for b in P4["blk"]))
        scale_c4 = {"metric": "ADMM iterations/s", "value": k4 / (R4["ms_total"] / 1e3), "unit": "iter/s", "n_gpus": args.gpus,
                    "steps": k4, "warmup": 3, "ms_per_step": R4["ms_total"] / k4, "scaling": "strong", "config": cfg4,
                    "stage_ms_per_iter": R4["stage"], "init_s": R4["init_s"], "gpu_launches": R4["launches"],
                    "roofline": {"kernel": "projection stage: sym_gemm (FP64 DMMA sign iteration, blocks n > 168) + proj_jacobi_kernel",
                                 "bound": "tensor", "achieved": f4 / world / (R4["stage"]["projection"] * 1e-3) / 1e12, "peak": fp64_peak,
                                 "unit": "TFLOP/s", "frac": f4 / world / (R4["stage"]["projection"] * 1e-3) / 1e12 / fp64_peak,
                                 "alg_flop_per_launch": f4 / world, "peak_source": fp64_src}}
        del P4
    if job.dist is not None:
        job.dist.barrier()
        job.dist.destroy_process_group()
    if rank != 0:
        return

    n, m = P["vec_len"], P["con_num"]
    hbm, hbm_src = measured_peaks()
    value = args.steps / (R["ms_total"] / 1e3)
    proj_ms = R["stage"]["projection"]
    alg_bytes = 56 * n                      # fused projection stage: reads Xb, X, Rd1, C; writes Xproj, S, SmC
    f_alg = float(sum((20.0 / 3.0) * float(b) ** 3 for b in P["blk"]))
    tf = f_alg / world / (proj_ms * 1e-3) / 1e12
    traffic, traffic_src = ncu_traffic(args.workload, args)
    line = {"metric": "ADMM iterations/s", "value": value, "unit": "iter/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": R["ms_total"] / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
            "clocks": clocks,
            "e2e": {"value": R["e2e_steps"] / R["e2e_dt"], "unit": "iter/s", "h2d_bytes_per_step": 8 * (2 * n + m),
                    "d2h_bytes_per_step": 8 * (2 * n + m), "steps": R["e2e_steps"],
                    "how": "per step: cuadmm_solver_set_XyS (pinned host -> device), cuadmm_solver_solve(max_iter=1, "
                           "if_first=0), cuadmm_solver_get_X/y/S (device -> pinned host); wall clock"},
            "gpu_launches": R["launches"],
            "stage_ms_per_iter": R["stage"], "ysolve": R["ysolve"], "init_s": R["init_s"]}
    if args.workload == "c2b":
        line["roofline"] = {
            "kernel": "proj_jacobi_kernel (fused svec->smat, one-sided Jacobi eig, clamp, rebuild, smat->svec, S/SmC "
                      "epilogue; all size classes of one projection stage)",
            "bound": "latency", "achieved": tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": tf / fp64_peak,
            "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": fp64_src, "alg_flop_per_launch": f_alg / world, "launch_ms": proj_ms,
            "hbm": {"achieved": alg_bytes / world / (proj_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                    "frac": alg_bytes / world / (proj_ms * 1e-3) / 1e9 / hbm, "alg_bytes_per_launch": alg_bytes / world,
                    "peak_source": hbm_src},
            "note": "The stage is bound by the serial rotation depth of the Jacobi sweeps and by instruction issue, by neither "
                    "roof (SURVEY 8d): `frac` is F_alg = (20/3) sum n^3 per second against the FP64 DGEMM peak; the `hbm` "
                    "sub-record is the same launch against the HBM roof (56 B per svec entry)"}
    else:
        # C3 / C4 / C5: the projection is dominated by the large blocks (n > 168), i.e. by the FP64 tensor-core (DMMA)
        # products of the sign iteration: tensor-bound, F_alg = (20/3) n^3 per block (SURVEY 8d)
        line["roofline"] = {"kernel": "projection stage: sym_gemm (FP64 DMMA sign iteration, blocks n > 168) + proj_jacobi_kernel",
                            "bound": "tensor", "achieved": tf, "peak": fp64_peak, "unit": "TFLOP/s",
                            "frac": tf / fp64_peak, "traffic": None, "peak_source": fp64_src,
                            "alg_flop_per_launch": f_alg / world, "launch_ms": proj_ms,
                            "note": "the sign iteration executes ~5x F_alg in symmetric products of n^3 flop each"}
    if scale_c4 is not None:
        line["scale_c4"] = scale_c4
    if not args.no_cpu_baseline and args.gpus == 1:
        cores = os.cpu_count() or 1
        threads = min(30, cores)
        try:
            val, dt, ti, done = cpu_reference_iterations(P, 8, threads, budget_s=25.0)
            line["cpu_baseline"] = {"value": val, "unit": "iter/s", "cores": threads, "kind": "port",
                                    "sample": "%d sGS-ADMM iterations of the same workload (after 1 untimed, %.1f s): projection = "
                                              "LAPACK dsyevd + dgemm on a %d-thread std::thread pool in C++ (oracle/cpu_baseline.cpp), "
                                              "SpMV by scipy, A A^T solves by SuperLU (CHOLMOD-substitute)" % (done, dt, threads)}
        except Exception as ex:   # the baseline is informational; never lose the GPU line over it
            line["cpu_baseline"] = {"value": None, "unit": "iter/s", "cores": threads, "kind": "port", "sample": "failed: %s" % ex}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
