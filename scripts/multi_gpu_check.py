"""torchrun worker: the sharded solver on N GPUs must reproduce the single-GPU trajectory.
   torchrun --nproc-per-node N scripts/multi_gpu_check.py"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch, torch.distributed as dist
import cuadmm_b200 as cu
from cuadmm_b200.synthetic import chain_sdp, c2b_blocks
rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local); os.environ["CUADMM_DEVICE"] = str(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
if rank == 0:
    idt.copy_(torch.frombuffer(bytearray(cu.unique_id()), dtype=torch.uint8))
dist.broadcast(idt, 0)
job_id = bytes(idt.cpu().numpy().tolist())
nblk = int(os.environ.get("NBLK", "200")); con = int(os.environ.get("CON", "40000")); iters = int(os.environ.get("ITERS", "60"))
P = chain_sdp(c2b_blocks(nblk, 6, 60, 0), con, seed=0)
def make(distributed):
    s = cu.Solver(verbose=False)
    if distributed: s.set_distributed(rank, world, job_id)
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"], P["C_idx"], P["C_val"], P["blk"])
    return s
sd = make(True)
sd.solve(iters, 1e-12, 500, 50, 100, 11000, 1.05)
Xd, yd, Sd = sd.X, sd.y, sd.S
r = sd.run_iterations(30, sgs=True)
if rank == 0:
    s1 = make(False)
    s1.solve(iters, 1e-12, 500, 50, 100, 11000, 1.05)
    X1, S1 = s1.X, s1.S
    r1 = s1.run_iterations(30, sgs=True)
    ok = True
    for k in ["errRp", "errRd", "pobj", "dobj", "sig"]:
        a, b = sd.history(k), s1.history(k)
        err = np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-12))
        print(k, "max rel diff vs 1 GPU", err)
        ok = ok and err < 1e-7
    ex = np.linalg.norm(Xd - X1) / np.linalg.norm(X1); es = np.linalg.norm(Sd - S1) / np.linalg.norm(S1)
    print("X rel diff", ex, "S rel diff", es)
    ok = ok and ex < 1e-8 and es < 1e-8
    print("MULTI_GPU_OK" if ok else "MULTI_GPU_MISMATCH", "world", world, "ms/iter sharded", r["total_ms"] / 30, "single", r1["total_ms"] / 30)
dist.barrier()
dist.destroy_process_group()
