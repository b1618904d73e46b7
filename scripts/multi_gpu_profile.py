"""torchrun worker: stage breakdown of the sharded solver (run_iterations_ex) on the bench workload.
   torchrun --nproc-per-node N scripts/multi_gpu_profile.py"""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch, torch.distributed as dist
import cuadmm_b200 as cu
from cuadmm_b200.synthetic import chain_sdp, c2b_blocks
rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
P = chain_sdp(c2b_blocks(2000, 6, 60, 0), 700000, seed=0)
s = cu.Solver(verbose=False); s.set_device(local)
if world > 1:
    idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        idt.copy_(torch.frombuffer(bytearray(cu.unique_id()), dtype=torch.uint8))
    dist.broadcast(idt, 0)
    s.set_distributed(rank, world, bytes(idt.cpu().numpy().tolist()))
s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"], P["C_idx"], P["C_val"], P["blk"])
s.solve(1, -1.0, 500, 50, 100, 1 << 30, 1.05)
s.run_iterations(30, sgs=True)
r = s.run_iterations(100, sgs=True)
e = s.run_iterations_ex(50, sgs=True)
if rank == 0:
    print(json.dumps({"world": world, "ms_per_iter": r["total_ms"] / 100,
                      "profiled": {k: v / 50 for k, v in e.items()}}), flush=True)
s.close()
if world > 1:
    dist.barrier(); dist.destroy_process_group()
