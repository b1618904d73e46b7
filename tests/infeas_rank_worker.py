"""Worker of the sharded infeasibility tests (tests/test_gpu_infeas.py): one process per rank, launched by
test_gpu_multi.launch (ranks share GPU 0 when there is only one).  Every rank solves a feasible typed problem (1,500 iterations), a primal
infeasible and a dual infeasible one sharded with the check on at interval 50; rank 0 also solves them on one GPU and
compares stop iteration, stop reason and certificates.  The dual certificate is gathered collectively on every rank."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np  # noqa: E402
import cuadmm_b200 as cu  # noqa: E402
import infeas_util as iu  # noqa: E402

rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"])
job = bytes.fromhex(os.environ["JOB_ID"])
dev = rank % max(cu.device_count(), 1)
CASES = [("typed", iu.feasible_problems()["typed"], 2, (1500, 1e-6, 500, 50, 100, 11000, 1.05)),
         ("mix_classes_primal", iu.problems()["mix_classes_primal"][0], 3, (3000, 1e-6, 500, 50, 100, 11000, 1.05)),
         ("mix_dual", iu.problems()["mix_dual"][0], 4, (3000, 1e-6, 500, 50, 100, 11000, 1.05))]


def solve(P, args, distributed):
    s = cu.Solver(verbose=False)
    s.set_device(dev)
    if distributed:
        s.set_distributed(rank, world, job)
    s.set_infeasibility_check(50, 1e-7)
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
           P["C_idx"], P["C_val"], P["blk"], blk_types=P["types"])
    s.solve(*args)
    cert = s.certificate(0 if s.stop_reason == 3 else 1) if s.stop_reason in (3, 4) else None
    return s.info_iter_num, s.stop_reason, cert, s.infeasibility_stats()


ok = True
for name, P, reason, args in CASES:
    it, rs, cert, stats = solve(P, args, True)
    if rank == 0:
        it1, rs1, cert1, stats1 = solve(P, args, False)
        print("world", world, name, "sharded: reason %d at %d, single GPU: reason %d at %d" % (rs, it, rs1, it1))
        print("  checks %d / %d, projections %d+%d / %d+%d" % (stats["checks"], stats1["checks"], stats["primal_projections"],
              stats["dual_projections"], stats1["primal_projections"], stats1["dual_projections"]))
        ok = ok and rs == rs1 == reason and it == it1
        if cert is not None:
            v, r = cert
            v1, r1 = cert1
            err = float(np.linalg.norm(v - v1) / np.linalg.norm(v1))
            print("  certificate rel diff %.2e, ratio %.3e vs %.3e" % (err, r, r1))
            ok = ok and err <= 1e-10 and max(r, r1) <= 1e-7
print("rank", rank, "done")
if rank == 0 and ok:
    print("INFEAS_RANK_OK")
sys.exit(0 if ok else 1)
