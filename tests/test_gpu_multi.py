"""Multi-rank parity: the block-sharded solver (one process per rank, peer-memory transport) must reproduce the
single-GPU trajectory, iterates, y and stop iteration.  With one GPU the
ranks share it (CUDA IPC works between processes on the same device), so the sharded data path — SpMV rows pushed
to the reducing rank, slice reduction, split dense-tail GEMVs, gather by owner — is exercised on every box."""
import os
import subprocess
import sys

import pytest

import cuadmm_b200 as cu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def launch(world, worker, timeout=600, **extra_env):
    """one process per rank running tests/<worker> with a fresh job id; the processes and their outputs"""
    job = cu.unique_id().hex()
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), JOB_ID=job, CUADMM_PEER_TIMEOUT_S="20", **extra_env)
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", worker)], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=timeout)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
        outs.append(o)
    return procs, outs


@pytest.mark.parametrize("world,case", [(2, "sgs"), (2, "admm"), (2, "tol"), (2, "restart"), (3, "sgs"), (2, "mixed")])
def test_sharded_solver_matches_single_gpu(world, case):
    if cu.device_count() < 1:
        pytest.skip("needs a GPU")
    procs, outs = launch(world, "multi_rank_worker.py", CASE=case)
    assert "MULTI_RANK_OK" in outs[0], "\n".join(o[-3000:] for o in outs)
    assert all(p.returncode == 0 for p in procs), "\n".join(o[-3000:] for o in outs)
