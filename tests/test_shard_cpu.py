"""Multi-GPU host logic on CPU: block sharding, local index maps and column slices, and the data path
of one sharded operator application with a world_size-2 gloo all-reduce (no GPU needed)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import cuadmm_b200 as cu
from cuadmm_b200.synthetic import chain_sdp, c2b_blocks, svec_offsets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shards_partition_the_svec_vector():
    blk = c2b_blocks(300, 6, 60, 1)
    off = svec_offsets(blk)
    world = 4
    shards = [cu.Shard(blk, world, r) for r in range(world)]
    allglob = np.concatenate([s.loc2glob for s in shards])
    assert sorted(allglob.tolist()) == list(range(int(off[-1])))          # disjoint cover
    owner = shards[0].owner
    for r, s in enumerate(shards):
        assert np.array_equal(s.owner, owner)
        ids = np.nonzero(owner == r)[0]
        assert np.array_equal(s.local_block_ids, ids) and np.array_equal(s.local_blk, blk[ids])
        exp = np.concatenate([np.arange(off[k], off[k + 1]) for k in ids])
        assert np.array_equal(s.loc2glob, exp)                            # blocks keep their order and layout
    cost = np.array([float(b) ** 3 for b in blk])
    loads = np.array([cost[owner == r].sum() for r in range(world)])
    assert loads.max() / loads.mean() < 1.05


def test_column_slices_reassemble_the_operator():
    P = chain_sdp(c2b_blocks(60, 6, 30, 2), 900, seed=3)
    m, n = P["con_num"], P["vec_len"]
    A = sp.csr_matrix((P["vals"], P["row_ids"], P["col_ptrs"]), shape=(m, n))
    rng = np.random.default_rng(0)
    x = rng.standard_normal(n); y = rng.standard_normal(m)
    world = 3
    acc = np.zeros(m); aty = np.zeros(n)
    for r in range(world):
        s = cu.Shard(P["blk"], world, r)
        cp, ri, v = s.slice_csc(P["col_ptrs"], P["row_ids"], P["vals"])
        Ag = sp.csr_matrix((v, ri, cp), shape=(m, s.vec_len_local))
        acc += Ag @ x[s.loc2glob]                 # what the reduction over the ranks sums
        aty[s.loc2glob] = Ag.T @ y                # A^T y needs no communication
    assert np.allclose(acc, A @ x, rtol=0, atol=1e-12 * np.abs(A @ x).max())
    assert np.allclose(aty, A.T @ y, rtol=0, atol=1e-12 * np.abs(A.T @ y).max())


CUADMM_EINVAL = -1


def test_job_ids_need_no_gpu():
    # cuadmm_nccl_unique_id stays for callers of the removed NCCL transport and makes the same kind of id
    ids = [cu.unique_id(), cu.unique_id(), cu.nccl_unique_id(), cu.nccl_unique_id()]
    assert all(isinstance(i, bytes) and len(i) == 128 for i in ids)
    assert len(set(ids)) == 4


@pytest.mark.parametrize("comm", [None, "peer", "nccl"])
def test_set_distributed_rejects_the_removed_nccl_transport(monkeypatch, comm):
    # a job launched with CUADMM_COMM=nccl must fail, not run the peer-memory transport under the NCCL label
    if comm is None:
        monkeypatch.delenv("CUADMM_COMM", raising=False)
    else:
        monkeypatch.setenv("CUADMM_COMM", comm)
    s = cu.Solver(verbose=False)
    if comm == "nccl":
        with pytest.raises(cu.CuadmmError) as e:
            s.set_distributed(0, 2, cu.unique_id())
        assert e.value.code == CUADMM_EINVAL and "NCCL transport was removed" in str(e.value)
    else:
        s.set_distributed(0, 2, cu.unique_id())
    s.close()


WORKER = r'''
import os, sys
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "oracle"))
import numpy as np, scipy.sparse as sp, torch, torch.distributed as dist
import cuadmm_b200 as cu, oracle_np as onp
from cuadmm_b200.synthetic import chain_sdp
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
blk = np.array([5, 8, 3, 12, 6, 6, 9, 7, 4, 10], np.int32)
P = chain_sdp(blk, 60, seed=4)
m, n = P["con_num"], P["vec_len"]
normA, vals = onp.get_normA(P["col_ptrs"], P["vals"])
A = sp.csr_matrix((vals, P["row_ids"], P["col_ptrs"]), shape=(m, n))
s = cu.Shard(blk, world, rank)
cp, ri, v = s.slice_csc(P["col_ptrs"], P["row_ids"], vals)
Ag = sp.csr_matrix((v, ri, cp), shape=(m, s.vec_len_local))
lin = onp.AATSolver(A, 1e-15)                       # replicated y-solve
rng = np.random.default_rng(1)
Xb = rng.standard_normal(n)
# one sharded half-iteration: local projection of the owned blocks, partial A x, all-reduce, y-solve
Xp_loc = onp.project_svec(s.local_blk, Xb[s.loc2glob])
part = torch.from_numpy(Ag @ Xp_loc)
dist.all_reduce(part)
y = lin.solve(part.numpy())
ref_Xp = onp.project_svec(blk, Xb)
ref_y = lin.solve(A @ ref_Xp)
assert np.allclose(Xp_loc, ref_Xp[s.loc2glob], rtol=0, atol=1e-13)
assert np.allclose(y, ref_y, rtol=1e-10, atol=1e-12 * np.abs(ref_y).max())
full = torch.zeros(n, dtype=torch.float64); full[torch.from_numpy(s.loc2glob)] = torch.from_numpy(Xp_loc)
dist.all_reduce(full)                               # gather_full
assert np.allclose(full.numpy(), ref_Xp, rtol=0, atol=1e-13)
sys.stdout.write("RANK%dOK\n" % rank); sys.stdout.flush()
'''


def test_two_rank_gloo_data_path(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29517", str(script), ROOT],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    assert "RANK0OK" in out.stdout and "RANK1OK" in out.stdout
