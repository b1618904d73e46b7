"""Linear ('l') and free ('u') blocks on the GPU: the linear-cone projection kernel inside typed plans, the solver on
typed problems against the typed oracle (tests/cones_util.py) and against scipy's LP solver, cuadmm_exe on a typed TXT
directory, and the block-sharded solver on 2 and 3 ranks."""
import os
import subprocess

import numpy as np
import pytest

import cuadmm_b200 as cu
import cones_util as cz
import oracle_np as onp
from test_gpu_multi import launch
from util_problems import ROOT, parse_log

pytestmark = pytest.mark.gpu

# PSD blocks {1, 7, 40, 100, 200 (dense path)} between linear and free blocks; odd lengths put later blocks at odd
# offsets, the 9,000-entry 'l' block spans several chunks of the kernel
MIX = [("l", 37), ("s", 1), ("u", 5), ("s", 7), ("l", 1), ("s", 40), ("u", 1000), ("s", 100), ("l", 9003),
       ("s", 200), ("u", 3), ("l", 2)]


def _plan(blocks, **kw):
    return cu.Plan([n for _, n in blocks], device=0, types="".join(t for t, _ in blocks), **kw)


def _check_projection(blocks, x, out, rank=0):
    blk = [n for _, n in blocks]
    types = "".join(t for t, _ in blocks)
    off = cz.svec_offsets(blk, types)
    for k, (t, n) in enumerate(blocks):
        seg, xin = out[off[k]:off[k + 1]], x[off[k]:off[k + 1]]
        if t == "l":
            assert np.array_equal(seg, np.maximum(xin, 0.0)), k
        elif t == "u":
            assert np.array_equal(seg, xin), k
        else:
            ref = onp.project_svec_rank([n], xin, rank) if rank else onp.project_svec([n], xin)
            assert np.max(np.abs(seg - ref)) <= 1e-9 * max(1.0, np.linalg.norm(ref)), (k, n)


def _typed_input(blocks, seed):
    rng = np.random.default_rng(seed)
    parts = []
    for t, n in blocks:
        if t == "s":
            G = rng.standard_normal((n, n))
            parts.append(onp.svec((G + G.T) / 2))
        else:
            parts.append(rng.standard_normal(n))
    return np.concatenate(parts)


@pytest.mark.parametrize("blocks", [MIX, [("l", 5000)], [("u", 777)], [("u", 3), ("l", 4097), ("u", 1), ("l", 9)]],
                         ids=["mix", "l_only", "u_only", "l_and_u"])
def test_typed_projection_without_epilogue(blocks):
    p = _plan(blocks)
    x = _typed_input(blocks, 1)
    out, eig, sweeps = p.project_eig_host(x)
    _check_projection(blocks, x, out)
    # eigenvalue slots of 'l' / 'u' blocks are NaN, their sweep counts 0; 's' blocks as before
    o = 0
    for k, (t, n) in enumerate(blocks):
        if t != "s":
            assert np.all(np.isnan(eig[o:o + n])) and sweeps[k] == 0
        else:
            assert not np.any(np.isnan(eig[o:o + n]))
        o += n
    assert len(eig) == sum(n for _, n in blocks)
    out2 = p.project_host(x)
    _check_projection(blocks, x, out2)
    assert p.last_launches >= 1
    if all(t != "s" for t, _ in blocks):
        assert p.last_launches == 1        # one launch for every linear chunk, no Jacobi class at all


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("blocks", [MIX, [("u", 3), ("l", 4097), ("u", 1), ("l", 9)]], ids=["mix", "l_and_u"])
def test_typed_projection_with_epilogue(blocks, offset):
    import torch
    p = _plan(blocks)
    x = _typed_input(blocks, 2)
    L = len(x)
    rng = np.random.default_rng(3)
    X, Rd1, Cv = rng.standard_normal(L), rng.standard_normal(L), rng.standard_normal(L)
    Cv[::7] = 0.0
    sig = 1.7
    # offset 1: every vector starts 8 bytes past a 16-byte boundary (the kernel's scalar path)
    def dev(v):
        t = torch.zeros(L + 1, dtype=torch.float64, device="cuda")
        t[offset:offset + L] = torch.from_numpy(v)
        return t
    dXb, dX, dR, dC = dev(x), dev(X), dev(Rd1), dev(Cv)
    dP, dS, dSmC = dev(np.zeros(L)), dev(np.full(L, np.nan)), dev(np.full(L, np.nan))
    dsig = torch.tensor([sig], dtype=torch.float64, device="cuda")
    ptr = lambda t: t.data_ptr() + 8 * offset
    p.project_epilogue_device(ptr(dXb), ptr(dP), ptr(dX), ptr(dR), ptr(dC), ptr(dS), ptr(dSmC), dsig.data_ptr())
    torch.cuda.synchronize()
    host = lambda t: t[offset:offset + L].cpu().numpy()
    out, S, SmC = host(dP), host(dS), host(dSmC)
    _check_projection(blocks, x, out)
    off = cz.svec_offsets([n for _, n in blocks], "".join(t for t, _ in blocks))
    for k, (t, n) in enumerate(blocks):
        sl = slice(off[k], off[k + 1])
        if t == "u":
            assert np.all(S[sl] == 0.0) and np.array_equal(SmC[sl], 0.0 - Cv[sl])
        elif t == "l":
            Sref = (out[sl] - X[sl]) / sig - Rd1[sl]
            assert np.array_equal(S[sl], Sref) and np.array_equal(SmC[sl], Sref - Cv[sl])
        else:
            Sref = (out[sl] - X[sl]) / sig - Rd1[sl]
            assert np.max(np.abs(S[sl] - Sref)) <= 1e-12 * max(1.0, np.linalg.norm(Sref))


def test_rank_limit_with_linear_blocks():
    blocks = [("l", 11), ("s", 12), ("u", 4), ("s", 30), ("l", 3)]
    p = _plan(blocks)
    p.set_rank_limit(3)
    x = _typed_input(blocks, 4)
    _check_projection(blocks, x, p.project_host(x), rank=3)


def test_all_psd_launch_count_unchanged():
    blk = [1, 7, 40, 100, 200, 7, 1]
    a = cu.Plan(blk, device=0)
    b = cu.Plan(blk, device=0, types="s" * len(blk))
    x = _typed_input([("s", n) for n in blk], 5)
    ra, rb = a.project_host(x), b.project_host(x)
    assert a.last_launches == b.last_launches
    # (two plans of the n = 200 block's sign iteration agree to rounding, not bit for bit)
    assert np.linalg.norm(ra - rb) <= 1e-12 * np.linalg.norm(rb)
    # adding linear blocks adds exactly one launch
    c = _plan([("s", n) for n in blk] + [("l", 100), ("u", 5)])
    c.project_host(np.concatenate([x, np.ones(105)]))
    assert c.last_launches == a.last_launches + 1


# ------------------------------------------------------------------ solver
def _solver(P, **kw):
    s = cu.Solver(verbose=False)
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
           P["C_idx"], P["C_val"], P["blk"], blk_types=P.get("types"), **kw)
    return s


def _compare_histories(s, o, n, rtol):
    for key in ["errRp", "errRd", "pobj", "dobj", "relgap", "sig"]:
        a, b = s.history(key)[:n], np.array(o.hist[key][:n])
        scale = np.maximum(np.abs(b), 1e-12 if key.startswith("err") or key == "relgap" else 1e-9)
        assert np.max(np.abs(a - b) / scale) < rtol, key


TYPED = [("s", 5), ("l", 30), ("s", 8), ("u", 6), ("s", 3), ("l", 12), ("s", 20), ("u", 9)]


@pytest.mark.parametrize("mode,graph", [("sgs", True), ("admm", True), ("sgs", False)])
def test_typed_solver_matches_oracle_iteration_by_iteration(mode, graph, monkeypatch):
    if not graph:
        monkeypatch.setenv("CUADMM_NO_GRAPH", "1")
    P = cz.typed_synthetic(TYPED, 60, seed=3)
    switch = 11000 if mode == "sgs" else 1
    iters = 60
    s = _solver(P)
    s.solve(iters, 1e-12, 500, 50, 100, switch, 1.05)
    o = cz.oracle_for(P)
    X, y, S, it = o.solve(iters, 1e-12, 500, 50, 100, switch, 1.05)
    assert s.info_iter_num == it == iters
    _compare_histories(s, o, iters, 1e-7)
    assert np.linalg.norm(s.X - X) <= 1e-8 * np.linalg.norm(X)
    assert np.linalg.norm(s.S - S) <= 1e-8 * max(np.linalg.norm(S), 1e-12)
    Aty = lambda yy: o.A.T @ (yy * o.normA / o.Cscale)
    assert np.linalg.norm(Aty(s.y) - Aty(y)) <= 1e-7 * max(np.linalg.norm(Aty(y)), 1e-12)
    free = o._free
    assert np.all(s.S[free] == 0.0)


def test_one_linear_block_equals_scalar_psd_blocks():
    # the same LP written as n 1x1 PSD blocks and as one 'l' block of n entries
    P = cz.random_lp(300, 0, 80, seed=7, density=0.05)
    n = int(P["blk"][0])
    Q = dict(P, blk=np.ones(n, np.int32), types=None)
    a, b = _solver(P), _solver(Q)
    a.solve(4000, 1e-7, 500, 50, 100, 11000, 1.05)
    b.solve(4000, 1e-7, 500, 50, 100, 11000, 1.05)
    assert a.info_iter_num == b.info_iter_num
    worst = 0.0
    for key in ["errRp", "errRd", "pobj", "dobj", "relgap", "sig"]:
        ha, hb = a.history(key), b.history(key)
        worst = max(worst, float(np.max(np.abs(ha - hb) / np.maximum(np.abs(hb), 1e-300))))
    dX = np.linalg.norm(a.X - b.X) / np.linalg.norm(b.X)
    dS = np.linalg.norm(a.S - b.S) / np.linalg.norm(b.S)
    # observed on a B200: 1207 iterations in both, history, X and S bit-identical (max differences 0): the 1x1 Jacobi
    # path returns max(x, 0) exactly.  The bound allows for per-iteration rounding that grows over the run.
    print("1x1 's' vs 'l': iterations %d, history max rel %.3e, X %.3e, S %.3e" % (a.info_iter_num, worst, dX, dS))
    assert worst <= 1e-10 and dX <= 1e-10 and dS <= 1e-10


def test_typed_synthetic_converges_to_known_optimum():
    P = cz.typed_synthetic([("s", 5), ("l", 30), ("s", 8), ("u", 6), ("s", 3), ("l", 12)], 40, seed=4)
    s = _solver(P)
    s.solve(20000, 1e-6, 500, 50, 100, 11000, 1.05)
    o = cz.oracle_for(P)
    X, y, S, it = o.solve(20000, 1e-6, 500, 50, 100, 11000, 1.05)
    assert it < 20000
    assert abs(s.info_iter_num - it) <= max(1, int(0.02 * it))
    pobj = s.history("pobj")[-1]
    assert abs(pobj - P["pstar"]) <= 1e-4 * (1 + abs(P["pstar"]))
    assert max(s.history("errRp")[-1], s.history("errRd")[-1], s.history("relgap")[-1]) < 1e-6
    _check_dual_slack(s.S, P)


def _check_dual_slack(S, P):
    off = cz.svec_offsets(P["blk"], P["types"])
    for k, t in enumerate(P["types"]):
        seg = S[off[k]:off[k + 1]]
        if t == "u":
            assert np.all(seg == 0.0)
        elif t == "l":
            # the 'l' slack is the PSD blocks' arithmetic (Xproj - X)/sig - Rd1, not a clamp: nonnegative to rounding
            assert seg.min() >= -1e-10 * max(1.0, np.abs(seg).max())


@pytest.mark.parametrize("n_free", [0, 8])
def test_lp_matches_linprog(n_free):
    P = cz.random_lp(40, n_free, 15, seed=1)
    f = cz.linprog_objective(P)
    s = _solver(P)
    s.solve(20000, 1e-6, 500, 50, 100, 11000, 1.05)
    assert abs(s.history("pobj")[-1] - f) <= 1e-4 * (1 + abs(f))
    o = cz.oracle_for(P)
    X, y, S, it = o.solve(20000, 1e-6, 500, 50, 100, 11000, 1.05)
    assert abs(s.info_iter_num - it) <= max(1, int(0.02 * it))
    _check_dual_slack(s.S, P)


def test_exe_on_typed_txt_directory(tmp_path):
    P = cz.typed_synthetic(TYPED, 50, seed=2)
    d = str(tmp_path / "typed")
    cz.write_txt(P, d)
    assert "l 30" in open(os.path.join(d, "blk.txt")).read() and "u 6" in open(os.path.join(d, "blk.txt")).read()
    exe = os.path.join(ROOT, "cuadmm_b200", "lib", "cuadmm_exe")
    out = subprocess.run([exe, d + "/", "--max-iter", "300", "--tol", "1e-5"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    assert "vector length: %d" % P["vec_len"] in out.stdout
    assert parse_log(out.stdout)
    X = np.loadtxt(os.path.join(d, "X_opt.txt"))
    prob = cu.Problem(d + "/")
    assert prob.blk_types == P["types"]
    s = cu.Solver(verbose=False)
    s.init_from_problem(prob)
    s.solve(300, 1e-5, 0, 50, 100, 5000, 1.05)
    assert X.shape == (P["vec_len"],) and np.allclose(X, s.X, rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_typed_solver_matches_single_gpu(world):
    procs, outs = launch(world, "cones_rank_worker.py")
    assert "CONES_RANK_OK" in outs[0], "\n".join(o[-3000:] for o in outs)
    assert all(p.returncode == 0 for p in procs), "\n".join(o[-3000:] for o in outs)
