"""Parity at the sizes BASELINE.json names (round-1 verdict, "close the parity holes"):
  * large blocks (C3 n = 4000, the n = 800 / 200 blocks of C4) against Baseline A — the reference's own cuSOLVER
    projection stage compiled from the unmodified reference sources into oracle/_ref — run here on the GPU box,
    1e-9 relative Frobenius (north_star's tolerance for the projected X);
  * ten solver iterations at the full C2b size against the ADMM oracle;
  * the stop iterations of the bundled examples against the reference's committed logs;
  * the MEX-shaped entry cuadmm_solve_matlab_like against the Solver API.
"""
import ctypes as C
import os

import numpy as np
import pytest

import cuadmm_b200 as cu
import oracle_np as onp
from conftest import random_svec, ip, dp
from util_problems import GOLD, load_fixture, make_solver, parse_log, synthetic_sdp

pytestmark = pytest.mark.gpu
X_TOL = 1e-9


def _baseline_A(oref, blk, x):
    h = oref.ref_proj_create(ip(blk), len(blk), 15)
    out = np.zeros_like(x)
    oref.ref_proj_run(C.c_void_p(h), dp(x), dp(out), 1)
    oref.ref_proj_destroy(C.c_void_p(h))
    return out


def test_c3_n4000_against_reference_cusolver(request):
    # BASELINE configs[2]: one dense block n = 4000; cusolverDnXsyevd + gemm (src/solver.cu:540-564, 600-644) is the oracle,
    # and LAPACK dsyevd (numpy) the one that needs no reference build
    blk = np.array([4000], np.int32)
    x = random_svec(blk, seed=6)
    ours = cu.Plan(blk).project_host(x)
    lap = onp.project_svec(blk, x)
    assert np.linalg.norm(ours - lap) <= X_TOL * np.linalg.norm(lap)
    ref = _baseline_A(request.getfixturevalue("oref"), blk, x)      # skips here when the reference build is absent
    assert np.linalg.norm(ours - ref) <= X_TOL * np.linalg.norm(ref)


def test_c4_large_blocks_against_reference_cusolver(request):
    # BASELINE configs[3] block shapes; the reference routes n = 200 and n = 800 through Xsyevd ("large"), whose
    # accuracy is ~1e-13, so those blocks are compared at 1e-9; its batched Jacobi (small blocks) stops at 1e-6
    blk = np.concatenate([np.full(6, 800), np.full(12, 200), np.full(10, 50), np.full(20, 10)]).astype(np.int32)
    np.random.default_rng(1).shuffle(blk)
    x = random_svec(blk, seed=9)
    plan = cu.Plan(blk)
    ours = plan.project_host(x)
    lap = onp.project_svec(blk, x)
    assert np.linalg.norm(ours - lap) <= X_TOL * np.linalg.norm(lap)
    ref = _baseline_A(request.getfixturevalue("oref"), blk, x)      # skips here when the reference build is absent
    sizes, nums, is_large = plan.sizes()
    large = {int(s) for s, l in zip(sizes, is_large) if l}
    assert {200, 800} <= large
    off = onp.svec_offsets(blk)
    for k, n in enumerate(blk):
        a, b = ours[off[k]:off[k + 1]], ref[off[k]:off[k + 1]]
        tol = X_TOL if int(n) in large else 1e-5
        assert np.linalg.norm(a - b) <= tol * np.linalg.norm(b), (k, int(n))


@pytest.mark.parametrize("coeffs", ["unit", "gauss"])
def test_c2b_full_size_ten_iterations_against_oracle(coeffs):
    """BASELINE configs[1] at full size (2,000 blocks n ~ U{6..60}, m = 700,000): iteration by iteration against the oracle.
    "unit": +-1 constraint coefficients (moment-consistency rows as in the SPOT data): A A^T is well conditioned apart
    from exactly redundant rows, and the trajectories must agree to 1e-7.
    "gauss": the bench workload itself.  Its N(0,1) coefficients along long chains make A A^T numerically singular with a
    continuum of pivots between 1e-16 and 1e-11: two SuperLU factorisations of A A^T + 1e-15 I that differ only in the
    column ordering already disagree by 2.8e-5 in A^T y (scripts/pivot_tol_probe.py, DESIGN.md section 5), so nothing
    tighter than that can be asked of ANY implementation of the reference's solve; the primal residual, which does not
    depend on y, still agrees to 1e-7."""
    from cuadmm_b200.synthetic import c2b_blocks, chain_sdp
    P = chain_sdp(c2b_blocks(2000, 6, 60, 0), 700000, seed=0, coeffs=coeffs)
    blk = np.ascontiguousarray(P["blk"], np.int32)
    iters = 10
    s = make_solver(P)
    s.solve(iters, 1e-12, 500, 50, 100, 11000, 1.05)
    o = onp.ADMMOracle(P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
                       P["C_idx"], P["C_val"], blk, project=lambda v: onp.project_svec_cpp(blk, v, min(30, os.cpu_count() or 1)))
    X, y, S, it = o.solve(iters, 1e-12, 500, 50, 100, 11000, 1.05)
    assert s.info_iter_num == it == iters
    tol = {"unit": dict(errRp=1e-7, errRd=1e-7, pobj=1e-7, dobj=1e-7, relgap=1e-6, sig=1e-12, X=1e-8),
           "gauss": dict(errRp=1e-7, errRd=2e-4, pobj=5e-3, dobj=5e-4, relgap=1e-4, sig=1e-12, X=3e-2)}[coeffs]
    for key in ["errRp", "errRd", "pobj", "dobj", "relgap", "sig"]:
        a, b = s.history(key), np.array(o.hist[key])
        assert np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-9)) < tol[key], key
    assert np.linalg.norm(s.X - X) <= tol["X"] * np.linalg.norm(X)
    if coeffs == "unit":
        assert np.linalg.norm(s.S - S) <= 1e-8 * np.linalg.norm(S)


@pytest.mark.parametrize("name,log,stop_iter", [("ros_2000", "ros_2000_sgs.log", 12732), ("pusht_n10", "pusht_n10_sgs.log", 6149)])
def test_stop_iteration_matches_reference_log(name, log, stop_iter):
    # the committed sGS logs were produced with solve(.., tol 1e-3, switch_admm 11000 = solver.h:242 default): the run
    # must stop at exactly the iteration the reference's own run stopped at (time-to-KKT parity, north_star: +-2 %)
    rows = parse_log(os.path.join(GOLD, log))
    assert rows[-1]["it"] == stop_iter
    P = load_fixture(name)
    s = make_solver(P)
    s.solve(20000, 1e-3, 0, 50, 100, 11000, 1.05)
    assert abs(s.info_iter_num - stop_iter) <= int(0.02 * stop_iter), s.info_iter_num
    assert s.info_iter_num == stop_iter, s.info_iter_num
    last = rows[-1]
    assert abs(s.history("pobj")[-1] - last["pobj"]) <= 2e-4 * abs(last["pobj"]) + 1e-9


def test_matlab_like_entry_matches_solver_api():
    # MATLAB/cuadmm_MATLAB.cu:197-433: At_stack sparse (size_t jc / ir), b / C_stack sparse columns, blk_vec doubles,
    # X0 / y0 / S0 dense (never null: always a warm start with the passed vectors), info arrays per iteration
    P = synthetic_sdp([6, 9, 4, 14, 21], m=60, seed=8)
    rng = np.random.default_rng(0)
    X0 = 0.1 * rng.standard_normal(P["vec_len"]); y0 = 0.1 * rng.standard_normal(P["con_num"]); S0 = 0.1 * rng.standard_normal(P["vec_len"])
    iters = 40
    X, y, S, info = cu.solve_matlab_like(15, iters, 1e-12, P["col_ptrs"].astype(np.int64), P["row_ids"].astype(np.int64), P["vals"],
                                         P["b_idx"].astype(np.int64), P["b_val"], P["C_idx"].astype(np.int64), P["C_val"],
                                         P["blk"].astype(np.float64), X0, y0, S0, 1.7, 500, 50, 100, 11000, 1.05)
    s = make_solver(P, X=X0, y=y0, S=S0, sig=1.7)
    s.solve(iters, 1e-12, 500, 50, 100, 11000, 1.05)
    assert info["iter_num"] == s.info_iter_num == iters and info["total_time"] > 0
    for key in ["pobj", "dobj", "errRp", "errRd", "relgap", "sig", "bscale", "Cscale"]:
        assert np.allclose(info[key], s.history(key), rtol=1e-9, atol=1e-14), key
    assert np.allclose(X, s.X, rtol=1e-9, atol=1e-12) and np.allclose(S, s.S, rtol=1e-9, atol=1e-12)
    assert np.allclose(y, s.y, rtol=1e-7, atol=1e-10)
    # and against the oracle started from the same point
    o = onp.ADMMOracle(P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
                       P["C_idx"], P["C_val"], P["blk"], X=X0, y=y0, S=S0, sig=1.7)
    Xo, yo, So, it = o.solve(iters, 1e-12, 500, 50, 100, 11000, 1.05)
    assert np.linalg.norm(X - Xo) <= 1e-8 * np.linalg.norm(Xo)
