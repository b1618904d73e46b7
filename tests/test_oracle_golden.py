"""Pins the oracle (oracle/oracle_host.c, oracle/oracle_np.py) against the golden vectors and
known-answer tests the reference's own test-suite holds for the hot path (SURVEY 8c), and against
the unmodified reference compiled into oracle/_ref where that is available.  CPU only."""
import math
import os

import numpy as np
import pytest

import oracle_np as onp
from conftest import ip, dp, oracle_maps, ROOT


# ---- svec maps --------------------------------------------------------------------------------
def test_get_maps_duo_golden(ohost):
    # reference test/utils_test.hpp:19-63  (blk {5,4}, LARGE=5)
    blk = np.array([5, 4], np.int32)
    L = 25
    B = np.zeros(L, np.int32); M1 = np.zeros(L, np.int32); M2 = np.zeros(L, np.int32)
    ohost.oracle_get_maps_duo(ip(blk), 2, 5, ip(B), ip(M1), ip(M2))
    assert B.tolist() == [0] * 15 + [1] * 10
    assert M1.tolist() == [0, 5, 6, 10, 11, 12, 15, 16, 17, 18, 20, 21, 22, 23, 24,
                           0, 4, 5, 8, 9, 10, 12, 13, 14, 15]
    assert M2.tolist() == [0, 1, 6, 2, 7, 12, 3, 8, 13, 18, 4, 9, 14, 19, 24,
                           0, 1, 5, 2, 6, 10, 3, 7, 11, 15]


def test_get_maps_golden_2small_4large(ohost):
    # reference test/kernels_test.hpp:339-341: blk {2,4} -> 2 small (1 matrix, 2-17 > 1.4 false), 4 small?
    # the literal maps there put the 2x2 in pool 1 and the 4x4 in pool 0
    B = [1, 1, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0]
    M1 = [0, 2, 3, 0, 4, 5, 8, 9, 10, 12, 13, 14, 15]
    M2 = [0, 1, 3, 0, 1, 5, 2, 6, 10, 3, 7, 11, 15]
    # these are the duo maps for LARGE=4 (analyze_blk_duo): get_maps_duo reproduces them
    blk = np.array([2, 4], np.int32)
    b = np.zeros(13, np.int32); m1 = np.zeros(13, np.int32); m2 = np.zeros(13, np.int32)
    ohost.oracle_get_maps_duo(ip(blk), 2, 4, ip(b), ip(m1), ip(m2))
    assert b.tolist() == B and m1.tolist() == M1 and m2.tolist() == M2


def test_analyze_blk_duo_golden(ohost):
    # reference test/utils_test.hpp:65-82
    import ctypes as C
    blk = np.array([5, 4, 4, 5, 5], np.int32)
    L, S, nm, nl = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    rc = ohost.oracle_analyze_blk_duo(ip(blk), 5, C.byref(L), C.byref(S), C.byref(nm), C.byref(nl))
    assert rc == 0 and (L.value, S.value, nm.value, nl.value) == (5, 4, 3, 2)


def test_is_large_heuristic(ohost):
    # src/matrix_sizes.cu:14-19 and the fitted table of plots/single_batched_comparison.ipynb
    assert ohost.oracle_is_large_mat(33, 1000) == 1
    assert ohost.oracle_is_large_mat(32, 20) == 0
    assert ohost.oracle_is_large_mat(32, 10) == 1      # 15 > 14
    assert ohost.oracle_is_large_mat(18, 1) == 0       # 1 > 1.4 false
    assert ohost.oracle_is_large_mat(19, 1) == 1       # 2 > 1.4
    assert ohost.oracle_is_large_mat(17, 0) == 0


def _planarhand_blk():
    # examples/SPOT/data/TXT/PlanarHand_N=1_MOMENT/blk.txt, committed as a fixture
    return np.loadtxt(os.path.join(ROOT, "tests", "golden", "planarhand_n1_blk.txt"), dtype=np.int32)


def test_matrix_sizes_planarhand_log(ohost):
    # golden: examples/benchmarks/PlanarHand_N=1_MOMENT/cuADMM.log:9-35 (MatrixSizes printout)
    blk = _planarhand_blk()
    n = len(blk)
    sizes = np.zeros(n, np.int32); nums = np.zeros(n, np.int32)
    ns = ohost.oracle_analyze_blk(ip(blk), n, ip(sizes), ip(nums))
    arr = lambda k: np.zeros(k + 2, np.int32)
    ls, ln, lm, lw, ss, sn, sm, sw = (arr(ns) for _ in range(8))
    tot = np.zeros(6, np.int32)
    packed = ohost.oracle_matrix_sizes(ip(sizes), ip(nums), ns, ip(ls), ip(ln), ip(lm), ip(lw),
                                       ip(ss), ip(sn), ip(sm), ip(sw), ip(tot))
    nl, nsm = packed & 0xffff, packed >> 16
    assert ls[:nl].tolist() == [28, 55, 66, 91, 120]
    assert lm[:nl + 1].tolist() == [0, 2352, 8402, 21470, 46313, 89513]
    assert ss[:nsm].tolist() == [7, 10, 11, 13, 15]
    assert sm[:nsm + 1].tolist() == [0, 245, 1445, 4591, 6957, 18432]
    assert int(sum(int(b) * (int(b) + 1) // 2 for b in blk)) == 55179


def test_oracle_maps_vs_reference_build(ohost, oref):
    rng = np.random.default_rng(0)
    cases = [[5, 4], [2, 4], [3, 4, 1, 2], [1], [40, 3, 3, 40, 17, 18, 19], _planarhand_blk().tolist(),
             rng.integers(1, 45, 200).tolist()]
    for blk in cases:
        blk = np.array(blk, np.int32)
        L = int(sum(int(n) * (int(n) + 1) // 2 for n in blk))
        B, M1, M2 = oracle_maps(ohost, blk)
        rB = np.zeros(L, np.int32); rM1 = np.zeros(L, np.int32); rM2 = np.zeros(L, np.int32)
        oref.ref_get_maps(ip(blk), len(blk), L, ip(rB), ip(rM1), ip(rM2))
        assert np.array_equal(B, rB) and np.array_equal(M1, rM1) and np.array_equal(M2, rM2)


def test_sqrt2_constants(ohost):
    # test/kernels_test.hpp:218-222; the literals are what the reference build returns (ref_sqrt2, ref_sqrt2inv)
    # (EXPECT_DOUBLE_EQ there tolerates 4 ulp; the Newton fixed point is 1 ulp below sqrt(2))
    assert ohost.oracle_sqrt2() == onp.SQRT2 == 1.414213562373095
    assert abs(onp.SQRT2 - math.sqrt(2.0)) <= 2.3e-16
    assert onp.SQRT2INV == 0.7071067811865476


# ---- svec <-> smat ----------------------------------------------------------------------------
def test_matrices_to_vector_golden(ohost):
    # test/kernels_test.hpp:224-307
    mom = np.array([1, 2, 3, 4, 2, 5, 6, 7, 3, 6, 8, 9, 4, 7, 9, 10], float)
    loc = np.array([2, 3, 4, 5, 3, 6, 7, 8, 4, 7, 9, 10, 5, 8, 10, 11], float)
    M1 = [0, 1, 2, 3, 5, 6, 7, 10, 11, 15]
    M2 = [0, 4, 8, 12, 5, 9, 13, 10, 14, 15]
    M1 = np.array(M1 + M1, np.int32); M2 = np.array(M2 + M2, np.int32)
    B = np.array([0] * 10 + [1] * 10, np.int32)
    out = np.zeros(20)
    ohost.oracle_matrices_to_vector(dp(out), dp(mom), dp(loc), ip(B), ip(M1), ip(M2), 20)
    s2 = onp.SQRT2
    assert out.tolist() == [1, 2 * s2, 3 * s2, 4 * s2, 5, 6 * s2, 7 * s2, 8, 9 * s2, 10,
                            2, 3 * s2, 4 * s2, 5 * s2, 6, 7 * s2, 8 * s2, 9, 10 * s2, 11]


def test_svec_roundtrip_matches_numpy_oracle(ohost):
    # round trip exactness (test/kernels_test.hpp:310-556) + agreement of the two oracle halves
    rng = np.random.default_rng(1)
    blk = np.array([3, 4, 1, 2, 40], np.int32)
    B, M1, M2 = oracle_maps(ohost, blk)
    L = len(B)
    x = rng.standard_normal(L)
    large = np.zeros(40 * 40 + 1); small = np.zeros(9 + 16 + 1 + 4 + 1)
    ohost.oracle_vector_to_matrices(dp(x), dp(large), dp(small), ip(B), ip(M1), ip(M2), L)
    back = np.zeros(L)
    ohost.oracle_matrices_to_vector(dp(back), dp(large), dp(small), ip(B), ip(M1), ip(M2), L)
    assert np.allclose(back, x, rtol=0, atol=4e-16 * np.abs(x).max())
    off = onp.svec_offsets(blk)
    M40 = onp.smat(x[off[4]:off[5]], 40)
    assert np.array_equal(M40.ravel(order="F"), large[:1600])
    assert np.array_equal(onp.svec(M40), back[off[4]:off[5]])


def test_mul_diag_batch_golden(ohost):
    # test/kernels_test.hpp:122-216 (column-major column scaling)
    mat = np.arange(1, 26, dtype=float)
    vec = np.array([1, 2, 3, 4, 5], float)
    out = np.zeros(25)
    ohost.oracle_mul_diag_batch(dp(out), dp(mat), dp(vec), 5, 25)
    exp = mat.reshape(5, 5) * vec[:, None]
    assert np.array_equal(out, exp.ravel())


# ---- eig / projection -------------------------------------------------------------------------
def test_eig_known_answers():
    # test/eig_cpu_test.hpp:7-66, test/cusolver_test.hpp:33-92,116-187 (reference tolerance 1e-5)
    A4 = np.array([[4, 1, 2, 2], [1, 4, 1, 2], [2, 1, 4, 1], [2, 2, 1, 4]], float)
    w, Q = onp.eig_dsyevd(A4)
    exp = [0.5 * (5 - math.sqrt(5)), 0.5 * (11 - math.sqrt(37)), 0.5 * (5 + math.sqrt(5)), 0.5 * (11 + math.sqrt(37))]
    assert np.allclose(w, exp, rtol=1e-14)
    assert np.allclose(w, [1.38197, 2.45862, 3.61803, 8.54138], atol=1e-5)
    assert np.allclose(Q @ np.diag(w) @ Q.T, A4, atol=1e-13)
    w2, _ = onp.eig_dsyevd(np.array([[2, 1], [1, 3.0]]))
    assert np.allclose(w2, [(5 - math.sqrt(5)) / 2, (5 + math.sqrt(5)) / 2], rtol=1e-14)
    w3, _ = onp.eig_dsyevd(np.array([[3, 1, 2], [1, 3, 1], [2, 1, 3.0]]))
    assert np.allclose(w3, [1, 4 - math.sqrt(3), 4 + math.sqrt(3)], rtol=1e-14)


def test_projection_properties():
    rng = np.random.default_rng(2)
    blk = [1, 2, 7, 33]
    x = np.concatenate([onp.svec((G + G.T) / 2) for G in (rng.standard_normal((n, n)) for n in blk)])
    p = onp.project_svec(blk, x)
    assert np.allclose(onp.project_svec(blk, p), p, atol=1e-13)          # idempotent
    assert np.allclose(p - onp.project_svec(blk, -x), x, atol=1e-13)     # Moreau: x = P(x) - P(-x)
    assert abs(p @ (p - x)) < 1e-12                                      # <P(x), P(x)-x> = 0


def test_thread_ranges_restates_reference_split():
    # src/duo_solver.cu:346-371
    assert onp.thread_ranges(14, 4) == [(0, 4), (4, 7), (7, 10), (10, 14)]
    assert onp.thread_ranges(7, 2) == [(0, 3), (3, 7)]
    assert sum(b - a for a, b in onp.thread_ranges(80, 30)) == 80


# ---- sparse -----------------------------------------------------------------------------------
def test_normA_golden(ohost):
    # test/kernels_test.hpp:35-83 with test/data/sparse_matrix_coo.txt ((row col val) per line)
    rows = np.array([0, 2, 1, 3, 2, 3], np.int32)   # after COO_to_CSC, see fixture below
    coo = np.loadtxt(os.path.join(ROOT, "tests", "golden", "ref_sparse_matrix_coo.txt"))
    r, c, v = coo[:, 0].astype(np.int32), coo[:, 1].astype(np.int32), coo[:, 2].copy()
    cp = np.zeros(5, np.int32)
    ohost.oracle_coo_to_csc(ip(cp), ip(c), ip(r), dp(v), len(v), 4)
    normA = np.zeros(4)
    ohost.oracle_get_normA(ip(cp), dp(v), dp(normA), 4)
    assert normA.tolist() == [math.sqrt(10.0 * 10 + 30.0 * 30), math.sqrt(20.0 * 20 + 60.0 * 60), 40.0, 50.0]
    n0, n1 = math.sqrt(1000.0), math.sqrt(4000.0)
    assert v.tolist() == [10.0 / n0, 30.0 / n0, 20.0 / n1, 60.0 / n1, 1.0, 1.0]
    nA2, v2 = onp.get_normA(cp, np.array([10.0, 30, 20, 60, 40, 50]))
    assert nA2.tolist() == normA.tolist() and v2.tolist() == v.tolist()


def test_coo_to_csc_golden(ohost):
    # test/io_test.hpp:92-109 on random input.  The (col, row) pairs are unique, so the reference's COO_to_CSC has one
    # possible result: the triplets in (col, row) order, which is scipy's sorted CSC, values and columns included
    rng = np.random.default_rng(3)
    nnz, ncol, nrow = 500, 40, 300
    cols = rng.integers(0, ncol, nnz).astype(np.int32); cols[0] = 0
    rows = rng.permutation(nrow * ncol)[:nnz].astype(np.int32) % nrow
    # make (col,row) unique so the unstable sorts agree
    key = np.unique(cols.astype(np.int64) * nrow + rows)
    cols = (key // nrow).astype(np.int32); rows = (key % nrow).astype(np.int32); nnz = len(key)
    perm = rng.permutation(nnz)
    cols, rows = cols[perm].copy(), rows[perm].copy()
    vals = rng.standard_normal(nnz)
    c1, r1, v1 = cols.copy(), rows.copy(), vals.copy(); cp1 = np.zeros(ncol + 1, np.int32)
    ohost.oracle_coo_to_csc(ip(cp1), ip(c1), ip(r1), dp(v1), nnz, ncol)
    import scipy.sparse as sp
    M = sp.csc_matrix((vals, (rows, cols)), shape=(nrow, ncol)); M.sort_indices()
    assert np.array_equal(M.indptr, cp1) and np.array_equal(M.indices, r1) and np.array_equal(M.data, v1)
    assert np.array_equal(np.repeat(np.arange(ncol), np.diff(M.indptr)), c1)


def test_spmv_golden(ohost):
    # test/cusparse_test.hpp:41-94: CSR 4x4 example; the reference writes expected = 2*A*x + 3*y but
    # never asserts it (and its last row uses x[0] instead of x[1]); asserted here with the right x.
    rowptr = np.array([0, 1, 2, 5, 6], np.int32)
    colind = np.array([0, 1, 0, 2, 3, 1], np.int32)
    val = np.array([10, 20, 30, 40, 50, 60], float)
    x = np.array([1, 2, 3, 4], float); y = np.array([5, 6, 7, 8], float)
    ohost.oracle_spmv_csr(4, ip(rowptr), ip(colind), dp(val), C_double(2.0), dp(x), C_double(3.0), dp(y))
    assert y.tolist() == [2 * 10.0 + 15, 2 * 40.0 + 18, 2 * (30.0 + 120 + 200) + 21, 2 * 120.0 + 24]


def C_double(v):
    import ctypes
    return ctypes.c_double(v)


def test_permutation_golden(ohost):
    # test/kernels_test.hpp:4-33 (scatter) and test/utils_test.hpp:8-17
    perm = np.array([6, 4, 1, 3, 0, 5, 2, 8, 7, 9], np.int32)
    v2 = np.arange(10, dtype=float); v1 = np.zeros(10)
    ohost.oracle_perform_permutation(dp(v1), dp(v2), ip(perm), 10)
    assert all(v1[perm[i]] == v2[i] for i in range(10))
    p = np.array([10, 6, 2, 4, 0, 8, 1, 3, 5, 7, 9], np.int32)
    inv = np.zeros(11, np.int32)
    ohost.oracle_inverse_permutation(ip(inv), ip(p), 11)
    # what the reference's get_inverse_permutation returns for p: a permutation has exactly one inverse
    assert all(p[inv[i]] == i for i in range(11)) and inv.tolist() == [4, 6, 2, 7, 3, 8, 1, 9, 5, 10, 0]


def test_ysolve_golden():
    # test/cholesky_cpu_test.hpp:3-55: A = 11^T + I (4x4) => A A^T = 6*11^T + I, rhs = 25 -> y = 1
    import scipy.sparse as sp
    A = sp.csr_matrix(np.ones((4, 4)) + np.eye(4))
    assert np.array_equal((A @ A.T).toarray(), 6 * np.ones((4, 4)) + np.eye(4))
    sol = onp.AATSolver(A, 1e-16).solve(np.full(4, 25.0))
    assert np.allclose(sol, 1.0, atol=1e-12)
