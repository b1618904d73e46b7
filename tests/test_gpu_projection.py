"""GPU parity of the PSD projection (through the C ABI) against the LAPACK dsyevd oracle.
Tolerances are BASELINE.json's: eigenvalues 1e-10 relative, projected X 1e-9 relative Frobenius."""
import os

import numpy as np
import pytest

import cuadmm_b200 as cu
import oracle_np as onp
from conftest import random_svec, ROOT, ip, dp

pytestmark = pytest.mark.gpu

X_TOL = 1e-9
EIG_TOL = 1e-10


def _check(blk, x, x_tol=X_TOL):
    blk = np.asarray(blk, np.int32)
    p = cu.Plan(blk, device=0)
    out, eig, sweeps = p.project_eig_host(x)
    ref, reig = onp.project_svec(blk, x, want_eig=True)
    off = onp.svec_offsets(blk)
    eoff = np.concatenate([[0], np.cumsum(blk)])
    worst = 0.0
    for k in range(len(blk)):
        a, b = out[off[k]:off[k + 1]], ref[off[k]:off[k + 1]]
        xin = x[off[k]:off[k + 1]]
        scale = max(np.linalg.norm(b), 1e-6 * np.linalg.norm(xin), 1e-300)
        worst = max(worst, np.linalg.norm(a - b) / scale)
        e, re_ = eig[eoff[k]:eoff[k + 1]], reig[eoff[k]:eoff[k + 1]]
        escale = max(np.abs(re_).max(), 1e-300)
        # n <= 168: eigenvalues of the shared-memory Jacobi kernel that also produced X.  168 < n <= 1024: X comes from the
        # dense sign iteration (no eigenvalues), the eigenvalues of this debug entry from the global-memory Jacobi kernel
        if blk[k] <= 1024:
            assert np.abs(e - re_).max() / escale < EIG_TOL, (k, blk[k])
        else:
            assert np.all(np.isnan(e))
    assert worst < x_tol, worst
    assert sweeps.max() < 40
    return out, p


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 6, 7, 8, 10, 13, 15, 16, 17, 21, 28, 31, 32, 33, 45, 55, 60, 64, 65,
                               66, 91, 96, 97, 120, 128, 129, 150, 168])
def test_single_block_sizes(n):
    _check([n], random_svec([n], seed=n))


def test_known_answer_matrices():
    # test/eig_cpu_test.hpp:7-66, test/cusolver_test.hpp:116-187
    A4 = np.array([[4, 1, 2, 2], [1, 4, 1, 2], [2, 1, 4, 1], [2, 2, 1, 4]], float)
    A2 = np.array([[2, 1], [1, 3.0]])
    A3 = np.array([[3, 1, 2], [1, 3, 1], [2, 1, 3.0]])
    blk = [4, 2, 3]
    x = np.concatenate([onp.svec(A4), onp.svec(A2), onp.svec(A3)])
    p = cu.Plan(blk)
    out, eig, _ = p.project_eig_host(x)
    assert np.allclose(out, x, rtol=0, atol=1e-13)          # all PSD already
    s5, s37, s3 = np.sqrt(5), np.sqrt(37), np.sqrt(3)
    exp = [0.5 * (5 - s5), 0.5 * (11 - s37), 0.5 * (5 + s5), 0.5 * (11 + s37), (5 - s5) / 2, (5 + s5) / 2, 1, 4 - s3, 4 + s3]
    assert np.allclose(eig, exp, rtol=1e-13)


def test_large_blocks_dense_sign_path():
    # n > 168: GEMM-only matrix-sign projection (csrc/dense_proj.cu)
    _check([200], random_svec([200], seed=200))
    _check([169, 3, 250], random_svec([169, 3, 250], seed=1))
    _check([512, 300, 40], random_svec([512, 300, 40], seed=2))
    _check([1000], random_svec([1000], seed=3))


def test_large_blocks_both_tile_shapes_in_one_plan(monkeypatch):
    # blocks up to n = 2048 run on 64 x 64 tiles, larger ones on 128 x 128 tiles (two work lists per product, csrc/dense_proj.cu);
    # a plan that holds both, plus shared-memory Jacobi blocks, against LAPACK — and the same blocks with the threshold moved
    blk = [2100, 300, 40, 700]
    x = random_svec(blk, seed=7)
    out, _ = _check(blk, x)
    for thr in ("0", "100000"):              # everything on 128-tiles / everything on 64-tiles
        monkeypatch.setenv("CUADMM_SG_SMALL_MAX", thr)
        alt = cu.Plan(np.asarray(blk, np.int32), device=0).project_host(x)
        assert np.linalg.norm(alt - out) <= 1e-12 * np.linalg.norm(out)


def test_large_blocks_degenerate_spectra():
    rng = np.random.default_rng(5)
    n = 300
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    mats = []
    lam = np.concatenate([np.ones(n // 2), -np.ones(n - n // 2)]); mats.append((Q * lam) @ Q.T)
    lam = np.zeros(n); lam[:5] = [5, 4, 3, 2, 1]; lam[-3:] = [-1, -2, -3]; lam[5:-3] = 1e-8 * rng.standard_normal(n - 8)
    mats.append((Q * lam) @ Q.T)                                  # low rank + tiny noise (late ADMM iterates)
    mats.append(np.zeros((n, n)))
    mats.append(-np.eye(n) * 3.0)
    v = rng.standard_normal(n); mats.append(np.outer(v, v))
    lam = np.geomspace(1e-9, 1, n) * np.where(np.arange(n) % 2, 1, -1); mats.append((Q * lam) @ Q.T)   # 9 decades
    blk = [n] * len(mats)
    x = np.concatenate([onp.svec((M + M.T) / 2) for M in mats])
    out = cu.Plan(blk).project_host(x)
    ref = onp.project_svec(blk, x)
    off = onp.svec_offsets(blk)
    for k in range(len(blk)):
        a, b, xin = out[off[k]:off[k + 1]], ref[off[k]:off[k + 1]], x[off[k]:off[k + 1]]
        assert np.linalg.norm(a - b) <= 1e-9 * max(np.linalg.norm(b), 1e-3 * np.linalg.norm(xin)) + 1e-300, k


def test_mixed_blocks_planarhand_layout():
    blk = np.loadtxt(os.path.join(ROOT, "tests", "golden", "planarhand_n1_blk.txt"), dtype=np.int32)
    _check(blk, random_svec(blk, seed=0))


def test_c2b_synthetic_2000_blocks():
    rng = np.random.default_rng(0)
    blk = rng.integers(6, 61, 2000).astype(np.int32)
    x = random_svec(blk, seed=0)
    out, p = _check(blk, x)
    # size-independent properties at full size
    out2 = p.project_host(out)
    assert np.linalg.norm(out2 - out) <= 1e-11 * np.linalg.norm(out)          # idempotent
    neg = p.project_host(-x)
    assert np.linalg.norm((out - neg) - x) <= 1e-11 * np.linalg.norm(x)      # Moreau decomposition
    assert abs(out @ (out - x)) <= 1e-10 * (x @ x)                            # complementarity


def test_degenerate_spectra():
    rng = np.random.default_rng(3)
    mats = []
    blk = []
    for n in [2, 6, 10, 16, 32, 33, 60, 100]:
        Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
        lam = np.concatenate([np.ones(n // 2), -np.ones(n - n // 2)])                 # +-1 clusters
        mats.append((Q * lam) @ Q.T); blk.append(n)
        lam = np.zeros(n); lam[0] = 5; lam[-1] = -3; lam[1:-1] = 1e-9 * rng.standard_normal(n - 2)
        mats.append((Q * lam) @ Q.T); blk.append(n)                                   # low rank + noise
        mats.append(np.eye(n) * 2.5); blk.append(n)                                   # multiple of I
        mats.append(-np.eye(n)); blk.append(n)
        mats.append(np.zeros((n, n))); blk.append(n)                                  # zero block
        v = rng.standard_normal(n); mats.append(-np.outer(v, v)); blk.append(n)       # rank-1 negative
        mats.append(np.outer(v, v)); blk.append(n)                                    # rank-1 positive
    mats.append(np.array([[0, 1.0], [1, 0]])); blk.append(2)
    x = np.concatenate([onp.svec((M + M.T) / 2) for M in mats])
    p = cu.Plan(blk)
    out = p.project_host(x)
    ref = onp.project_svec(blk, x)
    off = onp.svec_offsets(blk)
    for k in range(len(blk)):
        a, b, xin = out[off[k]:off[k + 1]], ref[off[k]:off[k + 1]], x[off[k]:off[k + 1]]
        assert np.linalg.norm(a - b) <= 1e-9 * max(np.linalg.norm(b), 1e-3 * np.linalg.norm(xin)) + 1e-300, (k, blk[k])


def test_scaling_invariance_and_extremes():
    blk = [7, 20, 40]
    x = random_svec(blk, seed=9)
    p = cu.Plan(blk)
    base = p.project_host(x)
    # exact power-of-two scalings: the kernel prescales by 2^-exponent, so nothing may over/underflow
    for e in [-900, -500, -60, 60, 500, 900]:
        out = p.project_host(np.ldexp(x, e))
        assert np.linalg.norm(np.ldexp(out, -e) - base) <= 1e-13 * np.linalg.norm(base), e
    for s10 in [1e-150, 1e150]:
        out = p.project_host(x * s10)
        assert np.linalg.norm(out / s10 - base) <= 1e-12 * np.linalg.norm(base)
    assert np.all(np.isnan(p.project_host(np.full_like(x, np.nan))))


def test_empty_and_ragged():
    p = cu.Plan([], device=0)
    assert p.project_host(np.zeros(0)).shape == (0,)
    blk = [1] * 100 + [2] * 50 + [33] + [1]
    _check(blk, random_svec(blk, seed=4))


def test_svec_smat_kernels_bit_exact(ohost):
    import torch
    rng = np.random.default_rng(11)
    blk = np.array([3, 4, 1, 2, 40, 40, 7, 7, 7, 33], np.int32)
    p = cu.Plan(blk, device=0)
    B, M1, M2 = p.maps()
    L = p.vec_len
    x = rng.standard_normal(L)
    tot = p.totals()
    large = np.zeros(max(int(tot[2]), 1)); small = np.zeros(max(int(tot[5]), 1))
    ohost.oracle_vector_to_matrices(dp(x), dp(large), dp(small), ip(B), ip(M1), ip(M2), L)
    dx = torch.from_numpy(x).cuda()
    dl = torch.zeros(len(large), dtype=torch.float64, device="cuda")
    ds = torch.zeros(len(small), dtype=torch.float64, device="cuda")
    p.svec_to_smat_device(dx.data_ptr(), dl.data_ptr(), ds.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(dl.cpu().numpy(), large) and np.array_equal(ds.cpu().numpy(), small)
    back = np.zeros(L)
    ohost.oracle_matrices_to_vector(dp(back), dp(large), dp(small), ip(B), ip(M1), ip(M2), L)
    dback = torch.zeros(L, dtype=torch.float64, device="cuda")
    p.smat_to_svec_device(dl.data_ptr(), ds.data_ptr(), dback.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(dback.cpu().numpy(), back)


def test_device_pointer_entry_matches_host_entry():
    import torch
    blk = [10, 33, 5]
    x = random_svec(blk, seed=2)
    p = cu.Plan(blk)
    p.set_warm_start(False)          # cold Jacobi every call: the two entries must agree bit for bit
    ref = p.project_host(x)
    dx = torch.from_numpy(x).cuda(); dy = torch.empty_like(dx)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        p.project_device(dx.data_ptr(), dy.data_ptr(), s.cuda_stream)
    s.synchronize()
    assert np.array_equal(dy.cpu().numpy(), ref)


def test_against_reference_cusolver_build(request):
    """Baseline A (the reference's own cuSOLVER stage, oracle/_ref) on the same input.  Its batched
    Jacobi stops at tol 1e-6 (include/cuadmm/cusolver.h:113), so agreement is only expected at ~1e-6."""
    blk = np.array([6] * 40 + [10] * 40 + [13] * 30 + [32] * 25 + [45, 45, 60], np.int32)
    x = random_svec(blk, seed=5)
    ours = cu.Plan(blk).project_host(x)
    lap = onp.project_svec(blk, x)
    assert np.linalg.norm(ours - lap) / np.linalg.norm(lap) < 1e-12
    oref = request.getfixturevalue("oref")      # skips here when the reference build is absent
    h = oref.ref_proj_create(ip(blk), len(blk), 15)
    out_ref = np.zeros_like(x)
    import ctypes as C
    oref.ref_proj_run(C.c_void_p(h), dp(x), dp(out_ref), 1)
    oref.ref_proj_destroy(C.c_void_p(h))
    assert np.linalg.norm(out_ref - lap) / np.linalg.norm(lap) < 1e-5


def test_warm_start_matches_cold_and_oracle():
    """The plan warm-starts Jacobi from the eigenbasis of its previous call.  Project a sequence of
    slowly drifting inputs (as successive ADMM iterates are), then an unrelated one: every result must
    match the LAPACK oracle as tightly as a cold plan does, and the sweep count must drop."""
    blk = [6, 17, 33, 60, 60, 96, 128, 150]
    rng = np.random.default_rng(5)
    x = random_svec(blk, seed=11)
    warm = cu.Plan(blk)
    cold = cu.Plan(blk); cold.set_warm_start(False)
    sweeps_warm, sweeps_cold = [], []
    for it in range(6):
        xi = x + (1e-3 * it) * random_svec(blk, seed=100 + it)
        ow, _, sw = warm.project_eig_host(xi)
        oc, _, sc = cold.project_eig_host(xi)
        ref = onp.project_svec(blk, xi)
        scale = np.abs(ref).max()
        assert np.abs(ow - ref).max() <= 1e-11 * scale      # stop rule: all |cos| <= 1e-11 (north_star tolerance: 1e-9)
        assert np.abs(oc - ref).max() <= 1e-11 * scale
        sweeps_warm.append(sw.max()); sweeps_cold.append(sc.max())
    assert max(sweeps_warm[1:]) < min(sweeps_cold[1:]), (sweeps_warm, sweeps_cold)
    y = random_svec(blk, seed=77)                      # unrelated input: still correct, just not faster
    ow, _, _ = warm.project_eig_host(y)
    ref = onp.project_svec(blk, y)
    assert np.abs(ow - ref).max() <= 1e-11 * np.abs(ref).max()
    z = np.zeros_like(y)                               # zero block keeps the stored basis valid
    assert np.array_equal(warm.project_host(z), z)
    ow, _, _ = warm.project_eig_host(x)
    ref = onp.project_svec(blk, x)
    assert np.abs(ow - ref).max() <= 1e-11 * np.abs(ref).max()


def _identities(blk, x):
    """size-independent properties of Pi_+: idempotence, Moreau decomposition x = Pi(x) - Pi(-x), orthogonality"""
    p = cu.Plan(np.asarray(blk, np.int32))
    a = p.project_host(x)
    b = p.project_host(-x)
    aa = p.project_host(a)
    nx = np.linalg.norm(x)
    assert np.linalg.norm(aa - a) <= 1e-11 * nx
    assert np.linalg.norm(a - b - x) <= 1e-12 * nx
    assert abs(a @ b) <= 1e-12 * nx * nx
    return a


def test_c4_block_mix_identities_and_oracle_sample():
    # BASELINE configs[3] block mix {10, 50, 200, 800} at 1/20 of the block count, shuffled like the full case
    blk = np.concatenate([np.full(300, 10), np.full(150, 50), np.full(45, 200), np.full(5, 800)]).astype(np.int32)
    np.random.default_rng(0).shuffle(blk)
    x = random_svec(blk, seed=4)
    a = _identities(blk, x)
    off = onp.svec_offsets(blk)
    picks = [int(np.flatnonzero(blk == n)[0]) for n in (10, 50, 200, 800)] + [int(np.flatnonzero(blk == 200)[-1])]
    for k in picks:
        ref = onp.project_svec(blk[k:k + 1], x[off[k]:off[k + 1]])
        assert np.linalg.norm(a[off[k]:off[k + 1]] - ref) <= X_TOL * np.linalg.norm(ref), (k, blk[k])


def test_c3_single_block_n4000_identities():
    # BASELINE configs[2]: one dense block n = 4000 (a CPU eigendecomposition of this size is left to the bench baseline)
    blk = np.array([4000], np.int32)
    _identities(blk, random_svec(blk, seed=6))


def test_fixed_rank_projection():
    """max_dense_vector_zero_mask + get_eig_rank_mask (the reference's fixed-rank projection, src/duo_solver.cu:843-850):
    only the eig_rank largest eigenvalues survive the clamp"""
    blk = np.array([4, 9, 16, 17, 30, 33, 48, 64, 70, 100, 150], np.int32)
    x = random_svec(blk, seed=21)
    p = cu.Plan(blk)
    for rank in (1, 3, 8, 200):
        p.set_rank_limit(rank)
        out = p.project_host(x)
        ref = onp.project_svec_rank(blk, x, rank)
        assert np.linalg.norm(out - ref) <= X_TOL * np.linalg.norm(ref), rank
    p.set_rank_limit(0)
    assert np.linalg.norm(p.project_host(x) - onp.project_svec(blk, x)) <= X_TOL * np.linalg.norm(x)
    big = cu.Plan(np.array([200, 10], np.int32))
    big.set_rank_limit(2)
    with pytest.raises(cu.CuadmmError):
        big.project_host(random_svec([200, 10], seed=1))
