"""Host logic of the product (block analysis, partition, maps, C-ABI surface) — runs without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import cuadmm_b200 as cu
from conftest import ip, oracle_maps, ROOT


CASES = [[5, 4], [2, 4], [3, 4, 1, 2], [1], [40, 3, 3, 40, 17, 18, 19], [6] * 1999, [10] * 30 + [55] * 3]


@pytest.mark.parametrize("blk", CASES)
def test_maps_bit_exact_vs_oracle(ohost, blk):
    p = cu.Plan(blk, device=-1)
    B, M1, M2 = p.maps()
    oB, oM1, oM2 = oracle_maps(ohost, blk)
    assert np.array_equal(B, oB) and np.array_equal(M1, oM1) and np.array_equal(M2, oM2)
    assert p.vec_len == sum(n * (n + 1) // 2 for n in blk)


def test_maps_and_partition_bit_exact_vs_reference_build(ohost, request):
    rng = np.random.default_rng(7)
    planar = np.loadtxt(os.path.join(ROOT, "tests", "golden", "planarhand_n1_blk.txt"), dtype=np.int32)
    lists = [np.array(blk, np.int32) for blk in CASES + [planar.tolist(), rng.integers(1, 60, 500).tolist()]]
    # the same lists against the C restatement of analyze_blk / MatrixSizes / get_maps, which needs no reference build
    for blk in lists:
        p = cu.Plan(blk, device=-1)
        assert all(np.array_equal(a, b) for a, b in zip(p.maps(), oracle_maps(ohost, blk)))
        n = len(blk)
        sizes = np.zeros(n, np.int32); nums = np.zeros(n, np.int32)
        ns = ohost.oracle_analyze_blk(ip(blk), n, ip(sizes), ip(nums))
        ls, ln, lm, lw, ss, sn, sm, sw = (np.zeros(ns + 2, np.int32) for _ in range(8))
        tot = np.zeros(6, np.int32)
        packed = ohost.oracle_matrix_sizes(ip(sizes), ip(nums), ns, ip(ls), ip(ln), ip(lm), ip(lw), ip(ss), ip(sn), ip(sm),
                                           ip(sw), ip(tot))
        nl, nsm = packed & 0xffff, packed >> 16
        s, c, l = p.sizes()
        assert s.tolist() == sizes[:ns].tolist() and c.tolist() == nums[:ns].tolist()
        assert l.tolist() == [ohost.oracle_is_large_mat(int(a), int(b)) for a, b in zip(sizes[:ns], nums[:ns])]
        assert p.totals().tolist() == tot.tolist()
        assert p.start_indices(0).tolist() == lm[:nl + 1].tolist() and p.start_indices(1).tolist() == lw[:nl + 1].tolist()
        assert p.start_indices(2).tolist() == sm[:nsm + 1].tolist() and p.start_indices(3).tolist() == sw[:nsm + 1].tolist()
    oref = request.getfixturevalue("oref")      # skips here when the reference build is absent
    for blk in lists:
        p = cu.Plan(blk, device=-1)
        L = p.vec_len
        B, M1, M2 = p.maps()
        rB = np.zeros(L, np.int32); rM1 = np.zeros(L, np.int32); rM2 = np.zeros(L, np.int32)
        oref.ref_get_maps(ip(blk), len(blk), L, ip(rB), ip(rM1), ip(rM2))
        assert np.array_equal(B, rB) and np.array_equal(M1, rM1) and np.array_equal(M2, rM2)
        n = len(blk)
        sizes = np.zeros(n, np.int32); nums = np.zeros(n, np.int32); lg = np.zeros(n, np.int32)
        tot = np.zeros(6, np.int32)
        ls = np.zeros(n + 2, np.int32); lw = np.zeros(n + 2, np.int32); ss = np.zeros(n + 2, np.int32); sw = np.zeros(n + 2, np.int32)
        nl, nsm = C.c_int(), C.c_int()
        ns = oref.ref_analyze(ip(blk), n, ip(sizes), ip(nums), ip(lg), ip(tot), ip(ls), ip(lw), ip(ss), ip(sw),
                              C.byref(nl), C.byref(nsm))
        s, c, l = p.sizes()
        assert s.tolist() == sizes[:ns].tolist() and c.tolist() == nums[:ns].tolist() and l.tolist() == lg[:ns].tolist()
        assert p.totals().tolist() == tot.tolist()
        assert p.start_indices(0).tolist() == ls[:nl.value + 1].tolist()
        assert p.start_indices(1).tolist() == lw[:nl.value + 1].tolist()
        assert p.start_indices(2).tolist() == ss[:nsm.value + 1].tolist()
        assert p.start_indices(3).tolist() == sw[:nsm.value + 1].tolist()


def test_planarhand_partition_matches_committed_log():
    # examples/benchmarks/PlanarHand_N=1_MOMENT/cuADMM.log:9-35
    blk = np.loadtxt(os.path.join(ROOT, "tests", "golden", "planarhand_n1_blk.txt"), dtype=np.int32)
    p = cu.Plan(blk, device=-1)
    assert p.vec_len == 55179 and p.nblk == 122
    assert p.start_indices(0).tolist() == [0, 2352, 8402, 21470, 46313, 89513]
    assert p.start_indices(2).tolist() == [0, 245, 1445, 4591, 6957, 18432]


def test_cost_partition_balanced_and_deterministic():
    rng = np.random.default_rng(0)
    blk = rng.integers(6, 61, 2000)
    p = cu.Plan(blk, device=-1)
    o1, c1 = p.partition(8)
    o2, c2 = p.partition(8)
    assert np.array_equal(o1, o2) and set(o1.tolist()) == set(range(8))
    assert c1.max() / c1.mean() < 1.02          # LPT on 2000 blocks balances to ~1 block
    # the reference's equal-count split (src/duo_solver.cu:270-295) is far worse on mixed sizes
    order = np.argsort(-blk, kind="stable")
    eq = np.zeros(8); per = len(blk) // 8
    for g in range(8):
        eq[g] = (blk[g * per:(g + 1) * per].astype(float) ** 3).sum()
    assert c1.max() / c1.mean() <= eq.max() / eq.mean()
    o, c = cu.Plan([100, 1, 1, 1], device=-1).partition(2)
    assert o[0] != o[1] and o[1] == o[2] == o[3]


def test_edge_cases():
    p = cu.Plan([], device=-1)
    assert p.vec_len == 0 and p.nblk == 0
    with pytest.raises(cu.CuadmmError):
        cu.Plan([3, 0], device=-1)
    with pytest.raises(cu.CuadmmError):
        cu.Plan([3, -2], device=-1)


def test_no_cpu_fallback_without_device():
    if cu.device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(cu.CuadmmError) as e:
        cu.Plan([3, 4], device=0)
    assert e.value.code == -2
    p = cu.Plan([3, 4], device=-1)
    with pytest.raises(cu.CuadmmError) as e:
        p.project_host(np.zeros(p.vec_len))
    assert e.value.code == -2
    with pytest.raises(cu.CuadmmError):
        cu.SpMV(1, 1, [0, 1], [0], [1.0])


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "cuadmm_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = sorted(set(re.findall(r"\b(cuadmm_[a-z_A-Z0-9]+)\s*\(", hdr)))
    assert len(names) > 30
    missing = [n for n in names if not hasattr(cu.lib, n)]
    assert not missing, f"declared in include/cuadmm_b200.h but not exported: {missing}"


def test_host_sparse_helpers(ohost):
    import scipy.sparse as sp
    rng = np.random.default_rng(5)
    M = sp.random(50, 30, density=0.1, random_state=5, format="csc")
    M.sort_indices()
    normA, v = cu.normA_host(M.indptr, M.data)
    v2 = M.data.copy(); n2 = np.zeros(30)
    from conftest import dp
    ohost.oracle_get_normA(ip(M.indptr.astype(np.int32)), dp(v2), dp(n2), 30)
    assert np.array_equal(normA, n2) and np.array_equal(v, v2)
    rp, ci, vv = cu.csc_to_csr_host(50, 30, M.indptr, M.indices, M.data)
    R = M.tocsr(); R.sort_indices()
    assert np.array_equal(rp, R.indptr) and np.array_equal(ci, R.indices) and np.array_equal(vv, R.data)


def test_eig_rank_mask_golden(ohost):
    # test/utils_test.hpp:84-99 of the reference: batch 2, size 4, rank 2
    exp = np.array([0, 0, 1, 1, 0, 0, 1, 1], np.int32)
    assert np.array_equal(cu.eig_rank_mask(2, 4, 2), exp)
    m = np.zeros(8, np.int32)
    ohost.oracle_eig_rank_mask(ip(m), 2, 4, 2)
    assert np.array_equal(m, exp)
    for b, n, r in [(1, 1, 0), (3, 7, 7), (5, 6, 1), (2, 9, 4)]:
        m = np.zeros(b * n, np.int32)
        ohost.oracle_eig_rank_mask(ip(m), b, n, r)
        assert np.array_equal(cu.eig_rank_mask(b, n, r), m)
