"""The y-solve's dense-tail relabelling on the host (cuadmm_debug_tail_order, no GPU): the tail unknowns are relabelled
in a postorder of the tail's elimination tree, so the structure of L22^-1 (entry (i, j) only when j is a descendant of
i) stays lower triangular and falls into far fewer 64 x 64 tiles than in the order the ordering leaves the tail in."""
import ctypes

import numpy as np
import pytest

import cuadmm_b200 as cu
from cuadmm_b200.synthetic import c2b_blocks, chain_sdp


def _tail_order(P):
    m, n = P["con_num"], P["vec_len"]
    rp = np.ascontiguousarray(P["col_ptrs"], np.int32)
    ci = np.ascontiguousarray(P["row_ids"], np.int32)
    v = np.ascontiguousarray(P["vals"], np.float64)
    n_lead = ctypes.c_int64(0)
    parent, pos = np.zeros(m, np.int32), np.zeros(m, np.int32)
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rc = cu.lib.cuadmm_debug_tail_order(ctypes.c_int64(m), ctypes.c_int64(n), ptr(rp), ptr(ci), ptr(v), ctypes.c_double(1e-15),
                                        ctypes.byref(n_lead), ptr(parent), ptr(pos))
    assert rc == 0
    r = m - n_lead.value
    return parent[:r], pos[:r]


def _pairs(parent):
    """(ancestor-or-self i, j) for every tail row j: the structural non-zeros of L22^-1"""
    j = np.arange(len(parent))
    rows, cols = [j], [j]
    cur = parent[j]
    while len(j):
        keep = cur >= 0
        j, cur = j[keep], cur[keep]
        rows.append(cur); cols.append(j)
        cur = parent[cur]
    return np.concatenate(rows), np.concatenate(cols)


def _check(parent, pos):
    r = len(parent)
    assert np.array_equal(np.sort(pos), np.arange(r))                   # a relabelling
    # postorder: a node follows its whole subtree, which fills the size[i] - 1 slots right before it
    size = np.ones(r, np.int64)
    for i in range(r):                                                  # parent > child in an elimination tree
        assert parent[i] < 0 or parent[i] > i
        if parent[i] >= 0:
            size[parent[i]] += size[i]
    i, j = _pairs(parent)
    assert np.all((pos[j] <= pos[i]) & (pos[j] > pos[i] - size[i]))
    # so the permuted pattern is lower triangular
    assert np.all(pos[i] >= pos[j])
    nt = (r + 63) // 64
    before = np.zeros((nt, nt), bool); after = np.zeros((nt, nt), bool)
    before[i // 64, j // 64] = True
    after[pos[i] // 64, pos[j] // 64] = True
    assert not np.triu(after, 1).any()
    return len(i), int(before.sum()), int(after.sum()), nt * (nt + 1) // 2


def test_tail_postorder_small_chain():
    P = chain_sdp(c2b_blocks(100, 6, 60, 3), 30000, seed=1)
    parent, pos = _tail_order(P)
    assert len(parent) > 64
    nnz, before, after, lower = _check(parent, pos)
    assert after < before <= lower


def test_tail_postorder_c2b():
    # the bench operator (C2b): 2,000 blocks n ~ U{6..60}, m = 700,000
    P = chain_sdp(c2b_blocks(2000, 6, 60, 0), 700000, seed=0)
    parent, pos = _tail_order(P)
    assert len(parent) == 10228 and int((parent < 0).sum()) == 40
    nnz, before, after, lower = _check(parent, pos)
    assert nnz == 1901276 and lower == 12880
    assert before == 8054                    # 62.5 % of the lower tiles in the order of the ordering
    assert after == 710                      # 5.5 % in postorder

