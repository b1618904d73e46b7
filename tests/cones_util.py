"""Typed blocks ('s' PSD, 'l' nonnegative orthant, 'u' free) for the tests: the numpy reference of the typed projection
and ADMM iteration, the typed TXT reader, and problem generators with known optima.  Test infrastructure only.

The reference oracle (oracle/oracle_np.py) knows PSD blocks only; everything here is built on it:
  * project_typed: 's' blocks through onp.project_block (LAPACK dsyevd), 'l' -> max(x, 0), 'u' -> x;
  * TypedADMMOracle: onp.ADMMOracle with that projection and the one rule of the free cone, S = 0 exactly on 'u'
    entries after every projection (the dual cone of R^n is {0}).  The formula S = (Xproj - X)/sig - Rd1 gives the
    same value up to rounding there; the solver stores the exact zero, and so does this oracle."""
import numpy as np
import scipy.sparse as sp

import oracle_np as onp


def entries(t, n):
    return n * (n + 1) // 2 if t == "s" else n


def svec_offsets(blk, types=None):
    if types is None:
        return onp.svec_offsets(blk)
    return np.concatenate([[0], np.cumsum([entries(t, int(n)) for t, n in zip(types, blk)])]).astype(np.int64)


def project_typed(blk, types, Xb, eig_rank=0):
    off = svec_offsets(blk, types)
    out = np.empty_like(Xb)
    for k, (t, n) in enumerate(zip(types, blk)):
        x = Xb[off[k]:off[k + 1]]
        if t == "l":
            out[off[k]:off[k + 1]] = np.maximum(x, 0.0)
        elif t == "u":
            out[off[k]:off[k + 1]] = x
        elif eig_rank > 0:
            out[off[k]:off[k + 1]] = onp.project_svec_rank([int(n)], x, eig_rank)
        else:
            out[off[k]:off[k + 1]] = onp.project_svec([int(n)], x)
    return out


class TypedADMMOracle(onp.ADMMOracle):
    """onp.ADMMOracle over typed blocks (same arguments, plus types = one letter per block, None: all 's')."""

    def __init__(self, vec_len, con_num, At_col_ptrs, At_row_ids, At_vals, b_idx, b_val, C_idx, C_val, blk,
                 types=None, **kw):
        types = "s" * len(blk) if types is None else "".join(types)
        off = svec_offsets(blk, types)
        self._free = np.zeros(vec_len, bool)
        for k, t in enumerate(types):
            if t == "u":
                self._free[off[k]:off[k + 1]] = True
        self._zero_free = False          # the initial S (given or zero) is taken as it is, like the solver's init
        kw.setdefault("project", lambda v: project_typed(blk, types, v))
        super().__init__(vec_len, con_num, At_col_ptrs, At_row_ids, At_vals, b_idx, b_val, C_idx, C_val, blk, **kw)
        self.types = types
        self._zero_free = True

    # every S the iteration computes (ADMMOracle.solve: S = (Xproj - X)/sig - Rd1) goes through this setter
    @property
    def S(self):
        return self._S

    @S.setter
    def S(self, v):
        if self._zero_free:
            v = np.array(v, dtype=np.float64)
            v[self._free] = 0.0
        self._S = v


def oracle_for(P, **kw):
    return TypedADMMOracle(P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
                           P["C_idx"], P["C_val"], P["blk"], types=P.get("types"), **kw)


def read_problem_txt(prefix):
    """onp.read_problem_txt with the block letters: returns its dict plus types, vec_len from the typed counts"""
    P = onp.read_problem_txt(prefix)
    types = []
    for line in open(prefix + "blk.txt"):
        t = line.split()
        if len(t) == 2 and t[0].isalpha():
            types.append(t[0])
        elif len(t) == 1:
            types.append("s")
    P["types"] = "".join(types)
    P["vec_len"] = int(svec_offsets(P["blk"], P["types"])[-1])
    return P


def write_txt(P, prefix):
    """SDPT3-style TXT files with the block letters"""
    import os
    from util_problems import write_txt as write_s
    write_s(P, prefix)
    types = P.get("types") or "s" * len(P["blk"])
    with open(os.path.join(prefix, "blk.txt"), "w") as f:
        for t, n in zip(types, P["blk"]):
            f.write(f"{t} {int(n)}\n")


def _finish(A, xstar, sstar, ystar, blk, types):
    A = sp.csr_matrix(A)
    A.sum_duplicates(); A.sort_indices()
    b = A @ xstar
    C = sstar + A.T @ ystar
    nzb = np.nonzero(b)[0]; nzc = np.nonzero(C)[0]
    return dict(blk=np.asarray(blk, np.int32), types="".join(types), vec_len=len(xstar), con_num=A.shape[0],
                col_ptrs=A.indptr.astype(np.int32), row_ids=A.indices.astype(np.int32), vals=A.data.astype(np.float64),
                b_idx=nzb.astype(np.int32), b_val=b[nzb], C_idx=nzc.astype(np.int32), C_val=C[nzc],
                xstar=xstar, sstar=sstar, pstar=float(C @ xstar), A=A, b=b, C=C)


def _primal_dual_pair(t, n, rng):
    """x*, s* of one block: complementary and in the cone / dual cone"""
    if t == "s":
        Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
        r = max(1, n // 3)
        lam = np.zeros(n); lam[:r] = rng.uniform(0.5, 2.0, r)
        mu = np.zeros(n); mu[r:] = rng.uniform(0.5, 2.0, n - r)
        return onp.svec((Q * lam) @ Q.T), onp.svec((Q * mu) @ Q.T)
    if t == "l":
        pos = rng.random(n) < 0.5
        return np.where(pos, rng.uniform(0.5, 2.0, n), 0.0), np.where(pos, 0.0, rng.uniform(0.5, 2.0, n))
    return rng.standard_normal(n), np.zeros(n)


def typed_synthetic(blocks, m, seed=0, nnz_per_con=3):
    """synthetic_sdp (tests/util_problems.py) over typed blocks [(letter, n), ...]: constraints with a few random entries
    in at most two blocks, b = A x*, C = s* + A^T y*, x* and s* complementary ('l': each entry has x* > 0 = s* or
    x* = 0 < s*; 'u': x* random, s* = 0, so C_u = (A^T y*)_u).  Feasible with the known optimum p* = <C, x*>."""
    rng = np.random.default_rng(seed)
    types = [t for t, _ in blocks]
    blk = [int(n) for _, n in blocks]
    off = svec_offsets(blk, types)
    xs, ss = zip(*[_primal_dual_pair(t, n, rng) for t, n in blocks])
    xstar, sstar = np.concatenate(xs), np.concatenate(ss)
    rows, cols, vals = [], [], []
    for i in range(m):
        k = 1 + rng.poisson(nnz_per_con - 1)
        b1, b2 = rng.integers(0, len(blk), 2)
        idx = set()
        for _ in range(k):
            bsel = b1 if rng.random() < 0.5 else b2
            idx.add(int(rng.integers(off[bsel], off[bsel + 1])))
        for j in sorted(idx):
            rows.append(i); cols.append(j); vals.append(rng.standard_normal())
    A = sp.csr_matrix((vals, (rows, cols)), shape=(m, int(off[-1])))
    return _finish(A, xstar, sstar, rng.standard_normal(m), blk, types)


def random_lp(n_nonneg, n_free, m, seed=0, density=0.3):
    """min c^T x, A x = b, x_l >= 0, x_u free as one 'l' block followed (n_free > 0) by one 'u' block.  Feasible
    (b = A x*, x* >= 0 on the 'l' part) and bounded (c = A^T y* + s*, s* >= 0 on 'l', 0 on 'u')."""
    rng = np.random.default_rng(seed)
    blocks = [("l", n_nonneg)] + ([("u", n_free)] if n_free else [])
    n = n_nonneg + n_free
    xs, ss = zip(*[_primal_dual_pair(t, k, rng) for t, k in blocks])
    A = sp.random(m, n, density=density, random_state=rng, data_rvs=rng.standard_normal, format="lil")
    # every variable in at least one constraint, every constraint with at least two variables
    for j in range(n):
        A[rng.integers(m), j] = rng.standard_normal()
    for i in range(m):
        for j in rng.choice(n, 2, replace=False):
            A[i, j] = rng.standard_normal()
    return _finish(A, np.concatenate(xs), np.concatenate(ss), rng.standard_normal(m), [k for _, k in blocks],
                   [t for t, _ in blocks])


def linprog_objective(P):
    """optimum of the LP by scipy's HiGHS; 'u' variables unbounded"""
    from scipy.optimize import linprog
    bounds = []
    for t, n in zip(P["types"], P["blk"]):
        assert t in "lu"
        bounds += [(0, None) if t == "l" else (None, None)] * int(n)
    r = linprog(P["C"], A_eq=P["A"].toarray(), b_eq=P["b"], bounds=bounds, method="highs")
    assert r.status == 0, r.message
    return float(r.fun)
