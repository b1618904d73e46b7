"""The infeasibility check of the solver (INTEGRATION.md §10) on the numpy oracle, and small infeasible problems with
known certificates.  Test infrastructure only.

check_oracle runs cones_util.TypedADMMOracle and applies, after every `interval`-th iteration, the test the solver's
check kernels apply, in the same scaled space (A_s, b_s, C_s, the scaled X and y):
  dy = y_k - y_{k-p}, dX = X_k - X_{k-p}, A_s dX = Rp_{k-p} - Rp_k;
  primal: beta = b_s'dy > GAMMA |b_s| |dy| and |Pi_K(A_s'dy)| <= eps beta;
  dual:   kappa = -<C_s, dX> > GAMMA |C_s| |dX| and max(|A_s dX|, |dX - Pi_K(dX)|) <= eps kappa.
A check in an iteration whose stop test fires (converged, or the last iteration) does not run, as on the solver."""
import numpy as np
import scipy.sparse as sp

import cones_util as cz
import oracle_np as onp

GAMMA = 1e-8


class _Fired(Exception):
    pass


class _CheckedOracle(cz.TypedADMMOracle):
    """TypedADMMOracle with the check after every `interval`-th iteration (_residuals runs once at the start point and
    once at the end of every iteration, after Rp)"""

    def _residuals(self):
        super()._residuals()
        if not hasattr(self, "_k"):
            self._k = 0
            self._snap = (self.X.copy(), self.y.copy(), self.Rp.copy())
            return
        self._k += 1
        k = self._k
        if k % self.interval or max(self.maxfeas, self.relgap) < self.stop_tol or k + 1 > self.max_iter:
            return
        X0, y0, Rp0 = self._snap
        dX, dy, Adx = self.X - X0, self.y - y0, Rp0 - self.Rp
        self._snap = (self.X.copy(), self.y.copy(), self.Rp.copy())
        beta, kappa = float(self.b @ dy), -float(self.C @ dX)
        cos_p = beta / max(np.linalg.norm(self.b) * np.linalg.norm(dy), 1e-300)
        cos_d = kappa / max(np.linalg.norm(self.C) * np.linalg.norm(dX), 1e-300)
        pr = dr = np.inf
        if beta > GAMMA * np.linalg.norm(self.b) * np.linalg.norm(dy):
            pr = np.linalg.norm(self.project(self.At @ dy)) / beta
            self.min_cos_p = min(self.min_cos_p, cos_p)
        if kappa > GAMMA * np.linalg.norm(self.C) * np.linalg.norm(dX):
            dr = max(np.linalg.norm(Adx), np.linalg.norm(dX - self.project(dX))) / kappa
            self.min_cos_d = min(self.min_cos_d, cos_d)
        self.min_pr, self.min_dr = min(self.min_pr, pr), min(self.min_dr, dr)
        fired = (pr <= self.eps) | ((dr <= self.eps) << 1)
        if fired:
            self.result = dict(reason=3 if fired & 1 else 4, iter=k, fired=fired, pratio=pr, dratio=dr, dy=dy, dX=dX,
                               beta=beta, kappa=kappa)
            raise _Fired()


def check_oracle(P, interval=50, eps=1e-7, max_iter=3000, stop_tol=1e-6, switch_admm=11000):
    """runs the oracle with the check; returns a dict: reason (1 converged or 2 max_iter when nothing fired, 3 / 4),
    iter, the ratios, the certificate directions in scaled space, and the smallest ratios and guard cosines
    (b_s'dy / |b_s||dy|, -<C_s, dX> / |C_s||dX|) of the candidates that passed the guard"""
    o = _CheckedOracle.__new__(_CheckedOracle)
    o.interval, o.eps, o.stop_tol, o.max_iter = interval, eps, stop_tol, max_iter
    o.min_pr = o.min_dr = o.min_cos_p = o.min_cos_d = np.inf
    o.result = None
    _CheckedOracle.__init__(o, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"],
                            P["b_val"], P["C_idx"], P["C_val"], P["blk"], types=P.get("types"))
    try:
        _, _, _, it = o.solve(max_iter, stop_tol, 500, 50, 100, switch_admm, 1.05)
        r = dict(reason=2 if it >= max_iter else 1, iter=it)
    except _Fired:
        r = o.result
    r.update(min_pratio=o.min_pr, min_dratio=o.min_dr, min_cos_p=o.min_cos_p, min_cos_d=o.min_cos_d, oracle=o)
    return r


def make(types, blk, rows, b, C):
    """a problem dict (the keys of cones_util's generators) from dense constraint rows over the typed svec vector"""
    off = cz.svec_offsets(blk, types)
    A = sp.csr_matrix(np.array(rows, float).reshape(len(rows), int(off[-1])))
    A.sort_indices()
    b, C = np.asarray(b, float), np.asarray(C, float)
    nzb, nzc = np.nonzero(b)[0], np.nonzero(C)[0]
    return dict(blk=np.array(blk, np.int32), types=types, vec_len=int(off[-1]), con_num=A.shape[0],
                col_ptrs=A.indptr.astype(np.int32), row_ids=A.indices.astype(np.int32), vals=A.data,
                b_idx=nzb.astype(np.int32), b_val=b[nzb], C_idx=nzc.astype(np.int32), C_val=C[nzc], A=A, b=b, C=C)


def _trace_row(blk, types, k):
    """the row <I, X_k> of block k over the typed svec vector"""
    off = cz.svec_offsets(blk, types)
    row = np.zeros(int(off[-1]))
    row[off[k]:off[k + 1]] = onp.svec(np.eye(int(blk[k])))
    return row


def _mix():
    """primal infeasible through its 'l' block, with PSD blocks in several Jacobi size classes: tr X_k = 1 on every
    's' block, sum of the 'l' block = -1, the 'u' entries fixed"""
    blocks = [("s", 3), ("l", 10), ("s", 20), ("u", 3), ("s", 40), ("s", 100)]
    types, blk = "".join(t for t, _ in blocks), [n for _, n in blocks]
    off = cz.svec_offsets(blk, types)
    rows, b = [], []
    for k, t in enumerate(types):
        if t == "s":
            rows.append(_trace_row(blk, types, k)); b.append(1.0)
        elif t == "l":
            r = np.zeros(int(off[-1])); r[off[k]:off[k + 1]] = 1.0; rows.append(r); b.append(-1.0)
        else:
            for j in range(int(off[k]), int(off[k + 1])):
                r = np.zeros(int(off[-1])); r[j] = 1.0; rows.append(r); b.append(0.5)
    C = np.concatenate([_trace_row(blk, types, k)[off[k]:off[k + 1]] if t == "s" else np.ones(int(off[k + 1] - off[k]))
                        for k, t in enumerate(types)])
    return make(types, blk, rows, b, C)


def _mix_dual():
    """unbounded in two blocks ('s' 3x3: min -X00 - X11 with X22 = 1, X01 = 0; 'l': min -x0 with x0 = x1, x2 = 1) next
    to two bounded PSD blocks (tr X = 1, C = I), so that every rank of a sharded solver owns a part of d"""
    blocks = [("s", 3), ("s", 5), ("l", 3), ("s", 4)]
    types, blk = "".join(t for t, _ in blocks), [n for _, n in blocks]
    off = cz.svec_offsets(blk, types)
    n = int(off[-1])

    def row(k, local):
        r = np.zeros(n); r[off[k]:off[k + 1]] = local; return r
    rows = [row(0, [0, 0, 0, 0, 0, 1]), row(0, [0, 1, 0, 0, 0, 0]), _trace_row(blk, types, 1),
            row(2, [1, -1, 0]), row(2, [0, 0, 1]), _trace_row(blk, types, 3)]
    b = [1, 0, 1, 0, 1, 1]
    C = np.concatenate([-onp.svec(np.diag([1., 1, 0])), onp.svec(np.eye(5)), [-1, 0, 0], onp.svec(np.eye(4))])
    return make(types, blk, rows, b, C)


def _dense_block(n=200):
    """one PSD block on the dense sign path (n > 168) with tr X = -1"""
    return make("s", [n], [_trace_row([n], "s", 0)], [-1.0], onp.svec(np.eye(n)))


def problems():
    """name -> (problem, expected stop reason)"""
    r = np.sqrt(2)
    return {
        # x >= 0, x0 + x1 = -1
        "lp_primal": (make("l", [4], [[1, 1, 0, 0], [0, 0, 1, -1]], [-1, 1], [1, 2, 0, 1]), 3),
        # 3x3 PSD, tr X = -1
        "sdp_primal": (make("s", [3], [[1, 0, 1, 0, 0, 1], [0, r / 2, 0, 0, 0, 0]], [-1, 0.3], onp.svec(np.eye(3))), 3),
        # s + l + u, infeasible through the 'l' block
        "mixed_primal": (make("slu", [2, 2, 1], [[1, 0, 1, 0, 0, 0], [0, 0, 0, 1, 1, 0], [0, 0, 0, 0, 0, 1]], [1, -2, 3],
                              [1, 0, 1, 1, 1, 0]), 3),
        # min -x0, x0 = x1, x2 = 1, x >= 0 (unbounded)
        "lp_dual": (make("l", [3], [[1, -1, 0], [0, 0, 1]], [0, 1], [-1, 0, 0]), 4),
        # min -X00 - X11, X22 = 1, X01 = 0 (unbounded)
        "sdp_dual": (make("s", [3], [[0, 0, 0, 0, 0, 1], [0, 1, 0, 0, 0, 0]], [1, 0], -onp.svec(np.diag([1., 1, 0]))), 4),
        "dense_primal": (_dense_block(), 3),
        "mix_classes_primal": (_mix(), 3),
        "mix_dual": (_mix_dual(), 4),
    }


def feasible_problems():
    """the typed synthetic, the same with every constraint duplicated (null(A') of dimension m) and a random LP"""
    P = cz.typed_synthetic([("s", 5), ("l", 30), ("s", 8), ("u", 6), ("s", 3), ("l", 12)], 40, seed=4)
    A = sp.vstack([P["A"], P["A"]]).tocsr()
    A.sort_indices()
    b = np.concatenate([P["b"], P["b"]])
    nzb = np.nonzero(b)[0]
    D = dict(P, col_ptrs=A.indptr.astype(np.int32), row_ids=A.indices.astype(np.int32), vals=A.data,
             con_num=A.shape[0], b_idx=nzb.astype(np.int32), b_val=b[nzb], A=A, b=b)
    return {"typed": P, "typed_duplicated": D, "lp": cz.random_lp(40, 8, 15, seed=1)}


def dual_cone_violation(P, v):
    """per block of the typed layout: the largest eigenvalue ('s'), the largest entry ('l'), the largest |entry| ('u')
    of v; v in -K* makes every one of them <= 0 (0 on 'u')"""
    off = cz.svec_offsets(P["blk"], P["types"])
    out = []
    for k, t in enumerate(P["types"]):
        seg = v[off[k]:off[k + 1]]
        if t == "s":
            out.append(float(np.linalg.eigvalsh(onp.smat(seg, int(P["blk"][k])))[-1]))
        elif t == "l":
            out.append(float(seg.max()))
        else:
            out.append(float(np.abs(seg).max()))
    return max(out)


def primal_cone_distance(P, d):
    """|d - Pi_K(d)| over the typed layout"""
    return float(np.linalg.norm(d - cz.project_typed(P["blk"], P["types"], d)))
