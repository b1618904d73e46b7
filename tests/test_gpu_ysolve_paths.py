"""Every kernel path of the y-solve against an extended-precision reference.

The ordering, the elimination tree, the subtree split, the packing decisions, the collapsed chains and the dense-tail cut
depend only on the sparsity pattern of A A^T, not on eps.  An operator built with eps = 1 therefore runs exactly the
kernel configuration it runs at eps = 1e-15, on a system whose condition number is a few tens to hundreds, and can be
held to a forward error of 1e-12 and a backward error of 1e-14 instead of the 1e-6 residual that the numerically singular
eps = 1e-15 system allows (DESIGN 5).  Every test asserts the path counters (YSolve.paths()) of the paths it claims to
cover, so a retuned threshold that moves its work to another path fails the test instead of passing vacuously.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import oracle_np as onp

FWD_TOL = 1e-12        # ||y - y_ref||_2 / ||y_ref||_2, with kappa_hat <= 1e3
BWD_TOL = 1e-14        # ||r - M y||_inf / (||M||_inf ||y||_inf + ||r||_inf)
KAPPA_MAX = 1e3


# ---------------------------------------------------------------- reference
def _n2(v):
    return np.sqrt(np.sum(v * v))


class Reference:
    """M = A A^T + eps I formed in long double (u = 1.1e-19 on x86-64), factored in double with SuperLU as
    oracle_np.AATSolver does, then iterative refinement with the residual computed in long double."""

    def __init__(self, A, eps, steps=3):
        m = A.shape[0]
        Al = sp.csr_matrix(A).astype(np.longdouble)
        self.M = (Al @ Al.T + np.longdouble(eps) * sp.eye(m, dtype=np.longdouble, format="csr")).tocsr()
        self.lu = spla.splu(self.M.astype(np.float64).tocsc(), permc_spec="MMD_AT_PLUS_A", diag_pivot_thresh=0.0,
                            options=dict(SymmetricMode=True))
        self.norm_inf = float(np.max(np.asarray(abs(self.M).sum(axis=1))))
        self.kappa = self.norm_inf / eps      # Gershgorin: lambda_max <= ||M||_inf and lambda_min >= eps
        self.steps = steps

    def solve(self, r):
        rl = np.asarray(r, np.longdouble)
        y = self.lu.solve(np.asarray(r, np.float64)).astype(np.longdouble)
        for _ in range(self.steps):
            y += self.lu.solve((rl - self.M @ y).astype(np.float64))
        return y

    def errors(self, r, y, y_ref=None):
        """(forward, backward) error of y, both evaluated in long double"""
        if y_ref is None:
            y_ref = self.solve(r)
        yl, rl = np.asarray(y, np.longdouble), np.asarray(r, np.longdouble)
        fwd = _n2(yl - y_ref) / _n2(y_ref)
        bwd = np.max(np.abs(rl - self.M @ yl)) / (self.norm_inf * np.max(np.abs(yl)) + np.max(np.abs(rl)))
        return float(fwd), float(bwd)


def _check(R, r, y, what):
    assert R.kappa <= KAPPA_MAX, (what, R.kappa)
    assert np.all(np.isfinite(y)), what
    fwd, bwd = R.errors(r, y)
    print(f"[ysolve-paths] {what}: forward {fwd:.2e} backward {bwd:.2e} kappa_hat {R.kappa:.1f}")
    assert fwd <= FWD_TOL and bwd <= BWD_TOL, (what, fwd, bwd)
    return fwd, bwd


def test_reference_matches_dense_solve():
    """the reference helper itself, against LAPACK on the dense matrix (m = 300)"""
    from cuadmm_b200.synthetic import chain_sdp
    P = chain_sdp(np.array([6, 9, 12, 7, 10, 8], np.int32), 300, seed=3)
    A = sp.csr_matrix((P["vals"], P["row_ids"], P["col_ptrs"]), shape=(P["con_num"], P["vec_len"]))
    eps = 0.25
    R = Reference(A, eps)
    Md = (A @ A.T).toarray() + eps * np.eye(300)
    assert np.linalg.cond(Md) <= R.kappa <= KAPPA_MAX
    r = np.random.default_rng(4).standard_normal(300)
    y_ref = R.solve(r)
    y_dense = np.linalg.solve(Md, r)
    assert _n2(y_dense - y_ref) / _n2(y_ref) <= 1e-14
    fwd, bwd = R.errors(r, y_dense, y_ref)
    assert fwd <= 1e-14 and bwd <= 1e-15
    # refinement reaches the long-double floor; one unrefined double solve does not
    assert R.errors(r, y_ref, y_ref)[1] <= 1e-18
    assert Reference(A, eps, steps=0).errors(r, R.lu.solve(r), y_ref)[0] > 1e-18


# ---------------------------------------------------------------- operators and helpers
def _csr(P, normalise=True):
    vals = onp.get_normA_fast(P["col_ptrs"], P["vals"])[1] if normalise else P["vals"]
    A = sp.csr_matrix((vals, P["row_ids"], P["col_ptrs"]), shape=(P["con_num"], P["vec_len"]))
    A.sort_indices()
    return A


def _ysolve(A, eps):
    import cuadmm_b200 as cu
    return cu.YSolve(A.shape[0], A.shape[1], A.indptr, A.indices, A.data, eps=eps)


_STRUCTURAL = ("n_sub", "n_sub_pack", "n_sub_warp", "n_sub_cta", "pk_rows", "pk_n_heavy", "pk_has_ext", "collapsed",
               "levels", "narrow_phases", "wide_phases", "top_long_slots")


def _structure(paths):
    """the counters that depend on the sparsity pattern only (chunk, record and tile counts also see the exact zeros
    that pinned pivots put into L and into the chain inverses)"""
    return dict(fwd={k: paths["fwd"][k] for k in _STRUCTURAL}, bwd={k: paths["bwd"][k] for k in _STRUCTURAL},
                n_tail=paths["tail"]["n_tail"])


def _largest_subtree_rows(A, perm, n_lead, cap=12000, min_size=2):
    """constraint indices of the largest subtree that choose_subtrees (ysolve.cu) cuts from the elimination tree of the
    lead part; perm[new] = old is the solve's permutation (YSolve.perm(); lead unknowns are in the factor's order)"""
    m = A.shape[0]
    inv = np.empty(m, np.int64); inv[perm] = np.arange(m)
    G = sp.triu(sp.csr_matrix((A @ A.T).astype(bool)), k=1).tocoo()
    i, j = np.minimum(inv[G.row], inv[G.col]), np.maximum(inv[G.row], inv[G.col])
    keep = i < n_lead
    U = sp.csc_matrix((np.ones(int(keep.sum()), np.int8), (i[keep], j[keep])), shape=(m, m))
    indptr, indices = U.indptr.tolist(), U.indices.tolist()
    parent, anc = [-1] * m, [-1] * m          # elimination tree (Liu, path compression), lead columns only matter
    for k in range(m):
        for q in range(indptr[k], indptr[k + 1]):
            v = indices[q]
            while v != -1 and v < k:
                nxt = anc[v]; anc[v] = k
                if nxt == -1:
                    parent[v] = k
                v = nxt
    size = [1] * m
    for v in range(n_lead):
        p = parent[v]
        if 0 <= p < n_lead:
            size[p] += size[v]
    sub = [-1] * m
    roots = []
    for v in range(n_lead - 1, -1, -1):
        p = parent[v]
        if not (p < 0 or p >= n_lead or sub[p] < 0):
            sub[v] = sub[p]
            continue
        parent_fits = 0 <= p < n_lead and size[p] <= cap
        if size[v] <= cap and not parent_fits and size[v] >= min_size:
            sub[v] = len(roots); roots.append(v)
    sub = np.array(sub[:n_lead])
    big = int(np.argmax([size[v] for v in roots]))
    return perm[:n_lead][sub == big]


def _equal_bits(a, b):
    return np.array_equal(a.view(np.int64), b.view(np.int64))


# ---------------------------------------------------------------- a. the bench operator at eps = 1
BENCH_M = 700000


@pytest.fixture(scope="module")
def bench():
    from cuadmm_b200.synthetic import chain_sdp, c2b_blocks
    A = _csr(chain_sdp(c2b_blocks(2000, 6, 60, 0), BENCH_M, seed=0))
    ys = _ysolve(A, 1.0)
    paths = ys.paths()
    ys15 = _ysolve(A, 1e-15)
    paths15 = ys15.paths()
    ys15.close()
    return dict(A=A, ys=ys, paths=paths, paths15=paths15, R=Reference(A, 1.0))


@pytest.mark.gpu
def test_bench_operator_paths(bench):
    p, p15 = bench["paths"], bench["paths15"]
    print(f"[ysolve-paths] bench eps=1:     {p}")
    print(f"[ysolve-paths] bench eps=1e-15: {p15}")
    assert _structure(p) == _structure(p15)
    nt = (p["tail"]["n_tail"] + 63) // 64
    for w in ("fwd", "bwd"):
        s = p[w]
        assert s["n_sub_pack"] > 0 and s["n_sub_warp"] > 0 and s["n_sub_cta"] == 0, (w, s)
        assert s["collapsed"] > 0 and s["levels"] > 0, (w, s)
        assert s["max_chunks"] >= 5, (w, s)        # > 2 x the chunk ring: the ring's mbarrier parity wraps back
    # a forward subtree depends on its own descendants only; the backward sweep's rows reach up into the top part and
    # the tail, the collapsed chains' rows into hundreds of ancestors (a warp each in pk_gather_kernel)
    assert p["fwd"]["pk_has_ext"] == 0 and p["bwd"]["pk_has_ext"] == 1 and p["bwd"]["pk_n_heavy"] > 0
    # the bench's top part is one or two wide levels per sweep: the narrow-run kernel is covered by the forced variants
    # and the star forest below
    assert p["tail"]["n_tail"] > 0 and p["tail"]["postorder_fallback"] == 0
    assert 0 < p["tail"]["tiles_lower"] < nt * (nt + 1) // 2 and 0 < p["tail"]["tiles_upper"] < nt * (nt + 1) // 2


def _bench_rhs(bench, kind):
    A, ys = bench["A"], bench["ys"]
    m, n = A.shape
    rng = np.random.default_rng(11)
    if kind == "normal":
        return rng.standard_normal(m)
    if kind == "range":
        return A @ rng.standard_normal(n)
    r = np.zeros(m)
    n_tail = bench["paths"]["tail"]["n_tail"]
    perm = ys.perm()
    if kind == "tail":
        rows = perm[m - n_tail:]
    else:       # the largest packed subtree
        rows = _largest_subtree_rows(A, perm, m - n_tail)
        assert 32 < len(rows) <= 12000
    r[rows] = rng.standard_normal(len(rows))
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["normal", "range", "subtree", "tail"])
def test_bench_operator_solve(bench, kind):
    r = _bench_rhs(bench, kind)
    _check(bench["R"], r, bench["ys"].solve_host(r), f"bench {kind}")


# ---------------------------------------------------------------- b. forced variants on a mid-size operator
@pytest.fixture(scope="module")
def mid():
    from cuadmm_b200.synthetic import chain_sdp, c2b_blocks
    A = _csr(chain_sdp(c2b_blocks(300, 6, 60, 1), 100000, seed=1))
    r = np.random.default_rng(5).standard_normal(A.shape[0])
    ys = _ysolve(A, 1.0)
    return dict(A=A, r=r, ys=ys, paths=ys.paths(), y=ys.solve_host(r), R=Reference(A, 1.0))


# (environment, check of the counters against the default build's, bit-equal to the default build)
_VARIANTS = {
    "default": ({}, lambda p, d: p["tail"]["n_tail"] > 0 and all(
        p[w]["n_sub_pack"] > 0 and p[w]["n_sub_warp"] > 0 and p[w]["collapsed"] > 0 and p[w]["levels"] > 0
        for w in ("fwd", "bwd")), True),
    "subtree_cap_0": ({"CUADMM_SWEEP_SUBTREE_CAP": "0"}, lambda p, d: all(
        p[w]["n_sub"] == 0 and p[w]["pk_rows"] == 0 and p[w]["levels"] > d[w]["levels"] for w in ("fwd", "bwd")), False),
    "subtree_cap_8": ({"CUADMM_SWEEP_SUBTREE_CAP": "8"}, lambda p, d: all(
        p[w]["n_sub_pack"] == 0 and p[w]["n_sub_warp"] > 0 and p[w]["collapsed"] == 0 for w in ("fwd", "bwd")), False),
    "subtree_cap_32": ({"CUADMM_SWEEP_SUBTREE_CAP": "32"}, lambda p, d: all(
        p[w]["n_sub_warp"] > 0 and p[w]["collapsed"] == 0 for w in ("fwd", "bwd")), False),
    "subtree_cap_33": ({"CUADMM_SWEEP_SUBTREE_CAP": "33"}, lambda p, d: all(
        p[w]["n_sub_pack"] > 0 and p[w]["n_sub_warp"] > 0 for w in ("fwd", "bwd")), False),
    "subtree_cap_200": ({"CUADMM_SWEEP_SUBTREE_CAP": "200"}, lambda p, d: all(
        p[w]["n_sub_pack"] > 0 and p[w]["n_sub_warp"] > 0 and p[w]["collapsed"] > 0 for w in ("fwd", "bwd")), False),
    "subtree_min_1000": ({"CUADMM_SWEEP_SUBTREE_MIN": "1000"}, lambda p, d: all(
        p[w]["n_sub_warp"] == 0 and p[w]["n_sub_pack"] > 0 and p[w]["levels"] > d[w]["levels"] for w in ("fwd", "bwd")),
        False),
    "chain_max_0": ({"CUADMM_SWEEP_CHAIN_MAX": "0"}, lambda p, d: all(
        p[w]["collapsed"] == 0 and p[w]["n_sub_pack"] == d[w]["n_sub_pack"] for w in ("fwd", "bwd")), False),
    "chain_max_384": ({"CUADMM_SWEEP_CHAIN_MAX": "384"}, lambda p, d: p == d, True),
    # above the chain slots that the shared-memory budget reserves: clamped to them
    "chain_max_768": ({"CUADMM_SWEEP_CHAIN_MAX": "768"}, lambda p, d: p == d, True),
    "narrow_slots_0": ({"CUADMM_SWEEP_NARROW_SLOTS": "0"}, lambda p, d: all(
        p[w]["narrow_phases"] == 0 and p[w]["wide_phases"] == p[w]["levels"] > 0 for w in ("fwd", "bwd")), True),
    "narrow_slots_1e9": ({"CUADMM_SWEEP_NARROW_SLOTS": "1000000000"}, lambda p, d: all(
        p[w]["narrow_phases"] == 1 and p[w]["wide_phases"] == 0 for w in ("fwd", "bwd")), True),
    "init_threads_1": ({"CUADMM_INIT_THREADS": "1"}, lambda p, d: p == d, True),
    "max_tail_0": ({"CUADMM_YSOLVE_MAX_TAIL": "0"}, lambda p, d: p["tail"]["n_tail"] == 0, False),
    "max_tail_300": ({"CUADMM_YSOLVE_MAX_TAIL": "300", "CUADMM_YSOLVE_MIN_DEPTH": "4"},
                     lambda p, d: 0 < p["tail"]["n_tail"] <= 300, False),
    "tail_order": ({"CUADMM_YSOLVE_TAIL_POSTORDER": "0"}, lambda p, d: p["tail"]["n_tail"] == d["tail"]["n_tail"] and
                   p["tail"]["postorder_fallback"] == 0 and p["tail"]["tiles_lower"] > d["tail"]["tiles_lower"], False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(_VARIANTS))
def test_forced_variant(mid, monkeypatch, name):
    env, check, bit_equal = _VARIANTS[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ys = _ysolve(mid["A"], 1.0)
    p = ys.paths()
    print(f"[ysolve-paths] mid {name}: {p}")
    assert check(p, mid["paths"]), (p, mid["paths"])
    y = ys.solve_host(mid["r"])
    _check(mid["R"], mid["r"], y, f"mid {name}")
    if bit_equal:      # only the launch structure changed, not any row's summation order
        assert _equal_bits(y, mid["y"])


# ---------------------------------------------------------------- c. star forest: record and kernel boundaries
STAR_K = (1, 2, 24, 25, 31, 32, 767, 768, 769, 1500)
PATH_ROWS = 5000


def _star_forest(path_rows=0, seed=7):
    """disconnected stars: hub constraint h shares a distinct svec entry with each of its k leaves, every leaf has an
    entry of its own.  Leaves are eliminated first, so a star is one subtree whose hub row has k in-subtree entries.
    Optionally one path of path_rows constraints (consecutive ones share an entry), longer than the subtree cap, for
    the top kernels.  Hub coefficients are scaled by 1/sqrt(k) so that kappa_hat stays near 1 + sqrt(k)."""
    rng = np.random.default_rng(seed)
    rows, cols, vals = [], [], []
    con = col = 0

    def coef(n, scale=1.0):
        return scale * rng.uniform(0.5, 1.0, n) * rng.choice([-1.0, 1.0], n)

    for k in STAR_K:
        hub = con
        shared = col + np.arange(k)
        own = col + k + np.arange(k)
        rows += [np.full(k, hub)]; cols += [shared]; vals += [coef(k, 1.0 / np.sqrt(k))]
        leaves = hub + 1 + np.arange(k)
        rows += [leaves, leaves]; cols += [shared, own]; vals += [coef(k), coef(k)]
        con += k + 1; col += 2 * k
    if path_rows:
        path = con + np.arange(path_rows)
        rows += [path, path]; cols += [col + np.arange(path_rows), col + 1 + np.arange(path_rows)]
        vals += [coef(path_rows), coef(path_rows)]
        con += path_rows; col += path_rows + 1
    A = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(con, col))
    A.sort_indices()
    return A


@pytest.mark.gpu
@pytest.mark.parametrize("path_rows", [0, PATH_ROWS])
def test_star_forest_boundaries(path_rows):
    A = _star_forest(path_rows)
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("CUADMM_SWEEP_SUBTREE_CAP", "1600")     # every star is a subtree, the path is not
        mp.setenv("CUADMM_SWEEP_CHAIN_MAX", "0")          # no chain inverse: long records are the hub rows only
        mp.setenv("CUADMM_YSOLVE_MAX_TAIL", "0")          # the path's top levels stay in the sweeps
        ys = _ysolve(A, 1.0)
    p = ys.paths()
    print(f"[ysolve-paths] star forest, path of {path_rows}: {p}")
    f, b = p["fwd"], p["bwd"]
    # forward: a hub row has k in-subtree entries.  k <= 31: warp-packed (<= 32 rows); k = 32..768: CTA-packed;
    # k > 768 (kPkMaxRowEntries): the generic CTA-per-subtree kernel.  Backward: every row has at most one in-subtree
    # entry (a leaf's on its hub), so every star is packed
    assert f["n_sub_cta"] == 2 and b["n_sub_cta"] == 0, p
    for s in (f, b):
        assert s["collapsed"] == 0, s
    assert p["tail"]["n_tail"] == 0
    if path_rows == 0:
        assert f["n_sub_warp"] == 5 and f["n_sub_pack"] == 3 and b["n_sub_warp"] == 5 and b["n_sub_pack"] == 5, p
        # short (4-lane) records up to 24 entries, warp-wide from 25: the hubs of k = 25, 31, 32, 767, 768
        assert f["long_records"] == 5 and b["long_records"] == 0, p
        assert f["levels"] == 0 and b["levels"] == 0, p
    else:
        # the path's subtrees are CTA-packed, its upper part runs in the top kernels
        assert f["n_sub_warp"] == 5 and f["n_sub_pack"] > 3, p
        for s in (f, b):
            assert s["levels"] > 0 and s["narrow_phases"] > 0, s
    R = Reference(A, 1.0)
    rng = np.random.default_rng(8)
    for what, r in (("normal", rng.standard_normal(A.shape[0])), ("range", A @ rng.standard_normal(A.shape[1]))):
        _check(R, r, ys.solve_host(r), f"star forest, path of {path_rows}, {what}")


@pytest.mark.gpu
def test_later_object_with_smaller_subtrees(bench):
    """the packed kernel's dynamic shared-memory limit is a property of the kernel, shared by every y-solve on the
    device: creating one with smaller subtrees (the star forest's largest packed one has 769 rows, the bench's thousands) must
    not lower it below what an existing one launches with"""
    ys = bench["ys"]
    r = np.random.default_rng(24).standard_normal(ys.m)
    y = ys.solve_host(r)
    small = _ysolve(_star_forest(), 1.0)
    assert _equal_bits(ys.solve_host(r), y)
    small.close()


# ---------------------------------------------------------------- d. state between solves
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mid", "bench"])
def test_nan_solve_leaves_no_state(request, name):
    """a clean solve after one whose right-hand side holds NaN equals a fresh object's solve bit for bit: nothing of
    x, z, the packed rows' w, the chain scratch slots or the tail's intermediate vector is read before it is written"""
    o = request.getfixturevalue(name)
    ys = o["ys"]
    r = np.random.default_rng(21).standard_normal(ys.m)
    bad = r.copy(); bad[::5] = np.nan
    assert np.isnan(ys.solve_host(bad)).any()
    y = ys.solve_host(r)
    assert not np.isnan(y).any()
    fresh = _ysolve(o["A"], 1.0)
    assert _equal_bits(y, fresh.solve_host(r))
    fresh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mid", "bench"])
def test_side_stream_equals_host_entry(request, name):
    """solve_device on a non-default stream (the subtree kernels fork to the solve's side stream and join back)"""
    import torch
    o = request.getfixturevalue(name)
    ys = o["ys"]
    r = np.random.default_rng(22).standard_normal(ys.m)
    y_host = ys.solve_host(r)
    d_r = torch.from_numpy(r).cuda()
    d_y = torch.full_like(d_r, float("nan"))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            ys.solve_device(d_r.data_ptr(), d_y.data_ptr(), s.cuda_stream)
    s.synchronize()
    assert _equal_bits(d_y.cpu().numpy(), y_host)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mid", "bench"])
def test_power_of_two_scaling_is_exact(request, name):
    o = request.getfixturevalue(name)
    ys = o["ys"]
    r = np.random.default_rng(23).standard_normal(ys.m)
    y = ys.solve_host(r)
    for e in (200, -200):
        assert _equal_bits(ys.solve_host(np.ldexp(r, e)), np.ldexp(y, e))
