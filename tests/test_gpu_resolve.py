"""Re-solves with new b and C on an initialised solver (cuadmm_solver_update_data): a cold update against a fresh init
with the same data, a warm update against a fresh init at the previous solution, the committed PushT_N=10 log through an
update, rejected input, and the sharded solver on 2 and 3 ranks against the single-GPU update."""
import os

import numpy as np
import pytest

import cuadmm_b200 as cu
import cones_util as cz
from test_gpu_multi import launch
from util_problems import GOLD, load_fixture, parse_log

pytestmark = pytest.mark.gpu

CUADMM_EINVAL = -1
# all 's', with one block on the dense sign path (n > 168); and the typed mix of tests/test_gpu_cones.py
PSD = [("s", 6), ("s", 20), ("s", 200), ("s", 40), ("s", 13), ("s", 90)]
TYPED = [("s", 5), ("l", 30), ("s", 8), ("u", 6), ("s", 3), ("l", 12), ("s", 20), ("u", 9)]
CASES = {"psd": (PSD, 400), "typed": (TYPED, 60)}


def _problem(case, seed=3):
    blocks, m = CASES[case]
    P = cz.typed_synthetic(blocks, m, seed=seed)
    if case == "psd":
        P["types"] = None
    return P


def _triplets(v):
    i = np.nonzero(v)[0]
    return i.astype(np.int32), v[i]


def new_data(P, seed, w=0.1, drop=0.0):
    """b2 = A x2, C2 = S2 + A^T y* with x2, S2 convex combinations of the problem's x*, s* and another primal-dual pair
    in the same cones: feasible again, with a new optimum.  drop > 0 leaves out that share of the triplets (a new
    pattern), and the first C triplet is preceded by a stale value for the same index, which the later one replaces."""
    blocks = list(zip(P["types"] or "s" * len(P["blk"]), P["blk"]))
    Q = cz.typed_synthetic(blocks, 1, seed=seed)
    x2 = (1 - w) * P["xstar"] + w * Q["xstar"]
    C2 = P["C"] + w * (Q["sstar"] - P["sstar"])
    bi, bv = _triplets(P["A"] @ x2)
    ci, cv = _triplets(C2)
    if drop:
        rng = np.random.default_rng(seed)
        kb, kc = rng.random(len(bi)) >= drop, rng.random(len(ci)) >= drop
        bi, bv, ci, cv = bi[kb], bv[kb], ci[kc], cv[kc]
    ci, cv = np.concatenate([ci[:1], ci]), np.concatenate([[1e3], cv])
    return bi, bv, ci, cv


def fresh(P, data=None, **kw):
    bi, bv, ci, cv = data if data is not None else (P["b_idx"], P["b_val"], P["C_idx"], P["C_val"])
    s = cu.Solver(verbose=False)
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], bi, bv, ci, cv, P["blk"],
           blk_types=P.get("types"), **kw)
    return s


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)) if len(b) else 0.0


def compare_to_fresh(s, f, P, tol_hist=1e-11, tol_vec=1e-10, control=None, exact=False):
    """s (updated) against f (fresh init).  init and update_data load b and C through one device path, so where nothing
    on the way is run-to-run dependent (exact=True) every history and X, S and y are equal bit for bit.
    Otherwise histories are compared relative to their largest entry: a difference in the last bits of a scale moves a
    residual by a roughly constant absolute amount, so entry by entry a residual that fell by eight orders would show
    it magnified eight orders.  control: a second fresh init of the same data.  Blocks n > 168 (dense sign path) sum
    |A|_F^2 with floating-point atomicAdd, so two fresh inits differ from each other run to run; the update may then
    differ from f by up to 10x what the control does, never by less than the tolerances."""
    assert s.info_iter_num == f.info_iter_num
    if exact:
        for key in cu.Solver.HIST:
            assert np.array_equal(s.history(key), f.history(key)), key
        for name in ["X", "S", "y"]:
            assert np.array_equal(getattr(s, name), getattr(f, name)), name
    for key in ["errRp", "errRd", "pobj", "dobj", "sig", "relgap"]:
        a, b = s.history(key), f.history(key)
        err = _rel(a, b)
        ctrl = _rel(control.history(key), b) if control is not None else 0.0
        pointwise = float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))
        print("  %-6s rel diff %.2e (entry by entry %.2e; fresh vs fresh %.2e)" % (key, err, pointwise, ctrl))
        assert err < max(1e-9 if key == "relgap" else tol_hist, 10 * ctrl), key
    A = P["A"]
    for name, g in [("X", lambda t: t.X), ("S", lambda t: t.S), ("Aty", lambda t: A.T @ t.y)]:
        a, b = g(s), g(f)
        err = float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))
        ctrl = float(np.linalg.norm(g(control) - b) / max(np.linalg.norm(b), 1e-300)) if control is not None else 0.0
        print("  %-6s rel diff %.2e (fresh vs fresh %.2e)" % (name, err, ctrl))
        assert err < max(tol_vec, 10 * ctrl), name
    if P.get("types"):
        off = cz.svec_offsets(P["blk"], P["types"])
        for k, t in enumerate(P["types"]):
            if t == "u":
                assert np.all(s.S[off[k]:off[k + 1]] == 0.0)


def _run_args(mode, iters=60):
    return (iters, 1e-12, 500, 50, 100, 11000 if mode == "sgs" else 1, 1.05)


@pytest.mark.parametrize("graph", [True, False], ids=["graph", "no_graph"])
@pytest.mark.parametrize("mode", ["sgs", "admm"])
@pytest.mark.parametrize("case", ["psd", "typed"])
def test_cold_update_equals_fresh_init(case, mode, graph, monkeypatch):
    if not graph:
        monkeypatch.setenv("CUADMM_NO_GRAPH", "1")
    P = _problem(case)
    data = new_data(P, seed=11, drop=0.1)
    s = fresh(P)
    s.solve(*_run_args(mode, 300))                    # dirty state: sigma, windows, Jacobi bases, best iterate
    s.update_data(*data, keep_iterate=False, sig=1.3)
    assert s.info_iter_num == 0
    s.solve(*_run_args(mode))
    f = fresh(P, data, sig=1.3)
    f.solve(*_run_args(mode))
    g = fresh(P, data, sig=1.3)
    g.solve(*_run_args(mode))
    assert s.info_iter_num == 60
    compare_to_fresh(s, f, P, control=g, exact=case == "typed")
    assert s.times()["update"] > 0


def test_warm_update_equals_fresh_init_at_previous_solution():
    P = _problem("psd", seed=5)
    run = (20000, 1e-6, 500, 50, 100, 11000, 1.05)
    s = fresh(P)
    s.solve(*run)
    X, y, S = s.X, s.y, s.S
    sig = float(s.history("sig")[-1])
    data = new_data(P, seed=12, w=0.05)
    s.update_data(*data, keep_iterate=True, sig=sig)
    s.solve(*run)
    f = fresh(P, data, X_vals=X, y_vals=y, S_vals=S, sig=sig)
    f.solve(*run)
    c = fresh(P, data)
    c.solve(*run)
    it_w, it_f = s.info_iter_num, f.info_iter_num
    print("warm update %d iterations, fresh init at the previous solution %d, cold %d" % (it_w, it_f, c.info_iter_num))
    assert it_f < 20000
    assert abs(it_w - it_f) <= max(1, int(0.02 * it_f))
    for key in ["pobj", "dobj"]:
        a, b = s.history(key)[-1], f.history(key)[-1]
        assert abs(a - b) <= 1e-6 * abs(b), key


def test_iterate_kept_before_any_solve():
    # keep_iterate right after init: the start point is init's X0, y0, S0 (held scaled until a solve), unscaled first
    P = _problem("psd")
    rng = np.random.default_rng(1)
    X0, y0, S0 = 0.1 * rng.standard_normal(P["vec_len"]), rng.standard_normal(P["con_num"]), 0.1 * rng.standard_normal(P["vec_len"])
    data = new_data(P, seed=13)
    s = fresh(P, X_vals=X0, y_vals=y0, S_vals=S0)
    s.update_data(*data, keep_iterate=True, sig=1.0)
    s.solve(*_run_args("sgs"))
    f = fresh(P, data, X_vals=X0, y_vals=y0, S_vals=S0)
    f.solve(*_run_args("sgs"))
    compare_to_fresh(s, f, P, tol_hist=1e-9, tol_vec=1e-9)


def test_reference_log_through_an_update():
    # the solve after a cold update to the true data stops where the reference's own run stopped
    P = load_fixture("pusht_n10")
    rows = parse_log(os.path.join(GOLD, "pusht_n10_sgs.log"))
    assert rows[-1]["it"] == 6149
    rng = np.random.default_rng(0)
    s = cu.Solver(verbose=False)
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], 1.1 * P["b_val"],
           P["C_idx"], P["C_val"] * (1 + 0.05 * rng.standard_normal(len(P["C_val"]))), P["blk"], None, None, None, 1.0)
    s.solve(300, 1e-3, 0, 50, 100, 11000, 1.05)
    s.update_data(P["b_idx"], P["b_val"], P["C_idx"], P["C_val"], keep_iterate=False, sig=1.0)
    s.solve(20000, 1e-3, 0, 50, 100, 11000, 1.05)
    assert s.info_iter_num == 6149, s.info_iter_num
    assert abs(s.history("pobj")[-1] - rows[-1]["pobj"]) <= 2e-4 * abs(rows[-1]["pobj"]) + 1e-9


def test_bad_input_leaves_solver_usable():
    P = _problem("typed")
    data = new_data(P, seed=11, drop=0.1)
    s = fresh(P)
    s.solve(*_run_args("admm", 100))
    bi, bv, ci, cv = data
    for bad in [(bi, bv, np.append(ci, P["vec_len"]).astype(np.int32), np.append(cv, 1.0)),
                (np.append(bi, -1).astype(np.int32), np.append(bv, 1.0), ci, cv),
                (np.append(bi, P["con_num"]).astype(np.int32), np.append(bv, 1.0), ci, cv)]:
        with pytest.raises(cu.CuadmmError) as e:
            s.update_data(*bad, keep_iterate=False, sig=1.3)
        assert e.value.code == CUADMM_EINVAL
    assert s.info_iter_num == 100                      # the rejected calls changed nothing
    s.update_data(*data, keep_iterate=False, sig=1.3)
    s.solve(*_run_args("sgs"))
    f = fresh(P, data, sig=1.3)
    f.solve(*_run_args("sgs"))
    compare_to_fresh(s, f, P, exact=True)


@pytest.mark.parametrize("world", [2, 3], ids=["2-peer", "3-peer"])
def test_sharded_update_matches_single_gpu(world):
    procs, outs = launch(world, "resolve_rank_worker.py")
    print(outs[0])
    assert "RESOLVE_RANK_OK" in outs[0], "\n".join(o[-3000:] for o in outs)
    assert all(p.returncode == 0 for p in procs), "\n".join(o[-3000:] for o in outs)
