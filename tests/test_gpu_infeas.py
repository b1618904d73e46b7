"""Infeasibility detection on the GPU (cuadmm_solver_set_infeasibility_check): small infeasible problems against the
numpy reference of the check (tests/infeas_util.py) with their certificates verified in the caller's units, the solve
unchanged bit for bit on the bundled fixtures when the check is on and never fires, an infeasible re-solve of PushT_N=10
through update_data, and run-to-run reproducibility of the certificates."""
import numpy as np
import pytest
import scipy.sparse as sp

import cuadmm_b200 as cu
import infeas_util as iu
from cuadmm_b200.synthetic import c2b_blocks, chain_sdp
from test_gpu_multi import launch
from util_problems import load_fixture

pytestmark = pytest.mark.gpu

CUADMM_EINVAL = -1
RUN = (3000, 1e-6, 500, 50, 100, 11000, 1.05)


def _solver(P, interval=0, eps=1e-7, verbose=False):
    s = cu.Solver(verbose=verbose)
    if interval:
        s.set_infeasibility_check(interval, eps)
    s.init(15, 30, P["vec_len"], P["con_num"], P["col_ptrs"], P["row_ids"], P["vals"], P["b_idx"], P["b_val"],
           P["C_idx"], P["C_val"], P["blk"], blk_types=P.get("types"))
    return s


def _check_certificate(P, s, reason, eps):
    vec, ratio = s.certificate(0 if reason == 3 else 1)
    assert 0.0 <= ratio <= eps
    A, b, C = P["A"], P["b"], P["C"]
    if reason == 3:
        assert vec.shape == (P["con_num"],)
        assert abs(b @ vec - 1) <= 1e-12
        # A'y-bar in -K* up to the ratio: |Pi_K(A'y-bar)| = ratio / bscale <= ratio bounds every eigenvalue / entry
        assert iu.dual_cone_violation(P, A.T @ vec) <= 1.01 * ratio + 1e-15
    else:
        assert vec.shape == (P["vec_len"],)
        assert abs(C @ vec + 1) <= 1e-12
        normA = np.sqrt(np.asarray(A.multiply(A).sum(axis=1)).ravel()).clip(min=1.0)
        assert np.linalg.norm(A @ vec) <= 1.01 * normA.max() * ratio + 1e-15
        assert iu.primal_cone_distance(P, vec) <= 1.01 * ratio + 1e-15
    if reason == 4:                  # both tests firing at one check stop with reason 3
        with pytest.raises(cu.CuadmmError) as e:
            s.certificate(0)
        assert e.value.code == CUADMM_EINVAL
    return vec, ratio


@pytest.mark.parametrize("name", list(iu.problems()))
def test_detection_matches_reference(name):
    P, reason = iu.problems()[name]
    s = _solver(P, 50)
    s.solve(*RUN)
    r = iu.check_oracle(P, interval=50, eps=1e-7, max_iter=RUN[0], stop_tol=RUN[1])
    print(name, "GPU: reason %d at %d; reference: reason %d at %d" % (s.stop_reason, s.info_iter_num, r["reason"], r["iter"]))
    assert s.stop_reason == r["reason"] == reason
    # observed on a B200: the same check as the reference on every problem (350, 50, 350, 300, 300, 50, 350, 300)
    assert s.info_iter_num == r["iter"]
    assert s.info_iter_num % 50 == 0 and len(s.history("pobj")) == s.info_iter_num
    _check_certificate(P, s, reason, 1e-7)
    # the iteration is the one without the check: the same history up to the detection
    if name != "dense_primal":                # the dense sign path is not reproducible bit for bit run to run
        off = _solver(P)
        off.solve(*RUN)
        assert off.stop_reason == 2 and off.info_iter_num == RUN[0]
        for key in cu.Solver.HIST:
            assert np.array_equal(s.history(key), off.history(key)[:s.info_iter_num]), key


def test_verbose_stop_line(capfd):
    P, _ = iu.problems()["lp_dual"]
    s = _solver(P, 50, verbose=True)
    s.solve(*RUN)
    out = capfd.readouterr().out
    assert "Solver ended: dual infeasible" in out and "converged" not in out


def test_certificates_are_reproducible():
    for name in ["lp_primal", "sdp_dual", "mix_classes_primal"]:
        P, reason = iu.problems()[name]
        got = []
        for _ in range(2):
            s = _solver(P, 50)
            s.solve(*RUN)
            got.append((s.info_iter_num, s.stop_reason, s.certificate(0 if reason == 3 else 1)))
        (i0, r0, (v0, q0)), (i1, r1, (v1, q1)) = got
        assert i0 == i1 and r0 == r1 == reason
        assert v0.tobytes() == v1.tobytes() and q0 == q1, name


def test_update_data_and_set_XyS_discard_the_certificate():
    P, _ = iu.problems()["lp_primal"]
    s = _solver(P, 50)
    s.solve(*RUN)
    assert s.stop_reason == 3
    s.certificate(0)
    s.update_data(P["b_idx"], P["b_val"], P["C_idx"], P["C_val"])
    with pytest.raises(cu.CuadmmError):
        s.certificate(0)
    s.solve(*RUN)
    assert s.stop_reason == 3
    s.certificate(0)
    s.set_XyS(s.X, s.y, s.S, 1.0)
    with pytest.raises(cu.CuadmmError):
        s.certificate(0)
    s.update_data(P["b_idx"], P["b_val"], P["C_idx"], P["C_val"])
    s.set_infeasibility_check(0)              # off from the next solve: runs to max_iter
    s.solve(*RUN)
    assert s.stop_reason == 2 and s.info_iter_num == RUN[0]


def _same_solve(a, b):
    assert a.info_iter_num == b.info_iter_num and a.stop_reason == b.stop_reason
    for key in cu.Solver.HIST:
        assert np.array_equal(a.history(key), b.history(key)), key
    for name in ["X", "y", "S"]:
        assert np.array_equal(getattr(a, name), getattr(b, name)), name


FIXTURES = {
    # name: (problem, solve arguments, expected stop iteration, expected stop reason)
    "planarhand_sgs": (lambda: load_fixture("planarhand_n1"), (5000, 1e-3, 0, 50, 100, 11000, 1.05), 800, 1),
    "planarhand_admm": (lambda: load_fixture("planarhand_n1"), (5000, 1e-3, 0, 50, 100, 0, 1.05), 878, 1),
    "ros_2000": (lambda: load_fixture("ros_2000"), (20000, 1e-3, 0, 50, 100, 11000, 1.05), 12732, 1),
    "pusht_n10": (lambda: load_fixture("pusht_n10"), (20000, 1e-3, 0, 50, 100, 11000, 1.05), 6149, 1),
    "pendulum_n80": (lambda: load_fixture("pendulum_n80"), (3000, 1e-12, 0, 50, 100, 11000, 1.05), 3000, 2),
    "typed": (lambda: iu.feasible_problems()["typed"], (20000, 1e-6, 500, 50, 100, 11000, 1.05), None, 1),
    "c2b_200": (lambda: chain_sdp(c2b_blocks(2000, 6, 60, 0), 700000, seed=0), (200, 1e-12, 500, 50, 100, 11000, 1.05),
                200, 2),
}


@pytest.mark.parametrize("name", list(FIXTURES))
def test_check_that_never_fires_changes_nothing(name):
    make, args, stop_iter, reason = FIXTURES[name]
    P = make()
    off = _solver(P)
    off.solve(*args)
    on = _solver(P, 50)
    on.solve(*args)
    st = on.infeasibility_stats()
    print(name, "stop", off.info_iter_num, off.stop_reason, "checks %d, projections run %d / %d, smallest ratios %.3g / %.3g, "
          "smallest guard values %.3g / %.3g" % (st["checks"], st["primal_projections"], st["dual_projections"],
                                                 st["min_primal_ratio"], st["min_dual_ratio"], st["min_primal_guard"],
                                                 st["min_dual_guard"]))
    if stop_iter is not None:
        assert off.info_iter_num == stop_iter
    assert off.stop_reason == reason
    _same_solve(on, off)
    # the check after the stopping iteration does nothing: the stop test of that iteration fired first
    assert st["checks"] == (off.info_iter_num - 1) // 50
    assert off.infeasibility_stats()["checks"] == 0
    assert min(st["min_primal_ratio"], st["min_dual_ratio"]) > 1e-7
    if name == "typed":
        # the check's projections ran beside the iteration's plan (on the numpy reference this problem passes the primal
        # guard with ratios near 1), and the iterates above are still bit-identical
        assert st["primal_projections"] > 0 and np.isfinite(st["min_primal_ratio"])
    for which in (0, 1):
        with pytest.raises(cu.CuadmmError):
            on.certificate(which)


def test_pusht_infeasible_update_and_back():
    P = load_fixture("pusht_n10")
    args = (20000, 1e-3, 0, 50, 100, 11000, 1.05)
    # constraint 17146 is X[5168] = 1 on a diagonal entry of a PSD block: b = -1 makes the problem primal infeasible
    row, j = 17146, 5168
    cp, ri = P["col_ptrs"], P["row_ids"]
    assert cp[row + 1] - cp[row] == 1 and ri[cp[row]] == j
    b = np.zeros(P["con_num"]); b[P["b_idx"]] = P["b_val"]
    assert b[row] == 1.0
    b_bad = b.copy(); b_bad[row] = -1.0
    nz = np.nonzero(b_bad)[0].astype(np.int32)
    s = _solver(P, 50)
    s.solve(*args)
    assert s.stop_reason == 1 and s.info_iter_num == 6149
    s.update_data(nz, b_bad[nz], P["C_idx"], P["C_val"], keep_iterate=False)
    s.solve(*args)
    print("PushT_N=10 with b[%d] = -1: reason %d after %d iterations, %.3f s" % (row, s.stop_reason, s.info_iter_num,
                                                                                s.times()["solve"]))
    assert s.stop_reason == 3 and s.info_iter_num < args[0]
    A = sp.csr_matrix((P["vals"], P["row_ids"], P["col_ptrs"]), shape=(P["con_num"], P["vec_len"]))
    Q = dict(P, A=A, b=b_bad, C=None, types="s" * len(P["blk"]))
    _check_certificate(Q, s, 3, 1e-7)
    # back to the true data with a cold update: the solve of a solver that never saw the infeasible data
    s.update_data(P["b_idx"], P["b_val"], P["C_idx"], P["C_val"], keep_iterate=False)
    s.solve(*args)
    f = _solver(P)
    f.solve(*args)
    assert f.info_iter_num == 6149
    _same_solve(s, f)


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_check_matches_single_gpu(world):
    procs, outs = launch(world, "infeas_rank_worker.py")
    print(outs[0])
    assert "INFEAS_RANK_OK" in outs[0], "\n".join(o[-3000:] for o in outs)
    assert all(p.returncode == 0 for p in procs), "\n".join(o[-3000:] for o in outs)
