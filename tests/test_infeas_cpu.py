"""Infeasibility detection without a GPU: the argument checks of cuadmm_solver_set_infeasibility_check, the state of a
solver that has not solved, and the numpy reference of the check (tests/infeas_util.py) on small infeasible problems,
whose certificates are verified in the caller's units, and on feasible ones, where it must never fire."""
import numpy as np
import pytest

import cuadmm_b200 as cu
import infeas_util as iu

CUADMM_EINVAL = -1


@pytest.mark.parametrize("interval,eps", [(-1, 1e-7), (-50, 1e-7), (50, 0.0), (50, -1e-7), (50, 1.0), (50, 2.0),
                                          (1, float("nan"))])
def test_bad_arguments_are_rejected(interval, eps):
    s = cu.Solver()
    with pytest.raises(cu.CuadmmError) as e:
        s.set_infeasibility_check(interval, eps)
    assert e.value.code == CUADMM_EINVAL


def test_good_arguments_and_off():
    s = cu.Solver()
    s.set_infeasibility_check(50, 1e-7)
    s.set_infeasibility_check(1, 0.5)
    s.set_infeasibility_check(0, 0.0)            # off: eps is not looked at
    s.set_infeasibility_check(0, 5.0)


def test_check_and_sharding_in_either_order():
    s = cu.Solver()
    s.set_distributed(0, 2, cu.unique_id())
    s.set_infeasibility_check(50, 1e-7)
    t = cu.Solver()
    t.set_infeasibility_check(50, 1e-7)
    t.set_distributed(0, 2, cu.unique_id())


def test_no_stats_before_a_solve():
    st = cu.Solver().infeasibility_stats()
    assert st["checks"] == 0 and st["primal_projections"] == 0 and st["dual_projections"] == 0


def test_no_stop_reason_or_certificate_before_a_solve():
    s = cu.Solver()
    assert s.stop_reason == 0
    s.set_infeasibility_check(50)
    for which in (0, 1):
        with pytest.raises(cu.CuadmmError) as e:
            s.certificate(which)
        assert e.value.code == CUADMM_EINVAL


def _unscaled_certificate(P, r):
    """the certificate in the caller's units as the solver returns it: y-bar = dy ./ normA / (bscale beta),
    d = dX / (Cscale kappa)"""
    o = r["oracle"]
    if r["reason"] == 3:
        return r["dy"] / o.normA / (o.bscale * r["beta"])
    return r["dX"] / (o.Cscale * r["kappa"])


@pytest.mark.parametrize("name", list(iu.problems()))
def test_reference_detects_infeasible_problems(name):
    P, reason = iu.problems()[name]
    r = iu.check_oracle(P, interval=50, eps=1e-7, max_iter=3000)
    print(name, "reason", r["reason"], "at", r["iter"], "ratios %.2e %.2e" % (r["pratio"], r["dratio"]))
    assert r["reason"] == reason
    assert r["iter"] % 50 == 0 and r["iter"] <= 1000
    c = _unscaled_certificate(P, r)
    A, b, C = P["A"], P["b"], P["C"]
    if reason == 3:
        assert abs(b @ c - 1) <= 1e-12
        assert iu.dual_cone_violation(P, A.T @ c) <= 1e-7
    else:
        assert abs(C @ c + 1) <= 1e-12
        assert np.linalg.norm(A @ c) <= 1e-7 * max(1.0, np.abs(A).max())
        assert iu.primal_cone_distance(P, c) <= 1e-7


@pytest.mark.parametrize("name", list(iu.feasible_problems()))
@pytest.mark.parametrize("interval", [10, 50])
def test_reference_never_fires_on_feasible_problems(name, interval):
    P = iu.feasible_problems()[name]
    r = iu.check_oracle(P, interval=interval, eps=1e-7, max_iter=3000, stop_tol=1e-8)
    print(name, interval, "stop", r["reason"], r["iter"], "smallest ratios %.2e %.2e, smallest guard cosines %.2e %.2e"
          % (r["min_pratio"], r["min_dratio"], r["min_cos_p"], r["min_cos_d"]))
    assert r["reason"] in (1, 2)
    assert min(r["min_pratio"], r["min_dratio"]) > 0.1
