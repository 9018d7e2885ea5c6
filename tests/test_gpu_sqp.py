"""GPU parity: the on-device Dubins SQP driver (config 4) against the numpy restatement of the same loop
(oracle/sqp_dubins.py: src/cholesky_solver.jl:109-153 + src/sqp.jl:72-94)."""
import numpy as np
import pytest

from lqr_b200.sqp import DubinsSQP

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


@pytest.mark.parametrize("N,batch", [(11, 5), (11, 70), (201, 3)])
def test_full_step_iterates_match_oracle(handle, oracle_mod, N, batch):
    """line_search = 0: every iterate is a deterministic function of the KKT solves -> tight agreement."""
    from oracle import sqp_dubins as S
    Z0, x0, xf, o = S.turn90_problem(batch, N=N)
    o["line_search"] = 0
    Zo, fpo, fdo, ito, solves_o = S.solve(Z0, x0, xf, o)
    s = DubinsSQP(x0, xf, N=N, tf=o["dt"] * (N - 1), iters=10, line_search=False, handle=handle)
    Z = s.solve_(Z0)
    assert _rel(Z, Zo) <= 1e-9
    assert np.array_equal(s.iters, ito) and s.kkt_solves == solves_o
    assert np.allclose(s.feas_p, fpo, rtol=1e-4, atol=1e-12) and np.allclose(s.feas_d, fdo, rtol=1e-4, atol=1e-10)


def test_line_search_converges_like_reference_tolerances(handle, oracle_mod):
    """With the L1-merit line search + SOC: converges within 10 iterations to feas_p, feas_d < 1e-5
    (src/cholesky_solver.jl:111,131-137) and lands on the oracle's solution."""
    from oracle import sqp_dubins as S
    Z0, x0, xf, o = S.turn90_problem(64, N=11)
    Zo, fpo, fdo, ito, _ = S.solve(Z0, x0, xf, o)
    s = DubinsSQP(x0, xf, N=11, tf=3.0, handle=handle)
    Z = s.solve_(Z0)
    assert (s.feas_p < 1e-5).all() and (s.feas_d < 2e-5).all()
    assert (s.iters <= 10).all() and s.kkt_solves >= 64 * 8
    assert _rel(Z, Zo) <= 1e-6


def test_hard_start_exercises_backtracking(handle, oracle_mod):
    """A perturbed initial guess towards goals twice as far with headings off by up to several radians: the oracle's
    trace shows second-order-correction steps and back-tracking on part of the batch.  The device run lands on the
    oracle's end point with the same iteration counts, ends feasible-ish and lowers the merit (mu = 1) of almost every
    instance."""
    from oracle import sqp_dubins as S
    Z0, x0, xf, o = S.hard_turn_problem(32, 21, 3.0, 100.0, 0.5, 2.0, 3.0, seed=0)
    Zo, _, _, ito, _, tr = S.solve(Z0, x0, xf, o, trace=True)
    assert (tr["branch"] == S.BR_SOC).sum() >= 3 and (tr["branch"] >= 2).sum() >= 3
    s = DubinsSQP(x0, xf, N=21, tf=3.0, Qf=o["qf_diag"], iters=10, handle=handle)
    Z = s.solve_(Z0)
    assert np.isfinite(Z).all()
    assert np.median(s.feas_p) < 1e-3
    assert (np.linalg.norm(Z - Zo, axis=1) <= 1e-9 * np.linalg.norm(Zo, axis=1)).all()
    assert np.array_equal(s.iters, ito)
    mu = 1.0
    phi0 = S.cost(Z0, xf, o) + mu * S.c_norm1(Z0, x0, xf, o)
    phi1 = S.cost(Z, xf, o) + mu * S.c_norm1(Z, x0, xf, o)
    assert (phi1 <= phi0 + 1e-9).mean() > 0.9


def test_fused_path_matches_three_kernel_path(handle):
    """The fused linearise+KKT kernel (default) and the linearise -> packed data -> generic KKT path walk the same
    iterates: same per-instance iteration counts, same solve count, solutions equal to rounding."""
    from lqr_b200 import problems
    Z0, x0, xf, o = problems.dubins_turn90(200, N=41)
    rng = np.random.default_rng(1)
    Z0 = Z0 + 0.2 * rng.standard_normal(Z0.shape)  # every accepted step of this batch is the alpha = 1 step; the SOC and
    # back-tracking stages of both paths are held to the oracle in test_gpu_sqp_line_search.py
    s1 = DubinsSQP(x0, xf, N=41, tf=3.0, iters=10, handle=handle)
    Z1 = s1.solve_(Z0)
    assert handle.last_kernel.startswith(("dubins_sqp_step", "dubins_kkt_fused"))
    handle.set_option("sqp_fused", 0)
    try:
        s2 = DubinsSQP(x0, xf, N=41, tf=3.0, iters=10, handle=handle)
        Z2 = s2.solve_(Z0)
        assert handle.last_kernel.startswith("kkt_tpi<3,2")
    finally:
        handle.set_option("sqp_fused", 1)
    assert s1.kkt_solves == s2.kkt_solves and np.array_equal(s1.iters, s2.iters)
    assert _rel(Z1, Z2) <= 1e-9


def test_end_point_matches_scipy_slsqp(handle):
    """Independent of the oracle's SQP loop: SciPy's SLSQP on the same nonlinear program, from the same initial guess."""
    from oracle import sqp_dubins as S
    Z0, x0, xf, o = S.turn90_problem(3, N=11, seed=2)
    s = DubinsSQP(x0, xf, N=11, tf=3.0, handle=handle)
    Z = s.solve_(Z0)
    assert (s.feas_p < 1e-5).all()
    for i in range(3):
        z, f, cv = S.slsqp_solution(Z0, x0, xf, o, i)
        assert abs(f - S.cost(Z[i:i + 1], xf[i:i + 1], o)[0]) <= 1e-6 * abs(f)
        assert np.linalg.norm(z - Z[i]) <= 1e-4 * np.linalg.norm(z)
