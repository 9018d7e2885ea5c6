"""CPU tests of oracle/dare.py: the structured doubling against scipy.linalg.solve_discrete_are, and the gradient
formulas against complex-step derivatives of the complex128 doubling itself."""
import numpy as np
import pytest
import scipy.linalg as sl

from lqr_b200 import problems
from oracle import dare as od

SHAPES = [(1, 1), (3, 2), (4, 1), (6, 3), (8, 4), (12, 4), (16, 8), (24, 6), (32, 8), (48, 16), (64, 16)]


def _instance(n, m, unstable, seed):
    p = problems.dare_lti_riccati(n, m, 2, 1, seed=seed, unstable=unstable)
    return p["A"][0], p["B"][0], p["Q"][0], p["R"][0]


@pytest.mark.parametrize("unstable", [False, True], ids=["stable", "unstable"])
@pytest.mark.parametrize("n,m", SHAPES)
def test_sda_matches_scipy(n, m, unstable):
    A, B, Q, R = _instance(n, m, unstable, seed=n + 7 * m + unstable)
    P, K, steps, ok = od.dare(A, B, Q, R)
    assert ok and steps <= 16, steps
    P0 = sl.solve_discrete_are(A, B, Q, R)
    K0 = od.gain(A, B, R, P0)
    tol = 1e-10 if n <= 16 else 1e-9
    assert np.linalg.norm(P - P0) <= tol * np.linalg.norm(P0)
    assert np.linalg.norm(K - K0) <= tol * np.linalg.norm(K0)
    assert np.array_equal(P, P.T)
    res = np.linalg.norm(Q + A.T @ P @ A - A.T @ P @ B @ K - P) / np.linalg.norm(P)
    assert res <= (1e-12 if n <= 16 else 1e-10), res
    assert max(abs(np.linalg.eigvals(A - B @ K))) < 1.0


def test_sda_reports_no_stabilising_solution():
    A, B, Q, R = _instance(4, 1, True, seed=3)
    _, _, steps, ok = od.dare(A, 0.0 * B, Q, R)
    assert not ok and steps < od.MAX_STEPS  # H overflows long before the cap


def _complex_step(n, m, unstable, seed, cot):
    rng = np.random.default_rng(seed + 1)
    A, B, Q, R = _instance(n, m, unstable, seed)
    P, K, steps, ok = od.dare(A, B, Q, R)
    assert ok
    dP = rng.standard_normal((n, n)) if "P" in cot else None
    dK = rng.standard_normal((m, n)) if "K" in cot else None
    g, _, ok = od.dare_grad(A, B, R, P, dP, dK)
    assert ok
    fixed = steps + 2

    def loss(X):
        Qs, Rs = 0.5 * (X["Q"] + X["Q"].T), 0.5 * (X["R"] + X["R"].T)
        Pc, _, _ = od.sda(X["A"], X["B"], Qs, Rs, steps=fixed)
        val = 0.0
        if dP is not None:
            val = val + np.sum(dP * Pc)
        if dK is not None:
            val = val + np.sum(dK * od.gain(X["A"], X["B"], Rs, Pc))
        return val

    X0 = {k: v.astype(np.complex128) for k, v in dict(A=A, B=B, Q=Q, R=R).items()}
    for name in "ABQR":
        cs = np.zeros(X0[name].shape)
        for ij in np.ndindex(cs.shape):
            X = {k: v.copy() for k, v in X0.items()}
            X[name][ij] += 1e-30j
            cs[ij] = loss(X).imag / 1e-30
        err = np.max(np.abs(g[name] - cs)) / np.max(np.abs(cs))
        assert err <= 1e-11, (name, err)


@pytest.mark.parametrize("cot", ["P", "K", "PK"])
@pytest.mark.parametrize("n,m,unstable", [(1, 1, False), (4, 1, True), (6, 3, True), (8, 4, False), (12, 4, False)])
def test_gradient_matches_complex_step(n, m, unstable, cot):
    """Element by element, relative to the largest derivative of each array.  The complex-step derivative is that of
    the doubling in complex128, so it carries the doubling's own rounding: on an open-loop unstable (12, 4) draw with
    ||P|| ~ 900 it is off by 1.3e-10 where a 40-digit evaluation puts the formulas within 1.3e-12.  Such draws are
    covered by the GPU tests against the oracle, not here."""
    _complex_step(n, m, unstable, seed=n, cot=cot)
