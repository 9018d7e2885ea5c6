"""The gradient oracle of the Riccati solve (oracle/riccati_grad.py) against central finite differences of the C
oracle's forward solve, element by element for every argument, on small LTV and LTI problems (CPU only)."""
import numpy as np
import pytest

import oracle
from oracle.riccati_grad import riccati_grad
from lqr_b200 import problems

H = 1e-6
ARGS = ("A", "B", "Q", "R", "q", "r", "Qf", "qf", "x0")
SYMMETRIC = ("Q", "R", "Qf")


def _z(prob):
    X, U, _, _, info = oracle.riccati(prob)
    assert (info == 0).all()
    n, m, N = prob["n"], prob["m"], prob["N"]
    b = X.shape[0]
    body = np.concatenate([X[:, :-1], U], axis=2).reshape(b, -1)
    return np.concatenate([body, X[:, -1]], axis=1)


def _fd(prob, W):
    """Central differences of l = sum(W * Z) for every element of every argument of instance 0, all perturbed
    copies solved as one batch.  A symmetric matrix is perturbed at (i, j) and (j, i) together."""
    base = {k: np.asarray(prob[k])[:1] for k in ARGS}
    dirs = []
    for k in ARGS:
        shape = base[k].shape[1:]
        for idx in np.ndindex(*shape):
            if k in SYMMETRIC and idx[-2] > idx[-1]:
                continue
            E = np.zeros(shape)
            E[idx] = 1.0
            if k in SYMMETRIC:
                t = idx[:-2] + (idx[-1], idx[-2])
                E[t] = 1.0
            dirs.append((k, idx, E))
    batch = {k: np.repeat(base[k], 2 * len(dirs), axis=0) for k in ARGS}
    for d, (k, _, E) in enumerate(dirs):
        batch[k][2 * d] += H * E
        batch[k][2 * d + 1] -= H * E
    p = dict(prob, **batch)
    loss = (_z(p) * W).sum(axis=1)
    return [(k, idx, (loss[2 * d] - loss[2 * d + 1]) / (2 * H)) for d, (k, idx, _) in enumerate(dirs)]


@pytest.mark.parametrize("lti", [False, True])
def test_gradient_oracle_matches_finite_differences(lti):
    n, m, N = 3, 2, 5
    prob = problems.random_lqr_riccati(n, m, N, 1, seed=11, dt=0.1, lti=lti)
    W = np.random.default_rng(5).standard_normal((1, N * n + (N - 1) * m))
    g = riccati_grad(prob, W)
    worst = 0.0
    for k, idx, fd in _fd(prob, W):
        an = g[k][(0,) + idx]
        if k in SYMMETRIC and idx[-2] != idx[-1]:
            an = an + g[k][(0,) + idx[:-2] + (idx[-1], idx[-2])]
        scale = max(1.0, np.abs(g[k]).max())
        worst = max(worst, abs(an - fd) / scale)
        assert abs(an - fd) <= 1e-6 * scale, (k, idx, an, fd)
    assert worst < 1e-6


def test_gradient_oracle_symmetric_blocks_and_costates():
    """The matrix gradients of Q, R, Qf are symmetric, and dx0 equals the costate recursion
    lam^_{-1} = Q_0 x^_0 + q^_0 + A_0' lam^_0 run on the adjoint solution."""
    n, m, N = 4, 2, 6
    prob = problems.random_lqr_riccati(n, m, N, 2, seed=3, dt=0.1)
    W = np.random.default_rng(1).standard_normal((2, N * n + (N - 1) * m))
    g = riccati_grad(prob, W)
    for k in SYMMETRIC:
        np.testing.assert_allclose(g[k], np.swapaxes(g[k], -1, -2), rtol=0, atol=1e-14)
    # x^ = dq (the adjoint trajectory); run the costate recursion of the adjoint problem by hand
    for i in range(2):
        Xh = np.vstack([g["q"][i], g["qf"][i][None]])
        lh = prob["Qf"][i] @ Xh[-1] + W[i, (N - 1) * (n + m):]
        for k in range(N - 2, -1, -1):
            lh = prob["Q"][i, k] @ Xh[k] + W[i, k * (n + m):k * (n + m) + n] + prob["A"][i, k].T @ lh
        np.testing.assert_allclose(g["x0"][i], lh, rtol=1e-9, atol=1e-9)
