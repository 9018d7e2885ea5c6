"""The gradient oracle of the Riccati solve (oracle/riccati_grad.py) against central finite differences of the C
oracle's forward solve, element by element for every argument, on small LTV and LTI problems (CPU only)."""
import numpy as np
import pytest

import oracle
from oracle.riccati_grad import _split, riccati_grad
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


# ------------------------------------------------------------------ open-loop unstable, long horizons
def _unstable(N):
    """dare_lti_riccati's open-loop unstable (6, 3) instance (ρ(A) = 1.18) with random q, r, qf"""
    prob = problems.dare_lti_riccati(6, 3, N, 1, seed=1, unstable=True)
    prob["q"] = np.random.default_rng(1).standard_normal((1, 6))
    prob["r"] = np.random.default_rng(2).standard_normal((1, 3))
    prob["qf"] = np.random.default_rng(3).standard_normal((1, 6))
    return prob


def _refined_z(prob):
    from oracle import dense_kkt
    z, _ = dense_kkt.kkt_truth(dense_kkt.riccati_as_kkt(prob), 0)
    return z


def test_gradient_oracle_matches_finite_differences_of_the_refined_solve_on_an_unstable_horizon():
    """sum(g * D) against central differences of l = dZ·Z along a random direction D of every argument, Z from the
    refined solve itself (dense_kkt.kkt_truth), on the open-loop unstable problem at N = 201: the oracle is sound on
    the inputs of tests/test_gpu_riccati_grad_stability.py, so a 1e-9 verdict there is about the kernel"""
    N = 201
    prob = _unstable(N)
    assert np.abs(np.linalg.eigvals(prob["A"][0])).max() > 1.15
    W = np.random.default_rng(4).standard_normal((1, N * 6 + (N - 1) * 3))
    g = riccati_grad(prob, W)
    rng = np.random.default_rng(5)
    D = {k: rng.standard_normal(np.shape(prob[k])) for k in ARGS}
    for k in SYMMETRIC:
        D[k] = D[k] + np.swapaxes(D[k], -1, -2)
    h = 1e-5

    def loss(s):
        return float(_refined_z(dict(prob, **{k: prob[k] + s * h * D[k] for k in ARGS})) @ W[0])
    fd = (loss(1) - loss(-1)) / (2 * h)
    an = sum(float((g[k] * D[k]).sum()) for k in ARGS)
    np.testing.assert_allclose(an, fd, rtol=1e-7)


def _costate_sweep(prob, z, zh, dz, K, closed):
    """float64 restatement of riccati_grad_kernel's backward sweep for instance 0 of an LTI problem: the costates of
    the forward and the adjoint problem and from them ∂A, ∂B (sums over the knots) and ∂x0.  ``closed``: the
    closed-loop recursion λ_{k-1} = Q x_k + q − K_kᵀ(R u_k + r) + (A − B K_k)ᵀλ_k, else the open-loop one
    λ_{k-1} = Q x_k + q + Aᵀλ_k (the adjoint problem's with x̂, û, dZ)."""
    n, m, N = prob["n"], prob["m"], prob["N"]
    A, Bm, Q, R, Qf = (prob[s][0] for s in ("A", "B", "Q", "R", "Qf"))
    q, r, qf = prob["q"][0], prob["r"][0], prob["qf"][0]
    X, U = _split(z, n, m, N)
    Xh, Uh = _split(zh, n, m, N)
    dX, dU = _split(dz, n, m, N)
    lam, lamh = Qf @ X[-1] + qf, Qf @ Xh[-1] + dX[-1]
    gA, gB = np.zeros((n, n)), np.zeros((n, m))
    for k in range(N - 2, -1, -1):
        gA += np.outer(lam, Xh[k]) + np.outer(lamh, X[k])
        gB += np.outer(lam, Uh[k]) + np.outer(lamh, U[k])
        if closed:
            Acl = A - Bm @ K[k]
            lam = Q @ X[k] + q - K[k].T @ (R @ U[k] + r) + Acl.T @ lam
            lamh = Q @ Xh[k] + dX[k] - K[k].T @ (R @ Uh[k] + dU[k]) + Acl.T @ lamh
        else:
            lam = Q @ X[k] + q + A.T @ lam
            lamh = Q @ Xh[k] + dX[k] + A.T @ lamh
    return dict(A=gA, B=gB, x0=lamh)


def test_closed_loop_costate_recursion_reproduces_the_oracle_where_the_open_loop_one_diverges():
    """The recursion riccati_grad_kernel runs, restated in float64 and fed the best input any forward kernel could
    give it (the refined Z and Ẑ rounded to double, riccati_ld's K), on the unstable problem at N = 401: the
    closed-loop form matches the oracle to 1e-12; the open-loop form is off by orders of magnitude (the error of λ_k
    grows like ρ(A)^N)."""
    from oracle import riccati_ld
    n, m, N = 6, 3, 401
    prob = _unstable(N)
    dZ = np.random.default_rng(0).standard_normal((1, N * n + (N - 1) * m))
    go = riccati_grad(prob, dZ)
    body = dZ[:, :(N - 1) * (n + m)].reshape(1, N - 1, n + m)
    adj = dict(prob, lti=False, q=body[:, :, :n], r=body[:, :, n:], qf=dZ[:, (N - 1) * (n + m):], x0=np.zeros((1, n)))
    for k in ("A", "B", "Q", "R"):
        adj[k] = np.repeat(prob[k][:, None], N - 1, axis=1)
    z, zh = _refined_z(prob), _refined_z(adj)
    K = np.asarray(riccati_ld.riccati(prob)[2][0], dtype=np.float64)

    def err(g, k):
        return np.linalg.norm(g[k] - go[k][0]) / np.linalg.norm(go[k][0])
    closed = _costate_sweep(prob, z, zh, dZ[0], K, closed=True)
    openl = _costate_sweep(prob, z, zh, dZ[0], K, closed=False)
    for k in ("A", "B", "x0"):
        assert err(closed, k) <= 1e-12, (k, err(closed, k))
    assert err(openl, "A") > 1e-3 and err(openl, "x0") > 1e-3, (err(openl, "A"), err(openl, "x0"))
