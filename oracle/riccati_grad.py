"""CPU ORACLE (test infrastructure): gradients of a loss l(Z) through the Riccati solve.

The forward problem (SURVEY App. A, LTV-affine) and its adjoint LQR (same A, B, Q, R, Qf; linear terms q^_k =
dZ[x_k], r^_k = dZ[u_k], q^f = dZ[x_{N-1}]; x^0 = 0) are both solved as the global KKT system of
``dense_kkt.riccati_as_kkt`` with the extended-precision refined solve, whose multipliers are the costates:
with L = cost + lam_{-1}'(x0 - x_0) + sum_k lam_k'(A_k x_k + B_k u_k - x_{k+1}) the dynamics multipliers are lam_k
and the initial-condition multiplier is -lam_{-1}.  Then

    dA_k = lam_k x^_k' + lam^_k x_k'      dB_k = lam_k u^_k' + lam^_k u_k'
    dQ_k = (x^_k x_k' + x_k x^_k') / 2    dR_k = (u^_k u_k' + u_k u^_k') / 2      dQf likewise at x_{N-1}
    dq_k = x^_k   dr_k = u^_k   dqf = x^_{N-1}   dx0 = lam^_{-1}          (LTI: sums over the knots)

Everything is math order; the keys and shapes are those of the problem dict.
"""
from __future__ import annotations

import numpy as np

from . import dense_kkt


def _split(z, n, m, N):
    body = z[:(N - 1) * (n + m)].reshape(N - 1, n + m)
    return np.vstack([body[:, :n], z[None, (N - 1) * (n + m):]]), body[:, n:]


def _costates(lam, n, N):
    """multipliers [mu; lam_0; ...; lam_{N-2}] -> (lam_{-1}, lam (N-1, n))"""
    return -lam[:n], lam[n:n + (N - 1) * n].reshape(N - 1, n)


def riccati_grad(prob: dict, dZ):
    """Gradients of l(Z) for every instance of a math-order Riccati problem dict; dZ (b, NN) in Primals order."""
    n, m, N = prob["n"], prob["m"], prob["N"]
    b = prob["x0"].shape[0]
    lti = bool(prob.get("lti", False))
    dZ = np.asarray(dZ, dtype=np.float64).reshape(b, -1)
    adj = dict(prob)
    body = dZ[:, :(N - 1) * (n + m)].reshape(b, N - 1, n + m)
    adj.update(lti=False, q=body[:, :, :n], r=body[:, :, n:], qf=dZ[:, (N - 1) * (n + m):], x0=np.zeros((b, n)))
    for k in ("A", "B", "Q", "R"):
        if lti:
            adj[k] = np.repeat(np.asarray(prob[k])[:, None], N - 1, axis=1)
    fk, ak = dense_kkt.riccati_as_kkt(prob), dense_kkt.riccati_as_kkt(adj)
    kn = (b,) if lti else (b, N - 1)
    g = dict(A=np.zeros(kn + (n, n)), B=np.zeros(kn + (n, m)), Q=np.zeros(kn + (n, n)), R=np.zeros(kn + (m, m)),
             q=np.zeros(kn + (n,)), r=np.zeros(kn + (m,)), Qf=np.zeros((b, n, n)), qf=np.zeros((b, n)),
             x0=np.zeros((b, n)))
    for i in range(b):
        z, lam = dense_kkt.kkt_truth(fk, i)
        zh, lamh = dense_kkt.kkt_truth(ak, i)
        X, U = _split(z, n, m, N)
        Xh, Uh = _split(zh, n, m, N)
        _, L = _costates(lam, n, N)
        lh0, Lh = _costates(lamh, n, N)
        gA = np.einsum("ki,kj->kij", L, Xh[:-1]) + np.einsum("ki,kj->kij", Lh, X[:-1])
        gB = np.einsum("ki,kj->kij", L, Uh) + np.einsum("ki,kj->kij", Lh, U)
        gQ = 0.5 * (np.einsum("ki,kj->kij", Xh[:-1], X[:-1]) + np.einsum("ki,kj->kij", X[:-1], Xh[:-1]))
        gR = 0.5 * (np.einsum("ki,kj->kij", Uh, U) + np.einsum("ki,kj->kij", U, Uh))
        parts = dict(A=gA, B=gB, Q=gQ, R=gR, q=Xh[:-1], r=Uh)
        for k, v in parts.items():
            g[k][i] = v.sum(axis=0) if lti else v
        g["Qf"][i] = 0.5 * (np.outer(Xh[-1], X[-1]) + np.outer(X[-1], Xh[-1]))
        g["qf"][i] = Xh[-1]
        g["x0"][i] = lh0
    return g
