"""CPU ORACLE of lqrb_dare_f64 / lqrb_dare_grad_f64 (DESIGN §4.11): the structured doubling algorithm for the discrete
algebraic Riccati equation P = Q + A'PA - A'PB (R + B'PB)^-1 B'PA, its gain K = (R + B'PB)^-1 B'PA, and the gradient of
a loss l(P, K) through both.  One instance per call, numpy; everything also runs in complex128 (pass ``steps`` for the
fixed step count a complex-step derivative needs), so the tests can hold the gradient formulas against complex-step
derivatives of the doubling itself.
"""
from __future__ import annotations

import numpy as np

EPS = 2.0 ** -52  # the kernels' stopping rule: ||dH||_F <= EPS ||H||_F
MAX_STEPS = 64


def _sym(X):
    return 0.5 * (X + X.T)


def _fro2(X):
    with np.errstate(over="ignore", invalid="ignore"):  # a diverging iteration overflows; the caller tests isfinite
        return float(np.sum(np.abs(X) ** 2))


def sda(A, B, Q, R, steps: int | None = None):
    """Structured doubling: A_0 = A, G_0 = B R^-1 B', H_0 = Q; with W = I + G_k H_k,
    A_{k+1} = A_k W^-1 A_k, G_{k+1} = G_k + A_k W^-1 G_k A_k', H_{k+1} = H_k + A_k' H_k W^-1 A_k, G and H symmetrised.
    Stops when the increment of H is below EPS relative (at most MAX_STEPS), or after exactly ``steps``.
    Returns (P, steps taken, converged)."""
    n = A.shape[0]
    Ak, Gk, Hk = A.copy(), B @ np.linalg.solve(R, B.T), Q.copy()
    Gk = _sym(Gk)
    cap = MAX_STEPS if steps is None else steps
    for k in range(1, cap + 1):
        W = np.eye(n) + Gk @ Hk
        X = np.linalg.solve(W, np.concatenate([Ak, Gk], axis=1))
        X1, X2 = X[:, :n], X[:, n:]
        dH = Ak.T @ (Hk @ X1)
        Hk = _sym(Hk + dH)
        Gk = _sym(Gk + (Ak @ X2) @ Ak.T)
        Ak = Ak @ X1
        if steps is None:
            dd, hh = _fro2(dH), _fro2(Hk)
            if not (np.isfinite(dd) and np.isfinite(hh)):
                return Hk, k, False
            if dd <= EPS * EPS * hh:
                return Hk, k, True
    return Hk, cap, steps is not None


def gain(A, B, R, P):
    """K = (R + B'PB)^-1 B'PA  (u = -K x)"""
    return np.linalg.solve(R + B.T @ P @ B, B.T @ P @ A)


def stein(M, S, steps: int | None = None):
    """Y = M Y M' + S by Smith doubling: Y <- Y + M Y M', M <- M M from Y = S, M = M; the stopping rule of sda.
    Returns (Y, steps taken, converged)."""
    Y, Mk = S.copy(), M.copy()
    cap = MAX_STEPS if steps is None else steps
    for k in range(1, cap + 1):
        D = (Mk @ Y) @ Mk.T
        Y = _sym(Y + D)
        if steps is None:
            dd, yy = _fro2(D), _fro2(Y)
            if not (np.isfinite(dd) and np.isfinite(yy)):
                return Y, k, False
            if dd <= EPS * EPS * yy:
                return Y, k, True
        Mk = Mk @ Mk
    return Y, cap, steps is not None


def dare(A, B, Q, R, steps: int | None = None):
    """(P, K, steps, converged) of one instance; Q and R are read as given (symmetrise them first)."""
    P, k, ok = sda(A, B, Q, R, steps)
    return P, gain(A, B, R, P), k, ok


def dare_grad(A, B, R, P, dP=None, dK=None, steps: int | None = None):
    """Gradient of l(P, K) for the cotangents dP = dl/dP, dK = dl/dK (either may be None): with Gc = R + B'PB,
    Acl = A - BK,
        Yk = Gc^-1 dK, Gbar = -sym(Yk K'), S = sym(dP) + B Gbar B' + sym(B Yk A'), Y = Acl Y Acl' + S,
        gQ = Y, gR = K Y K' + Gbar, gA = 2 P Acl Y + P B Yk, gB = -2 P Acl Y K' + P A Yk' + 2 P B Gbar.
    Returns (dict(A, B, Q, R), Stein steps, converged).  gQ and gR are the symmetric gradients (Q and R enter through
    their symmetric parts)."""
    n, m = B.shape
    dt = np.result_type(A, B, R, P)
    dP = np.zeros((n, n), dt) if dP is None else dP
    dK = np.zeros((m, n), dt) if dK is None else dK
    Gc = R + B.T @ P @ B
    K = np.linalg.solve(Gc, B.T @ P @ A)
    Acl = A - B @ K
    Yk = np.linalg.solve(Gc, dK)
    Gb = -_sym(Yk @ K.T)
    S = _sym(dP) + B @ Gb @ B.T + _sym(B @ Yk @ A.T)
    Y, k, ok = stein(Acl, S, steps)
    V = P @ Acl @ Y
    g = dict(Q=Y, R=_sym(K @ Y @ K.T) + Gb, A=2 * V + P @ B @ Yk,
             B=-2 * V @ K.T + P @ A @ Yk.T + 2 * P @ B @ Gb)
    return g, k, ok
