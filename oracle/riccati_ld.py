"""CPU ORACLE (test infrastructure): the Riccati recursion in extended precision (x87 long double).

The C oracle (``oracle/lqr_oracle.c``) runs the recursion in double precision in the reference's operation order, so
on an ill-conditioned control block ``E = R + B'PB`` it is itself only accurate to about cond(E) x 1e-16.  This module
is the truth those verdicts are measured against: the same recursion (src/dynamic_programming.jl:28-72, generalised
to per-knot data and affine terms as in the C oracle) with every operation in ``np.longdouble``, ``E`` factored by a
hand-written Cholesky (numpy.linalg has no long double) and ``P`` symmetrised at every knot.  It is vectorised over
the batch and meant for the small horizons and batches of the tests.
"""
from __future__ import annotations

import numpy as np

LD = np.longdouble


def _require_extended():
    if np.finfo(LD).eps > 1e-18:
        raise RuntimeError("numpy.longdouble is not an extended-precision type on this platform")


def _knot(a, k, lti):
    return a if lti else a[:, k]


def _cholesky(E):
    """Lower Cholesky factors L = U' of a stack of symmetric (b, m, m) matrices (upper triangle read, as potrf('U'))
    and the potrf info of each: 0, or the 1-based index of the first non-positive pivot.  A failed factor is carried
    on with NaN."""
    b, m, _ = E.shape
    L = np.zeros_like(E)
    info = np.zeros(b, dtype=np.int32)
    for j in range(m):
        s = E[:, j, j] - np.einsum("bk,bk->b", L[:, j, :j], L[:, j, :j])
        bad = ~(s > 0)
        info[(info == 0) & bad] = j + 1
        d = np.sqrt(np.where(bad, LD(np.nan), s))
        L[:, j, j] = d
        for i in range(j + 1, m):
            L[:, i, j] = (E[:, j, i] - np.einsum("bk,bk->b", L[:, i, :j], L[:, j, :j])) / d
    return L, info


def _chol_solve(L, G):
    """E^-1 G for E = L L' (b, m, m) and right-hand sides G (b, m, c)."""
    m = L.shape[1]
    Y = np.zeros_like(G)
    for i in range(m):
        Y[:, i] = (G[:, i] - np.einsum("bk,bkc->bc", L[:, i, :i], Y[:, :i])) / L[:, i, i, None]
    X = np.zeros_like(G)
    for i in reversed(range(m)):
        X[:, i] = (Y[:, i] - np.einsum("bk,bkc->bc", L[:, i + 1:, i], X[:, i + 1:])) / L[:, i, i, None]
    return X


def riccati(prob: dict):
    """Batched Riccati solve of a math-order problem dict (``lqr_b200.problems.riccati_*``; ``lti`` and absent
    ``q``/``r``/``qf`` allowed).  Returns X (b,N,n), U (b,N-1,m), K (b,N-1,m,n), kff (b,N-1,m) in long double and
    info (b,) with the C oracle's code: (k+1)*1000 + pivot for the first failed factorisation of the backward sweep."""
    _require_extended()
    n, m, N = prob["n"], prob["m"], prob["N"]
    lti = bool(prob.get("lti", False))
    x0 = np.asarray(prob["x0"], dtype=LD)
    b = x0.shape[0]
    kn = () if lti else (N - 1,)
    A, B, Q, R = (np.asarray(prob[s], dtype=LD) for s in ("A", "B", "Q", "R"))
    q = np.zeros((b,) + kn + (n,), LD) if prob.get("q") is None else np.asarray(prob["q"], dtype=LD)
    r = np.zeros((b,) + kn + (m,), LD) if prob.get("r") is None else np.asarray(prob["r"], dtype=LD)
    P = np.asarray(prob["Qf"], dtype=LD).copy()
    p = np.zeros((b, n), LD) if prob.get("qf") is None else np.asarray(prob["qf"], dtype=LD).copy()
    K = np.zeros((b, N - 1, m, n), LD)
    kff = np.zeros((b, N - 1, m), LD)
    info = np.zeros(b, dtype=np.int32)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        for k in range(N - 2, -1, -1):
            Ak, Bk, Qk, Rk = (_knot(a, k, lti) for a in (A, B, Q, R))
            Bt = np.swapaxes(Bk, -1, -2)
            E = Rk + Bt @ P @ Bk
            G = Bt @ P @ Ak
            rr = _knot(r, k, lti) + np.einsum("bji,bj->bi", Bk, p)
            L, st = _cholesky(E)
            info[(info == 0) & (st != 0)] = (k + 1) * 1000 + st[(info == 0) & (st != 0)]
            Kf = _chol_solve(L, np.concatenate([G, rr[:, :, None]], axis=2))
            K[:, k], kff[:, k] = Kf[:, :, :n], Kf[:, :, n]
            P = Qk + np.swapaxes(Ak, -1, -2) @ P @ Ak - np.swapaxes(G, -1, -2) @ K[:, k]
            P = 0.5 * (P + np.swapaxes(P, -1, -2))
            p = _knot(q, k, lti) + np.einsum("bji,bj->bi", Ak, p) - np.einsum("bji,bj->bi", K[:, k], rr)
        X = np.zeros((b, N, n), LD)
        U = np.zeros((b, N - 1, m), LD)
        X[:, 0] = x0
        for k in range(N - 1):
            U[:, k] = -np.einsum("bij,bj->bi", K[:, k], X[:, k]) - kff[:, k]
            X[:, k + 1] = (np.einsum("bij,bj->bi", _knot(A, k, lti), X[:, k])
                           + np.einsum("bij,bj->bi", _knot(B, k, lti), U[:, k]))
    return X, U, K, kff, info
