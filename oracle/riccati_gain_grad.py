"""CPU ORACLE (test infrastructure): gradients of a loss l(K, kff) of the Riccati gains, and of l(Z, K, kff).

The forward recursion is the library's LTV-affine Riccati (SURVEY App. A) with P' = P_{k+1}, p' = p_{k+1}:

    G = R + B'P'B,  H = B'P'A,  h = r + B'p',  K = G^-1 H,  kff = G^-1 h
    P = sym(Q + A'P'A - H'K),  p = q + A'p' - K'h,  P_{N-1} = Qf,  p_{N-1} = qf

Its reverse mode runs forward over the knots, k = 0 ... N-2, from Pb = 0, pb = 0 (P_0, p_0 feed nothing), with
Acl = A - BK, v = p' - P'B kff, Y = G^-1 Kb_k, y = G^-1 kb_k and Gb = -sym(Y K' + y kff'):

    Qb_k += Pb                       qb_k += pb
    Ab_k += 2 P'Acl Pb + v pb' + P'B Y
    Bb_k += -2 P'Acl Pb K' - P'Acl pb kff' - v (K pb)' + P'A Y' + 2 P'B Gb + p' y'
    Rb_k += K Pb K' + sym((K pb) kff') + Gb          rb_k += -K pb + y
    Pb'  = Acl Pb Acl' - sym((Acl pb)(B kff)') + B Gb B' + sym(B Y A')        pb' = Acl pb + B y

and at the end Qfb = Pb, qfb = pb (x0 gets nothing).  Everything runs in long double with the hand Cholesky of
``riccati_ld`` for the G solves, vectorised over the batch.  Keys and shapes are those of ``riccati_grad``.
"""
from __future__ import annotations

import numpy as np

from .riccati_grad import riccati_grad
from .riccati_ld import LD, _chol_solve, _cholesky, _knot, _require_extended


def _t(a):
    return np.swapaxes(a, -1, -2)


def _sym(a):
    return 0.5 * (a + _t(a))


def _outer(u, v):
    return u[:, :, None] * v[:, None, :]


def _mv(M, v):
    return np.einsum("bij,bj->bi", M, v)


def gain_grad(prob: dict, dK=None, dkff=None):
    """Gradients of l(K, kff) for every instance of a math-order Riccati problem dict, from dK = dl/dK (b, N-1, m, n)
    and dkff = dl/dkff (b, N-1, m); either may be None (zero).  Returns float64 arrays."""
    _require_extended()
    n, m, N = prob["n"], prob["m"], prob["N"]
    lti = bool(prob.get("lti", False))
    b = np.asarray(prob["x0"]).shape[0]
    kn = () if lti else (N - 1,)
    A, B, Q, R = (np.asarray(prob[s], dtype=LD) for s in ("A", "B", "Q", "R"))
    q = np.zeros((b,) + kn + (n,), LD) if prob.get("q") is None else np.asarray(prob["q"], dtype=LD)
    r = np.zeros((b,) + kn + (m,), LD) if prob.get("r") is None else np.asarray(prob["r"], dtype=LD)
    Kb = np.zeros((b, N - 1, m, n), LD) if dK is None else np.asarray(dK, dtype=LD)
    kb = np.zeros((b, N - 1, m), LD) if dkff is None else np.asarray(dkff, dtype=LD)
    P = _sym(np.asarray(prob["Qf"], dtype=LD))
    p = np.zeros((b, n), LD) if prob.get("qf") is None else np.asarray(prob["qf"], dtype=LD).copy()
    tape = [None] * (N - 1)
    for k in range(N - 2, -1, -1):
        Ak, Bk, Qk, Rk = (_knot(a, k, lti) for a in (A, B, Q, R))
        G = Rk + _t(Bk) @ P @ Bk
        H = _t(Bk) @ P @ Ak
        h = _knot(r, k, lti) + np.einsum("bji,bj->bi", Bk, p)
        L, _ = _cholesky(G)
        Kf = _chol_solve(L, np.concatenate([H, h[:, :, None]], axis=2))
        K, kff = Kf[:, :, :n], Kf[:, :, n]
        tape[k] = (P, p, K, kff, L)
        P = _sym(Qk + _t(Ak) @ P @ Ak - _t(H) @ K)
        p = _knot(q, k, lti) + np.einsum("bji,bj->bi", Ak, p) - np.einsum("bji,bj->bi", K, h)
    g = {s: np.zeros((b,) + kn + shp, LD) for s, shp in
         (("A", (n, n)), ("B", (n, m)), ("Q", (n, n)), ("R", (m, m)), ("q", (n,)), ("r", (m,)))}
    Pb, pb = np.zeros((b, n, n), LD), np.zeros((b, n), LD)
    for k in range(N - 1):
        Ak, Bk = _knot(A, k, lti), _knot(B, k, lti)
        Pn, pn, K, kff, L = tape[k]
        Acl = Ak - Bk @ K
        v = pn - _mv(Pn @ Bk, kff)
        Kp = _mv(K, pb)
        Y = _chol_solve(L, Kb[:, k])
        y = _chol_solve(L, kb[:, k, :, None])[:, :, 0]
        Gb = -_sym(Y @ _t(K) + _outer(y, kff))
        PAcl = Pn @ Acl
        gA = 2 * PAcl @ Pb + _outer(v, pb) + Pn @ Bk @ Y
        gB = (-2 * PAcl @ Pb @ _t(K) - _outer(_mv(PAcl, pb), kff) - _outer(v, Kp) + Pn @ Ak @ _t(Y)
              + 2 * Pn @ Bk @ Gb + _outer(pn, y))
        gR = K @ Pb @ _t(K) + _sym(_outer(Kp, kff)) + Gb
        parts = dict(A=gA, B=gB, Q=Pb, R=gR, q=pb, r=y - Kp)
        for s, val in parts.items():
            if lti:
                g[s] += val
            else:
                g[s][:, k] += val
        Pb, pb = (Acl @ Pb @ _t(Acl) - _sym(_outer(_mv(Acl, pb), _mv(Bk, kff))) + Bk @ Gb @ _t(Bk)
                  + _sym(Bk @ Y @ _t(Ak))), _mv(Acl, pb) + _mv(Bk, y)
    out = {s: v.astype(np.float64) for s, v in g.items()}
    out.update(Qf=Pb.astype(np.float64), qf=pb.astype(np.float64), x0=np.zeros((b, n)))
    return out


def riccati_total_grad(prob: dict, dZ=None, dK=None, dkff=None):
    """Gradients of l(Z, K, kff): the Z part of ``riccati_grad`` (when dZ is given) plus the gains part."""
    g = gain_grad(prob, dK, dkff)
    if dZ is not None:
        gz = riccati_grad(prob, dZ)
        g = {s: g[s] + gz[s] for s in g}
    return g
