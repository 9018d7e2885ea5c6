"""CPU ORACLE (test infrastructure): gradients of a loss l(dz, mult) through the constrained KKT solve.

The solve returns x = [dz; mult] with K x = -[g; d], K = [H D'; D 0] (``dense_kkt.assemble``).  With the cotangents
x_bar = [dz_bar; mult_bar], the same K solved with g := dz_bar and [c; d] := mult_bar returns x^ = -K^-1 x_bar =
[z^; nu^] = dl/d[g; d] (K is symmetric), and dl/dK = x^ x'.  Split per knot (z_k = [x_k; u_k], multipliers mu_k of
C_k z_k + c_k = 0 and lam_k of D1_k z_k + D2_{k+1} z_{k+1} + d_k = 0; hats likewise):

    dq_k = x^_k   dr_k = u^_k   dd_k = lam^_k   dc_k = mu^_k
    dQ_k = (x^_k x_k' + x_k x^_k') / 2          dR_k = (u^_k u_k' + u_k u^_k') / 2    (DIAG: their diagonals only)
    dHux_k = u^_k x_k' + u_k x^_k'              (DENSE)
    dA_k = lam^_k x_k' + lam_k x^_k'            dB_k = lam^_k u_k' + lam_k u^_k'
    dC_k = mu^_k z_k' + mu_k z^_k'              dD2_{k+1} = lam^_k z_{k+1}' + lam_k z^_{k+1}'   (explicit D2)

Both solves are the extended-precision refined solve, one instance at a time, unless ``sols`` gives them: a list of
(z, mult, z^, nu^) per instance (for example from another solver, to measure what its error does to the gradient).  Everything is math order; the keys
and shapes are those of the problem dict (D2, C, c: per-knot lists; Hux, D2: None where the problem has none).
"""
from __future__ import annotations

import numpy as np

from . import dense_kkt


def kkt_grad(prob: dict, dz_bar=None, mult_bar=None, sols=None):
    """Gradients for every instance of a math-order KKT problem dict; dz_bar (b, NN), mult_bar (b, P), either None;
    sols: the forward and adjoint solutions per instance in place of the refined solves."""
    n, m, N = prob["n"], prob["m"], prob["N"]
    p = [int(x) for x in prob["p"]]
    mode = int(prob.get("hess_mode", 1))
    b = np.asarray(prob["q"]).shape[0]
    NN, P = N * n + (N - 1) * m, sum(p) + (N - 1) * n
    dzb = np.zeros((b, NN)) if dz_bar is None else np.asarray(dz_bar, dtype=np.float64).reshape(b, NN)
    mb = np.zeros((b, P)) if mult_bar is None else np.asarray(mult_bar, dtype=np.float64).reshape(b, P)
    ws = [n + (m if k < N - 1 else 0) for k in range(N)]
    explicit = prob.get("D2") is not None
    g = dict(Q=np.zeros((b, N, n, n)), R=np.zeros((b, N - 1, m, m)), Hux=np.zeros((b, N - 1, m, n)) if mode == 0 else None,
             q=np.zeros((b, N, n)), r=np.zeros((b, N - 1, m)), A=np.zeros((b, N - 1, n, n)), B=np.zeros((b, N - 1, n, m)),
             d=np.zeros((b, N - 1, n)), D2=[np.zeros((b, n, ws[k])) for k in range(1, N)] if explicit else None,
             C=[np.zeros((b, p[k], ws[k])) for k in range(N)], c=[np.zeros((b, p[k])) for k in range(N)])
    for i in range(b):
        if sols is None:
            H, gv, D, dv = dense_kkt.assemble(prob, i)
            z, mult = dense_kkt.solve_refined(H, gv, D, dv)
            zh, mh = dense_kkt.solve_refined(H, dzb[i], D, mb[i])
        else:
            z, mult, zh, mh = sols[i]
        zs = [z[k * (n + m):k * (n + m) + ws[k]] for k in range(N)]
        zhs = [zh[k * (n + m):k * (n + m) + ws[k]] for k in range(N)]
        mus, lams, muhs, lamhs, off = [], [], [], [], 0
        for k in range(N):
            mus.append(mult[off:off + p[k]])
            muhs.append(mh[off:off + p[k]])
            off += p[k]
            if k < N - 1:
                lams.append(mult[off:off + n])
                lamhs.append(mh[off:off + n])
                off += n
        for k in range(N):
            x, xh = zs[k][:n], zhs[k][:n]
            gQ = 0.5 * (np.outer(xh, x) + np.outer(x, xh))
            g["Q"][i, k] = np.diag(np.diag(gQ)) if mode == 2 else gQ
            g["q"][i, k] = xh
            g["C"][k][i] = np.outer(muhs[k], zs[k]) + np.outer(mus[k], zhs[k])
            g["c"][k][i] = muhs[k]
            if k == N - 1:
                continue
            u, uh = zs[k][n:], zhs[k][n:]
            gR = 0.5 * (np.outer(uh, u) + np.outer(u, uh))
            g["R"][i, k] = np.diag(np.diag(gR)) if mode == 2 else gR
            g["r"][i, k] = uh
            if mode == 0:
                g["Hux"][i, k] = np.outer(uh, x) + np.outer(u, xh)
            g["A"][i, k] = np.outer(lamhs[k], x) + np.outer(lams[k], xh)
            g["B"][i, k] = np.outer(lamhs[k], u) + np.outer(lams[k], uh)
            g["d"][i, k] = lamhs[k]
            if explicit:
                g["D2"][k][i] = np.outer(lamhs[k], zs[k + 1]) + np.outer(lams[k], zhs[k + 1])
    return g
