"""CPU ORACLE of lqrb_admm_cache_f64 / lqrb_admm_solve_f64 (DESIGN §4.12): box-constrained LTI MPC by ADMM on the cached
infinite-horizon Riccati factor of the rho-augmented costs (the algorithm of TinyMPC, Nguyen et al., ICRA 2024).  One
instance per call, numpy, in the iteration order of the kernel, so that both agree at a fixed iteration count.

Problem (x_1 = x0):
    min  sum_{k=1}^{N-1} 1/2 |x_k - xr_k|_Q^2 + 1/2 |u_k - ur_k|_R^2  +  1/2 |x_N - xr_N|_Qf^2
    s.t. x_{k+1} = A x_k + B u_k,  umin_k <= u_k <= umax_k (k = 1..N-1),  xmin_k <= x_k <= xmax_k (k = 2..N)
    with Qf = Pt - rho I,  Pt = DARE(A, B, Q + rho I, R + rho I).
"""
from __future__ import annotations

import numpy as np

from . import dare as od


def cache(A, B, Q, R, rho):
    """The cached factor of one instance: dict(A, B, Q, R, Qf, K, C1, C2, rho, ok).  Q and R are read through their upper
    triangles, as the kernels do."""
    n, m = B.shape
    Q = np.triu(Q) + np.triu(Q, 1).T
    R = np.triu(R) + np.triu(R, 1).T
    Rt = R + rho * np.eye(m)
    P, K, _, ok = od.dare(A, B, Q + rho * np.eye(n), Rt)
    C1 = np.linalg.inv(Rt + B.T @ P @ B)
    return dict(A=A, B=B, Q=Q, R=R, Qf=P - rho * np.eye(n), K=K, C1=0.5 * (C1 + C1.T), C2=(A - B @ K).T, rho=rho, ok=ok)


def solve(c, x0, N, xref=None, uref=None, umin=None, umax=None, xmin=None, xmax=None, max_iter=100, eps_pri=0.0,
          eps_dual=0.0, state=None):
    """ADMM with scaled duals on the cache ``c`` of one instance.  xref (N, n), uref (N-1, m), umin / umax (N-1, m),
    xmin / xmax (N-1, n) (knots 2..N) may be None (0, resp. -inf / +inf).  ``state`` = (z, y, v, g) warm-starts the
    iteration (z, y (N-1, m); v, g (N-1, n), v and g at knots 2..N); None starts from zeros.
    Returns dict(X (N, n), U (N-1, m), iters, r_pri, r_dual, converged, state=(z, y, v, g))."""
    A, B, Q, R, Qf, K, C1, C2, rho = (c[k] for k in ("A", "B", "Q", "R", "Qf", "K", "C1", "C2", "rho"))
    n, m = B.shape
    xref = np.zeros((N, n)) if xref is None else np.asarray(xref, dtype=np.float64)
    uref = np.zeros((N - 1, m)) if uref is None else np.asarray(uref, dtype=np.float64)
    umin = np.full((N - 1, m), -np.inf) if umin is None else umin
    umax = np.full((N - 1, m), np.inf) if umax is None else umax
    xmin = np.full((N - 1, n), -np.inf) if xmin is None else xmin
    xmax = np.full((N - 1, n), np.inf) if xmax is None else xmax
    if state is None:
        z, y, v, g = np.zeros((N - 1, m)), np.zeros((N - 1, m)), np.zeros((N - 1, n)), np.zeros((N - 1, n))
    else:
        z, y, v, g = (np.array(s, dtype=np.float64) for s in state)
    qref = -(xref[1:N - 1] @ Q.T)          # knots 2..N-1
    pref = -(Qf @ xref[N - 1])             # knot N
    rref = -(uref @ R.T)                   # knots 1..N-1
    X, U, d = np.zeros((N, n)), np.zeros((N - 1, m)), np.zeros((N - 1, m))
    r_pri = r_dual = np.inf
    it, converged = 0, False
    while it < max_iter:
        it += 1
        # 1-2: linear terms and the backward pass (v, g index knot k + 1 at row k - 1 ... stored for knots 2..N)
        p = pref - rho * (v[N - 2] - g[N - 2])
        rt = rref - rho * (z - y)
        for k in range(N - 2, -1, -1):     # knot k + 1 = N-1 .. 1
            d[k] = C1 @ (B.T @ p + rt[k])
            if k > 0:
                p = (qref[k - 1] - rho * (v[k - 1] - g[k - 1])) + C2 @ p - K.T @ rt[k]
        # 3: forward pass
        X[0] = x0
        for k in range(N - 1):
            U[k] = -K @ X[k] - d[k]
            X[k + 1] = A @ X[k] + B @ U[k]
        # 4-6: slacks, duals, residuals
        z_prev, v_prev = z, v
        z = np.clip(U + y, umin, umax)
        v = np.clip(X[1:] + g, xmin, xmax)
        y = y + U - z
        g = g + X[1:] - v
        r_pri = max(np.max(np.abs(U - z)), np.max(np.abs(X[1:] - v)))
        r_dual = rho * max(np.max(np.abs(z - z_prev)), np.max(np.abs(v - v_prev)))
        if r_pri <= eps_pri and r_dual <= eps_dual:
            converged = True
            break
    return dict(X=X, U=U, iters=it, r_pri=r_pri, r_dual=r_dual, converged=converged, state=(z, y, v, g))


def primals(X, U):
    """X (N, n), U (N-1, m) -> the Primals order [x1; u1; ...; xN]"""
    return np.concatenate([np.concatenate([X[:-1], U], axis=1).reshape(-1), X[-1]])
