"""CPU tests of oracle/admm.py, the statement of lqrb_admm_cache_f64 / lqrb_admm_solve_f64 the GPU tests pin to: the
converged iteration against three exact solutions of the same problem, stable and open-loop unstable.
  - no bounds: the unconstrained LQR with Qf = Pt - rho I, from the C oracle's Riccati recursion (stable draws; on the
    open-loop unstable ones its unsymmetrised recursion, the reference's form, drifts by 1e-4, and the refined dense KKT
    solve is the pin);
  - input bounds: the box QP of the condensed problem, by bounded-variable least squares;
  - state and input bounds: the equality-constrained QP with the converged active set, by the refined dense KKT solve,
    with the multipliers rho y, rho g of the sign their bound requires and zero off the active set (the KKT conditions).
"""
import numpy as np
import pytest
import scipy.optimize as so
import scipy.sparse as sp

from lqr_b200 import problems
from oracle import admm as oa
from oracle import dense_kkt

CASES = [(4, 1, False), (4, 1, True), (6, 3, True), (12, 4, False), (12, 4, True)]
RHO = 1.0
N = 30


def _instance(n, m, unstable, seed):
    p = problems.dare_lti_riccati(n, m, N, 1, seed=seed, unstable=unstable)
    rng = np.random.default_rng(seed + 1)
    A, B, Q, R = (p[k][0] for k in "ABQR")
    return A, B, Q, R, 3.0 * p["x0"][0], 0.5 * rng.standard_normal((N, n)), 0.2 * rng.standard_normal((N - 1, m))


def _bounds(c, x0, xref, uref, state_bounds, N=N):
    """input bounds at 0.4 of the largest unconstrained |u_j| (per component); with state_bounds, input bounds at 0.7 and
    a box on the first state component at 0.8 of its largest unconstrained excursion from knot 9 on (tighter pairs
    leave the unstable draws infeasible or slow)"""
    n, m = c["B"].shape
    r = oa.solve(c, x0, N, xref, uref, max_iter=20000, eps_pri=1e-11, eps_dual=1e-11)
    ub = (0.7 if state_bounds else 0.4) * np.abs(r["U"]).max(axis=0)
    b = dict(umin=np.broadcast_to(-ub, (N - 1, m)).copy(), umax=np.broadcast_to(ub, (N - 1, m)).copy())
    if state_bounds:
        xb = 0.8 * np.abs(r["X"][8:, 0]).max()
        b["xmin"], b["xmax"] = np.full((N - 1, n), -np.inf), np.full((N - 1, n), np.inf)
        b["xmin"][7:, 0], b["xmax"][7:, 0] = -xb, xb
    return b


def _condensed(c, x0, xref, uref):
    """H, g of the cost in U = (u_1..u_{N-1}): x_{k+1} = A^k x0 + sum_j A^(k-1-j) B u_j"""
    A, B, Q, R, Qf = (c[k] for k in ("A", "B", "Q", "R", "Qf"))
    n, m = B.shape
    Su, Sx = np.zeros(((N - 1) * n, (N - 1) * m)), np.zeros(((N - 1) * n, n))
    P = np.eye(n)
    for k in range(N - 1):
        P = A @ P
        Sx[k * n:(k + 1) * n] = P
        for j in range(k + 1):
            Su[k * n:(k + 1) * n, j * m:(j + 1) * m] = np.linalg.matrix_power(A, k - j) @ B
    Qb = np.kron(np.eye(N - 1), Q)
    Qb[-n:, -n:] = Qf
    Rb = np.kron(np.eye(N - 1), R)
    H = Su.T @ Qb @ Su + Rb
    g = Su.T @ Qb @ (Sx @ x0 - xref[1:].reshape(-1)) - Rb @ uref.reshape(-1)
    return 0.5 * (H + H.T), g


def _kkt(c, x0, xref, uref, rows, N=N):
    """Global H, g, D, d of the problem with equality rows (Primals index, value) added to x_1 = x0 and the dynamics"""
    A, B, Q, R, Qf = (c[k] for k in ("A", "B", "Q", "R", "Qf"))
    n, m = B.shape
    NN, w = N * n + (N - 1) * m, n + m
    H = sp.lil_matrix((NN, NN))
    g = np.zeros(NN)
    for k in range(N):
        ix = slice(k * w, k * w + n)
        H[ix, ix] = Qf if k == N - 1 else Q
        g[ix] = -(Qf if k == N - 1 else Q) @ xref[k]
        if k < N - 1:
            iu = slice(k * w + n, (k + 1) * w)
            H[iu, iu] = R
            g[iu] = -R @ uref[k]
    D = sp.lil_matrix((n + (N - 1) * n + len(rows), NN))
    d = np.zeros(D.shape[0])
    D[:n, :n] = np.eye(n)
    d[:n] = -x0
    for k in range(N - 1):
        r0 = n + k * n
        D[r0:r0 + n, k * w:k * w + n] = A
        D[r0:r0 + n, k * w + n:(k + 1) * w] = B
        D[r0:r0 + n, (k + 1) * w:(k + 1) * w + n] = -np.eye(n)
    for i, (col, val) in enumerate(rows):
        D[n + (N - 1) * n + i, col] = 1.0
        d[n + (N - 1) * n + i] = -val
    return sp.csc_matrix(H), g, sp.csc_matrix(D), d


@pytest.mark.parametrize("n,m,unstable", CASES)
def test_unbounded_equals_lqr_with_the_cached_terminal_cost(oracle_mod, n, m, unstable):
    A, B, Q, R, x0, xref, uref = _instance(n, m, unstable, seed=n + m + unstable)
    c = oa.cache(A, B, Q, R, RHO)
    assert c["ok"] and np.all(np.linalg.eigvalsh(c["Qf"] - Q) > 0)  # Qf = Pt - rho I >= Q
    r = oa.solve(c, x0, N, xref, uref, max_iter=20000, eps_pri=1e-13, eps_dual=1e-13)
    assert r["converged"], r["iters"]
    if unstable:
        dz, _ = dense_kkt.solve_refined(*_kkt(c, x0, xref, uref, []))
    else:
        rep = lambda M: np.repeat(M[None, None], N - 1, axis=1)  # noqa: E731
        prob = dict(n=n, m=m, N=N, lti=False, A=rep(A), B=rep(B), Q=rep(Q), R=rep(R), q=-(xref[None, :-1] @ Q.T),
                    r=-(uref[None] @ R.T), Qf=c["Qf"][None], qf=-(c["Qf"] @ xref[-1])[None], x0=x0[None])
        X, U, _, _, info = oracle_mod.riccati(prob)
        assert info[0] == 0
        dz = oa.primals(X[0], U[0])
    assert np.abs(oa.primals(r["X"], r["U"]) - dz).max() <= 1e-9 * np.abs(dz).max()


@pytest.mark.parametrize("n,m,unstable", CASES)
def test_input_bounds_equal_the_condensed_box_qp(n, m, unstable):
    A, B, Q, R, x0, xref, uref = _instance(n, m, unstable, seed=2 * n + m + unstable)
    c = oa.cache(A, B, Q, R, RHO)
    b = _bounds(c, x0, xref, uref, state_bounds=False)
    eps = 1e-10
    r = oa.solve(c, x0, N, xref, uref, max_iter=50000, eps_pri=eps, eps_dual=eps, **b)
    assert r["converged"], r["iters"]
    act = np.mean((r["state"][0] == b["umin"]) | (r["state"][0] == b["umax"]))
    assert act >= 0.05, act  # the bounds bind on a good share of knots
    H, g = _condensed(c, x0, xref, uref)
    L = np.linalg.cholesky(H).T  # H = L'L
    ls = so.lsq_linear(L, -np.linalg.solve(L.T, g), bounds=(b["umin"].reshape(-1), b["umax"].reshape(-1)),
                       method="bvls", tol=1e-15)
    U = ls.x.reshape(N - 1, m)
    # the ADMM error is bounded by the stopping residuals times the conditioning of the condensed Hessian
    tol = 1e3 * eps * np.linalg.cond(H) ** 0.5 * max(1.0, np.abs(U).max())
    assert np.abs(r["U"] - U).max() <= tol, (np.abs(r["U"] - U).max(), tol)


@pytest.mark.parametrize("n,m,unstable", CASES)
def test_state_and_input_bounds_satisfy_the_kkt_conditions(n, m, unstable):
    A, B, Q, R, x0, xref, uref = _instance(n, m, unstable, seed=3 * n + m + unstable)
    c = oa.cache(A, B, Q, R, RHO)
    b = _bounds(c, x0, xref, uref, state_bounds=True)
    eps = 1e-10
    r = oa.solve(c, x0, N, xref, uref, max_iter=20000, eps_pri=eps, eps_dual=eps, **b)
    assert r["converged"], r["iters"]
    z, y, v, gg = r["state"]
    w = n + m
    rows, mult = [], []
    for k in range(N - 1):
        for j in range(m):
            if z[k, j] == b["umin"][k, j] or z[k, j] == b["umax"][k, j]:
                rows.append((k * w + n + j, z[k, j]))
                mult.append(RHO * y[k, j])
        for i in range(n):
            if v[k, i] == b["xmin"][k, i] or v[k, i] == b["xmax"][k, i]:
                rows.append(((k + 1) * w + i, v[k, i]))
                mult.append(RHO * gg[k, i])
    assert any(col % w == 0 for col, _ in rows), "the state bound does not bind"
    assert any(col % w >= n for col, _ in rows), "no input bound binds"
    dz, lam = dense_kkt.solve_refined(*_kkt(c, x0, xref, uref, rows))
    scale = max(1.0, np.abs(dz).max())
    assert np.abs(oa.primals(r["X"], r["U"]) - dz).max() <= 1e-6 * scale
    lam_act = lam[n + (N - 1) * n:]
    lscale = max(1.0, np.abs(lam).max())
    assert np.abs(lam_act - np.array(mult)).max() <= 1e-6 * lscale
    # the sign each bound requires, and zero off the active set
    tol = 1e-6 * lscale
    assert np.all(RHO * y[z == b["umax"]] >= -tol) and np.all(RHO * y[z == b["umin"]] <= tol)
    assert np.all(RHO * gg[v == b["xmax"]] >= -tol) and np.all(RHO * gg[v == b["xmin"]] <= tol)
    free_u = (z > b["umin"]) & (z < b["umax"])
    free_x = (v > b["xmin"]) & (v < b["xmax"])
    assert np.abs(RHO * y[free_u]).max(initial=0.0) <= tol and np.abs(RHO * gg[free_x]).max(initial=0.0) <= tol


def test_fixed_count_warm_start_continues_the_cold_iteration():
    A, B, Q, R, x0, xref, uref = _instance(6, 3, True, seed=5)
    c = oa.cache(A, B, Q, R, RHO)
    b = _bounds(c, x0, xref, uref, state_bounds=True)
    r1 = oa.solve(c, x0, N, xref, uref, max_iter=7, **b)
    r2 = oa.solve(c, x0, N, xref, uref, max_iter=5, state=r1["state"], **b)
    r3 = oa.solve(c, x0, N, xref, uref, max_iter=12, **b)
    assert np.array_equal(r2["X"], r3["X"]) and np.array_equal(r2["U"], r3["U"])
