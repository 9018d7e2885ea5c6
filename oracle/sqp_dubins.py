"""CPU ORACLE (test infrastructure): the Dubins SQP loop restated in numpy.

Outer loop as solve!/step! (src/cholesky_solver.jl:109-153), QP step through the oracle's block-Cholesky
KKT chain, globalisation as the in-repo spec src/sqp.jl:72-94 (L1 merit, eta=1e-4, rho=0.5, <=10 trials,
second-order correction at alpha=1).  The penalty rule (TO.update_penalty!, un-vendored) is
mu <- max(mu, 1.1*||lambda||_inf); the Dubins RK3 model is re-derived (not reference-pinned).
"""
from __future__ import annotations

import numpy as np

import oracle
from lqr_b200 import problems

n, m = 3, 2


def rk3_step(X, U, dt):
    th, v, om = X[..., 2], U[..., 0], U[..., 1]
    th2, th3 = th + 0.5 * dt * om, th + dt * om
    cb = (np.cos(th) + 4 * np.cos(th2) + np.cos(th3)) / 6
    sb = (np.sin(th) + 4 * np.sin(th2) + np.sin(th3)) / 6
    return np.stack([X[..., 0] + dt * v * cb, X[..., 1] + dt * v * sb, th + dt * om], -1)


def split(Z, N):
    b = Z.shape[0]
    body = Z[:, :(N - 1) * (n + m)].reshape(b, N - 1, n + m)
    X = np.concatenate([body[:, :, :n], Z[:, None, (N - 1) * (n + m):]], axis=1)
    return X, body[:, :, n:]


def cost(Z, xf, o):
    X, U = split(Z, o["N"])
    e = X - xf[:, None]
    return (0.5 * o["q_diag"] * o["dt"] * (e[:, :-1] ** 2).sum((1, 2)) + 0.5 * o["r_diag"] * o["dt"] * (U ** 2).sum((1, 2))
            + 0.5 * o["qf_diag"] * (e[:, -1] ** 2).sum(1))


def constraints(Z, x0, xf, o):
    """[c_1; d_1; ...; d_{N-1}; c_N] pieces: c1 (b,n), d (b,N-1,n), cN (b,n)."""
    X, U = split(Z, o["N"])
    return X[:, 0] - x0, rk3_step(X[:, :-1], U, o["dt"]) - X[:, 1:], X[:, -1] - xf


def c_norm1(Z, x0, xf, o):
    c1, d, cN = constraints(Z, x0, xf, o)
    return np.abs(c1).sum(1) + np.abs(d).sum((1, 2)) + np.abs(cN).sum(1)


def linearize(Z, x0, xf, o):
    N, dt = o["N"], o["dt"]
    b = Z.shape[0]
    X, U = split(Z, N)
    A, B = problems.dubins_rk3_jacobians(X[:, :-1, 2], U[..., 0], U[..., 1], dt)
    e = X - xf[:, None]
    Q = np.zeros((b, N, n, n))
    Q[:, :-1] = o["q_diag"] * dt * np.eye(n)
    Q[:, -1] = o["qf_diag"] * np.eye(n)
    q = np.concatenate([o["q_diag"] * dt * e[:, :-1], o["qf_diag"] * e[:, -1:]], axis=1)
    R = np.broadcast_to(o["r_diag"] * dt * np.eye(m), (b, N - 1, m, m)).copy()
    r = o["r_diag"] * dt * U
    c1, d, cN = constraints(Z, x0, xf, o)
    p, Cs, cs = problems._init_goal_blocks(b, n, m, N, c1, cN)
    return dict(n=n, m=m, N=N, p=p, hess_mode=problems.HESS_DIAG, Q=Q, R=R, Hux=None, q=q, r=r, A=A, B=B, d=d,
                D2=None, C=Cs, c=cs)


def gradient_flat(prob):
    b, N = prob["q"].shape[0], prob["N"]
    g = np.zeros((b, N * n + (N - 1) * m))
    body = g[:, :(N - 1) * (n + m)].reshape(b, N - 1, n + m)
    body[:, :, :n] = prob["q"][:, :-1]
    body[:, :, n:] = prob["r"]
    g[:, (N - 1) * (n + m):] = prob["q"][:, -1]
    return g


# branch codes of the trace: which trial an instance accepted in one iteration
BR_FROZEN, BR_REJECTED, BR_FULL, BR_SOC = -2, -1, 0, 1  # 2..10: back-tracking trial i, alpha = rho^(i-1)


def _margin(lhs, rhs):
    """Relative distance of a merit comparison from its threshold (NaN compares as 0: no margin)."""
    with np.errstate(invalid="ignore"):
        return np.nan_to_num(np.abs(lhs - rhs) / np.maximum(np.maximum(np.abs(lhs), np.abs(rhs)), 1e-300), nan=0.0)


def solve(Z0, x0, xf, o, trace=False):
    """Returns Z, feas_p, feas_d, iters, kkt_solves (per-instance bookkeeping like the device driver).

    trace=True appends a dict of per-iteration arrays (the arithmetic is the same, Z is bit-identical):
      Z          (iters, b, NN)  the iterate after iteration k + 1 (what a run with iters = k + 1 returns)
      branch     (iters, b)      BR_FROZEN (converged before this iteration), BR_FULL (alpha = 1), BR_SOC,
                                 2..10 (accepted at back-tracking trial i), BR_REJECTED (every trial rejected)
      margin     (iters, b, 11)  relative margin of each merit comparison evaluated (alpha = 1, SOC, trials 2..10),
                                 NaN where the instance did not evaluate it; 0 where a side is NaN
      conv_margin (iters, b, 2)  relative margins of feas_p vs eps_p and feas_d vs eps_d in the convergence test
      mu         (iters, b)      the merit penalty after its update
      kkt_solves (iters,)        the running count of KKT solves, SOC solves included
    """
    Z = Z0.copy()
    b = Z.shape[0]
    mu = np.ones(b)
    conv = np.zeros(b, bool)
    iters = np.zeros(b, np.int32)
    lam = None
    solves = 0
    tr = dict(Z=[], branch=[], margin=[], conv_margin=[], mu=[], kkt_solves=[])
    for _ in range(o["iters"]):
        prob = linearize(Z, x0, xf, o)
        c1, d, cN = constraints(Z, x0, xf, o)
        feas_p = np.maximum(np.abs(c1).max(1), np.maximum(np.abs(d).max((1, 2)), np.abs(cN).max(1)))
        feas_d = residual_norm(prob, lam)
        if trace:
            tr["conv_margin"].append(np.where(conv[:, None], np.nan, np.stack(
                [_margin(feas_p, o["eps_p"]), _margin(feas_d, o["eps_d"])], -1)))
        conv |= (feas_p < o["eps_p"]) & (feas_d < o["eps_d"])
        dz, lam_new, info = oracle.kkt_solve(prob)
        solves += b
        act = ~conv
        lam = np.where(act[:, None], lam_new, lam if lam is not None else 0 * lam_new)
        iters[act] += 1
        br = np.where(conv, BR_FROZEN, BR_REJECTED)
        mg = np.full((b, 11), np.nan)
        if not o["line_search"]:
            Z[act] += dz[act]
            br[act] = BR_FULL
        else:
            mu = np.where(act, np.maximum(mu, 1.1 * np.abs(lam_new).max(1)), mu)
            g = gradient_flat(prob)
            cn0 = c_norm1(Z, x0, xf, o)
            phi0 = cost(Z, xf, o) + mu * cn0
            dphi0 = (g * dz).sum(1) - mu * cn0
            eta, rho = 1e-4, 0.5
            done = conv.copy()
            phi = lambda Zt: cost(Zt, xf, o) + mu * c_norm1(Zt, x0, xf, o)  # noqa: E731
            lhs, rhs = phi(Z + dz), phi0 + eta * dphi0
            if trace:
                mg[~done, 0] = _margin(lhs, rhs)[~done]
            ok = (lhs <= rhs) & ~done
            Z[ok] += dz[ok]
            done |= ok
            br[ok] = BR_FULL
            alpha = np.ones(b)
            if (~done).any():
                c1t, dt_, cNt = constraints(Z + dz, x0, xf, o)
                prob2 = dict(prob)
                p, Cs, cs = problems._init_goal_blocks(b, n, m, o["N"], c1t, cNt)
                prob2.update(d=dt_, c=cs)
                dzh, _, _ = oracle.kkt_solve(prob2, soc=True)
                solves += b
                lhs = phi(Z + dz + dzh)
                if trace:
                    mg[~done, 1] = _margin(lhs, rhs)[~done]
                ok = (lhs < rhs) & ~done
                Z[ok] += dz[ok] + dzh[ok]
                done |= ok
                br[ok] = BR_SOC
                alpha[~done] = rho
                for trial in range(2, 11):  # the reference's i = 2..10 (src/sqp.jl:76-92): alpha = rho^1..rho^9
                    if done.all():
                        break
                    lhs, rhs_a = phi(Z + alpha[:, None] * dz), phi0 + eta * alpha * dphi0
                    if trace:
                        mg[~done, trial] = _margin(lhs, rhs_a)[~done]
                    ok = (lhs <= rhs_a) & ~done
                    Z[ok] += alpha[ok, None] * dz[ok]
                    done |= ok
                    br[ok] = trial
                    alpha[~done] *= rho
        if trace:
            tr["Z"].append(Z.copy())
            tr["branch"].append(br)
            tr["margin"].append(mg)
            tr["mu"].append(mu.copy())
            tr["kkt_solves"].append(solves)
    prob = linearize(Z, x0, xf, o)
    c1, d, cN = constraints(Z, x0, xf, o)
    feas_p = np.maximum(np.abs(c1).max(1), np.maximum(np.abs(d).max((1, 2)), np.abs(cN).max(1)))
    out = (Z, feas_p, residual_norm(prob, lam), iters, solves)
    if trace:
        out += ({k: np.array(v) for k, v in tr.items()},)
    return out


def residual_norm(prob, lam):
    """residual(solver, recalculate=false): || (||g_k + D'lam restricted to knot k||)_k ||.
    Block-wise for the init + dynamics + goal pattern of this problem (multiplier order [mu_1; lam_1; ...;
    lam_{N-1}; mu_N], C_1 = [I 0], C_N = I, D2 = [-I 0]); residual_norm_assembled is the global-matrix form the
    tests hold it against."""
    g = gradient_flat(prob)
    if lam is None:
        return np.linalg.norm(g, axis=1)
    b, N = prob["q"].shape[0], prob["N"]
    L = lam[:, n:-n].reshape(b, N - 1, n)
    rx = np.einsum("bkji,bkj->bki", prob["A"], L)
    rx[:, 0] += lam[:, :n]
    rx[:, 1:] -= L[:, :-1]
    ru = np.einsum("bkji,bkj->bki", prob["B"], L)
    r = g.copy()
    body = r[:, :(N - 1) * (n + m)].reshape(b, N - 1, n + m)
    body[:, :, :n] += rx
    body[:, :, n:] += ru
    r[:, (N - 1) * (n + m):] += lam[:, -n:] - L[:, -1]
    return np.linalg.norm(r, axis=1)


def residual_norm_assembled(prob, lam):
    """The same number through the assembled global D (oracle/dense_kkt.py); slow, used to check the above."""
    from oracle import dense_kkt
    b = prob["q"].shape[0]
    out = np.zeros(b)
    g = gradient_flat(prob)
    for i in range(b):
        _, _, D, _ = dense_kkt.assemble(prob, i)
        out[i] = np.linalg.norm(g[i] + D.T @ lam[i])
    return out


def turn90_problem(batch, N=11, seed=2):
    """Config 4 generator (SURVEY §8d): x0 = 0, xf ~ [1.5,1.5,pi/2] + N(0,0.1^2), start from the u = 0.1
    rollout; tf = 3 as TO's turn90 (unpinned)."""
    rng = np.random.default_rng(seed)
    tf = 3.0
    o = dict(N=N, iters=10, dt=tf / (N - 1), q_diag=1e-2, r_diag=1e-2, qf_diag=100.0, eps_p=1e-5, eps_d=1e-5,
             line_search=1)
    x0 = np.zeros((batch, n))
    xf = np.array([1.5, 1.5, np.pi / 2]) + 0.1 * rng.standard_normal((batch, n))
    U = np.full((batch, N - 1, m), 0.1)
    X = np.zeros((batch, N, n))
    for k in range(N - 1):
        X[:, k + 1] = rk3_step(X[:, k], U[:, k], o["dt"])
    Z = np.zeros((batch, N * n + (N - 1) * m))
    body = Z[:, :(N - 1) * (n + m)].reshape(batch, N - 1, n + m)
    body[:, :, :n], body[:, :, n:] = X[:, :-1], U
    Z[:, (N - 1) * (n + m):] = X[:, -1]
    return Z, x0, xf, o


def hard_turn_problem(batch, N, tf, qf, z_sd, goal_scale, theta_sd, seed, keep=None):
    """A turn90 problem made hard for the line search: horizon tf, terminal weight qf, goal position scaled by
    goal_scale, goal heading + theta_sd * N(0,1), initial guess + z_sd * N(0,1).  keep: instance subset."""
    Z0, x0, xf, o = turn90_problem(batch, N=N, seed=seed)
    rng = np.random.default_rng(seed)
    xf = xf * np.array([goal_scale, goal_scale, 1.0])
    xf[:, 2] += theta_sd * rng.standard_normal(batch)
    Z0 = Z0 + z_sd * rng.standard_normal(Z0.shape)
    o = dict(o, dt=tf / (N - 1), qf_diag=qf)
    if keep is not None:
        Z0, x0, xf = Z0[keep], x0[keep], xf[keep]
    return Z0, x0, xf, o


def line_search_cases():
    """Frozen inputs on which the line search takes every branch: name -> (Z0, x0, xf, options).

    The first four reach the second-order correction and back-tracking trials 2..5 in hundreds of instance-iterations;
    the short horizons N = 3, 4, 5 with batches 33, 65 and 1 are the edges of the device's prefetch ring and partial
    warps and CTAs, and most of their instances converge (at different iterations) and freeze.  n3_far_start keeps
    the 18 instances of its draw whose every merit comparison is at least 1e-7 (relative) from its threshold and whose
    trajectory moves by less than 3e-12 under 1e-13 noise in the QP steps; they reach back-tracking trials 2..10, and
    one of them (index 6 of the subset) rejects all ten trials in some iterations."""
    far = [0, 5, 8, 16, 18, 20, 23, 25, 28, 30, 35, 38, 45, 47, 48, 55, 58, 63]
    return {
        "n11_far_goal": hard_turn_problem(128, 11, 3.0, 100.0, 1.0, 5.0, 3.0, seed=0),
        "n21_short_tf": hard_turn_problem(128, 21, 1.0, 100.0, 1.0, 3.0, 2.0, seed=0),
        "n6": hard_turn_problem(128, 6, 3.0, 100.0, 1.0, 2.0, 3.0, seed=0),
        "n41_qf1000": hard_turn_problem(128, 41, 2.0, 1000.0, 2.0, 4.0, 3.0, seed=0),
        "n3_b33": hard_turn_problem(33, 3, 3.0, 100.0, 0.5, 1.0, 0.0, seed=0),
        "n4_b65": hard_turn_problem(65, 4, 3.0, 100.0, 0.5, 1.0, 0.0, seed=0),
        "n5_b1": hard_turn_problem(1, 5, 3.0, 100.0, 1.0, 1.0, 1.0, seed=39),
        "n3_far_start": hard_turn_problem(65, 3, 3.0, 100.0, 10.0, 1.0, 3.0, seed=2, keep=far),
    }


def slsqp_solution(Z0, x0, xf, o, i):
    """Instance i of the same nonlinear program solved by SciPy's SLSQP (a third-party solver, finite-difference
    derivatives): an independent pin of the SQP driver's end point.  Returns (z, cost, max |constraint|)."""
    from scipy.optimize import minimize

    def f(z):
        return float(cost(z[None], xf[i:i + 1], o)[0])

    def c(z):
        c1, d, cN = constraints(z[None], x0[i:i + 1], xf[i:i + 1], o)
        return np.concatenate([c1.ravel(), d.ravel(), cN.ravel()])

    r = minimize(f, Z0[i], method="SLSQP", constraints=[dict(type="eq", fun=c)], options=dict(maxiter=1000, ftol=1e-15))
    assert r.success, r.message
    return r.x, float(r.fun), float(np.abs(c(r.x)).max())
