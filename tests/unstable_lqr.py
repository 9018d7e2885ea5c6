"""Open-loop unstable problem generators shared by the CPU oracle tests and the GPU stability tests (no GPU needed).

The unstable draw is dare_lti_riccati(unstable=True): A = I + 0.3 J / sqrt(n), B ~ N(0, 1), rho(A) ~ 1.1-1.5.  Draws
whose stationary (DARE) gain |K| exceeds K_BOUND are replaced: one actuator against many unstable modes can give |K| of
1e2-1e3, where double precision itself misses 1e-9 whatever the kernel does (test_gpu_riccati_grad_stability.py)."""
import numpy as np

from lqr_b200 import problems

K_BOUND = 50.0


def dare_gain_norm(A, B, Q, R):
    """|K| of the discrete algebraic Riccati equation's gain (SciPy's ordered-QZ solve)"""
    from scipy.linalg import solve_discrete_are
    P = solve_discrete_are(A, B, Q, R)
    return np.linalg.norm(np.linalg.solve(R + B.T @ P @ B, B.T @ P @ A))


def unstable_draw(n, m, Q, R, seed):
    """(A, B) of dare_lti_riccati(unstable=True) whose DARE gain for the stage cost (Q, R) is at most K_BOUND"""
    s = seed
    while True:
        p = problems.dare_lti_riccati(n, m, 2, 1, seed=s, unstable=True)
        if dare_gain_norm(p["A"][0], p["B"][0], Q, R) <= K_BOUND:
            return p["A"][0], p["B"][0]
        s += 10000


def destabilise(prob, seed):
    """A_k, B_k of the even instances of a KKT problem <- an unstable draw under 1 % relative noise per element and
    knot; the odd instances keep theirs.  The gain bound is taken with the knot-0 stage cost as the problem's Hessian
    mode reads it (diagonal mode: the diagonals)."""
    n, m, N = prob["n"], prob["m"], prob["N"]
    rng = np.random.default_rng(seed + 1)
    diag = int(prob.get("hess_mode", 1)) == 2
    for i in range(0, prob["q"].shape[0], 2):
        Q, R = prob["Q"][i, 0], prob["R"][i, 0]
        if diag:
            Q, R = np.diag(np.diag(Q)), np.diag(np.diag(R))
        A, Bm = unstable_draw(n, m, Q, R, seed + 17 * i)
        prob["A"][i] = A * (1.0 + 0.01 * rng.standard_normal((N - 1, n, n)))
        prob["B"][i] = Bm * (1.0 + 0.01 * rng.standard_normal((N - 1, n, m)))
    return prob


def free_final(prob):
    """Drop the goal rows of a KKT problem: p_N = 0 (initial condition, dynamics, stage rows, free final state)."""
    prob["p"] = prob["p"].copy()
    prob["p"][-1] = 0
    b = prob["q"].shape[0]
    prob["C"][-1] = np.zeros((b, 0, prob["n"]))
    prob["c"][-1] = np.zeros((b, 0))
    return prob


def unstable_kkt(n, m, N, batch, seed, mid_p=0, hess=1, goal=True):
    """random_lqr_kkt's costs, rows and d with unstable dynamics on the even instances; goal=False: p_N = 0"""
    prob = destabilise(problems.random_lqr_kkt(n, m, N, batch, seed=seed, mid_p=mid_p, hess_mode=hess), seed)
    return prob if goal else free_final(prob)


def spectral_radii(prob):
    """rho(A_0) of every instance"""
    return np.array([np.abs(np.linalg.eigvals(a[0])).max() for a in prob["A"]])


def unstable_riccati(n, m, N, batch, seed):
    """A Riccati problem (LTV, affine terms): dare_lti_riccati's unstable draw at the even instances (gain-bounded for
    their Q, R), its stable draw at the odd ones, A, B under 1 % relative noise per element and knot, random q, r, qf"""
    pu = problems.dare_lti_riccati(n, m, N, batch, seed=seed, unstable=True)
    ps = problems.dare_lti_riccati(n, m, N, batch, seed=seed + 1000, unstable=False)
    prob = dict(ps, lti=False)
    A, B = ps["A"].copy(), ps["B"].copy()
    for i in range(0, batch, 2):
        A[i], B[i] = unstable_draw(n, m, pu["Q"][i], pu["R"][i], seed + 17 * i)
        prob["Q"][i], prob["R"][i], prob["Qf"][i] = pu["Q"][i], pu["R"][i], pu["Qf"][i]
    rng = np.random.default_rng(seed + 2)
    prob.update(A=A[:, None] * (1.0 + 0.01 * rng.standard_normal((batch, N - 1, n, n))),
                B=B[:, None] * (1.0 + 0.01 * rng.standard_normal((batch, N - 1, n, m))),
                Q=np.repeat(prob["Q"][:, None], N - 1, axis=1), R=np.repeat(prob["R"][:, None], N - 1, axis=1),
                q=rng.standard_normal((batch, N - 1, n)), r=rng.standard_normal((batch, N - 1, m)),
                qf=rng.standard_normal((batch, n)))
    return prob
