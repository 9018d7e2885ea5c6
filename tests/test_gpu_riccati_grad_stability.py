"""GPU: the Riccati gradients on long horizons of open-loop unstable systems, against the refined solve.

The costates of the backward sweep run through a recursion.  Written open-loop, λ_{k-1} = Q_k x_k + q_k + A_kᵀλ_k,
any error in λ_k is multiplied by A_kᵀ at every knot: with ρ(A) = 1.18 it grows past 1e-3 relative at N = 201 and
past 1e11 at N = 401 even from the refined solutions (DESIGN §4.8), while the true costates stay bounded because the
optimal closed loop is stable.  The sweep therefore runs the closed-loop form (A_k − B_k K_k)ᵀ.  The generators of
the other gradient tests (dt = 0.05, N ≤ 41, the cartpole about its hanging rollout) are open-loop stable or nearly
so, and cannot tell the two forms apart; these inputs can:
  * unstable LTI: ``dare_lti_riccati(unstable=True)`` (ρ(A) ≈ 1.2–1.3, strong actuation) with random q, r, qf, so
    that λ carries the affine terms;
  * unstable LTV: the same A, B per knot with 1 % relative noise per knot, Q, R per knot under a 1 % diagonal
    congruence, fresh q_k, r_k;
  * near-marginal LTI control: the stable variant (ρ ≈ 1.02) at N = 1001.
Unstable and benign instances alternate in every batch (instances 0, 2 unstable, 1, 3 the stable variant), so that a
failure of one cannot hide behind the others.

Checks, per instance and per output array, relative norm error ≤ 1e-9 against the CPU oracles (oracle/riccati_grad.py
on the extended-precision refined solve, held against finite differences on these inputs in
tests/test_oracle_riccati_grad.py; oracle/riccati_gain_grad.py for the gains):
  * lqrb_riccati_grad_f64 on one shape per forward family that solves the adjoint problem, N = 101, 201, 401
    (101, 201 for n > 16), LTI and LTV;
  * lqrb_riccati_grad_gains_f64 with dZ, dK, dkff; with dK, dkff only; with dZ only (bitwise equal to
    lqrb_riccati_grad_f64);
  * the same LQR written as a KKT problem through lqrb_kkt_grad_f64 (its multipliers come out of the solve);
  * one backward pass of lqr_b200.autograd.riccati_solve(..., gains=True)."""
import contextlib
import functools

import numpy as np
import pytest

from lqr_b200 import ops, problems

pytestmark = pytest.mark.gpu

NAMES = ("A", "B", "Q", "R", "q", "r", "Qf", "qf", "x0")
TOL = 1e-9
B = 4  # instances per batch: unstable, benign, unstable, benign

# (n, m, expected kernel-name prefix, options, padded): one shape per forward family, as in
# test_gpu_riccati_conditioning.py
FAMILIES = [
    (4, 1, "riccati_tpi<4,1>", {}, False),
    (6, 3, "riccati_tpi<6,3>", {}, False),
    *[(n, m, f"riccati_dmma<{n},{m}>", {}, False) for n in (8, 12) for m in (1, 2, 3, 4)],
    (7, 2, "riccati_dmma<8,2>", {}, True),
    (10, 3, "riccati_dmma<12,3>", {}, True),
    (16, 8, "riccati_cta_dmma<16,8>", {}, False),
    (64, 16, "riccati_cta_dmma<64,16>", {}, False),
    (20, 6, "riccati_cta_dmma<24,8>", {}, True),
    (12, 4, "riccati_coop", {"riccati_variant": 2}, False),
    (10, 3, "riccati_coop", {"riccati_pad": 0}, False),
]
DEFAULTS = {"riccati_variant": 0, "riccati_pad": 1}


def _fid(f):
    return f"{f[2]}-{f[0]}x{f[1]}" + ("-padded" if f[4] else "") + ("-" + ",".join(f[3]) if f[3] else "")


def _horizons(n):
    return (101, 201, 401) if n <= 16 else (101, 201)


GRAD_CASES = [pytest.param(f, N, id=f"{_fid(f)}-N{N}") for f in FAMILIES for N in _horizons(f[0])]
# the gains call: every family but (64,16), whose long-double gain oracle alone takes tens of seconds
GAIN_CASES = [pytest.param(f, N, id=f"{_fid(f)}-N{N}") for f in FAMILIES if f[0] <= 24 for N in _horizons(f[0])[1:]]


@contextlib.contextmanager
def _options(handle, opts):
    for k, v in opts.items():
        handle.set_option(k, v)
    try:
        yield
    finally:
        for k in opts:
            handle.set_option(k, DEFAULTS[k])


def _check_kernel(handle, kern, padded):
    name = handle.last_kernel
    assert name.startswith(kern) and ("padded" in name) == padded, name


# ------------------------------------------------------------------ inputs
def _interleave(a, b):
    """instances a0, b0, a1, b1"""
    out = np.empty((a.shape[0] + b.shape[0],) + a.shape[1:])
    out[0::2], out[1::2] = a, b
    return out


def _dare_gain_norm(p, i):
    from scipy.linalg import solve_discrete_are
    A, Bm, R = p["A"][i], p["B"][i], p["R"][i]
    P = solve_discrete_are(A, Bm, p["Q"][i], R)
    return np.linalg.norm(np.linalg.solve(R + Bm.T @ P @ Bm, Bm.T @ P @ A))


# The unstable draws are kept where the stationary gain |K| <= 50.  One actuator against six to eight unstable modes
# ((12, 1)) can give |K| of 1e2-1e3; the gradient is then so sensitive that double precision misses 1e-9 whatever the
# costate recursion (the gain sweep, which never used the open-loop form, misses it too on those draws).
K_BOUND = 50.0


def _lti(n, m, N, seed, unstable=True):
    """B instances: the (un)stable dare_lti_riccati variant at the even indices, the stable one at the odd ones, with
    random q, r, qf"""
    s = seed
    while True:
        pu = problems.dare_lti_riccati(n, m, N, B // 2, seed=s, unstable=unstable)
        if all(_dare_gain_norm(pu, i) <= K_BOUND for i in range(B // 2)):
            break
        s += 10000
    ps = problems.dare_lti_riccati(n, m, N, B // 2, seed=seed + 1000, unstable=False)
    prob = dict(pu)
    for k in ("A", "B", "Q", "R", "Qf", "x0"):
        prob[k] = _interleave(pu[k], ps[k])
    rng = np.random.default_rng(seed + 1)
    prob.update(q=rng.standard_normal((B, n)), r=rng.standard_normal((B, m)), qf=rng.standard_normal((B, n)))
    return prob


def _ltv(n, m, N, seed):
    """_lti's batch with A, B per knot under 1 % relative noise per element, Q, R per knot under a 1 % diagonal
    congruence D_k Q D_k (stays SPD), and fresh q_k, r_k"""
    p = _lti(n, m, N, seed)
    rng = np.random.default_rng(seed + 2)

    def noisy(a):
        return a[:, None] * (1.0 + 0.01 * rng.standard_normal((B, N - 1) + a.shape[1:]))

    def congruent(a):
        d = 1.0 + 0.01 * rng.standard_normal((B, N - 1, a.shape[-1]))
        return a[:, None] * d[..., :, None] * d[..., None, :]
    p.update(lti=False, A=noisy(p["A"]), B=noisy(p["B"]), Q=congruent(p["Q"]), R=congruent(p["R"]),
             q=rng.standard_normal((B, N - 1, n)), r=rng.standard_normal((B, N - 1, m)))
    return p


@functools.lru_cache(maxsize=None)
def _case(n, m, N, lti, seed, unstable=True):
    """(problem, dZ, the oracle's gradient of l = dZ·Z), cached: the refined solve dominates every test here"""
    from oracle.riccati_grad import riccati_grad
    prob = _lti(n, m, N, seed, unstable) if lti else _ltv(n, m, N, seed)
    dZ = np.random.default_rng(seed + 3).standard_normal((B, N * n + (N - 1) * m))
    return prob, dZ, riccati_grad(prob, dZ)


def _seed(n, m, N):
    return 7 * n + m + N


def _z(X, U):
    b = X.shape[0]
    return np.concatenate([np.concatenate([X[:, :-1], U], axis=2).reshape(b, -1), X[:, -1]], axis=1)


def _solve(handle, prob, kern, opts, padded):
    with _options(handle, opts):
        X, U, _, _, info = ops.riccati_solve_problem(prob, want_gains=False, handle=handle)
    assert (info == 0).all(), info
    _check_kernel(handle, kern, padded)
    return _z(X, U)


def _errors(g, go, names=NAMES):
    """{(name, instance): relative norm error}"""
    out = {}
    for k in names:
        for i in range(B):
            out[(k, i)] = np.linalg.norm(g[k][i] - go[k][i]) / max(np.linalg.norm(go[k][i]), 1e-300)
    return out


def _assert_close(g, go, what, names=NAMES):
    errs = _errors(g, go, names)
    bad = {k: f"{e:.1e}" for k, e in errs.items() if not e <= TOL}
    assert not bad, (what, bad)


# ------------------------------------------------------------------ lqrb_riccati_grad_f64
@pytest.mark.parametrize("lti", [False, True], ids=["ltv", "lti"])
@pytest.mark.parametrize("fam,N", GRAD_CASES)
def test_riccati_grad_matches_oracle_on_unstable_horizons(handle, oracle_mod, fam, N, lti):
    n, m, kern, opts, padded = fam
    prob, dZ, go = _case(n, m, N, lti, _seed(n, m, N))
    Z = _solve(handle, prob, kern, opts, padded)
    with _options(handle, opts):
        g, info = ops.riccati_grad_problem(prob, Z, dZ, handle=handle)
    assert (info == 0).all(), info
    _check_kernel(handle, kern, padded)
    assert "riccati_grad<" in handle.last_kernel, handle.last_kernel
    _assert_close(g, go, handle.last_kernel)


@pytest.mark.parametrize("fam", [FAMILIES[1], FAMILIES[9], FAMILIES[12], FAMILIES[15]], ids=_fid)
def test_riccati_grad_near_marginal_lti_long_horizon(handle, oracle_mod, fam):
    """control: the stable variant (ρ(A) ≈ 1.02) at N = 1001"""
    n, m, kern, opts, padded = fam
    N = 1001
    prob, dZ, go = _case(n, m, N, True, _seed(n, m, N), unstable=False)
    assert np.abs(np.linalg.eigvals(prob["A"])).max() > 1.0
    Z = _solve(handle, prob, kern, opts, padded)
    with _options(handle, opts):
        g, info = ops.riccati_grad_problem(prob, Z, dZ, handle=handle)
    assert (info == 0).all(), info
    _assert_close(g, go, handle.last_kernel)


# ------------------------------------------------------------------ lqrb_riccati_grad_gains_f64
def _gain_cotangents(prob, seed):
    n, m, N = prob["n"], prob["m"], prob["N"]
    rng = np.random.default_rng(seed)
    return rng.standard_normal((B, N - 1, m, n)), rng.standard_normal((B, N - 1, m))


@pytest.mark.parametrize("lti", [False, True], ids=["ltv", "lti"])
@pytest.mark.parametrize("fam,N", GAIN_CASES)
def test_gains_call_with_every_cotangent_matches_oracle(handle, oracle_mod, fam, N, lti):
    from oracle.riccati_gain_grad import gain_grad
    n, m, kern, opts, padded = fam
    prob, dZ, gz = _case(n, m, N, lti, _seed(n, m, N))
    dK, dkff = _gain_cotangents(prob, N)
    Z = _solve(handle, prob, kern, opts, padded)
    with _options(handle, opts):
        g, info = ops.riccati_grad_gains_problem(prob, Z, dZ, dK, dkff, handle=handle)
    assert (info == 0).all(), info
    _check_kernel(handle, kern, padded)
    assert "riccati_gain_grad" in handle.last_kernel, handle.last_kernel
    gk = gain_grad(prob, dK, dkff)  # riccati_total_grad, with the cached Z part
    _assert_close(g, {k: gz[k] + gk[k] for k in NAMES}, handle.last_kernel)


@pytest.mark.parametrize("lti", [False, True], ids=["ltv", "lti"])
@pytest.mark.parametrize("fam,N", GAIN_CASES)
def test_gains_call_with_gain_cotangents_only_matches_oracle(handle, oracle_mod, fam, N, lti):
    """the gain sweep propagates P̄ through A − BK, so it needs no change on these inputs; this pins that"""
    from oracle.riccati_gain_grad import gain_grad
    n, m, kern, opts, padded = fam
    prob, _, _ = _case(n, m, N, lti, _seed(n, m, N))
    dK, dkff = _gain_cotangents(prob, N)
    with _options(handle, opts):
        g, info = ops.riccati_grad_gains_problem(prob, None, None, dK, dkff, handle=handle)
    assert (info == 0).all(), info
    assert handle.last_kernel.startswith("riccati_gain_grad"), handle.last_kernel
    go = gain_grad(prob, dK, dkff)
    assert not g["x0"].any()
    _assert_close(g, go, handle.last_kernel, names=NAMES[:-1])


@pytest.mark.parametrize("lti", [False, True], ids=["ltv", "lti"])
@pytest.mark.parametrize("fam,N", GAIN_CASES)
def test_gains_call_with_dz_only_is_bitwise_the_plain_call(handle, fam, N, lti):
    n, m, kern, opts, padded = fam
    prob = _lti(n, m, N, _seed(n, m, N)) if lti else _ltv(n, m, N, _seed(n, m, N))
    dZ = np.random.default_rng(N).standard_normal((B, N * n + (N - 1) * m))
    Z = _solve(handle, prob, kern, opts, padded)
    with _options(handle, opts):
        g1, i1 = ops.riccati_grad_problem(prob, Z, dZ, handle=handle)
        g2, i2 = ops.riccati_grad_gains_problem(prob, Z, dZ, None, None, handle=handle)
    _check_kernel(handle, kern, padded)
    assert np.array_equal(i1, i2) and (i1 == 0).all()
    for k in NAMES:
        assert np.array_equal(g1[k], g2[k]), k


# ------------------------------------------------------------------ lqrb_kkt_grad_f64 on the same LQR
@pytest.mark.parametrize("N", [101, 201])
@pytest.mark.parametrize("n,m,kern", [(4, 1, ("kkt_tpi<4,1",)), (12, 4, ("kkt_hw<12,4", "kkt_wp_dmma<12,4"))],
                         ids=["kkt_tpi-4x1", "kkt_hw_or_wp-12x4"])
def test_kkt_grad_of_the_unstable_lqr_matches_the_riccati_oracle(handle, oracle_mod, n, m, kern, N):
    """dense_kkt.riccati_as_kkt writes the LQR as a KKT system with initial-condition rows c_1 = -x0:
    lqrb_kkt_grad_f64's gA, gB, gR, gr; gQ_k, gq_k for k < N-1 and gQf, gqf at knot N-1; gx0 = -gc_1 against the
    Riccati gradient oracle"""
    from oracle import dense_kkt
    prob, dZ, go = _case(n, m, N, False, _seed(n, m, N))
    kp = dense_kkt.riccati_as_kkt(prob)
    dz, mult, info = ops.kkt_solve_problem(kp, handle=handle)
    assert (info == 0).all(), info
    gk, ginfo = ops.kkt_grad_problem(kp, dz, mult, dZ, None, handle=handle)
    assert (ginfo == 0).all(), ginfo
    assert handle.last_kernel.startswith(kern), handle.last_kernel
    g = dict(A=gk["A"], B=gk["B"], R=gk["R"], r=gk["r"], Q=gk["Q"][:, :N - 1], q=gk["q"][:, :N - 1],
             Qf=gk["Q"][:, N - 1], qf=gk["q"][:, N - 1], x0=-gk["c"][0])
    _assert_close(g, go, handle.last_kernel)


# ------------------------------------------------------------------ lqr_b200.autograd
def test_autograd_riccati_solve_with_gains_on_an_unstable_horizon(oracle_mod):
    import torch
    from lqr_b200.autograd import riccati_solve
    from oracle.riccati_gain_grad import gain_grad
    n, m, N = 6, 3, 201
    prob, _, _ = _case(n, m, N, False, _seed(n, m, N))
    t = {k: torch.tensor(prob[k], device="cuda", requires_grad=True) for k in NAMES}
    X, U, K, kff, info = riccati_solve(*(t[k] for k in NAMES), gains=True)
    assert (info == 0).all()
    rng = np.random.default_rng(5)
    W = [rng.standard_normal(tuple(a.shape)) for a in (X, U, K, kff)]
    sum((a * torch.from_numpy(w).cuda()).sum() for a, w in zip((X, U, K, kff), W)).backward()
    from oracle.riccati_grad import riccati_grad
    dZ = _z(W[0], W[1])
    gz, gk = riccati_grad(prob, dZ), gain_grad(prob, W[2], W[3])
    go = {k: gz[k] + gk[k] for k in NAMES}
    for k in ("Q", "R", "Qf"):  # riccati_solve differentiates through sym(Q), sym(R), sym(Qf)
        go[k] = 0.5 * (go[k] + np.swapaxes(go[k], -1, -2))
    _assert_close({k: t[k].grad.cpu().numpy() for k in NAMES}, go, "autograd.riccati_solve")
