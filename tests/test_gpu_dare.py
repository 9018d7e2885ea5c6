"""lqrb_dare_f64, lqrb_dare_grad_f64 and lqr_b200.autograd.dare_solve on the GPU: P and K against the CPU oracle
(oracle/dare.py, pinned against scipy and complex-step derivatives in tests/test_oracle_dare.py) and scipy for one shape
per launch shape and size class; the DARE residual; the fixed point of every Riccati family; the gradient against the
oracle and against lqrb_riccati_grad_gains_f64 over a long horizon; failed instances inside a batch; host, device and
chunked pointers; argument codes; the torch layer."""
import ctypes as C

import numpy as np
import pytest
import scipy.linalg as sl

from lqr_b200 import _lib, ops, problems
from oracle import dare as od

pytestmark = pytest.mark.gpu

SHAPES = [(1, 1), (3, 2), (4, 1), (6, 3), (8, 4), (12, 4), (16, 8), (24, 6), (32, 8), (48, 16), (64, 16)]


def _prob(n, m, b, unstable, seed):
    return problems.dare_lti_riccati(n, m, 2, b, seed=seed, unstable=unstable)


def _rel(a, b):
    return np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)


@pytest.mark.parametrize("unstable", [False, True], ids=["stable", "unstable"])
@pytest.mark.parametrize("n,m", SHAPES)
def test_dare_matches_oracle_and_scipy(handle, n, m, unstable):
    b = 6
    prob = _prob(n, m, b, unstable, seed=10 * n + m + unstable)
    P, K, iters, info = ops.dare_problem(prob, handle=handle)
    assert (info == 0).all(), info
    assert handle.last_kernel.startswith(f"dare<G={32 if n <= 24 else 256}>"), handle.last_kernel
    tol = 1e-10 if n <= 16 else 1e-9
    for i in range(b):
        A, B, Q, R = (prob[k][i] for k in "ABQR")
        Po, Ko, steps, ok = od.dare(A, B, Q, R)
        assert ok and 1 <= iters[i] <= 16, iters[i]
        Ps = sl.solve_discrete_are(A, B, Q, R)
        Ks = od.gain(A, B, R, Ps)
        assert _rel(P[i], Po) <= tol and _rel(K[i], Ko) <= tol, (i, _rel(P[i], Po), _rel(K[i], Ko))
        assert _rel(P[i], Ps) <= tol and _rel(K[i], Ks) <= tol, (i, _rel(P[i], Ps), _rel(K[i], Ks))
        assert np.array_equal(P[i], P[i].T)
        res = np.linalg.norm(Q + A.T @ P[i] @ A - A.T @ P[i] @ B @ K[i] - P[i]) / np.linalg.norm(P[i])
        assert res <= (1e-12 if n <= 16 else 1e-10), (i, res)


@pytest.mark.parametrize("n,m,variant,kern", [(4, 1, 0, "riccati_tpi"), (12, 4, 0, "riccati_dmma"),
                                              (32, 8, 0, "riccati_cta_dmma"), (10, 3, 0, "padded"),
                                              (6, 3, 2, "riccati_coop")])
def test_riccati_with_dare_terminal_cost_is_stationary(handle, n, m, variant, kern):
    """With Qf = P the finite-horizon recursion sits at its fixed point: every K_k equals K."""
    prob = problems.dare_lti_riccati(n, m, 30, 8, seed=n, unstable=True)
    P, K, _, info = ops.dare_problem(prob, handle=handle)
    assert (info == 0).all()
    prob["Qf"] = P
    handle.set_option("riccati_variant", variant)
    try:
        _, _, Kr, _, rinfo = ops.riccati_solve_problem(prob, handle=handle)
    finally:
        handle.set_option("riccati_variant", 0)
    assert (rinfo == 0).all() and kern in handle.last_kernel, handle.last_kernel
    for i in range(8):
        err = np.max(np.abs(Kr[i] - K[i][None])) / np.max(np.abs(K[i]))
        assert err <= 1e-10, (i, err)


def _cot(n, m, b, which, seed):
    rng = np.random.default_rng(seed)
    dP = rng.standard_normal((b, n, n)) if "P" in which else None
    dK = rng.standard_normal((b, m, n)) if "K" in which else None
    return dP, dK


@pytest.mark.parametrize("which", ["P", "K", "PK"])
@pytest.mark.parametrize("n,m", [(1, 1), (4, 1), (6, 3), (12, 4), (24, 6), (32, 8), (64, 16)])
def test_gradient_matches_oracle(handle, n, m, which):
    b = 4
    prob = _prob(n, m, b, True, seed=n + m)
    P, K, _, info = ops.dare_problem(prob, handle=handle)
    assert (info == 0).all()
    dP, dK = _cot(n, m, b, which, seed=n)
    g, ginfo = ops.dare_grad_problem(prob, P, dP, dK, handle=handle)
    assert (ginfo == 0).all(), ginfo
    assert handle.last_kernel.startswith("dare_grad<G="), handle.last_kernel
    for i in range(b):
        go, _, ok = od.dare_grad(prob["A"][i], prob["B"][i], prob["R"][i], P[i], None if dP is None else dP[i],
                                 None if dK is None else dK[i])
        assert ok
        for k in "ABQR":
            assert _rel(g[k][i], go[k]) <= 1e-10, (i, k, _rel(g[k][i], go[k]))


def test_gradient_matches_long_horizon_gain_gradient(handle):
    """Two device paths: the gradient of <dK, K_0> through an LTI horizon of N = 400 knots
    (lqrb_riccati_grad_gains_f64) is that of <dK, K> through the DARE when rho(Acl) <= 0.95."""
    n, m, N = 6, 3, 400
    prob = problems.dare_lti_riccati(n, m, N, 16, seed=5)
    P, K, _, info = ops.dare_problem(prob, handle=handle)
    rho = np.array([np.abs(np.linalg.eigvals(prob["A"][i] - prob["B"][i] @ K[i])).max() for i in range(16)])
    keep = np.nonzero(rho <= 0.95)[0]
    assert len(keep) >= 8 and (info == 0).all(), rho
    prob = {k: (v[keep] if isinstance(v, np.ndarray) else v) for k, v in prob.items()}
    b = len(keep)
    dK = np.random.default_rng(1).standard_normal((b, m, n))
    dKN = np.zeros((b, N - 1, m, n))
    dKN[:, 0] = dK
    gr, rinfo = ops.riccati_grad_gains_problem(prob, None, None, dKN, None, handle=handle)
    gd, dinfo = ops.dare_grad_problem(prob, P[keep], None, dK, handle=handle)
    assert (rinfo == 0).all() and (dinfo == 0).all()
    for k in "ABQR":
        assert _rel(gd[k], gr[k]) <= 1e-9, (k, _rel(gd[k], gr[k]))


def _bad_batch(n, m):
    prob = _prob(n, m, 9, True, seed=3)
    A, B, Q, R = (prob[k].copy() for k in "ABQR")
    A2, B2, Q2, R2 = (np.insert(x, [2, 4, 6], x[:3], axis=0) for x in (A, B, Q, R))
    A2[2], B2[2] = 1.5 * np.eye(n), 0.0   # unstable A, B = 0: not stabilisable
    R2[5] = -np.eye(m)           # indefinite R
    A2[8, 0, 0] = np.nan         # NaN input
    good = np.setdiff1d(np.arange(12), [2, 5, 8])
    return dict(A=A, B=B, Q=Q, R=R), dict(A=A2, B=B2, Q=Q2, R=R2), good


@pytest.mark.parametrize("n,m", [(6, 3), (32, 8)])
def test_failed_instances_leave_the_batch_alone(handle, n, m):
    clean, bad, good = _bad_batch(n, m)
    P0, K0, it0, info0 = ops.dare_problem(clean, handle=handle)
    P1, K1, it1, info1 = ops.dare_problem(bad, handle=handle)
    assert (info0 == 0).all()
    assert info1[2] == 1 and info1[5] == 1001 and info1[8] == 1, info1
    assert (info1[good] == 0).all()
    assert np.isnan(P1[[2, 5, 8]]).all() and np.isnan(K1[[2, 5, 8]]).all()
    assert np.array_equal(P1[good], P0) and np.array_equal(K1[good], K0) and np.array_equal(it1[good], it0)
    dP, dK = _cot(n, m, 12, "PK", seed=2)
    g0, ginfo0 = ops.dare_grad_problem(clean, P0, dP[good], dK[good], handle=handle)
    g1, ginfo1 = ops.dare_grad_problem(bad, P1, dP, dK, handle=handle)
    assert (ginfo0 == 0).all() and (ginfo1[good] == 0).all() and (ginfo1[[2, 5, 8]] != 0).all(), ginfo1
    for k in "ABQR":
        assert np.array_equal(g1[k][good], g0[k]) and np.isnan(g1[k][[2, 5, 8]]).all()


def test_gradient_reports_a_non_stabilising_p(handle):
    n, m = 4, 2
    prob = _prob(n, m, 2, True, seed=4)
    prob["A"] = np.broadcast_to(1.5 * np.eye(n), (2, n, n)).copy()
    P = np.zeros((2, n, n))  # P = 0: K = 0, Acl = A is unstable
    g, info = ops.dare_grad_problem(prob, P, np.ones((2, n, n)), None, handle=handle)
    assert (info == 1).all() and np.isnan(g["A"]).all()


@pytest.mark.parametrize("n,m", [(6, 3), (48, 16)])
def test_host_device_chunked_and_repeated_runs_are_bitwise_equal(handle, n, m):
    import torch
    b = 37
    prob = _prob(n, m, b, True, seed=7)
    dP, dK = _cot(n, m, b, "PK", seed=8)
    P, K, it, info = ops.dare_problem(prob, handle=handle)
    g, ginfo = ops.dare_grad_problem(prob, P, dP, dK, handle=handle)
    assert (info == 0).all() and (ginfo == 0).all()
    handle.set_option("host_chunk", 8)
    try:
        Pc, Kc, itc, _ = ops.dare_problem(prob, handle=handle)
        gc, _ = ops.dare_grad_problem(prob, P, dP, dK, handle=handle)
    finally:
        handle.set_option("host_chunk", 0)
    P2, K2, it2, _ = ops.dare_problem(prob, handle=handle)
    assert np.array_equal(Pc, P) and np.array_equal(Kc, K) and np.array_equal(itc, it)
    assert np.array_equal(P2, P) and np.array_equal(K2, K) and np.array_equal(it2, it)
    for k in "ABQR":
        assert np.array_equal(gc[k], g[k])
    # device-resident: torch tensors in the ABI's column-major layout
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(np.swapaxes(x, -1, -2))).cuda()
    A, B, Q, R = (dev(prob[k]) for k in "ABQR")
    Pd, Kd = torch.empty(b, n, n, dtype=torch.float64, device="cuda"), torch.empty(b, n, m, dtype=torch.float64, device="cuda")
    itd, infod = (torch.empty(b, dtype=torch.int32, device="cuda") for _ in range(2))
    ops.dare(handle, n, m, b, A, B, Q, R, Pd, Kd, itd, infod)
    handle.synchronize()
    assert np.array_equal(Pd.cpu().numpy().swapaxes(-1, -2), P) and np.array_equal(Kd.cpu().numpy().swapaxes(-1, -2), K)
    assert np.array_equal(itd.cpu().numpy(), it)
    gd = [torch.empty_like(x) for x in (A, B, Q, R)]
    ops.dare_grad(handle, n, m, b, A, B, R, Pd, dev(dP), dev(dK), *gd, infod)
    handle.synchronize()
    for k, x in zip("ABQR", gd):
        assert np.array_equal(x.cpu().numpy().swapaxes(-1, -2), g[k]), k


def test_argument_codes(handle):
    L, h = _lib.lib(), handle._h
    a = np.zeros(64 * 64 * 2)
    o = np.zeros(64 * 64 * 2)
    p = lambda x: x.ctypes.data

    def fwd(n=4, m=2, b=2, A=1, B=1, Q=1, R=1, P=1, K=1):
        s = lambda f: p(a) if f else None
        return L.lqrb_dare_f64(h, n, m, b, s(A), s(B), s(Q), s(R), p(o) if P else None, p(o) if K else None, None, None)

    assert fwd(n=0) == -2 and fwd(n=65) == -2 and fwd(m=0) == -3 and fwd(m=5) == -3 and fwd(b=-1) == -4
    assert fwd(A=0) == -5 and fwd(B=0) == -6 and fwd(Q=0) == -7 and fwd(R=0) == -8 and fwd(P=0, K=0) == -9
    assert fwd(b=0) == 0
    assert L.lqrb_dare_f64(None, 4, 2, 2, p(a), p(a), p(a), p(a), p(o), None, None, None) == -1

    def bwd(n=4, m=2, b=2, A=1, B=1, R=1, P=1, dP=1, dK=1, out=1):
        s = lambda f: p(a) if f else None
        g = p(o) if out else None
        return L.lqrb_dare_grad_f64(h, n, m, b, s(A), s(B), s(R), s(P), s(dP), s(dK), g, g, g, g, None)

    assert bwd(n=0) == -2 and bwd(n=65) == -2 and bwd(m=5) == -3 and bwd(b=-1) == -4
    assert bwd(A=0) == -5 and bwd(B=0) == -6 and bwd(R=0) == -7 and bwd(P=0) == -8 and bwd(dP=0, dK=0) == -9
    assert bwd(out=0) == -11 and bwd(b=0) == 0


# ------------------------------------------------------------------ torch
def _t(x):
    import torch
    return torch.tensor(x, dtype=torch.float64, device="cuda")


def test_gradcheck_broadcast():
    import torch
    from lqr_b200.autograd import dare_solve
    prob = _prob(3, 2, 3, False, seed=11)
    A = _t(prob["A"][:1]).requires_grad_()     # broadcast over the batch
    B, Q, R = (_t(prob[k]).requires_grad_() for k in "BQR")
    f = lambda A, B, Q, R: dare_solve(A, B, Q, R)[:2]
    assert torch.autograd.gradcheck(f, (A, B, Q, R), eps=1e-6, atol=1e-6, rtol=1e-5)


def test_mpc_pipeline_matches_central_differences():
    """dare_solve -> riccati_solve(Qf=P): a loss on the trajectory and the finite-horizon gains."""
    import torch
    from lqr_b200.autograd import dare_solve, riccati_solve
    n, m, N, b = 4, 2, 12, 3
    prob = _prob(n, m, b, True, seed=12)
    base = {k: _t(prob[k]) for k in ("A", "B", "Q", "R", "x0")}
    rng = np.random.default_rng(3)
    wX, wK = _t(rng.standard_normal((b, N, n))), _t(rng.standard_normal((b, N - 1, m, n)))
    dirs = {k: _t(rng.standard_normal(v.shape)) for k, v in base.items() if k != "x0"}

    def loss(d):
        P, K, info = dare_solve(d["A"], d["B"], d["Q"], d["R"])
        X, U, Kr, kff, rinfo = riccati_solve(d["A"], d["B"], d["Q"], d["R"], None, None, P, None, d["x0"], N=N,
                                             gains=True)
        assert (info == 0).all() and (rinfo == 0).all()
        return (wX * X).sum() + (wK * Kr).sum() + (K * K).sum()

    x = {k: v.clone().requires_grad_(k != "x0") for k, v in base.items()}
    loss(x).backward()
    analytic = sum((x[k].grad * dirs[k]).sum() for k in dirs).item()
    h = 1e-6
    with torch.no_grad():
        lp = loss({k: base[k] + h * dirs[k] if k in dirs else base[k] for k in base}).item()
        lm = loss({k: base[k] - h * dirs[k] if k in dirs else base[k] for k in base}).item()
    fd = (lp - lm) / (2 * h)
    assert abs(analytic - fd) <= 1e-6 * max(1.0, abs(fd)), (analytic, fd)


def test_loss_on_p_only_and_on_k_only(handle):
    import torch
    from lqr_b200.autograd import dare_solve
    n, m, b = 6, 3, 4
    prob = _prob(n, m, b, True, seed=13)
    P0, K0, _, _ = ops.dare_problem(prob, handle=handle)
    rng = np.random.default_rng(4)
    dP, dK = rng.standard_normal((b, n, n)), rng.standard_normal((b, m, n))
    for which in ("P", "K"):
        x = {k: _t(prob[k]).requires_grad_() for k in "ABQR"}
        P, K, _ = dare_solve(*(x[k] for k in "ABQR"))
        ((P * _t(dP)).sum() if which == "P" else (K * _t(dK)).sum()).backward()
        g, _ = ops.dare_grad_problem(prob, P0, dP if which == "P" else None, dK if which == "K" else None,
                                     handle=handle)
        for k in "ABQR":
            assert _rel(x[k].grad.cpu().numpy(), g[k]) <= 1e-12, (which, k)


def test_double_backward_and_cpu_tensors_raise():
    import torch
    from lqr_b200.autograd import dare_solve
    prob = _prob(3, 1, 2, False, seed=14)
    A, B, Q, R = (_t(prob[k]).requires_grad_() for k in "ABQR")
    P, K, _ = dare_solve(A, B, Q, R)
    (gA,) = torch.autograd.grad(P.sum() + K.sum(), A, create_graph=True)
    with pytest.raises(RuntimeError):
        gA.sum().backward()
    with pytest.raises(TypeError):
        dare_solve(*(torch.tensor(prob[k]) for k in "ABQR"))
