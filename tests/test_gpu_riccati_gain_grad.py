"""lqrb_riccati_grad_gains_f64 and lqr_b200.autograd.riccati_solve(..., gains=True) on the GPU: gradients of
l(Z, K, kff) through the Riccati solve against the CPU oracles (oracle/riccati_gain_grad.py, pinned against
complex-step derivatives in tests/test_oracle_riccati_gain_grad.py, plus oracle/riccati_grad.py for the Z part) for one
shape per lane configuration and forward family; bitwise agreement with lqrb_riccati_grad_f64 without gain
cotangents; finite differences through the library's own K, kff; host vs device pointers; argument codes; an
indefinite instance; determinism; torch gradcheck and stream ordering."""

import numpy as np
import pytest

from lqr_b200 import _lib, ops, problems

pytestmark = pytest.mark.gpu

NAMES = ("A", "B", "Q", "R", "q", "r", "Qf", "qf", "x0")


@pytest.fixture
def host_chunk(handle):
    def set_(v):
        handle.set_option("host_chunk", v)
    yield set_
    handle.set_option("host_chunk", 0)


def _z(X, U):
    b = X.shape[0]
    return np.concatenate([np.concatenate([X[:, :-1], U], axis=2).reshape(b, -1), X[:, -1]], axis=1)


def _cotangents(prob, seed, which):
    n, m, N = prob["n"], prob["m"], prob["N"]
    b = prob["x0"].shape[0]
    rng = np.random.default_rng(seed)
    dZ = rng.standard_normal((b, N * n + (N - 1) * m)) if which in ("Z", "all") else None
    dK = rng.standard_normal((b, N - 1, m, n)) if which in ("gains", "all") else None
    dkff = rng.standard_normal((b, N - 1, m)) if which in ("gains", "all") else None
    return dZ, dK, dkff


# one shape per lane configuration (G = 4, 8, 16, 32; R = 1, 2, 3) and per forward family (thread per instance,
# warp tensor-core, CTA tensor-core, padded, cooperative); (84, 1) is the largest n the solve accepts
CASES = [(4, 1), (3, 2), (6, 3), (8, 2), (12, 4), (16, 8), (24, 6), (40, 12), (64, 16), (70, 5), (84, 1)]


@pytest.mark.parametrize("which", ["Z", "gains", "all"])
@pytest.mark.parametrize("lti", [False, True])
@pytest.mark.parametrize("n,m", CASES)
def test_gradients_match_oracle(handle, oracle_mod, n, m, lti, which):
    from oracle.riccati_gain_grad import riccati_total_grad
    N = 12 if n <= 16 else 5
    prob = problems.random_lqr_riccati(n, m, N, 2, seed=n * 7 + m, dt=0.05, lti=lti)
    X, U, _, _, info = ops.riccati_solve_problem(prob, handle=handle)
    assert (info == 0).all()
    dZ, dK, dkff = _cotangents(prob, n + m, which)
    g, ginfo = ops.riccati_grad_gains_problem(prob, _z(X, U), dZ, dK, dkff, handle=handle)
    assert (ginfo == 0).all()
    if which != "Z":
        assert "riccati_gain_grad" in handle.last_kernel
    go = riccati_total_grad(prob, dZ, dK, dkff)
    for k in NAMES:
        if k == "x0" and dZ is None:
            assert not g[k].any()
            continue
        err = np.linalg.norm(g[k] - go[k]) / max(np.linalg.norm(go[k]), 1e-300)
        assert err <= 1e-9, (k, err)


@pytest.mark.parametrize("n,m,lti", [(4, 1, False), (12, 4, True), (40, 12, False)])
def test_gradients_without_affine_terms(handle, oracle_mod, n, m, lti):
    from oracle.riccati_gain_grad import riccati_total_grad
    prob = problems.random_lqr_riccati(n, m, 7, 2, seed=2, dt=0.05, lti=lti)
    prob.update(q=None, r=None, qf=None)
    X, U, _, _, _ = ops.riccati_solve_problem(prob, handle=handle)
    dZ, dK, dkff = _cotangents(prob, 3, "all")
    g, _ = ops.riccati_grad_gains_problem(prob, _z(X, U), dZ, dK, dkff, handle=handle)
    go = riccati_total_grad(prob, dZ, dK, dkff)
    for k in NAMES:
        assert np.linalg.norm(g[k] - go[k]) <= 1e-9 * np.linalg.norm(go[k]), k


@pytest.mark.parametrize("n,m,lti", [(4, 1, False), (12, 4, True), (64, 16, False)])
def test_without_gain_cotangents_bitwise_equal_to_riccati_grad(handle, n, m, lti):
    prob = problems.random_lqr_riccati(n, m, 9, 5, seed=4, dt=0.05, lti=lti)
    X, U, _, _, _ = ops.riccati_solve_problem(prob, handle=handle)
    Z = _z(X, U)
    dZ, _, _ = _cotangents(prob, 1, "Z")
    g1, i1 = ops.riccati_grad_problem(prob, Z, dZ, handle=handle)
    g2, i2 = ops.riccati_grad_gains_problem(prob, Z, dZ, None, None, handle=handle)
    assert np.array_equal(i1, i2)
    for k in NAMES:
        assert np.array_equal(g1[k], g2[k]), k


@pytest.mark.parametrize("n,m,lti", [(6, 3, False), (12, 4, True), (40, 12, False)])
def test_directional_finite_difference_through_the_library(handle, n, m, lti):
    """sum(g * D) against (l(p + hD) - l(p - hD)) / 2h with l = sum(dZ Z) + sum(dK K) + sum(dkff kff) from the
    library's own forward solve"""
    N = 8
    prob = problems.random_lqr_riccati(n, m, N, 2, seed=9, dt=0.05, lti=lti)
    X, U, _, _, _ = ops.riccati_solve_problem(prob, handle=handle)
    dZ, dK, dkff = _cotangents(prob, 5, "all")
    g, _ = ops.riccati_grad_gains_problem(prob, _z(X, U), dZ, dK, dkff, handle=handle)
    rng = np.random.default_rng(2)
    D = {k: rng.standard_normal(np.shape(prob[k])) for k in NAMES}
    for k in ("Q", "R", "Qf"):
        D[k] = D[k] + np.swapaxes(D[k], -1, -2)
    h = 1e-6

    def loss(s):
        p = dict(prob, **{k: prob[k] + s * h * D[k] for k in NAMES})
        X, U, K, kff, _ = ops.riccati_solve_problem(p, handle=handle)
        b = X.shape[0]
        return ((_z(X, U) * dZ).sum(axis=1) + (K * dK).reshape(b, -1).sum(axis=1)
                + (kff * dkff).reshape(b, -1).sum(axis=1))
    fd = (loss(1) - loss(-1)) / (2 * h)
    an = sum((g[k] * D[k]).reshape(2, -1).sum(axis=1) for k in NAMES)
    np.testing.assert_allclose(an, fd, rtol=1e-6)


def _flat(prob, Z, dZ, dK, dkff):
    f = ops.riccati_flatten(prob)
    ins = [f[k] for k in ("A", "B", "Q", "R", "q", "r", "Qf", "qf")]
    return ins + [Z, dZ, ops.cm(dK), dkff]


@pytest.mark.parametrize("which", ["gains", "all"])
def test_host_and_device_pointers_agree_bitwise_over_uneven_chunks(handle, host_chunk, which):
    import torch
    n, m, N, b = 6, 3, 20, 100
    prob = problems.random_lqr_riccati(n, m, N, b, seed=7, dt=0.05)
    X, U, _, _, _ = ops.riccati_solve_problem(prob, handle=handle)
    Z = _z(X, U)
    dZ, dK, dkff = _cotangents(prob, 7, which)
    g, _ = ops.riccati_grad_gains_problem(prob, Z, dZ, dK, dkff, handle=handle)  # host, default chunking
    ins = _flat(prob, Z, dZ, dK, dkff)
    host_chunk(32)  # 32 + 32 + 32 + 4 instances
    outs_h = [np.zeros_like(a) for a in ins[:8]] + [np.zeros((b, n))]
    info_h = np.zeros(b, dtype=np.int32)
    ops.riccati_grad_gains(handle, n, m, N, b, 0, *ins, *outs_h, info_h)
    dev = [None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in ins]
    outs_d = [torch.full(a.shape, 7.0, dtype=torch.float64, device="cuda") for a in outs_h]  # overwritten, not added
    info_d = torch.full((b,), 5, dtype=torch.int32, device="cuda")
    handle.set_stream(torch.cuda.current_stream().cuda_stream or 1)  # 1 = cudaStreamLegacy (torch's default stream)
    ops.riccati_grad_gains(handle, n, m, N, b, 0, *dev, *outs_d, info_d)
    torch.cuda.synchronize()
    handle.set_stream(None)
    for a, d in zip(outs_h, outs_d):
        assert np.array_equal(a, d.cpu().numpy())
    assert np.array_equal(info_h, info_d.cpu().numpy()) and not info_h.any()
    assert np.array_equal(np.swapaxes(outs_h[0], -1, -2), g["A"]) and np.array_equal(outs_h[8], g["x0"])


def test_null_outputs_and_batch_zero(handle):
    n, m, N, b = 4, 2, 9, 5
    prob = problems.random_lqr_riccati(n, m, N, b, seed=1, dt=0.05, lti=True)
    X, U, _, _, _ = ops.riccati_solve_problem(prob, handle=handle)
    Z = _z(X, U)
    dZ, dK, dkff = _cotangents(prob, 2, "all")
    g, _ = ops.riccati_grad_gains_problem(prob, Z, dZ, dK, dkff, handle=handle)
    ins = _flat(prob, Z, dZ, dK, dkff)
    gB, gQf = np.zeros_like(ins[1]), np.zeros_like(ins[6])
    ops.riccati_grad_gains(handle, n, m, N, b, _lib.FLAG_LTI, *ins, gB=gB, gQf=gQf)
    assert np.array_equal(np.swapaxes(gB, -1, -2), g["B"]) and np.array_equal(np.swapaxes(gQf, -1, -2), g["Qf"])
    gx0 = np.ones((b, n))
    ops.riccati_grad_gains(handle, n, m, N, 0, _lib.FLAG_LTI, *ins, gx0=gx0)  # batch 0: nothing to do
    assert (gx0 == 1).all()
    ins_g = ins[:8] + [None, None] + ins[10:]
    ops.riccati_grad_gains(handle, n, m, N, b, _lib.FLAG_LTI, *ins_g, gx0=gx0)  # no dZ: gx0 = 0
    assert not gx0.any()


def test_argument_codes(handle):
    n, m, N, b = 3, 1, 4, 2
    prob = problems.random_lqr_riccati(n, m, N, b, seed=1)
    NN = N * n + (N - 1) * m
    Z, dZ = np.zeros((b, NN)), np.zeros((b, NN))
    dK, dkff = np.zeros((b, N - 1, m, n)), np.zeros((b, N - 1, m))
    ins = _flat(prob, Z, dZ, dK, dkff)
    gx0 = np.zeros((b, n))
    L = _lib.lib()

    def rc(hp=True, n_=n, m_=m, N_=N, b_=b, flags=0, drop=(), outs=True):
        args = [_lib.ptr(a) for a in ins]
        for i in drop:
            args[i] = None
        g = [None] * 8 + [_lib.ptr(gx0) if outs else None]
        return L.lqrb_riccati_grad_gains_f64(handle._h if hp else None, n_, m_, N_, b_, flags, *args, *g, None)
    assert rc() == 0
    assert rc(hp=False) == -1
    assert rc(n_=0) == -2 and rc(n_=129) == -2
    assert rc(m_=0) == -3 and rc(m_=n + 1) == -3
    assert rc(N_=1) == -4
    assert rc(b_=-1) == -5
    assert rc(flags=1) == -6 and rc(flags=_lib.FLAG_SOC) == -6
    for i, code in ((0, -7), (1, -8), (2, -9), (3, -10), (6, -13), (8, -15)):
        assert rc(drop=(i,)) == code, code
    assert rc(drop=(9, 10, 11)) == -16
    assert rc(outs=False) == -19
    for drop in ((4,), (5,), (7,), (9,), (10,), (11,), (9, 10), (9, 11), (10, 11), (8, 9)):  # optional arguments
        assert rc(drop=drop) == 0, drop


@pytest.mark.parametrize("dz", [False, True])
def test_sizes_the_solve_rejects_are_rejected(dz):
    """n = 100 has no tuned kernel and is beyond the cooperative kernel's shared memory: the solve and the gradient
    both return -2, with or without the Z part"""
    n, m, N = 100, 4, 3
    prob = problems.random_lqr_riccati(n, m, N, 1, seed=1, dt=0.05)
    with pytest.raises(_lib.LqrbError, match="code -2"):
        ops.riccati_solve_problem(prob, want_gains=False)
    NN = N * n + (N - 1) * m
    with pytest.raises(_lib.LqrbError, match="code -2"):
        ops.riccati_grad_gains_problem(prob, np.zeros((1, NN)), np.ones((1, NN)) if dz else None,
                                       np.ones((1, N - 1, m, n)), None)


@pytest.mark.parametrize("which", ["gains", "all"])
def test_indefinite_instance_reports_info_and_leaves_neighbours(handle, which):
    n, m, N, b = 6, 3, 10, 7
    prob = problems.random_lqr_riccati(n, m, N, b, seed=4, dt=0.05)
    X, U, _, _, _ = ops.riccati_solve_problem(prob, handle=handle)
    Z = _z(X, U)
    dZ, dK, dkff = _cotangents(prob, 2, which)
    g, info = ops.riccati_grad_gains_problem(prob, Z, dZ, dK, dkff, handle=handle)
    assert not info.any()
    bad = {k: np.array(v, copy=True) if isinstance(v, np.ndarray) else v for k, v in prob.items()}
    bad["R"][3] = -bad["R"][3]
    _, _, _, _, finfo = ops.riccati_solve_problem(bad, handle=handle)
    gb, info = ops.riccati_grad_gains_problem(bad, Z, dZ, dK, dkff, handle=handle)
    assert info[3] != 0 and info[3] == finfo[3] and (np.delete(info, 3) == 0).all()
    keep = [i for i in range(b) if i != 3]
    for k in NAMES:
        assert np.array_equal(gb[k][keep], g[k][keep]), k


def test_run_to_run_determinism(handle):
    prob = problems.random_lqr_riccati(12, 4, 30, 70, seed=8, dt=0.05)
    X, U, _, _, _ = ops.riccati_solve_problem(prob, handle=handle)
    dZ, dK, dkff = _cotangents(prob, 8, "all")
    g1, _ = ops.riccati_grad_gains_problem(prob, _z(X, U), dZ, dK, dkff, handle=handle)
    g2, _ = ops.riccati_grad_gains_problem(prob, _z(X, U), dZ, dK, dkff, handle=handle)
    for k in NAMES:
        assert np.array_equal(g1[k], g2[k]), k


@pytest.mark.parametrize("lti", [False, True])
def test_autograd_gradcheck(lti):
    import torch
    from lqr_b200.autograd import riccati_solve
    n, m, N, b = 3, 2, 5, 2
    p = problems.random_lqr_riccati(n, m, N, b, seed=6, dt=0.1, lti=lti)
    t = {k: torch.tensor(p[k], device="cuda", requires_grad=True) for k in NAMES}
    t["A"] = torch.tensor(p["A"][:1], device="cuda", requires_grad=True)  # batch-broadcast
    t["Qf"] = torch.tensor(p["Qf"][:1], device="cuda", requires_grad=True)

    def f(*xs):
        X, U, K, kff, info = riccati_solve(*xs, N=N, gains=True)
        return X, U, K, kff

    def f_gains(*xs):
        _, _, K, kff, _ = riccati_solve(*xs, N=N, gains=True)
        return K, kff
    xs = tuple(t[k] for k in NAMES)
    assert torch.autograd.gradcheck(f, xs, eps=1e-6, atol=1e-7, rtol=1e-6)
    assert torch.autograd.gradcheck(f_gains, xs, eps=1e-6, atol=1e-7, rtol=1e-6)


def test_autograd_gains_outputs_and_unchanged_default(handle):
    import torch
    from lqr_b200.autograd import riccati_solve
    p = problems.random_lqr_riccati(8, 2, 15, 4, seed=12, dt=0.05)
    t = {k: torch.tensor(p[k], device="cuda", requires_grad=True) for k in NAMES}
    out = riccati_solve(*(t[k] for k in NAMES))
    assert len(out) == 3
    X, U, K, kff, info = riccati_solve(*(t[k] for k in NAMES), gains=True)
    assert K.shape == (4, 14, 2, 8) and kff.shape == (4, 14, 2) and not info.requires_grad
    Xh, Uh, Kh, kffh, _ = ops.riccati_solve_problem(p, handle=handle)
    assert np.array_equal(K.detach().cpu().numpy(), Kh) and np.array_equal(kff.detach().cpu().numpy(), kffh)
    assert torch.equal(X, out[0]) and torch.equal(U, out[1])
    WK = torch.randn(K.shape, dtype=torch.float64, device="cuda")
    (K * WK).sum().backward()
    g, _ = ops.riccati_grad_gains_problem(p, None, None, WK.cpu().numpy(), None, handle=handle)
    for k in NAMES:
        np.testing.assert_allclose(t[k].grad.cpu().numpy(), g[k], rtol=1e-11, atol=1e-13)
    with pytest.raises(TypeError):
        riccati_solve(*(torch.tensor(p[k]) for k in NAMES), gains=True)


def test_autograd_calls_on_two_streams_are_ordered():
    """as test_gpu_riccati_grad's stream test, through the gains: the call on s2 waits for the call on s1"""
    import torch
    from lqr_b200.autograd import riccati_solve
    ps = [problems.random_lqr_riccati(12, 4, 40, 64, seed=s, dt=0.05) for s in (13, 14)]

    def leaves(p):
        return {k: torch.tensor(p[k], device="cuda", requires_grad=True) for k in NAMES}

    def run(t):
        X, U, K, kff, _ = riccati_solve(*(t[k] for k in NAMES), gains=True)
        (X.square().sum() + K.square().sum() + kff.sum()).backward()
        return [X.detach(), K.detach()] + [t[k].grad for k in NAMES]
    ref = [run(leaves(p)) for p in ps]
    ins = [leaves(p) for p in ps]
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    e1, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(s1):
        torch.cuda._sleep(1_000_000_000)
        out1 = run(ins[0])
        e1.record()
    with torch.cuda.stream(s2):
        out2 = run(ins[1])
        e2.record()
    torch.cuda.synchronize()
    assert e1.elapsed_time(e2) >= 0, "the call on s2 finished before the earlier call on s1"
    for got, want in zip(out1 + out2, ref[0] + ref[1]):
        assert torch.equal(got, want)


def test_autograd_has_no_double_backward():
    import torch
    from lqr_b200.autograd import riccati_solve
    p = problems.random_lqr_riccati(4, 2, 6, 2, seed=3, dt=0.1)
    t = {k: torch.tensor(p[k], device="cuda", requires_grad=True) for k in NAMES}
    _, _, K, _, _ = riccati_solve(*(t[k] for k in NAMES), gains=True)
    (gA,) = torch.autograd.grad(K.square().sum(), t["A"], create_graph=True)
    with pytest.raises(RuntimeError):
        gA.sum().backward()
