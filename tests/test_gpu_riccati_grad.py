"""lqrb_riccati_grad_f64 and lqr_b200.autograd.riccati_solve on the GPU: gradients of l(Z) through the Riccati solve
against the CPU gradient oracle (oracle/riccati_grad.py: the adjoint formulas on the refined KKT solve, itself pinned
against finite differences in tests/test_oracle_riccati_grad.py) for one size of every kernel family, padded sizes,
the cooperative kernel, LTV / LTI, with and without affine terms; finite differences through the library's own
forward solve; host vs device pointers; argument errors; determinism; torch gradcheck."""

import numpy as np
import pytest

from lqr_b200 import _lib, ops, problems

pytestmark = pytest.mark.gpu

NAMES = ("A", "B", "Q", "R", "q", "r", "Qf", "qf", "x0")


@pytest.fixture
def variant(handle):
    """sets riccati_variant for one test and restores the default"""
    def set_(v):
        handle.set_option("riccati_variant", v)
    yield set_
    handle.set_option("riccati_variant", 0)


@pytest.fixture
def host_chunk(handle):
    def set_(v):
        handle.set_option("host_chunk", v)
    yield set_
    handle.set_option("host_chunk", 0)


def _solve_and_grad(handle, prob, seed=0):
    X, U, _, _, info = ops.riccati_solve_problem(prob, want_gains=False, handle=handle)
    assert (info == 0).all()
    b = X.shape[0]
    Z = np.concatenate([np.concatenate([X[:, :-1], U], axis=2).reshape(b, -1), X[:, -1]], axis=1)
    dZ = np.random.default_rng(seed).standard_normal(Z.shape)
    g, ginfo = ops.riccati_grad_problem(prob, Z, dZ, handle=handle)
    assert (ginfo == 0).all()
    return Z, dZ, g


def _check_against_oracle(prob, dZ, g, tol=1e-9):
    from oracle.riccati_grad import riccati_grad
    go = riccati_grad(prob, dZ)
    for k in NAMES:
        err = np.linalg.norm(g[k] - go[k]) / max(np.linalg.norm(go[k]), 1e-300)
        assert err <= tol, (k, err)


CASES = [(4, 1), (3, 2), (6, 3), (8, 2), (12, 4), (16, 8), (64, 16), (10, 3), (24, 6), (40, 12), (70, 5)]


@pytest.mark.parametrize("lti", [False, True])
@pytest.mark.parametrize("n,m", CASES)
def test_gradients_match_oracle(handle, oracle_mod, n, m, lti):
    N = 12 if n <= 16 else 6
    prob = problems.random_lqr_riccati(n, m, N, 3, seed=n * 7 + m, dt=0.05, lti=lti)
    _, dZ, g = _solve_and_grad(handle, prob, seed=n)
    _check_against_oracle(prob, dZ, g)


@pytest.mark.parametrize("n,m,lti", [(4, 1, False), (12, 4, True), (40, 12, False)])
def test_gradients_without_affine_terms(handle, oracle_mod, n, m, lti):
    prob = problems.random_lqr_riccati(n, m, 7, 2, seed=2, dt=0.05, lti=lti)
    prob.update(q=None, r=None, qf=None)
    _, dZ, g = _solve_and_grad(handle, prob, seed=3)
    _check_against_oracle(prob, dZ, g)


@pytest.mark.parametrize("n,m,lti", [(4, 1, False), (12, 4, True), (70, 5, False)])
def test_gradients_on_the_cooperative_kernel(handle, oracle_mod, variant, n, m, lti):
    variant(2)
    prob = problems.random_lqr_riccati(n, m, 6, 2, seed=5, dt=0.05, lti=lti)
    _, dZ, g = _solve_and_grad(handle, prob, seed=4)
    assert "riccati_coop" in handle.last_kernel and "riccati_grad" in handle.last_kernel
    _check_against_oracle(prob, dZ, g)


@pytest.mark.parametrize("batch", [1, 31, 33, 257])
def test_cartpole_batches(handle, oracle_mod, batch):
    prob = problems.riccati_cartpole_batch(batch, seed=batch, N=41)
    _, dZ, g = _solve_and_grad(handle, prob, seed=batch)
    _check_against_oracle(prob, dZ, g)


@pytest.mark.parametrize("n,m", [(64, 16), (40, 12), (70, 5)])
def test_directional_finite_difference_through_the_library(handle, n, m):
    """sum(g * D) against (l(p + hD) - l(p - hD)) / 2h with l = sum(dZ * Z) solved by the library itself"""
    N = 8
    prob = problems.random_lqr_riccati(n, m, N, 2, seed=9, dt=0.05)
    Z, dZ, g = _solve_and_grad(handle, prob, seed=1)
    rng = np.random.default_rng(2)
    D = {k: rng.standard_normal(np.shape(prob[k])) for k in NAMES}
    for k in ("Q", "R", "Qf"):
        D[k] = D[k] + np.swapaxes(D[k], -1, -2)
    h = 1e-6

    def loss(s):
        p = dict(prob, **{k: prob[k] + s * h * D[k] for k in NAMES})
        X, U, _, _, _ = ops.riccati_solve_problem(p, want_gains=False, handle=handle)
        b = X.shape[0]
        z = np.concatenate([np.concatenate([X[:, :-1], U], axis=2).reshape(b, -1), X[:, -1]], axis=1)
        return (z * dZ).sum(axis=1)
    fd = (loss(1) - loss(-1)) / (2 * h)
    an = sum((g[k] * D[k]).reshape(2, -1).sum(axis=1) for k in NAMES)
    np.testing.assert_allclose(an, fd, rtol=1e-6)


def _flat_inputs(prob, b):
    f = ops.riccati_flatten(prob)
    return f, [f[k] for k in ("A", "B", "Q", "R", "q", "r", "Qf", "qf")]


def _grad_buffers(prob, lib_like):
    return [np.zeros_like(a) for a in lib_like] + [np.zeros_like(prob["x0"])]


def test_host_and_device_pointers_agree_bitwise_over_uneven_chunks(handle, host_chunk):
    import torch
    n, m, N, b = 6, 3, 20, 100
    prob = problems.random_lqr_riccati(n, m, N, b, seed=7, dt=0.05)
    Z, dZ, g = _solve_and_grad(handle, prob, seed=7)  # host, default chunking
    f, ins = _flat_inputs(prob, b)
    host_chunk(32)  # 32 + 32 + 32 + 4 instances
    outs_h = _grad_buffers(prob, ins)
    info_h = np.zeros(b, dtype=np.int32)
    ops.riccati_grad(handle, n, m, N, b, 0, *ins, Z, dZ, *outs_h, info_h)
    dev = [torch.from_numpy(a).cuda() for a in ins]
    Zd, dZd = torch.from_numpy(Z).cuda(), torch.from_numpy(dZ).cuda()
    outs_d = [torch.zeros(a.shape, dtype=torch.float64, device="cuda") for a in outs_h]
    info_d = torch.zeros(b, dtype=torch.int32, device="cuda")
    handle.set_stream(torch.cuda.current_stream().cuda_stream or 1)  # 1 = cudaStreamLegacy (torch's default stream)
    ops.riccati_grad(handle, n, m, N, b, 0, *dev, Zd, dZd, *outs_d, info_d)
    torch.cuda.synchronize()
    handle.set_stream(None)
    for a, d in zip(outs_h, outs_d):
        assert np.array_equal(a, d.cpu().numpy())
    assert np.array_equal(np.swapaxes(outs_h[0], -1, -2), g["A"]) and np.array_equal(outs_h[8], g["x0"])


def test_null_outputs_and_batch_zero(handle):
    n, m, N, b = 4, 2, 9, 5
    prob = problems.random_lqr_riccati(n, m, N, b, seed=1, dt=0.05, lti=True)
    Z, dZ, g = _solve_and_grad(handle, prob)
    f, ins = _flat_inputs(prob, b)
    gx0 = np.zeros((b, n))
    gB = np.zeros_like(f["B"])
    ops.riccati_grad(handle, n, m, N, b, _lib.FLAG_LTI, *ins, Z, dZ, gB=gB, gx0=gx0)
    assert np.array_equal(gx0, g["x0"]) and np.array_equal(np.swapaxes(gB, -1, -2), g["B"])
    ops.riccati_grad(handle, n, m, N, 0, _lib.FLAG_LTI, *ins, Z, dZ, gx0=gx0)  # batch 0: nothing to do
    # NO_AFFINE ignores q, r, qf even when given
    p0 = dict(prob, q=None, r=None, qf=None)
    Z0, dZ0, g0 = _solve_and_grad(handle, p0)
    gq = np.zeros_like(f["q"])
    ops.riccati_grad(handle, n, m, N, b, _lib.FLAG_LTI | _lib.FLAG_NO_AFFINE, *ins, Z0, dZ0, gq=gq, gx0=gx0)
    assert np.array_equal(gq, g0["q"]) and np.array_equal(gx0, g0["x0"])


def test_argument_codes(handle):
    n, m, N, b = 3, 1, 4, 2
    prob = problems.random_lqr_riccati(n, m, N, b, seed=1)
    f, ins = _flat_inputs(prob, b)
    NN = N * n + (N - 1) * m
    Z, dZ, gx0 = np.zeros((b, NN)), np.zeros((b, NN)), np.zeros((b, n))
    L = _lib.lib()

    def rc(hp=True, n_=n, m_=m, N_=N, b_=b, flags=0, drop=None, outs=True):
        args = [_lib.ptr(a) for a in ins] + [_lib.ptr(Z), _lib.ptr(dZ)]
        if drop is not None:
            args[drop] = None
        g = [None] * 8 + [_lib.ptr(gx0) if outs else None]
        return L.lqrb_riccati_grad_f64(handle._h if hp else None, n_, m_, N_, b_, flags, *args, *g, None)
    assert rc() == 0
    assert rc(hp=False) == -1
    assert rc(n_=0) == -2 and rc(n_=129) == -2
    assert rc(m_=0) == -3 and rc(m_=n + 1) == -3
    assert rc(N_=1) == -4
    assert rc(b_=-1) == -5
    assert rc(flags=1) == -6
    for i, code in ((0, -7), (1, -8), (2, -9), (3, -10), (6, -13), (8, -15), (9, -16)):
        assert rc(drop=i) == code, code
    for i in (4, 5, 7):  # q, r, qf may be NULL
        assert rc(drop=i) == 0
    assert rc(outs=False) == -17


def test_indefinite_instance_reports_info_and_leaves_neighbours(handle):
    n, m, N, b = 6, 3, 10, 7
    prob = problems.random_lqr_riccati(n, m, N, b, seed=4, dt=0.05)
    Z, dZ, g = _solve_and_grad(handle, prob, seed=2)
    bad = {k: np.array(v, copy=True) if isinstance(v, np.ndarray) else v for k, v in prob.items()}
    bad["R"][3] = -bad["R"][3]
    gb, info = ops.riccati_grad_problem(bad, Z, dZ, handle=handle)
    assert info[3] != 0 and (np.delete(info, 3) == 0).all()
    keep = [i for i in range(b) if i != 3]
    for k in NAMES:
        assert np.array_equal(gb[k][keep], g[k][keep]), k


def test_run_to_run_determinism(handle):
    prob = problems.random_lqr_riccati(12, 4, 30, 70, seed=8, dt=0.05)
    Z, dZ, g1 = _solve_and_grad(handle, prob, seed=8)
    g2, _ = ops.riccati_grad_problem(prob, Z, dZ, handle=handle)
    for k in NAMES:
        assert np.array_equal(g1[k], g2[k]), k


@pytest.mark.parametrize("lti", [False, True])
def test_autograd_gradcheck(lti):
    import torch
    from lqr_b200.autograd import riccati_solve
    n, m, N, b = 3, 2, 5, 2
    p = problems.random_lqr_riccati(n, m, N, b, seed=6, dt=0.1, lti=lti)
    t = {k: torch.tensor(p[k], device="cuda", requires_grad=True) for k in NAMES}
    # batch-broadcast parameters: one A, one Qf for the whole batch
    t["A"] = torch.tensor(p["A"][:1], device="cuda", requires_grad=True)
    t["Qf"] = torch.tensor(p["Qf"][:1], device="cuda", requires_grad=True)
    names = list(NAMES)

    def f(*xs):
        X, U, info = riccati_solve(*xs, N=N)
        return X, U
    assert torch.autograd.gradcheck(f, tuple(t[k] for k in names), eps=1e-6, atol=1e-7, rtol=1e-6)


def test_autograd_matches_library_and_rejects_cpu(handle):
    import torch
    from lqr_b200.autograd import riccati_solve
    p = problems.random_lqr_riccati(8, 2, 15, 4, seed=12, dt=0.05)
    t = {k: torch.tensor(p[k], device="cuda", requires_grad=True) for k in NAMES}
    X, U, info = riccati_solve(*(t[k] for k in NAMES))
    assert (info == 0).all() and not info.requires_grad
    W = torch.randn(X.shape, dtype=torch.float64, device="cuda")
    (X * W).sum().backward()
    b, N, n, m = 4, 15, 8, 2
    dZ = torch.zeros(b, N * n + (N - 1) * m, dtype=torch.float64, device="cuda")
    dZ[:, :(N - 1) * (n + m)].view(b, N - 1, n + m)[:, :, :n] = W[:, :N - 1]
    dZ[:, (N - 1) * (n + m):] = W[:, N - 1]
    Z, _, _ = _solve_and_grad(handle, p)
    g, _ = ops.riccati_grad_problem(p, Z, dZ.cpu().numpy(), handle=handle)
    for k in NAMES:
        np.testing.assert_allclose(t[k].grad.cpu().numpy(), g[k], rtol=1e-11, atol=1e-13)
    with pytest.raises(TypeError):
        riccati_solve(*(torch.tensor(p[k]) for k in NAMES))


def test_autograd_calls_on_two_streams_are_ordered():
    """riccati_solve calls share one handle and its scratch.  A call issued on stream s2 while the previous call, on s1,
    has not even started (s1 is held by a sleep kernel) must wait for it.  Checked by the order in which the two
    streams reach their end events, which does not depend on timing, and by the values of both calls against the same
    problems solved one after the other."""
    import torch
    from lqr_b200.autograd import riccati_solve
    ps = [problems.random_lqr_riccati(12, 4, 40, 64, seed=s, dt=0.05) for s in (13, 14)]

    def leaves(p):
        return {k: torch.tensor(p[k], device="cuda", requires_grad=True) for k in NAMES}

    def run(t):
        X, U, _ = riccati_solve(*(t[k] for k in NAMES))
        (X.square().sum() + U.sum()).backward()
        return [X.detach()] + [t[k].grad for k in NAMES]
    ref = [run(leaves(p)) for p in ps]
    ins = [leaves(p) for p in ps]  # made before the streams below: a pageable copy would wait for the sleep
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    e1, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(s1):
        torch.cuda._sleep(1_000_000_000)  # about half a second of the GPU clock
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
    X, U, _ = riccati_solve(*(t[k] for k in NAMES))
    (gA,) = torch.autograd.grad(X.square().sum(), t["A"], create_graph=True)
    with pytest.raises(RuntimeError):
        gA.sum().backward()


def test_sizes_the_solve_rejects_are_rejected_by_the_gradient():
    """n = 100 has no tuned kernel and is beyond the cooperative kernel's shared memory: both calls return -2"""
    n, m, N = 100, 4, 3
    prob = problems.random_lqr_riccati(n, m, N, 1, seed=1, dt=0.05)
    with pytest.raises(_lib.LqrbError, match="code -2"):
        ops.riccati_solve_problem(prob, want_gains=False)
    NN = N * n + (N - 1) * m
    with pytest.raises(_lib.LqrbError, match="code -2"):
        ops.riccati_grad_problem(prob, np.zeros((1, NN)), np.ones((1, NN)))
