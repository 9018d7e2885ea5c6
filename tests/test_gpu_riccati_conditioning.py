"""GPU: every Riccati kernel family on ill-conditioned control blocks Muu = R + B'PB, against the extended-precision
recursion (oracle/riccati_ld.py).

riccati_cta_dmma applies Muu^-1 by multiplication (Gauss-Jordan without pivoting) and riccati_dmma factors Muu in
every lane of a quad, where the reference factors it once (chol_solve!).  The generators the other Riccati tests use
keep Muu ~ R well conditioned, so these inputs are built here:
  * the cost rescalings of the KKT conditioning grid, applied to Q, Qf and R;
  * near-parallel cheap actuators: B[..., j] = B[..., 0] + c B[..., j] for j >= 1 and R scaled by rs;
  * R with a large eigenvalue spread under a random rotation.
Ill-conditioned and benign instances alternate in every batch.

Tolerance, per instance: the largest relative error of X, U, K, kff against the long-double truth must be
<= max(1e-10, 4 x the error of the C oracle, which runs the reference's operation order in double, on the same
instance) — the rule of test_gpu_conditioning.py.  Where Muu itself is ill-conditioned no double-precision solver can
reach 1e-10, and the second term asks the kernel to do as well as Cholesky does.

The info tests fix the code the header promises, (knot + 1) * 1000 + pivot, in the caller's pivot numbering, for every
family: Muu = R_k exactly at a knot with B_k = 0, and R_k indefinite at a chosen potrf pivot."""
import contextlib

import numpy as np
import pytest

from lqr_b200 import ops, problems
from oracle import riccati_ld
from tests.test_gpu_conditioning import SCALES

pytestmark = pytest.mark.gpu

# (n, m, N, expected kernel-name prefix, options, padded)
FAMILIES = [
    (4, 1, 40, "riccati_tpi<4,1>", {}, False),
    (6, 3, 40, "riccati_tpi<6,3>", {}, False),
    *[(n, m, 40 if n == 12 else 30, f"riccati_dmma<{n},{m}>", {}, False) for n in (8, 12) for m in (1, 2, 3, 4)],
    (7, 2, 30, "riccati_dmma<8,2>", {}, True),
    (10, 3, 40, "riccati_dmma<12,3>", {}, True),
    (5, 4, 30, "riccati_dmma<8,4>", {}, True),
    (16, 8, 30, "riccati_cta_dmma<16,8>", {}, False),
    (24, 8, 20, "riccati_cta_dmma<24,8>", {}, False),
    (64, 16, 12, "riccati_cta_dmma<64,16>", {}, False),
    (7, 7, 20, "riccati_cta_dmma<16,8>", {}, True),
    (20, 6, 20, "riccati_cta_dmma<24,8>", {}, True),
    (12, 4, 40, "riccati_coop", {"riccati_variant": 2}, False),
    (10, 3, 40, "riccati_coop", {"riccati_pad": 0}, False),
]
FAMILY_IDS = [f"{f[3]}-{f[0]}x{f[1]}" + ("-padded" if f[5] else "") + ("-" + ",".join(f[4]) if f[4] else "")
              for f in FAMILIES]
DEFAULTS = {"riccati_variant": 0, "riccati_pad": 1}

PARALLEL = [(c, rs) for c in (1e-2, 1e-4, 1e-6) for rs in (1e-4, 1e-6, 1e-8)]
SPREADS = [(1e4, None), (1e8, None), (1e12, None), (1e6, (1e-4, 1e-4))]  # (spread, (c, rs) of near-parallel B too)


@contextlib.contextmanager
def _options(handle, opts):
    for k, v in opts.items():
        handle.set_option(k, v)
    try:
        yield
    finally:
        for k in opts:
            handle.set_option(k, DEFAULTS[k])


def _solve(handle, prob, kern, opts, padded):
    with _options(handle, opts):
        out = ops.riccati_solve_problem(prob, handle=handle)
    name = handle.last_kernel
    assert name.startswith(kern) and ("padded" in name) == padded, name
    return out


# ------------------------------------------------------------------ inputs
def _rotation(rng, m):
    V, _ = np.linalg.qr(rng.standard_normal((m, m)))
    return V


def _near_parallel(prob, i, c, rs):
    B = prob["B"][i]
    B[..., 1:] = B[..., :1] + c * B[..., 1:]
    prob["R"][i] *= rs


def _spread_R(prob, i, spread, rng):
    m = prob["m"]
    V = _rotation(rng, m)
    R = V @ np.diag(np.logspace(0.0, -np.log10(spread), m)) @ V.T
    prob["R"][i] = 0.5 * (R + R.T)  # broadcast over the knots of an LTV problem


def _grid(kind, n, m, N, seed, lti=False):
    """A batch of 2 J + 1 instances: benign at even positions, the J ill-conditioned variants at odd ones."""
    params = {"scales": SCALES, "parallel": PARALLEL, "spread": SPREADS}[kind]
    prob = problems.random_lqr_riccati(n, m, N, 2 * len(params) + 1, seed=seed, lti=lti)
    rng = np.random.default_rng(seed)
    for j, par in enumerate(params):
        i = 2 * j + 1
        if kind == "scales":
            qs, rs = par
            prob["Q"][i] *= qs
            prob["Qf"][i] *= qs
            prob["R"][i] *= rs
        elif kind == "parallel":
            _near_parallel(prob, i, *par)
        else:
            spread, par2 = par
            _spread_R(prob, i, spread, rng)
            if par2 is not None:
                _near_parallel(prob, i, *par2)
    return prob


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.longdouble), np.asarray(b, dtype=np.longdouble)
    nb = np.linalg.norm(np.asarray(b, dtype=np.float64))
    return float(np.linalg.norm(np.asarray(a - b, dtype=np.float64)) / max(nb, 1e-300))


def _errors(out, truth):
    return np.array([max(_rel(o[i], t[i]) for o, t in zip(out[:4], truth[:4])) for i in range(out[0].shape[0])])


# ------------------------------------------------------------------ accuracy
@pytest.mark.parametrize("kind,lti", [("scales", False), ("parallel", False), ("spread", False), ("parallel", True)])
@pytest.mark.parametrize("n,m,N,kern,opts,padded", FAMILIES, ids=FAMILY_IDS)
def test_ill_conditioned_control_block(handle, oracle_mod, n, m, N, kern, opts, padded, kind, lti):
    prob = _grid(kind, n, m, N, seed=1000 + 17 * n + m + (500 if lti else 0), lti=lti)
    out = _solve(handle, prob, kern, opts, padded)
    ref = oracle_mod.riccati(prob)
    truth = riccati_ld.riccati(prob)
    assert (truth[4] == 0).all() and (ref[4] == 0).all() and (out[4] == 0).all(), (truth[4], ref[4], out[4])
    e, eo = _errors(out, truth), _errors(ref, truth)
    bad = np.flatnonzero(e > np.maximum(1e-10, 4.0 * eo))
    assert bad.size == 0, [(int(i), f"kernel {e[i]:.2e}", f"oracle {eo[i]:.2e}") for i in bad]


# ------------------------------------------------------------------ info codes
def _indefinite(m, j, rng):
    """A symmetric R = L D L' (L unit lower triangular) whose potrf pivots are D: the first non-positive one is j."""
    L = np.eye(m) + np.tril(0.3 * rng.standard_normal((m, m)), -1)
    d = rng.uniform(0.5, 2.0, m)
    d[j] = -0.5
    R = (L * d) @ L.T
    return 0.5 * (R + R.T)


def _pivots(m):
    return sorted({0, m // 2, m - 1})


@pytest.mark.parametrize("n,m,N,kern,opts,padded", FAMILIES, ids=FAMILY_IDS)
def test_info_code_names_knot_and_pivot(handle, oracle_mod, n, m, N, kern, opts, padded):
    """B_k = 0 makes Muu = R_k exactly; R_k is indefinite at pivot j.  The kernel's code must be the oracle's, the
    first failure of the backward sweep (the largest bad knot), with j counted among the caller's controls."""
    rng = np.random.default_rng(n * 31 + m)
    cases = [(k, j) for k in (N - 2, N // 2, 0) for j in _pivots(m)]
    batch = 2 * len(cases) + 3
    prob = problems.random_lqr_riccati(n, m, N, batch, seed=7 * n + m)
    want = np.zeros(batch, dtype=np.int32)
    for c, (k, j) in enumerate(cases):
        i = 2 * c + 1
        prob["B"][i, k] = 0.0
        prob["R"][i, k] = _indefinite(m, j, rng)
        want[i] = (k + 1) * 1000 + j + 1
    # two bad knots: the later one in time is met first by the backward sweep
    i = batch - 2
    for k, j in ((3, m - 1), (N - 4, 0)):
        prob["B"][i, k] = 0.0
        prob["R"][i, k] = _indefinite(m, j, rng)
    want[i] = (N - 3) * 1000 + 1
    info = _solve(handle, prob, kern, opts, padded)[4]
    assert np.array_equal(oracle_mod.riccati(prob)[4], want)
    assert np.array_equal(riccati_ld.riccati(prob)[4], want)
    assert np.array_equal(info, want), (info.tolist(), want.tolist())


@pytest.mark.parametrize("n,m,N,kern,opts,padded", FAMILIES, ids=FAMILY_IDS)
def test_info_code_lti(handle, oracle_mod, n, m, N, kern, opts, padded):
    """LTI with B = 0: Muu = R at every knot, so the sweep fails at its first knot, N - 2."""
    rng = np.random.default_rng(n + 5 * m)
    prob = problems.random_lqr_riccati(n, m, N, 3, seed=11 * n + m, lti=True)
    j = m // 2
    prob["B"][1] = 0.0
    prob["R"][1] = _indefinite(m, j, rng)
    want = np.array([0, (N - 1) * 1000 + j + 1, 0], dtype=np.int32)
    info = _solve(handle, prob, kern, opts, padded)[4]
    assert np.array_equal(oracle_mod.riccati(prob)[4], want)
    assert np.array_equal(info, want), (info.tolist(), want.tolist())


@pytest.mark.parametrize("n,m,N,kern,opts,padded", FAMILIES, ids=FAMILY_IDS)
def test_nan_instance_is_isolated(handle, n, m, N, kern, opts, padded):
    """A NaN in one instance's R is reported by that instance only and changes no bit of any other instance."""
    prob = problems.random_lqr_riccati(n, m, N, 5, seed=13 * n + m)
    clean = _solve(handle, prob, kern, opts, padded)
    assert (clean[4] == 0).all()
    prob["R"][2, N // 2, 0, m - 1] = prob["R"][2, N // 2, m - 1, 0] = np.nan
    dirty = _solve(handle, prob, kern, opts, padded)
    assert dirty[4][2] != 0 and (np.delete(dirty[4], 2) == 0).all(), dirty[4].tolist()
    for a, b in zip(clean[:4], dirty[:4]):
        assert np.array_equal(np.delete(a, 2, axis=0), np.delete(b, 2, axis=0))
