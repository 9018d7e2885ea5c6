"""GPU parity of the Dubins SQP line search, iteration by iteration, against the oracle's loop
(oracle/sqp_dubins.py, src/sqp.jl:72-94): the alpha = 1 test, the second-order-correction solve and trial, back-tracking
through alpha = rho^1..rho^9 and the convergence freeze, on every device path:

  fused          dubins_sqp_step_kernel + dubins_kkt_fused_kernel<SOC> + dubins_linesearch_kernel<true> (default)
  prefetch       the same with dubins_sqp_step_pf_kernel, the cp.async prefetch ring (sqp_prefetch = 1)
  three_kernel   dubins_linearize_kernel -> kkt_tpi (LQRB_FLAG_SOC for the correction) -> dubins_linesearch_kernel<false>
                 (sqp_fused = 0)

The inputs are oracle/sqp_dubins.line_search_cases(): tests/test_oracle.py checks that they reach every branch and that
every decision along them is at least 1e-9 (relative) from its threshold, so the device must take the oracle's
decisions and land on its iterates to rounding.  A run with iters = k restarts from Z0 with mu = 1, so its result is
the k-th iterate of the full run."""
import contextlib
import functools

import numpy as np
import pytest

from lqr_b200.sqp import DubinsSQP

pytestmark = pytest.mark.gpu

PATHS = {"fused": {}, "prefetch": {"sqp_prefetch": 1}, "three_kernel": {"sqp_fused": 0}}
DEFAULTS = {"sqp_fused": 1, "sqp_prefetch": 0}


def _cases():
    from oracle import sqp_dubins as S
    return S.line_search_cases()


CASES = list(_cases())


@functools.lru_cache(maxsize=None)
def _oracle(name):
    """(Z0, x0, xf, o) and the traced oracle run of a case."""
    from oracle import sqp_dubins as S
    Z0, x0, xf, o = _cases()[name]
    return (Z0, x0, xf, o), S.solve(Z0, x0, xf, o, trace=True)


@contextlib.contextmanager
def _path(handle, path):
    try:
        for k, v in PATHS[path].items():
            handle.set_option(k, v)
        yield
    finally:
        for k, v in DEFAULTS.items():
            handle.set_option(k, v)


def _run(handle, path, Z0, x0, xf, o, iters):
    N = o["N"]
    s = DubinsSQP(x0, xf, N=N, tf=o["dt"] * (N - 1), Q=o["q_diag"], R=o["r_diag"], Qf=o["qf_diag"], iters=iters,
                  eps_p=o["eps_p"], eps_d=o["eps_d"], handle=handle)
    assert s.opts["dt"] == o["dt"]
    s.solve_(Z0)
    if path == "three_kernel":
        assert handle.last_kernel.startswith("kkt_tpi<3,2"), handle.last_kernel
    else:  # the name is set by the step launch; the prefetching kernel reports the same family
        assert handle.last_kernel.startswith("dubins_sqp_step"), handle.last_kernel
    return s


def _rel_rows(a, b):
    return np.linalg.norm(a - b, axis=1) / np.maximum(np.linalg.norm(b, axis=1), 1e-300)


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("case", CASES)
def test_line_search_iterates_match_oracle(handle, oracle_mod, case, path):
    """Every iterate k = 1..10 of every instance within 1e-9 of the oracle's Z_k; the per-instance iteration count
    and the running KKT-solve count (which pins the iterations where the batch-wide SOC solve runs) exactly equal;
    feas_p / feas_d at the end as tight as the full-step test."""
    from oracle import sqp_dubins as S
    (Z0, x0, xf, o), (Zo, fpo, fdo, ito, solves_o, tr) = _oracle(case)
    with _path(handle, path):
        for k in range(1, o["iters"] + 1):
            s = _run(handle, path, Z0, x0, xf, o, k)
            err = _rel_rows(s.Z, tr["Z"][k - 1])
            assert err.max() <= 1e-9, (k, int(err.argmax()), err.max(), tr["branch"][:k, err.argmax()].tolist())
            assert np.array_equal(s.iters, (tr["branch"][:k] != S.BR_FROZEN).sum(0)), k
            assert s.kkt_solves == tr["kkt_solves"][k - 1], (k, s.kkt_solves, tr["kkt_solves"][k - 1])
    assert np.array_equal(s.iters, ito) and s.kkt_solves == solves_o
    assert np.allclose(s.feas_p, fpo, rtol=1e-4, atol=1e-12) and np.allclose(s.feas_d, fdo, rtol=1e-4, atol=1e-10)


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("case", [c for c in CASES if c in ("n6", "n3_b33", "n4_b65", "n5_b1", "n3_far_start")])
def test_converged_instances_stay_frozen(handle, oracle_mod, case, path):
    """An instance the oracle finds converged before iteration j + 1 (after j steps) returns the bit-identical iterate
    for every budget k >= j, and iters == j."""
    from oracle import sqp_dubins as S
    (Z0, x0, xf, o), (_, _, _, ito, _, tr) = _oracle(case)
    frozen = (tr["branch"] == S.BR_FROZEN).any(0)
    assert frozen.any()
    runs = {}
    with _path(handle, path):
        for k in range(int(ito[frozen].min()), o["iters"] + 1):
            s = _run(handle, path, Z0, x0, xf, o, k)
            runs[k] = (s.Z.copy(), s.iters.copy())
    for i in np.flatnonzero(frozen):
        j = int(ito[i])
        for k in range(j, o["iters"] + 1):
            assert runs[k][1][i] == j, (i, j, k)
            assert np.array_equal(runs[k][0][i], runs[j][0][i]), (i, j, k)


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("where", ["xf", "Z0"])
@pytest.mark.parametrize("case", ["n11_far_goal", "n4_b65"])
def test_nan_instance_is_isolated(handle, oracle_mod, case, where, path):
    """A NaN in one instance's goal or initial guess changes no bit of any other instance's Z, feas_p, feas_d or iters.

    The NaN instance's merit is NaN, so every comparison is false: it needs the SOC solve and runs the stage loop to
    trial 10 in every iteration, never accepts a step (Z is returned as given, NaN included), never converges
    (iters = the budget) and reports feas_d = NaN.  feas_p is the largest of its constraint values that are not NaN:
    the device reduces them with fmax, which skips a NaN operand."""
    from oracle import sqp_dubins as S
    (Z0, x0, xf, o), _ = _oracle(case)
    b, bad = Z0.shape[0], 3
    Zb, xfb = Z0.copy(), xf.copy()
    if where == "xf":
        xfb[bad, 1] = np.nan
    else:
        Zb[bad, 2 * 5 + 4] = np.nan  # omega on knot 2
    with _path(handle, path):
        ref = _run(handle, path, Z0, x0, xf, o, o["iters"])
        s = _run(handle, path, Zb, x0, xfb, o, o["iters"])
    keep = np.arange(b) != bad
    assert np.array_equal(s.Z[keep], ref.Z[keep])
    for a in ("feas_p", "feas_d", "iters"):
        assert np.array_equal(getattr(s, a)[keep], getattr(ref, a)[keep]), a
    assert np.array_equal(s.Z[bad], Zb[bad], equal_nan=True)
    assert s.iters[bad] == o["iters"]
    assert s.kkt_solves == 2 * b * o["iters"]
    assert np.isnan(s.feas_d[bad])
    with np.errstate(invalid="ignore"):
        c1, d, cN = S.constraints(Zb[bad:bad + 1], x0[bad:bad + 1], xfb[bad:bad + 1], o)
    fp = np.nanmax(np.abs(np.concatenate([c1.ravel(), d.ravel(), cN.ravel()])))
    assert np.isfinite(s.feas_p[bad]) and np.isclose(s.feas_p[bad], fp, rtol=1e-12, atol=1e-15), (s.feas_p[bad], fp)
