"""GPU: every KKT kernel family, its kept factor and its gradient on long horizons of open-loop unstable systems,
against the extended-precision global KKT solve (oracle/dense_kkt.py).

The block elimination carries the Schur block Cp of the state from knot to knot through A_k: any error in it, and in
particular an antisymmetric rounding residue, is amplified by about |A|^2 per knot.  The tuned kernels (kkt_hw, kkt_wp,
kkt_cta) therefore symmetrise Cp exactly before they pass it on.  The generators of the other KKT tests build
A_k = I + 0.01 J (|A| ~ 1), where that amplification cannot be seen; these inputs can:
  * random_lqr_kkt's costs, rows and d, with A_k, B_k of instances 0, 2 replaced by the open-loop unstable draw of
    dare_lti_riccati (A = I + 0.3 J / sqrt(n), B ~ N(0, 1), rho(A) ~ 1.1-1.5) under 1 % relative noise per knot (LTV);
    draws whose stationary gain |K| exceeds K_BOUND are replaced (tests/unstable_lqr.py);
  * instances 1, 3 keep the benign draw, so that unstable and benign instances alternate in every batch;
  * every family of test_gpu_kkt_conditioning.py (its stage rows and dense Hessians included), with goal rows and with
    a free final state (p_N = 0, which the tuned families solve on the padded path), at N = 101, 401, 1001 (n <= 12)
    and N = 101, 201 (n >= 16).

Tolerance, per instance: the relative error of dz and of the multipliers against the truth must be
<= max(1e-10, 4 x the error of the C oracle, which runs the reference's operation order, on the same instance), the
rule of test_gpu_kkt_conditioning.py.  tests/test_oracle.py holds the C oracle to the truth on these inputs; here
every instance used is checked to be within 1e-8 of it.  Each assertion message carries the conditioning estimate
(log2 of the worst pivot ratio, lqrb_kkt_last_condition) the tuned kernel reported for every instance."""
import functools

import numpy as np
import pytest

from lqr_b200 import ops
from tests.test_gpu_kkt_conditioning import COND_BITS, FAMILIES, FAMILY_IDS, _solve, errors, make_problem, truth
from tests.test_gpu_kkt_grad import FAMILIES as GRAD_FAMILIES, _family_problem, _rel_errors, _solve_and_grad
from tests.unstable_lqr import destabilise, free_final, spectral_radii, unstable_riccati

pytestmark = pytest.mark.gpu

B = 4  # instances per batch: unstable, benign, unstable, benign
ORACLE_PIN = 1e-8  # the C oracle against the truth, on every instance used


# ------------------------------------------------------------------ inputs
def make_unstable(n, m, N, mid_p=0, hess=1, form="", goal=True, seed=0, batch=B):
    """make_problem's batch (random_lqr_kkt) with unstable dynamics on the even instances; goal=False: p_N = 0"""
    prob = destabilise(make_problem(n, m, N, batch, seed, mid_p, hess, form), seed)
    return prob if goal else free_final(prob)


def _seed(n, m, N, mid_p, hess, goal):
    return 5000 + 31 * n + 7 * m + N + mid_p + 3 * hess + (0 if goal else 1)


@functools.lru_cache(maxsize=None)
def _case(n, m, N, mid_p, hess, form, goal, seed):
    """(problem, truth, C-oracle errors), cached: the refined solve dominates every test here"""
    import oracle
    prob = make_unstable(n, m, N, mid_p, hess, form, goal, seed)
    tr = truth(prob)
    dzo, multo, infoo = oracle.kkt_solve(prob)
    assert (infoo == 0).all(), infoo.tolist()
    eo = errors(dzo, multo, tr)
    assert (eo <= ORACLE_PIN).all(), eo.tolist()
    return prob, tr, eo


def _rule(eo):
    return np.maximum(1e-10, 4.0 * eo)


def _report(e, eo, bits, prob):
    """per instance: (index, rho(A_0), kernel error, C-oracle error, conditioning bits)"""
    rho = spectral_radii(prob)
    return [(i, f"rho {rho[i]:.2f}", f"kernel {e[i]:.1e}", f"oracle {eo[i]:.1e}",
             f"bits {int(bits[i]) if bits is not None else '-'}") for i in range(len(e))]


def _prefix(kern, goal, tuned):
    """The expected kernel-name prefix: without goal rows a tuned shape is padded, and the half-warp family has no free
    final form (the warp-per-instance kernel of the same size solves it)."""
    if goal or not tuned:
        return kern
    kern = kern.replace("kkt_hw<", "kkt_wp_dmma<")
    return kern[:kern.index(",", kern.index(",") + 1) + 1]


def _horizons(n):
    return (101, 401, 1001) if n <= 12 else (101, 201)


def _gid(goal):
    return "goal" if goal else "free"


CASES = [pytest.param(f, N, goal, id=f"{i}-N{N}-{_gid(goal)}") for f, i in zip(FAMILIES, FAMILY_IDS)
         for N in _horizons(f[0]) for goal in (True, False)]
TUNED_CASES = [c for c in CASES if c.values[0][9]]

# Known misses, measured on a B200 (instance: kernel error / C-oracle error, bits).  Strict: a case that starts to pass
# must leave this list.
KNOWN_MISSES = {
    "kkt_wp_dmma<12,1-12x1-ps0-h1-N1001-free": "instance 0 (rho 1.18) not flagged: 1.1e-10 / 2e-11",
    "kkt_wp_dmma<12,2-12x2-ps0-h1-N101-goal": "instance 2 (rho 1.25) not flagged (bits 5): 1.2e-10 / 4.0e-12",
}


def _params(cases):
    """Both accuracy checks miss on a known miss: the instance is not re-solved, so the default dispatch returns the
    tuned kernel's output."""
    return [pytest.param(*c.values, id=c.id, marks=[pytest.mark.xfail(strict=True, reason=KNOWN_MISSES[c.id])]
                         if c.id in KNOWN_MISSES else []) for c in cases]


# ------------------------------------------------------------------ 1. the default dispatch
@pytest.mark.parametrize("fam,N,goal", _params(CASES))
def test_default_dispatch_on_unstable_horizons(handle, fam, N, goal):
    n, m, _, mid_p, hess, form, kern, opts, padded, tuned = fam
    prob, tr, eo = _case(n, m, N, mid_p, hess, form, goal, _seed(n, m, N, mid_p, hess, goal))
    padded = padded or (tuned and not goal)
    (dz, mult, info, _), name = _solve(handle, prob, _prefix(kern, goal, tuned), opts, padded)
    bits, resolved = handle.kkt_last_condition(B) if tuned else (None, 0)
    e = errors(dz, mult, tr)
    msg = (name, _report(e, eo, bits, prob))
    assert (info == 0).all(), (info.tolist(), msg)
    assert (e <= _rule(eo)).all(), msg
    if tuned:
        assert resolved == int((bits >= COND_BITS).sum()), (resolved, msg)
        assert ("+kkt_coop[" in name) == (resolved > 0), msg
        if not padded:  # (a padded shape mixes the pad states' unit blocks into its estimate; see DESIGN §2)
            assert (bits[1::2] < COND_BITS).all(), msg


# ------------------------------------------------------------------ 2. the estimate's promise
@pytest.mark.parametrize("fam,N,goal", _params(TUNED_CASES))
def test_unflagged_instances_meet_the_rule_without_the_re_solve(handle, fam, N, goal):
    """kkt_refine = 0: the tuned kernel's own output.  Every instance the estimate leaves below kkt_cond_bits must meet
    the rule by itself, since the default dispatch does not re-solve it."""
    n, m, _, mid_p, hess, form, kern, opts, padded, tuned = fam
    prob, tr, eo = _case(n, m, N, mid_p, hess, form, goal, _seed(n, m, N, mid_p, hess, goal))
    padded = padded or not goal
    kern = _prefix(kern, goal, tuned)
    _solve(handle, prob, kern, opts, padded)
    bits, _ = handle.kkt_last_condition(B)  # kkt_refine = 0 records no estimate: these are the default call's
    (dz, mult, info, _), name = _solve(handle, prob, kern, dict(opts, kkt_refine=0), padded)
    assert "+kkt_coop" not in name, name
    e = errors(dz, mult, tr)
    msg = (name, _report(e, eo, bits, prob))
    assert (info == 0).all(), (info.tolist(), msg)
    assert ((e <= _rule(eo)) | (bits >= COND_BITS)).all(), msg


# ------------------------------------------------------------------ 3. against the Riccati recursion
# one shape per kernel family: riccati_as_kkt has no goal rows, so the tuned shapes run their free-final padded form
RICCATI_SHAPES = [
    (4, 1, 1001, "kkt_tpi<4,1,", {}, False),
    (6, 3, 401, "kkt_tpi<6,3,", {}, False),
    (12, 4, 1001, "kkt_wp_dmma<12,4,", {}, True),
    (8, 2, 401, "kkt_wp_dmma<8,2,", {}, True),
    (10, 3, 401, "kkt_wp_dmma<12,4,", {}, True),
    (16, 8, 201, "kkt_cta_dmma<16,8,", {}, True),
    (64, 16, 101, "kkt_cta_dmma<64,16,", {}, True),
    (12, 4, 401, "kkt_coop<", {"kkt_variant": 2}, False),
]


@pytest.mark.parametrize("n,m,N,kern,opts,padded", RICCATI_SHAPES,
                         ids=[f"{s[3].rstrip(',')}-{s[0]}x{s[1]}-N{s[2]}" for s in RICCATI_SHAPES])
def test_unstable_lqr_as_kkt_matches_the_riccati_solutions(handle, n, m, N, kern, opts, padded):
    """dare_lti_riccati(unstable=True) with per-knot noise and affine terms (unstable_lqr.unstable_riccati),
    written as a KKT problem with initial-condition rows only (dense_kkt.riccati_as_kkt): the KKT kernel's trajectory
    equals the library's Riccati solution and the extended-precision recursion (oracle/riccati_ld.py) to 1e-9.  The
    Riccati kernels are held to SciPy's DARE on these inputs (tests/test_gpu_riccati_conditioning.py)."""
    from oracle import dense_kkt, riccati_ld
    from tests.test_gpu_riccati_grad_stability import _z
    rp = unstable_riccati(n, m, N, B, 11 * n + m)
    kp = dense_kkt.riccati_as_kkt(rp)
    (dz, _, info, _), name = _solve(handle, kp, kern, opts, padded)
    assert (info == 0).all(), (info.tolist(), name)
    bits = handle.kkt_last_condition(rp["x0"].shape[0])[0] if padded else None
    X, U, _, _, rinfo = ops.riccati_solve_problem(rp, want_gains=False, handle=handle)
    assert (rinfo == 0).all(), rinfo
    Xl, Ul, _, _, linfo = riccati_ld.riccati(rp)
    assert (linfo == 0).all()
    Zr, Zl = _z(X, U), _z(np.asarray(Xl, dtype=np.float64), np.asarray(Ul, dtype=np.float64))
    rel = lambda a, b: np.linalg.norm(a - b, axis=1) / np.linalg.norm(b, axis=1)  # noqa: E731
    er, el = rel(dz, Zr), rel(dz, Zl)
    msg = (name, [f"{a:.1e}/{b:.1e}" for a, b in zip(er, el)], None if bits is None else bits.tolist())
    assert (er <= 1e-9).all() and (el <= 1e-9).all(), msg


# ------------------------------------------------------------------ 4. the kept factor
def _new_rhs(prob, seed):
    """the same matrices with fresh q, r, d, c"""
    rng = np.random.default_rng(seed)
    return dict(prob, q=rng.standard_normal(prob["q"].shape), r=rng.standard_normal(prob["r"].shape),
                d=0.1 * rng.standard_normal(prob["d"].shape),
                c=[0.1 * rng.standard_normal(ck.shape) for ck in prob["c"]])


@functools.lru_cache(maxsize=None)
def _factor_case(n, m, N, mid_p):
    import oracle
    prob = make_unstable(n, m, N, mid_p, 1, "", True, seed=_seed(n, m, N, mid_p, 1, True) + 1)
    out = []
    for rhs in (prob, _new_rhs(prob, n + N)):
        tr = truth(rhs)
        dzo, multo, infoo = oracle.kkt_solve(rhs)
        assert (infoo == 0).all()
        eo = errors(dzo, multo, tr)
        assert (eo <= ORACLE_PIN).all(), eo.tolist()
        out.append((rhs, tr, eo))
    return out


@pytest.mark.parametrize("n,m,N,mid_p", [(4, 1, 1001, 0), (12, 4, 401, 0), (10, 3, 401, 1)])
def test_kept_factor_on_unstable_horizons(handle, n, m, N, mid_p):
    """lqrb_kkt_factor_f64 once, lqrb_kkt_solve_factored_f64 for the problem's own right-hand side and a fresh one
    (kkt_coop's factor and substitution phases), each under the rule against its truth."""
    cases = _factor_case(n, m, N, mid_p)
    f = ops.kkt_flatten(cases[0][0])
    b, p, hm = f["batch"], f["p"], f["hess_mode"]
    info = np.zeros(b, dtype=np.int32)
    ops.kkt_factor(handle, n, m, N, b, p, hm, 0, f["Q"], f["R"], f["Hux"], f["A"], f["B"], f["D2"], f["C"], info)
    assert (info == 0).all(), info.tolist()
    for j, (rhs, tr, eo) in enumerate(cases):
        g = ops.kkt_flatten(rhs)
        dz, mult = np.zeros((b, tr[0][0].size)), np.zeros((b, tr[0][1].size))
        ops.kkt_solve_factored(handle, n, m, N, b, p, hm, False, 0, g["q"], g["r"], g["d"], g["c"], dz, mult, None,
                               info)
        assert (info == 0).all(), (j, info.tolist())
        e = errors(dz, mult, tr)
        assert (e <= _rule(eo)).all(), (j, handle.last_kernel, _report(e, eo, None, rhs))


# ------------------------------------------------------------------ 5. the gradient
def _adjoint_problem(prob, dzb, mb):
    """the KKT problem whose solve is the adjoint one: g := dz_bar, [c; d] := mult_bar (oracle/kkt_grad.py)"""
    n, m, N = prob["n"], prob["m"], prob["N"]
    b = dzb.shape[0]
    p = [int(x) for x in prob["p"]]
    q, r, d = np.zeros((b, N, n)), np.zeros((b, N - 1, m)), np.zeros((b, N - 1, n))
    c, off = [], 0
    for k in range(N):
        q[:, k] = dzb[:, k * (n + m):k * (n + m) + n]
        if k < N - 1:
            r[:, k] = dzb[:, k * (n + m) + n:(k + 1) * (n + m)]
        c.append(mb[:, off:off + p[k]])
        off += p[k]
        if k < N - 1:
            d[:, k] = mb[:, off:off + n]
            off += n
    return dict(prob, q=q, r=r, d=d, c=c)


def _grad_horizons(n):
    return (101, 401) if n < 16 else (101,)


GRAD_CASES = [pytest.param(fam, N, id=f"{fam}-N{N}") for fam in GRAD_FAMILIES
              for N in _grad_horizons(GRAD_FAMILIES[fam][0])]


@pytest.mark.parametrize("family,N", GRAD_CASES)
def test_kkt_grad_on_unstable_horizons(handle, oracle_mod, family, N):
    """lqrb_kkt_grad_f64 on an unstable batch of every family of test_gpu_kkt_grad.py: every output array within 1e-9
    (relative, norms over the whole batch) of oracle/kkt_grad.py.  Where the forward rule needs more than 1e-10 on any
    instance, the bound of every array is widened, for the whole batch, to 4 x the error of the same oracle built on
    the C oracle's forward and adjoint solves (the errors are batch norms, so the widening cannot be per instance)."""
    from oracle.kkt_grad import kkt_grad
    n, m, _, b, o, kern = GRAD_FAMILIES[family]
    prob = destabilise(_family_problem(n, m, N, b, o, seed=3 * n + m + N), seed=3 * n + m + N)
    dz, mult, dzb, mb, g = _solve_and_grad(handle, prob, seed=n)
    assert handle.last_kernel.startswith(kern), handle.last_kernel
    tuned = not kern.startswith(("kkt_tpi", "kkt_coop"))
    bits = handle.kkt_last_condition(b)[0].tolist() if tuned else None
    errs = _rel_errors(prob, dzb, mb, g)
    tr = truth(prob)
    dzo, multo, _ = oracle_mod.kkt_solve(prob)
    eo = errors(dzo, multo, tr)
    tol = dict.fromkeys(errs, 1e-9)
    if (4.0 * eo > 1e-10).any():
        zh, mh, _ = oracle_mod.kkt_solve(_adjoint_problem(prob, dzb, mb))
        go = kkt_grad(prob, dzb, mb, sols=[(dzo[i], multo[i], zh[i], mh[i]) for i in range(b)])
        for k, err in _rel_errors(prob, dzb, mb, go).items():
            tol[k] = max(tol[k], 4.0 * err)
    bad = {k: f"{e:.1e} > {tol[k]:.1e}" for k, e in errs.items() if not e <= tol[k]}
    assert not bad, (handle.last_kernel, bad, f"rho {spectral_radii(prob).round(2).tolist()}", f"bits {bits}",
                     f"forward oracle {eo.tolist()}")
