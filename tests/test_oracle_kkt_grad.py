"""The gradient oracle of the constrained KKT solve (oracle/kkt_grad.py) against central finite differences of the
refined dense solve, element by element for every input, on small problems: the three Hessian modes, stage rows
(uniform and a different count per knot), an explicit D2 and a free final state (CPU only)."""
import copy

import numpy as np
import pytest

from lqr_b200 import problems
from oracle import dense_kkt
from oracle.kkt_grad import kkt_grad

H = 1e-6
SYMMETRIC = ("Q", "R")


def _ragged(prob, seed, hi):
    """a random number (0..hi) of the stage rows on every interior knot"""
    rng = np.random.default_rng(seed)
    p = prob["p"].copy()
    for k in range(1, prob["N"] - 1):
        p[k] = int(rng.integers(0, hi + 1))
        prob["C"][k] = prob["C"][k][:, :p[k]]
        prob["c"][k] = prob["c"][k][:, :p[k]]
    prob["p"] = p
    return prob


def _free_final(prob):
    prob["p"] = prob["p"].copy()
    prob["p"][-1] = 0
    prob["C"][-1] = np.zeros((1, 0, prob["n"]))
    prob["c"][-1] = np.zeros((1, 0))
    return prob


def _leaves(prob):
    """(key, knot or None, instance-0 array) of every differentiable input"""
    for k in ("Q", "R", "Hux", "q", "r", "A", "B", "d"):
        if prob.get(k) is not None:
            yield k, None, prob[k][0]
    for k in ("D2", "C", "c"):
        if prob.get(k) is not None:
            for j, blk in enumerate(prob[k]):
                yield k, j, blk[0]


def _loss(prob, Wz, Wm):
    z, mult = dense_kkt.kkt_truth(prob, 0)
    return float(Wz @ z + Wm @ mult)


def _fd(prob, Wz, Wm):
    out = []
    for key, j, arr in _leaves(prob):
        for idx in np.ndindex(*arr.shape):
            if key in SYMMETRIC and idx[-2] > idx[-1]:
                continue
            vals = []
            for s in (1.0, -1.0):
                q = copy.deepcopy(prob)
                a = q[key][0] if j is None else q[key][j][0]
                a[idx] += s * H
                if key in SYMMETRIC and idx[-2] != idx[-1]:
                    a[idx[:-2] + (idx[-1], idx[-2])] += s * H
                vals.append(_loss(q, Wz, Wm))
            out.append((key, j, idx, (vals[0] - vals[1]) / (2 * H)))
    return out


CASES = {
    "blockdiag-stage-rows": dict(hess=1, mid_p=1),
    "dense": dict(hess=0, mid_p=1),
    "diag": dict(hess=2, mid_p=0),
    "ragged-p": dict(hess=1, mid_p=2, ragged=True),
    "explicit-D2": dict(hess=1, mid_p=0, d2x=True),
    "dense-ragged-D2-free-final": dict(hess=0, mid_p=2, ragged=True, d2x=True, free=True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_gradient_oracle_matches_finite_differences(case):
    c = CASES[case]
    n, m, N = 3, 2, 5
    prob = problems.random_lqr_kkt(n, m, N, 1, seed=4, dt=0.1, mid_p=c["mid_p"], hess_mode=c["hess"],
                                   explicit_D2=c.get("d2x", False))
    if c.get("ragged"):
        prob = _ragged(prob, 3, c["mid_p"])
    if c.get("free"):
        prob = _free_final(prob)
    NN, P = N * n + (N - 1) * m, int(np.sum(prob["p"])) + (N - 1) * n
    rng = np.random.default_rng(5)
    Wz, Wm = rng.standard_normal(NN), rng.standard_normal(P)
    g = kkt_grad(prob, Wz[None], Wm[None])
    for key, j, idx, fd in _fd(prob, Wz, Wm):
        ga = g[key] if j is None else g[key][j]
        an = ga[(0,) + idx]
        if key in SYMMETRIC and idx[-2] != idx[-1]:
            an = an + ga[(0,) + idx[:-2] + (idx[-1], idx[-2])]
        scale = max(1.0, np.abs(ga).max())
        assert abs(an - fd) <= 1e-6 * scale, (key, j, idx, an, fd)


def test_gradient_oracle_cotangent_parts_add_and_symmetric_blocks():
    """The gradient is linear in (dz_bar, mult_bar): the two halves given alone add up to both given together; the Q
    and R gradients are symmetric, and their off-diagonal part is zero under the diagonal Hessian mode."""
    n, m, N = 4, 2, 6
    for hess in (1, 2):
        prob = problems.random_lqr_kkt(n, m, N, 2, seed=9, dt=0.1, mid_p=1, hess_mode=hess)
        NN, P = N * n + (N - 1) * m, int(np.sum(prob["p"])) + (N - 1) * n
        rng = np.random.default_rng(1)
        Wz, Wm = rng.standard_normal((2, NN)), rng.standard_normal((2, P))
        both, gz, gm = kkt_grad(prob, Wz, Wm), kkt_grad(prob, Wz, None), kkt_grad(prob, None, Wm)
        for k in ("Q", "R", "q", "r", "A", "B", "d"):
            np.testing.assert_allclose(both[k], gz[k] + gm[k], rtol=1e-9, atol=1e-12)
        for k in SYMMETRIC:
            np.testing.assert_allclose(both[k], np.swapaxes(both[k], -1, -2), rtol=0, atol=1e-14)
            if hess == 2:
                off = both[k] * (1.0 - np.eye(both[k].shape[-1]))
                assert not off.any()
