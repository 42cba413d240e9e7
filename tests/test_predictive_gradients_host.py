"""CPU checks of the predictive-gradient path: the NumPy gradient oracle against central differences of the oracle's
own prediction (one level and the multi-fidelity chain rule), bounded L-BFGS-B against SciPy bit for bit, and the
logic of LBFGSBMaximizer on a stub owner with an analytic variance surface."""
import numpy as np
import pytest
from scipy.optimize import fmin_l_bfgs_b

from multifidelity_datafusion_gps_b200 import _lbfgsb
from multifidelity_datafusion_gps_b200.adaptation_maximizers import CandidateSetMaximizer, LBFGSBMaximizer
from oracle import gpy_oracle as go
from oracle import mfgp_oracle as mo
from tests import util
from tests.gradient_oracle import central_diff, level_gradients, mf_gradients


def _normwise(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


@pytest.mark.parametrize("kind", [go.KIND_RBF, go.KIND_COMPOSITE])
@pytest.mark.parametrize("E", [1, 3, 5])
def test_level_gradients_match_central_differences(kind, E):
    d = 2
    X, Y, theta = util.random_case(7 + E, 40, d, E, kind)
    Xq = np.random.default_rng(E).uniform(size=(25, d + E))
    dmean, dvar = level_gradients(kind, X, Y, d, theta, Xq)
    res = go.inference(kind, X, Y, d, theta, form="direct", want_grad=False)

    def pred(Z, which):
        mu, var = go.posterior_predict(kind, X, d, theta, res["L"], res["alpha"], Z, include_noise=False,
                                       form="direct")
        return (mu if which == 0 else var).ravel()

    assert np.all(pred(Xq, 1) > 1e-10)          # away from the clip: the latent variance is differentiable
    assert _normwise(dmean, central_diff(lambda Z: pred(Z, 0), Xq, 1e-5)) < 1e-6
    assert _normwise(dvar, central_diff(lambda Z: pred(Z, 1), Xq, 1e-5)) < 1e-6


def _lf_2d_grad(x):
    a0, a1 = util.A2
    s0, s1 = np.sin(x[:, 0] * a0), np.sin(x[:, 1] * a1)
    c = 1.2 * np.pi * 0.1
    return np.stack([a0 * np.cos(x[:, 0] * a0) * s1 - c * np.cos(x[:, 0] * np.pi * 0.1),
                     a1 * s0 * np.cos(x[:, 1] * a1) - c * np.cos(x[:, 1] * np.pi * 0.1)], axis=1)


@pytest.mark.parametrize("lf", ["callable", "data_driven"])
@pytest.mark.parametrize("n_der", [1, 2])
def test_mf_chain_rule_matches_central_differences(lf, n_der):
    rng = np.random.RandomState(5)
    if lf == "callable":
        m = mo.OracleMFGP(2, n_der, 0.01, util.hf_2d, f_low=util.lf_2d, form="direct")
        jac = _lf_2d_grad
    else:
        lf_X = rng.uniform(size=(60, 2))
        m = mo.OracleMFGP(2, n_der, 0.01, util.hf_2d, lf_X=lf_X, lf_Y=util.lf_2d(lf_X), form="direct",
                          lf_theta=np.array([1.5, 0.4, 1e-3]))
        lfm = m.lf_model
        jac = lambda Z: level_gradients(lfm.kind, lfm.X, lfm.Y, lfm.d, lfm.theta, Z)[0]
    m.fit(rng.uniform(size=(15, 2)), theta=np.array([1.0, 0.8, 1.0, 0.5, 0.1, 0.3, 1e-3]))
    hf = m.hf_model
    Xq = np.random.default_rng(9).uniform(0.05, 0.95, size=(20, 2))
    grads = level_gradients(hf.kind, hf.X, hf.Y, hf.d, hf.theta, m.augment(Xq))
    dmean, dvar = mf_gradients(grads, Xq, m.offsets, m.tau, jac)
    assert _normwise(dmean, central_diff(lambda Z: m.predict(Z)[0].ravel(), Xq, 1e-5)) < 1e-6
    assert _normwise(dvar, central_diff(lambda Z: m.predict(Z)[1].ravel(), Xq, 1e-5)) < 1e-6


# -- bounded L-BFGS-B --------------------------------------------------------------------------------------------------
def _fun(x):
    return (float(np.sum(np.sin(3.0 * x) + 0.1 * x ** 2) - x[0] * x[1]),
            3.0 * np.cos(3.0 * x) + 0.2 * x - np.r_[x[1], x[0], np.zeros(len(x) - 2)])


CASES = [
    (np.array([0.3, -1.2, 2.0]), [(0.0, 1.0), (-0.5, None), (None, 1.5)]),      # bounds become active
    (np.array([3.0, -3.0, 0.1]), [(0.0, 1.0)] * 3),                            # x0 outside the box
    (np.array([0.5, 0.5, 0.5]), [(-2.0, 2.0)] * 3),
    (np.array([0.3, -1.2, 2.0]), None),
]


def _same(a, b):
    return (np.array_equal(a[0], b[0]) and a[1] == b[1] and a[2]["funcalls"] == b[2]["funcalls"]
            and a[2]["nit"] == b[2]["nit"] and a[2]["warnflag"] == b[2]["warnflag"])


@pytest.mark.parametrize("case", range(len(CASES)))
def test_bounded_minimize_equals_fmin_l_bfgs_b(case):
    x0, bounds = CASES[case]
    ref = fmin_l_bfgs_b(_fun, x0, bounds=bounds, maxfun=80, maxiter=80)
    assert _same(ref, _lbfgsb.minimize(_fun, x0, maxfun=80, maxiter=80, bounds=bounds))
    if bounds is None:
        assert _same(ref, _lbfgsb.minimize(_fun, x0, maxfun=80, maxiter=80))


def test_bounded_lockstep_equals_fmin_l_bfgs_b():
    bounds = [(0.0, 1.0), (-0.5, 0.7), (-1.0, 1.5)]
    x0s = [np.array([0.3, -1.2, 2.0]), np.array([3.0, -3.0, 0.1]), np.array([0.5, 0.5, 0.5])]
    out = _lbfgsb.minimize_lockstep(lambda xs: [_fun(x) for x in xs], x0s, maxfun=80, maxiter=80, bounds=bounds)
    for x0, got in zip(x0s, out):
        assert _same(fmin_l_bfgs_b(_fun, x0, bounds=bounds, maxfun=80, maxiter=80), got)


# -- LBFGSBMaximizer on a stub owner -----------------------------------------------------------------------------------
class _StubOwner:
    """Variance surface v(x) = 0.1 + exp(-|x - c|^2 / w) with an analytic gradient."""

    def __init__(self, c, w=0.2):
        self.c, self.w = np.asarray(c, dtype=np.float64), w
        self.batch_calls = 0

    def _v(self, X):
        return 0.1 + np.exp(-np.sum((X - self.c) ** 2, axis=1) / self.w)

    def predict(self, X):
        X = np.atleast_2d(X)
        return np.zeros((len(X), 1)), self._v(X)[:, None]

    def variance_and_gradient(self, X):
        e = self._v(X) - 0.1
        return self._v(X), (-2.0 / self.w) * e[:, None] * (X - self.c)

    def acquisition_batch(self, cands, q, distributed=False):
        self.batch_calls += 1
        v = self._v(cands)
        idx = np.argsort(-v, kind="stable")[:q]
        return idx, v[idx]


def test_maximizer_finds_the_in_box_maximum():
    owner = _StubOwner([0.37, 0.81])
    mx = LBFGSBMaximizer(n_candidates=200, n_starts=4)
    x, fopt = mx.maximize(owner.predict, np.zeros(2), np.ones(2))
    assert np.max(np.abs(x - owner.c)) < 1e-4
    assert fopt == -owner.predict(x[None])[1][0, 0]
    assert owner.batch_calls == 1 and mx.last_rounds >= 1


def test_maximizer_respects_the_bounds_and_never_loses_to_start_0():
    owner = _StubOwner([1.3, -0.2])                # maximum outside the box: the answer sits on its corner
    lb, ub = np.zeros(2), np.ones(2)
    mx = LBFGSBMaximizer(n_candidates=300, n_starts=8)
    x, fopt = mx.maximize(owner.predict, lb, ub)
    assert np.all(x >= lb) and np.all(x <= ub)
    assert np.allclose(x, [1.0, 0.0], atol=1e-6)
    start0 = mx.candidates[mx.last_index]
    assert -fopt >= owner.predict(start0[None])[1][0, 0]


def test_foreign_callable_falls_back_to_the_candidate_argmax():
    owner = _StubOwner([0.37, 0.81])
    foreign = lambda X: owner.predict(X)           # not a bound method of an owner
    a = LBFGSBMaximizer(n_candidates=500, seed=3).maximize(foreign, np.zeros(2), np.ones(2))
    b = CandidateSetMaximizer(n_candidates=500, seed=3).maximize(foreign, np.zeros(2), np.ones(2))
    assert np.array_equal(a[0], b[0]) and a[1] == b[1]
    assert owner.batch_calls == 0


def test_n_starts_is_checked():
    with pytest.raises(ValueError):
        LBFGSBMaximizer(n_starts=0)
    with pytest.raises(ValueError):
        LBFGSBMaximizer(n_starts=65)
