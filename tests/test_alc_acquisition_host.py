"""Integrated-variance (ALC) acquisition without a GPU: the oracle's closed form against its definition, the scratch
size helper of the C-ABI, and the logic of ALCMaximizer on a stub owner."""
import numpy as np
import pytest

from oracle import mfgp_oracle as mo
from tests import alc_oracle
from tests import util

THETA_R = np.array([1.2, 0.9, 1e-3])
THETA_C = np.array([1.0, 0.8, 1.0, 0.5, 0.1, 0.3, 1e-3])


def _oracle_model(name):
    X_hf = np.random.RandomState(10).uniform(size=(12, 2))
    if name == "GPDF":           # RBF on d = 2 plus two delays: D = 7
        o = mo.OracleMFGP(2, 2, 0.001, util.hf_2d, f_low=util.lf_2d, use_composite_kernel=False, form="direct")
        theta = THETA_R
    elif name == "GPDFC":        # composite kernel, one delay: D = 5
        o = mo.OracleMFGP(2, 1, 0.001, util.hf_2d, f_low=util.lf_2d, use_composite_kernel=True, form="direct")
        theta = THETA_C
    else:                        # NARGP: composite kernel on [x, f_low(x)], D = 3
        o = mo.OracleMFGP(2, 0, 0.0, util.hf_2d, f_low=util.lf_2d, use_composite_kernel=True, form="direct")
        theta = THETA_C
    o.fit(X_hf, theta=theta)
    return o, theta


@pytest.mark.parametrize("name", ["GPDF", "GPDFC", "NARGP"])
def test_closed_form_equals_the_definition(name):
    o, theta = _oracle_model(name)
    hf = o.hf_model
    rng = np.random.default_rng(3)
    Xc, Xr = o.augment(rng.uniform(size=(40, 2))), o.augment(rng.uniform(size=(50, 2)))
    for w in (None, rng.uniform(size=50)):
        a = alc_oracle.closed_form(hf.kind, hf.X, hf.d, theta, Xc, Xr, w)
        b = alc_oracle.definition(hf.kind, hf.X, hf.d, theta, Xc, Xr, w)
        assert np.all(a > 0.0)
        assert np.max(np.abs(a - b)) <= 1e-10 * np.max(np.abs(a)), (name, np.max(np.abs(a - b)), np.max(a))


def test_alc_scratch_size_helper_is_pure_host_logic():
    """mfgp_alc_ws_bytes: 0 for invalid arguments; K(ref, X) and Tt_R (Rpad x npad each) plus at least one
    128-column chunk of Ks, Tt_C (npad each) and G (Rpad); monotone in C and R; the chunk capped at 1 GiB."""
    from multifidelity_datafusion_gps_b200 import _ffi
    lib = _ffi.load_library()
    f = lib.mfgp_alc_ws_bytes
    for args in ((0, 10, 10), (30, 0, 10), (30, 10, 0), (-1, 10, 10), (30, -5, 10), (30, 10, -1), (30, 10, 1 << 31)):
        assert f(*args) == 0, args
    for N, R in ((30, 1), (30, 300), (1024, 1024), (1000, 4096)):
        npad, rpad = (N + 127) // 128 * 128, (R + 127) // 128 * 128
        fixed = 2 * rpad * npad * 8
        assert f(N, 1, R) == fixed + 128 * (2 * npad + rpad) * 8
        assert f(N, 1 << 20, R) >= fixed + min(1 << 30, (1 << 20) * (2 * npad + rpad) * 8)
        assert f(N, 1 << 40, R) <= fixed + max(1 << 30, 128 * (2 * npad + rpad) * 8)
    prev = 0
    for C in (1, 127, 128, 129, 5000, 1 << 16, 1 << 20, 1 << 26):
        assert f(1024, C, 1024) >= prev
        prev = f(1024, C, 1024)
    prev = 0
    for R in (1, 128, 129, 300, 1024, 4096, 1 << 16):
        assert f(1024, 1 << 20, R) >= prev
        prev = f(1024, 1 << 20, R)


# -- ALCMaximizer on a stub owner -----------------------------------------------------------------------------------
class _Owner:
    """Stands in for a model: answers acquisition_alc with the oracle's closed form on un-augmented rows."""

    def __init__(self):
        rng = np.random.RandomState(1)
        self.X = rng.uniform(size=(8, 2))
        self.calls = []

    def predict(self, X):
        return np.zeros((len(X), 1)), np.ones((len(X), 1))

    def acquisition_alc(self, candidates, reference, weights=None, distributed=False):
        self.calls.append((candidates, reference, weights, distributed))
        a = alc_oracle.closed_form(0, self.X, 2, THETA_R, candidates, reference, weights)
        i = int(np.argmax(a))
        return i, float(a[i])


LB, UB = np.array([0.0, -1.0]), np.array([1.0, 2.0])


def test_default_reference_is_deterministic_inside_the_bounds_and_its_own_stream():
    from multifidelity_datafusion_gps_b200 import ALCMaximizer
    m1 = ALCMaximizer(n_candidates=500, n_reference=300, seed=5)
    ref = m1._reference(LB, UB)
    assert ref.shape == (300, 2) and np.all(ref >= LB) and np.all(ref <= UB)
    m2 = ALCMaximizer(n_candidates=500, n_reference=300, seed=5)
    cands2 = m2._candidates(LB, UB)                  # drawing the candidates first changes nothing
    assert np.array_equal(m2._reference(LB, UB), ref)
    assert np.array_equal(m1._candidates(LB, UB), cands2)
    from multifidelity_datafusion_gps_b200 import CandidateSetMaximizer
    assert np.array_equal(CandidateSetMaximizer(n_candidates=500, seed=5)._candidates(LB, UB), cands2)
    # not the candidates' stream: the reference rows are not the candidates' leading rows
    big = ALCMaximizer(n_candidates=300, n_reference=300, seed=5)
    assert not np.any(np.all(np.isclose(big._candidates(LB, UB)[:, None, :], ref[None, :, :]), axis=2))
    assert not np.array_equal(ALCMaximizer(n_reference=300, seed=6)._reference(LB, UB), ref)
    given = np.random.default_rng(0).uniform(size=(7, 2))
    assert np.array_equal(ALCMaximizer(reference=given)._reference(LB, UB), given)


def test_weights_are_validated():
    from multifidelity_datafusion_gps_b200 import ALCMaximizer
    ok = ALCMaximizer(n_reference=4, weights=[0.0, 1.0, 2.0, 0.5])
    assert ok.weights.dtype == np.float64 and ok.weights.shape == (4,)
    for bad in ([1.0, 1.0, 1.0], [1.0] * 5, [1.0, -1.0, 1.0, 1.0], [1.0, np.nan, 1.0, 1.0],
                [1.0, np.inf, 1.0, 1.0], [0.0] * 4, [[1.0] * 4]):
        with pytest.raises(ValueError):
            ALCMaximizer(n_reference=4, weights=bad)
    with pytest.raises(ValueError):
        ALCMaximizer(reference=np.zeros((3, 2)), weights=[1.0] * 4)
    for bad_ref in (np.zeros((0, 2)), np.zeros(3)):
        with pytest.raises(ValueError):
            ALCMaximizer(reference=bad_ref)
    with pytest.raises(ValueError):
        ALCMaximizer(n_reference=0)


def test_maximize_returns_the_best_candidate_and_the_negated_alc():
    from multifidelity_datafusion_gps_b200 import ALCMaximizer
    owner = _Owner()
    w = np.random.default_rng(2).uniform(size=64)
    mx = ALCMaximizer(n_candidates=200, n_reference=64, weights=w, seed=3, distributed=False)
    x, fopt = mx.maximize(owner.predict, LB, UB)
    cands, ref, weights, distributed = owner.calls[-1]
    assert cands is mx.candidates and ref is mx.reference and np.array_equal(weights, w) and distributed is False
    a = alc_oracle.closed_form(0, owner.X, 2, THETA_R, cands, ref, w)
    assert np.array_equal(x, cands[int(np.argmax(a))]) and fopt == -float(np.max(a)) and fopt < 0.0
    assert mx.last_index == int(np.argmax(a)) and mx.last_alc == -fopt
    X1, f1 = mx.maximize_batch(owner.predict, LB, UB, 1)
    assert X1.shape == (1, 2) and np.array_equal(X1[0], x) and f1.shape == (1,) and f1[0] == fopt


def test_batches_of_more_than_one_point_are_refused():
    from multifidelity_datafusion_gps_b200 import ALCMaximizer
    owner = _Owner()
    mx = ALCMaximizer(n_candidates=50, n_reference=16)
    for q in (2, 8):
        with pytest.raises(NotImplementedError):
            mx.maximize_batch(owner.predict, LB, UB, q)
    assert owner.calls == []


def test_a_foreign_predict_callable_is_refused():
    from multifidelity_datafusion_gps_b200 import ALCMaximizer
    mx = ALCMaximizer(n_candidates=50, n_reference=16)

    def predict(X):
        return np.zeros((len(X), 1)), np.ones((len(X), 1))

    class Plain:
        def predict(self, X):
            return predict(X)

    for f in (predict, Plain().predict):
        with pytest.raises(TypeError):
            mx.maximize(f, LB, UB)
