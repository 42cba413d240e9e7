"""GPU end-to-end tests through the reference-facing classes (NumPy in / NumPy out), mirroring the
reference's own scripts (tests/test_mfgp_adapt_2d.py, tests/test_mfgp_adapt_4d.py, tests/MFDF_tests.py)
against the CPU oracle."""
import numpy as np
import pytest

from oracle import gpy_oracle as go
from oracle import mfgp_oracle as mo
from tests import util

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg(gpu):
    import multifidelity_datafusion_gps_b200 as pkg
    return pkg


def _data(dim, seed=10, n_lf=100, n_hf=5, n_test=100):
    # tests/utils.py:11,30-35
    rs = np.random.RandomState(seed)
    X_lf = rs.uniform(size=(n_lf, dim))
    X_hf = rs.uniform(size=(n_hf, dim))
    X_test = rs.uniform(size=(n_test, dim))
    return X_lf, X_hf, X_test


THETA_C = np.array([1.0, 0.8, 1.0, 0.5, 0.1, 0.3, 1e-3])
THETA_R = np.array([1.2, 0.9, 1e-3])


def test_config1_nargp_1d_callable_lf_fixed_theta(pkg):
    # config 1: 1-D, f_low = sin 8 pi t, f_high = sin^2 8 pi t (src/data/exampleCurves1D.py:10-13)
    hf_X = np.linspace(0, 1, 10)[:, None]
    Xt = np.linspace(0, 1, 1000)[:, None]                       # src/abstractMFGP.py:288
    m = pkg.NARGP(1, util.f_high_1d, util.f_low_1d)
    m.fit(hf_X, theta=THETA_C)
    o = mo.OracleMFGP(1, 0, 0, util.f_high_1d, f_low=util.f_low_1d)
    o.fit(hf_X, theta=THETA_C)
    mean, var = m.predict(Xt)
    mu_ref, var_ref = o.predict(Xt)
    assert mean.shape == (1000, 1) and var.shape == (1000, 1)
    assert util.rel_err(mean, mu_ref) < 1e-8
    assert util.rel_err(var, var_ref, THETA_C[0] * THETA_C[2] + THETA_C[4]) < 1e-6
    assert np.isclose(m.get_mse(Xt, util.f_high_1d(Xt)), o.get_mse(Xt, util.f_high_1d(Xt)), rtol=1e-6)


def test_config1_nargp_1d_data_driven_lf(pkg):
    rs = np.random.RandomState(42)
    lf_X = rs.uniform(size=(50, 1))
    lf_Y = util.f_low_1d(lf_X)
    hf_X = np.linspace(0, 1, 10)[:, None]
    Xt = np.linspace(0, 1, 400)[:, None]
    lf_theta = np.array([1.0, 0.12, 1e-4])
    m = pkg.NARGP(1, util.f_high_1d, None, lf_X=lf_X, lf_Y=lf_Y)
    m.lf_model._set_params(lf_theta)          # fixed-theta parity: skip comparing optimiser paths
    m.fit(hf_X, theta=THETA_C)
    o = mo.OracleMFGP(1, 0, 0, util.f_high_1d, lf_X=lf_X, lf_Y=lf_Y, lf_theta=lf_theta)
    o.fit(hf_X, theta=THETA_C)
    assert util.rel_err(m.hf_model.X, o.hf_model.X) < 1e-9     # augmentation through the LF GP
    mean, var = m.predict(Xt)
    mu_ref, var_ref = o.predict(Xt)
    assert util.rel_err(mean, mu_ref) < 1e-8
    assert util.rel_err(var, var_ref, 1.1) < 1e-6
    # f_low attribute keeps the reference's contract: mean predictor of the LF GP
    assert util.rel_err(m.f_low(Xt[:9]), o.f_low(Xt[:9])) < 1e-8


@pytest.mark.parametrize("model", ["GPDF", "GPDFC"])
def test_config2_gpdf_2d_delays_fixed_theta(pkg, model):
    # tests/test_mfgp_adapt_2d.py:27: GPDF(dim=2, tau=0.001, num_derivatives=2) -> D = 7
    _, X_hf, X_test = _data(2)
    X_hf = np.vstack([X_hf, np.random.RandomState(3).uniform(size=(25, 2))])   # N_h 5 -> 30
    composite = model == "GPDFC"
    theta = THETA_C if composite else THETA_R
    cls = getattr(pkg, model)
    m = cls(2, 0.001, 2, util.hf_2d, util.lf_2d)
    m.fit(X_hf, theta=theta)
    assert m.hf_model.X.shape == (30, 7)
    o = mo.OracleMFGP(2, 2, 0.001, util.hf_2d, f_low=util.lf_2d, use_composite_kernel=composite)
    o.fit(X_hf, theta=theta)
    assert np.array_equal(m.hf_model.X, o.hf_model.X)
    mean, var = m.predict(X_test)
    mu_ref, var_ref = o.predict(X_test)
    assert util.rel_err(mean, mu_ref) < 1e-8
    assert util.rel_err(var, var_ref, 1.2) < 1e-6


def test_add_noise_refactorises_at_1e_6(pkg):
    _, X_hf, X_test = _data(2)
    m = pkg.GPDF(2, 0.001, 2, util.hf_2d, util.lf_2d, add_noise=True)
    m.fit(X_hf, theta=THETA_R)
    o = mo.OracleMFGP(2, 2, 0.001, util.hf_2d, f_low=util.lf_2d, use_composite_kernel=False, add_noise=True)
    o.fit(X_hf, theta=THETA_R)
    mean, var = m.predict(X_test)
    mu_ref, var_ref = o.predict(X_test)
    assert m.hf_model.likelihood.variance == 1e-6
    assert util.rel_err(mean, mu_ref) < 1e-7        # cond(K_y) ~ 1e6 at noise 1e-6
    assert util.rel_err(var, var_ref, 1.2) < 1e-6


def test_fit_reaches_oracle_likelihood(pkg):
    # optimiser trajectories are not comparable (global NumPy RNG, SciPy version); the achieved LML is
    np.random.seed(0)
    _, X_hf, _ = _data(2, n_hf=12)
    m = pkg.GPDF(2, 0.001, 2, util.hf_2d, util.lf_2d)
    m.fit(X_hf)
    o = mo.OracleMFGP(2, 2, 0.001, util.hf_2d, f_low=util.lf_2d, use_composite_kernel=False,
                      rng=np.random.RandomState(0))
    o.fit(X_hf)
    ours = m.hf_model.log_likelihood()
    theirs = o.hf_model.log_likelihood()
    assert ours >= theirs - 1e-6 * abs(theirs) - 1e-3
    # and the fitted theta evaluates to the same LML on the oracle.  An optimiser-chosen theta can be
    # badly conditioned (the optimiser drives the noise towards 0: cond(K_y) ~ 1e10), where neither
    # side can promise 1e-6: the bound is 1e-6 + a few cond(K_y) * eps (SURVEY.md section 7, "hard
    # parts"), and cond is part of the assertion message.
    theta = m.hf_model.param_array
    cond = np.linalg.cond(go.assemble_Ky(go.KIND_RBF, o.hf_model.X, 2, theta, form="direct"))
    tol = (1e-6 + 1e-14 * cond) * abs(ours) + 1e-9
    for form in ("direct", "gpy"):
        chk = go.inference(go.KIND_RBF, o.hf_model.X, o.hf_model.Y, 2, theta, want_grad=False, form=form)
        assert abs(chk["lml"] - ours) <= tol, (form, cond, chk["lml"], ours)


def test_adaptation_with_candidate_set_improves_mse_and_matches_oracle_argmax(pkg):
    # tests/MFDF_tests.py:10-26 asserts mse_after < mse_before; the arg-max index must be bit-exact
    np.random.seed(1)
    _, X_hf, X_test = _data(2, n_hf=6)
    cands = np.random.default_rng(0).uniform(size=(100000, 2))
    mx = pkg.CandidateSetMaximizer(candidates=cands)
    m = pkg.GPDF(2, 0.001, 2, util.hf_2d, util.lf_2d, adapt_maximizer=mx)
    m.fit(X_hf)
    Y_test = util.hf_2d(X_test)
    mse_before = m.get_mse(X_test, Y_test)
    # index parity at the fitted theta
    o = mo.OracleMFGP(2, 2, 0.001, util.hf_2d, f_low=util.lf_2d, use_composite_kernel=False)
    o.fit(X_hf, theta=m.hf_model.param_array)
    i_ref, x_ref, fopt_ref, gap = mo.candidate_argmax(o.predict, cands)
    idx, val = m.acquisition_argmax(cands)
    if gap > 1e-9:
        assert idx == i_ref
    assert abs(-val - fopt_ref) <= 1e-6 * abs(fopt_ref)
    m.adapt(5, eps=0.0)
    assert m.hf_X.shape == (11, 2) and m.adapt_steps == 5 and len(m.acquired_points) == 5
    assert m.get_mse(X_test, Y_test) < mse_before


def test_config3_nargp_4d_one_million_candidates(pkg):
    # BASELINE.json configs[2] at full size (tests/test_mfgp_adapt_4d.py:10-42): NARGP in 4-D (D = 5), 5 HF
    # points, callable lf_4d, 1 048 576 uniform candidates; the arg-max index is checked against the oracle
    # over ALL of them, bit-exact unless the top two variances tie
    _, X_hf, _ = _data(4)
    cands = np.random.default_rng(0).uniform(size=(1 << 20, 4))
    theta = np.array([1.0, 0.3, 1.0, 0.3, 0.1, 0.3, 1e-3])
    mx = pkg.CandidateSetMaximizer(candidates=cands)
    m = pkg.NARGP(4, util.hf_4d, util.lf_4d, adapt_maximizer=mx)
    m.fit(X_hf, theta=theta)
    o = mo.OracleMFGP(4, 0, 0, util.hf_4d, f_low=util.lf_4d)
    o.fit(X_hf, theta=theta)
    i_ref, x_ref, fopt_ref, gap = mo.candidate_argmax(o.predict, cands)
    idx, val = m.acquisition_argmax(cands)
    assert gap > 1e-9, "degenerate case: pick other candidates"
    assert idx == i_ref
    assert abs(-val - fopt_ref) <= 1e-6 * abs(fopt_ref)
    # through the plug-in (src/abstractMFGP.py:124-129), with the candidate set now resident on the device
    hits = getattr(m, "candidate_cache_hits", 0)
    x, fopt = m.get_input_with_highest_uncertainty(m)
    assert m.candidate_cache_hits == hits + 1 and mx.last_index == i_ref
    assert np.array_equal(x, x_ref) and fopt == -val


def test_resident_candidates_follow_the_model_state(pkg):
    # the cached augmented candidates must be rebuilt when the low-fidelity level changes, and only then
    lf_X, X_hf, _ = _data(2, n_hf=8)
    cands = np.random.default_rng(1).uniform(size=(30000, 2))
    m = pkg.NARGP(2, util.hf_2d, None, lf_X=lf_X, lf_Y=util.lf_2d(lf_X))
    m.lf_model._set_params(np.array([1.5, 0.4, 1e-3]))
    m.fit(X_hf, theta=THETA_C)
    a = m.acquisition_argmax(cands)
    assert m.acquisition_argmax(cands) == a and m.candidate_cache_hits == 1
    m.fit(np.vstack([X_hf, cands[a[0]]]), theta=THETA_C)          # HF refit: LF untouched -> still a hit
    b = m.acquisition_argmax(cands)
    assert m.candidate_cache_hits == 2 and b == m.acquisition_argmax(cands, cache=False)
    m.lf_model._set_params(np.array([1.2, 0.5, 1e-3]))            # LF change: stale rows must not be used
    m.fit(m.hf_X, theta=THETA_C)
    c = m.acquisition_argmax(cands)
    assert m.candidate_cache_hits == 2                            # a miss: the rows were rebuilt
    assert c == m.acquisition_argmax(cands, cache=False)
    cands2 = cands.copy()
    cands2[::7] = cands2[::7][:, ::-1]                            # different contents -> different key
    assert m.acquisition_argmax(cands2) == m.acquisition_argmax(cands2, cache=False)


def test_lf_level_optimize_reaches_oracle_likelihood(pkg):
    # A7 (src/abstractMFGP.py:96-104): the constructor trains the LF GP with one L-BFGS-B run from (1, 1, 1)
    # on the GPU objective; the achieved LML must not be worse than the oracle's run, and the oracle must
    # agree on the LML at the GPU's hyper-parameters (conditioning-aware bound as in
    # test_fit_reaches_oracle_likelihood: the optimiser drives the noise towards zero)
    for dim, n_lf, lf in ((1, 50, util.f_low_1d), (2, 60, util.lf_2d), (4, 100, util.lf_4d)):
        rs = np.random.RandomState(10 + dim)
        lf_X = rs.uniform(size=(n_lf, dim))
        lf_Y = lf(lf_X).reshape(-1, 1)
        m = pkg.NARGP(dim, lambda x: lf(x).reshape(-1, 1), None, lf_X=lf_X, lf_Y=lf_Y)
        o = go.OracleGPRegression(lf_X, lf_Y)
        o.optimize()
        ours, theirs = m.lf_model.log_likelihood(), o.log_likelihood()
        # both runs stop on a flat, ill-conditioned ridge (noise -> 1e-13): the oracle's own two distance forms
        # end 2.4e-6 apart on the 1-D curve, hence 1e-5 and not 1e-6
        assert ours >= theirs - 1e-5 * abs(theirs) - 1e-3, (dim, ours, theirs)
        theta = m.lf_model.param_array
        cond = np.linalg.cond(go.assemble_Ky(go.KIND_RBF, lf_X, dim, theta, form="direct"))
        chk = go.inference(go.KIND_RBF, lf_X, lf_Y, dim, theta, want_grad=False, form="direct")
        assert abs(chk["lml"] - ours) <= (1e-6 + 1e-14 * cond) * abs(ours) + 1e-9, (dim, cond, chk["lml"], ours)
        # and f_low is the trained GP's mean (src/abstractMFGP.py:104)
        Xs = rs.uniform(size=(20, dim))
        o.theta = theta.copy()
        o._post = None
        assert util.rel_err(m.f_low(Xs), o.predict(Xs)[0]) <= 1e-8 + 1e-15 * cond


def test_default_direct_maximizer_acquires_the_oracles_point(pkg):
    # the default maximizer (src/adaptation_maximizers/scipydirect_wrapper.py:16-31): original DIRECT,
    # 20 000 single-point predicts, no volume / side-length termination; same search over the oracle
    from scipy.optimize import direct
    hf_X = np.linspace(0, 1, 10)[:, None]
    m = pkg.NARGP(1, util.f_high_1d, util.f_low_1d)
    assert isinstance(m.adapt_maximizer, pkg.ScipyDirectMaximizer)
    m.fit(hf_X, theta=THETA_C)
    o = mo.OracleMFGP(1, 0, 0, util.f_high_1d, f_low=util.f_low_1d)
    o.fit(hf_X, theta=THETA_C)
    n_evals = [0]

    def f(x):
        n_evals[0] += 1
        return -float(o.predict(np.asarray(x)[None])[1][0, 0])
    ref = direct(f, [(0.0, 1.0)], eps=1e-4, maxfun=20000, maxiter=6000, locally_biased=False, vol_tol=0.0,
                 len_tol=0.0)
    x, fopt = m.get_input_with_highest_uncertainty(m)
    assert n_evals[0] >= 20000                                  # the whole budget, as scipydirect's defaults
    assert abs(fopt - ref.fun) <= 1e-6 * abs(ref.fun)
    # variance landscape has symmetric maxima: compare the acquired value, and the point when it is unique
    v_at = lambda t: float(o.predict(np.array([[t]]))[1][0, 0])
    assert abs(v_at(float(x[0])) - v_at(float(ref.x[0]))) <= 1e-6 * abs(ref.fun)


def test_f_low_probe_handles_group_only_callables_and_propagates_errors(pkg):
    X_hf = np.random.RandomState(3).uniform(size=(9, 2))
    calls = []

    def group_only(loc):                       # valid per (E, d) group only, as the reference calls it (:197)
        loc = np.asarray(loc)
        calls.append(loc.shape)
        assert loc.shape == (5, 2), "called with a stack of groups"
        return util.lf_2d(loc)

    m = pkg.GPDF(2, 0.01, 2, util.hf_2d, group_only)
    m.fit(X_hf, theta=THETA_R)
    ref = pkg.GPDF(2, 0.01, 2, util.hf_2d, util.lf_2d)
    ref.fit(X_hf, theta=THETA_R)
    assert np.array_equal(m.hf_model.X, ref.hf_model.X)

    def broken(loc):
        raise RuntimeError("bug inside the user's f_low")
    with pytest.raises(RuntimeError, match="bug inside"):
        pkg.GPDF(2, 0.01, 2, util.hf_2d, broken).fit(X_hf, theta=THETA_R)

    def not_rowwise(loc):                      # returns the right number of values for a stack, but mixes rows
        loc = np.asarray(loc)
        return np.cumsum(util.lf_2d(loc).ravel())[:, None] if len(loc) > 5 else util.lf_2d(loc)
    m3 = pkg.GPDF(2, 0.01, 2, util.hf_2d, not_rowwise)
    m3.fit(X_hf, theta=THETA_R)
    assert np.array_equal(m3.hf_model.X, ref.hf_model.X)


def test_two_threads_two_models_do_not_share_scratch(pkg):
    # one C-ABI handle and one scratch per (device, thread): concurrent predictions equal the serial ones
    import threading
    models = [_mc_models(pkg, seed=4)[0], _mc_models(pkg, n_l=140, n_h=40, seed=5)[0]]
    Xt = [np.random.default_rng(30 + i).uniform(size=(20000, 4)) for i in range(2)]
    serial = [mm.predict(x) for mm, x in zip(models, Xt)]
    out, errs = [None, None], []

    def work(i):
        try:
            for _ in range(5):
                out[i] = models[i].predict(Xt[i])
        except Exception as exc:      # surfaced below
            errs.append(exc)
    threads = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errs, errs
    for i in range(2):
        assert np.array_equal(out[i][0], serial[i][0]) and np.array_equal(out[i][1], serial[i][1])


def test_mc_without_delays_on_the_plain_rbf_kernel(pkg):
    # GPDF with num_derivatives = 0: one RBF over [x, f_low(x)] (E = 1) -- the K7 path must serve it too
    rs = np.random.RandomState(8)
    lf_X, hf_X = rs.uniform(size=(90, 2)), rs.uniform(size=(25, 2))
    lf_theta = np.array([1.5, 0.4, 1e-3])
    m = pkg.GPDF(2, 0.0, 0, util.hf_2d, None, lf_X=lf_X, lf_Y=util.lf_2d(lf_X))
    m.lf_model._set_params(lf_theta)
    m.fit(hf_X, theta=THETA_R)
    o = mo.OracleMFGP(2, 0, 0.0, util.hf_2d, lf_X=lf_X, lf_Y=util.lf_2d(lf_X), lf_theta=lf_theta,
                      use_composite_kernel=False)
    o.fit(hf_X, theta=THETA_R)
    Xt = rs.uniform(size=(300, 2))
    eps = np.random.default_rng(3).standard_normal((300, 24, 1))
    mean, var = m.predict_mc(Xt, n_samples=24, eps=eps)
    mu_ref, var_ref = o.predict_mc(Xt, eps)
    assert util.rel_err(mean, mu_ref) < 1e-8 and util.rel_err(var, var_ref, 1.2) < 1e-6


def test_mc_with_the_even_delay_pattern(pkg):
    # src/augm_iterators/even_augm_iterator.py:20-48 under MC propagation: 2*1*2 + 1 = 5 joint LF locations
    rs = np.random.RandomState(9)
    lf_X, hf_X = rs.uniform(size=(120, 2)), rs.uniform(size=(30, 2))
    lf_theta = np.array([1.5, 0.4, 1e-3])
    m = pkg.MultifidelityDataFusion("even", 2, 1, 0.05, util.hf_2d, lf_X=lf_X, lf_Y=util.lf_2d(lf_X),
                                    use_composite_kernel=True, augm_iterator="even")
    m.lf_model._set_params(lf_theta)
    m.fit(hf_X, theta=THETA_C)
    o = mo.OracleMFGP(2, 1, 0.05, util.hf_2d, lf_X=lf_X, lf_Y=util.lf_2d(lf_X), lf_theta=lf_theta,
                      offsets=mo.even_offsets(1, 2))
    o.fit(hf_X, theta=THETA_C)
    Xt = rs.uniform(size=(200, 2))
    eps = np.random.default_rng(4).standard_normal((200, 30, 5))
    mean, var = m.predict_mc(Xt, n_samples=30, eps=eps)
    mu_ref, var_ref = o.predict_mc(Xt, eps)
    assert util.rel_err(mean, mu_ref) < 1e-8 and util.rel_err(var, var_ref, 1.2) < 1e-6


def _mc_models(pkg, n_l=100, n_h=30, d=4, seed=4):
    rs = np.random.RandomState(seed)
    lf_X = rs.uniform(size=(n_l, d))
    hf_X = rs.uniform(size=(n_h, d))
    lf_theta = np.array([1.5, 0.6, 1e-3])
    th = np.array([1.0, 0.5, 1.0, 0.6, 0.1, 0.5, 1e-3])
    m = pkg.NARGP(d, util.hf_4d, None, lf_X=lf_X, lf_Y=util.lf_4d(lf_X))
    m.lf_model._set_params(lf_theta)
    m.fit(hf_X, theta=th)
    o = mo.OracleMFGP(d, 0, 0, util.hf_4d, lf_X=lf_X, lf_Y=util.lf_4d(lf_X), lf_theta=lf_theta)
    o.fit(hf_X, theta=th)
    return m, o


def test_mc_propagation_matches_oracle_with_supplied_normals(pkg):
    m, o = _mc_models(pkg)
    M, S = 500, 100
    Xt = np.random.default_rng(5).uniform(size=(M, 4))
    eps = np.random.default_rng(2).standard_normal((M, S, 1))
    mean, var = m.predict_mc(Xt, n_samples=S, eps=eps)
    mu_ref, var_ref = o.predict_mc(Xt, eps)
    assert util.rel_err(mean, mu_ref) < 1e-8
    assert util.rel_err(var, var_ref, 1.1) < 1e-6


@pytest.mark.parametrize("n_h,S", [(5, 100), (16, 9), (17, 40), (30, 7), (32, 33), (33, 100), (64, 9), (65, 100), (96, 40)])
def test_mc_propagation_across_the_fused_small_level_boundary(pkg, n_h, S):
    """N_h <= 16, <= 32 and <= 64 take the fused generator + contraction kernel (mc_small_kernel<16 / 32 / 64>), larger levels
    the general Ks + trmm_sumsq pair; ragged sample counts exercise the partial 8-column groups."""
    m, o = _mc_models(pkg, n_l=60, n_h=n_h, seed=11)
    M = 137
    Xt = np.random.default_rng(8).uniform(size=(M, 4))
    eps = np.random.default_rng(3).standard_normal((M, S, 1))
    mean, var = m.predict_mc(Xt, n_samples=S, eps=eps)
    mu_ref, var_ref = o.predict_mc(Xt, eps)
    assert util.rel_err(mean, mu_ref) < 1e-8
    assert util.rel_err(var, var_ref, 1.1) < 1e-6


def test_mc_one_sample_zero_eps_reproduces_predict(pkg):
    # SURVEY.md section 8a row A8: S = 1, eps = 0 must reproduce the reference predict()
    m, o = _mc_models(pkg)
    Xt = np.random.default_rng(6).uniform(size=(300, 4))
    mean, var = m.predict_mc(Xt, n_samples=1, eps=np.zeros((300, 1)))
    mu, v = m.predict(Xt)
    assert util.rel_err(mean, mu) < 1e-12 and util.rel_err(var, v, 1.1) < 1e-10
    mu_ref, var_ref = o.predict(Xt)
    assert util.rel_err(mean, mu_ref) < 1e-8


def test_mc_in_kernel_philox_matches_oracle_and_pce_mean(pkg):
    from multifidelity_datafusion_gps_b200 import ops
    m, o = _mc_models(pkg)
    nodes, w = mo.gauss_legendre_grid(3, 4)                      # 4^4 = 256 quadrature nodes
    M, S, seed = nodes.shape[0], 32, 2
    mean, var = m.predict_mc(nodes, n_samples=S, seed=seed, weights=w)
    eps = ops.fill_normal(seed, 0, M * S, "cuda:0").cpu().numpy().reshape(M, S, 1)
    mu_ref, var_ref = o.predict_mc(nodes, eps)
    assert util.rel_err(mean, mu_ref) < 1e-8
    assert util.rel_err(var, var_ref, 1.1) < 1e-6
    assert np.isclose(m.last_pce_mean, float(np.sum(w * mu_ref[:, 0])), rtol=1e-9)
    # sharding invariance: points [128, 256) evaluated alone with m0 = 128 give the same bits
    import torch
    dX = torch.from_numpy(nodes[128:]).to("cuda:0")
    mean2, var2, _ = m.predict_mc_device(dX, S, None, seed, 128)
    assert np.array_equal(mean2.cpu().numpy(), mean[128:, 0]) and np.array_equal(var2.cpu().numpy(), var[128:, 0])


def _mc_delay_models(pkg, model, n_l=120, n_h=30, seed=7):
    """GPDF / GPDFC in 2-D with delays (tau = 0.05, n = 2 -> E = 5, D = 7) on a data-driven LF GP."""
    rs = np.random.RandomState(seed)
    lf_X = rs.uniform(size=(n_l, 2))
    hf_X = rs.uniform(size=(n_h, 2))
    lf_theta = np.array([1.5, 0.4, 1e-3])
    composite = model == "GPDFC"
    theta = THETA_C if composite else THETA_R
    m = getattr(pkg, model)(2, 0.05, 2, util.hf_2d, None, lf_X=lf_X, lf_Y=util.lf_2d(lf_X))
    m.lf_model._set_params(lf_theta)
    m.fit(hf_X, theta=theta)
    o = mo.OracleMFGP(2, 2, 0.05, util.hf_2d, lf_X=lf_X, lf_Y=util.lf_2d(lf_X), lf_theta=lf_theta,
                      use_composite_kernel=composite)
    o.fit(hf_X, theta=theta)
    return m, o


@pytest.mark.parametrize("model", ["GPDF", "GPDFC"])
def test_mc_with_delays_samples_the_joint_lf_posterior(pkg, model):
    # SURVEY.md section 8a row A8 for E > 1: z_s = mu_l + chol(Sigma_l) eps_s with Sigma_l in R^(5x5)
    m, o = _mc_delay_models(pkg, model)
    M, S, E = 300, 40, 5
    Xt = np.random.default_rng(8).uniform(size=(M, 2))
    eps = np.random.default_rng(9).standard_normal((M, S, E))
    mean, var = m.predict_mc(Xt, n_samples=S, eps=eps)
    mu_ref, var_ref = o.predict_mc(Xt, eps)
    assert util.rel_err(mean, mu_ref) < 1e-8
    assert util.rel_err(var, var_ref, 1.2) < 1e-6
    # extra diagonal jitter on Sigma_l follows the oracle's
    mean_j, var_j = m.predict_mc(Xt, n_samples=S, eps=eps, lf_jitter=1e-4)
    mu_rj, var_rj = o.predict_mc(Xt, eps, jitter=1e-4)
    assert util.rel_err(mean_j, mu_rj) < 1e-8 and util.rel_err(var_j, var_rj, 1.2) < 1e-6
    assert util.rel_err(mean_j, mean) > 1e-7          # ... and it does change the result


def test_mc_with_delays_one_sample_zero_eps_reproduces_predict(pkg):
    m, o = _mc_delay_models(pkg, "GPDF")
    Xt = np.random.default_rng(10).uniform(size=(257, 2))
    mean, var = m.predict_mc(Xt, n_samples=1, eps=np.zeros((257, 1, 5)))
    mu, v = m.predict(Xt)
    assert util.rel_err(mean, mu) < 1e-12 and util.rel_err(var, v, 1.2) < 1e-10
    mu_ref, _ = o.predict(Xt)
    assert util.rel_err(mean, mu_ref) < 1e-8


def test_mc_with_delays_in_kernel_philox_and_sharding(pkg):
    from multifidelity_datafusion_gps_b200 import ops
    import torch
    m, o = _mc_delay_models(pkg, "GPDF")
    M, S, E, seed = 200, 16, 5, 11
    Xt = np.random.default_rng(12).uniform(size=(M, 2))
    mean, var = m.predict_mc(Xt, n_samples=S, seed=seed)
    eps = ops.fill_normal(seed, 0, M * S * E, "cuda:0").cpu().numpy().reshape(M, S, E)
    mu_ref, var_ref = o.predict_mc(Xt, eps)
    assert util.rel_err(mean, mu_ref) < 1e-8
    assert util.rel_err(var, var_ref, 1.2) < 1e-6
    # points [64, 200) alone with m0 = 64, and a scratch so small that the call runs in many chunks
    dX = torch.from_numpy(Xt[64:]).to("cuda:0")
    mean2, var2, _ = m.predict_mc_device(dX, S, None, seed, 64)
    assert np.array_equal(mean2.cpu().numpy(), mean[64:, 0]) and np.array_equal(var2.cpu().numpy(), var[64:, 0])
    small = 8 * (256 * (2 * 128 + 128 + 2 + 5 + 4) + 40 * (5 + 25 + max(5 * (2 + 256 + 1) + 15, S * (7 + 128 + 2))))
    mean3, var3, _ = m.predict_mc_device(dX, S, None, seed, 64, ws_bytes=small)
    assert np.array_equal(mean3.cpu().numpy(), mean2.cpu().numpy())
    assert np.array_equal(var3.cpu().numpy(), var2.cpu().numpy())


def test_assertions_mirror_reference(pkg):
    m = pkg.NARGP(2, util.hf_2d, util.lf_2d)
    with pytest.raises(AssertionError):
        m.fit(np.zeros((5, 3)))                                 # src/MFDataFusion.py:84
    with pytest.raises(AssertionError):
        m.fit(np.zeros(5))                                      # :83
    m.fit(np.random.RandomState(0).uniform(size=(5, 2)), theta=THETA_C)
    with pytest.raises(AssertionError):
        m.predict(np.zeros((4, 3)))                             # :152
    with pytest.raises(AssertionError):
        m.get_mse(np.zeros((4, 2)), np.zeros((3, 1)))           # :169
    with pytest.raises(AssertionError):
        pkg.NARGP(2, util.hf_2d, None)                          # src/abstractMFGP.py:93-95
    with pytest.raises(AssertionError):
        m.adapt(1, plot_mode="x")                               # src/MFDataFusion.py:138


def test_jitter_retry_on_duplicate_rows(pkg):
    # duplicated HF points with (almost) no noise -> first Cholesky fails, GPy's jitter schedule kicks in
    from multifidelity_datafusion_gps_b200 import gp
    X = np.repeat(np.random.RandomState(0).uniform(size=(6, 2)), 2, axis=0)
    Y = util.hf_2d(X)
    model = gp.GPRegression(X, Y)
    model._set_params(np.array([1.0, 1.0, 0.0]))
    model._dA.fill_(0)
    # K + 1e-8 I is numerically singular here or not; force the issue with a negative-definite shift
    try:
        model._ensure_posterior()
    except gp.NotPositiveDefinite:
        pytest.fail("jitter schedule exhausted")
    assert model.last_jitter >= 0.0
    mu, _ = model.predict(X)
    assert util.rel_err(mu, Y) < 1e-3


# ---- K9: PCE projection (SURVEY.md section 8f rank 2) ------------------------------------------------
@pytest.mark.parametrize("d,p,q", [(1, 0, 0), (1, 6, 9), (2, 5, 7), (3, 4, 4), (4, 8, 8), (5, 3, 3), (2, 20, 20)])
def test_pce_projection_matches_oracle(pkg, d, p, q):
    from oracle import pce_oracle as po
    from multifidelity_datafusion_gps_b200.gpc import LegendrePCE
    rng = np.random.default_rng(100 * d + p)
    lb, ub = -rng.uniform(0.5, 1.5, d), rng.uniform(0.5, 2.0, d)
    a = rng.uniform(0.5, 3.0, d)
    f = lambda x: np.prod(np.sin(x * a + 0.3), axis=1) + 0.25 * x[:, 0] ** 2
    pce = LegendrePCE(f, lb, ub, polynomial_order=p, quadrature_order=q)
    pce.calculate_coefficients()
    nodes, wts = po.tensor_grid(q + 1, lb, ub)
    ref = po.project(nodes, wts, f(nodes), lb, ub, po.multi_index(d, p))
    assert pce.coefficients.shape == ref.shape
    assert util.rel_err(pce.coefficients, ref) < 1e-13
    assert np.isclose(pce.get_mean(), ref[0], rtol=1e-13)
    assert np.isclose(pce.get_var(), np.sum(ref[1:] ** 2), rtol=1e-12, atol=1e-300)


def test_pce_reference_closed_forms_and_update_order(pkg):
    # the reference's own gPC check: hf_4d = prod sin(pi x_i) + 5 on [0,1]^4 (tests/test_mfgp_adapt_4d.py:56-66)
    from oracle import pce_oracle as po
    from multifidelity_datafusion_gps_b200.gpc import LegendrePCE
    pce = LegendrePCE(util.hf_4d, [0] * 4, [1] * 4, polynomial_order=4, quadrature_order=4)
    pce.calculate_coefficients()
    a4 = [np.pi] * 4
    assert abs(pce.get_mean() - po.analytical_mean(a4, 5.0)) < 1e-5
    pce.update_order(8)
    pce.update_function(util.hf_4d)
    assert abs(pce.get_mean() - po.analytical_mean(a4, 5.0)) < 1e-12
    assert abs(pce.get_var() - po.analytical_var(a4)) < 1e-4 * po.analytical_var(a4)
    assert pce.get_mean_var() == (pce.get_mean(), pce.get_var())


def test_pce_of_the_model_mean_stays_on_device_and_matches_oracle(pkg):
    from oracle import pce_oracle as po
    from multifidelity_datafusion_gps_b200.gpc import LegendrePCE
    m, o = _mc_models(pkg)
    pce = LegendrePCE(m.predict, [0] * 4, [1] * 4, polynomial_order=5, quadrature_order=5)
    pce.calculate_coefficients()                              # nodes -> K6 -> K9, no host round trip
    mean_ref, var_ref, c_ref = po.pce_mean_var(lambda x: o.predict(x)[0], [0] * 4, [1] * 4, 5, 5)
    assert util.rel_err(pce.coefficients, c_ref) < 1e-8
    # the reference's way of wiring it (src/gpc/mfgp_gpc.py:25): a host lambda around predict
    pce_host = LegendrePCE(lambda x: m.predict(x)[0], [0] * 4, [1] * 4, polynomial_order=5, quadrature_order=5)
    pce_host.calculate_coefficients()
    assert np.array_equal(pce_host.coefficients, pce.coefficients)
    # MC-propagated mean through the device hook; its c_0 is the fused PCE mean of K7
    f = lambda x: m.predict_mc(x, n_samples=8, seed=3)[0]
    f.device_predict = lambda dX: m.predict_mc_device(dX, 8, None, 3, 0)[0]
    pce_mc = LegendrePCE(f, [0] * 4, [1] * 4, polynomial_order=3, quadrature_order=3)
    pce_mc.calculate_coefficients()
    m.predict_mc(pce_mc.quad_points, n_samples=8, seed=3, weights=pce_mc.quad_weights)
    assert np.isclose(pce_mc.get_mean(), m.last_pce_mean, rtol=1e-12)


def test_mfgp_gpc_driver_runs_adaptation_rounds(pkg):
    # src/gpc/mfgp_gpc.py: rounds of 5 adaptation steps, statistics re-projected after each round
    from multifidelity_datafusion_gps_b200.gpc import LegendrePCE, MFGP_GPC
    _, X_hf, X_test = _data(2)
    cands = np.random.default_rng(1).uniform(size=(2000, 2))
    m = pkg.NARGP(2, util.hf_2d, util.lf_2d, adapt_maximizer=pkg.CandidateSetMaximizer(cands))
    m.fit(X_hf)
    pce = LegendrePCE(m.predict, [0, 0], [1, 1], polynomial_order=6, quadrature_order=6)
    drv = MFGP_GPC(m, pce, num_adapts=1, init_cost=5, X_test=X_test, Y_test=util.hf_2d(X_test))
    drv.adapt()
    assert len(drv.mean_history) == 2 and len(drv.var_history) == 2 and len(drv.mse_history) == 2
    assert drv.cost_history == [5, 5 + m.adapt_steps]
    assert m.hf_X.shape[0] == 5 + m.adapt_steps


def test_adaptation_with_bordered_updates_between_refits(pkg):
    # refit_every = 3: steps 1, 2 extend the factorisation at fixed theta, step 3 refits (SURVEY.md 8f rank 3)
    _, X_hf, X_test = _data(2)
    cands = np.random.default_rng(2).uniform(size=(3000, 2))
    m = pkg.NARGP(2, util.hf_2d, util.lf_2d, adapt_maximizer=pkg.CandidateSetMaximizer(cands))
    m.refit_every = 3
    m.fit(X_hf)
    theta0 = m.hf_model.param_array.copy()
    m.adapt(2)                                                    # two bordered updates, no refit
    assert m.hf_X.shape == (7, 2) and m.hf_Y.shape == (7, 1) and m.hf_model.N == 7
    assert np.array_equal(m.hf_model.param_array, theta0)
    o = mo.OracleMFGP(2, 0, 0, util.hf_2d, f_low=util.lf_2d)
    o.fit(m.hf_X, theta=theta0)                                   # full factorisation of the same 7 points
    mean, var = m.predict(X_test)
    mu_ref, var_ref = o.predict(X_test)
    assert util.rel_err(mean, mu_ref) < 1e-8 and util.rel_err(var, var_ref, 1.2) < 1e-6
    m.adapt(3)                                                    # third step of this call refits
    assert m.hf_model.N == 10 and not np.array_equal(m.hf_model.param_array, theta0)


def test_even_delay_pattern_is_selectable_and_matches_oracle(pkg):
    # src/augm_iterators/even_augm_iterator.py: 2*n*dim + 1 symmetric delays (here n = 1, dim = 2 -> E = 5)
    _, X_hf, X_test = _data(2)
    X_hf = np.vstack([X_hf, np.random.RandomState(5).uniform(size=(20, 2))])
    m = pkg.MultifidelityDataFusion("even", 2, 1, 0.01, util.hf_2d, f_low=util.lf_2d,
                                    use_composite_kernel=False, augm_iterator="even")
    assert isinstance(m.augm_iterator, pkg.EvenAugmentation) and m.augm_iterator.new_entries_count() == 5
    m.fit(X_hf, theta=THETA_R)
    o = mo.OracleMFGP(2, 1, 0.01, util.hf_2d, f_low=util.lf_2d, use_composite_kernel=False,
                      offsets=mo.even_offsets(1, 2))
    o.fit(X_hf, theta=THETA_R)
    assert np.array_equal(m.hf_model.X, o.hf_model.X)
    mean, var = m.predict(X_test)
    mu_ref, var_ref = o.predict(X_test)
    assert util.rel_err(mean, mu_ref) < 1e-8 and util.rel_err(var, var_ref, 1.2) < 1e-6
    # the presets keep the reference's default pattern
    assert isinstance(pkg.GPDF(2, 0.01, 1, util.hf_2d, util.lf_2d).augm_iterator, pkg.BackwardAugmentation)


def test_full_size_mc_sweep_properties(pkg):
    """BASELINE.json configs[4] at full size: M = 32^4 Gauss-Legendre nodes x S = 100 samples, N_h = 1024,
    N_l = 4096.  The oracle covers a 256-point subsample; the full sweep is pinned by invariances: the
    two halves evaluated separately (m0 = M/2, as two ranks would) and a different scratch size give the
    same bits, and the fused PCE mean equals sum w * mean."""
    import torch
    from multifidelity_datafusion_gps_b200 import gp
    rng = np.random.default_rng(1)
    Xh, Xl = rng.uniform(size=(1024, 4)), rng.uniform(size=(4096, 4))
    yh, yl = util.hf_4d(Xh), util.lf_4d(Xl)
    lf_theta = np.array([1.0, 0.3, 0.01 * yl.var()])
    hf_theta = np.array([1.0, 0.3, 1.0, 0.3, 0.1, 0.3, 0.01 * yh.var()])
    m = pkg.NARGP(4, util.hf_4d, None, lf_X=Xl[:8], lf_Y=yl[:8])
    m.lf_X, m.lf_Y = Xl, yl
    m.lf_model = gp.GPRegression(Xl, yl)
    m.lf_model._set_params(lf_theta)
    m.fit(Xh, theta=hf_theta)
    nodes, w = mo.gauss_legendre_grid(31, 4)                      # 32 nodes per dimension
    M, S, seed = nodes.shape[0], 100, 2
    assert M == 32 ** 4
    dX, dw = gp.to_device(nodes, 0), gp.to_device(w, 0)
    mean, var, wsum = m.predict_mc_device(dX, S, None, seed, 0, dw)
    assert torch.isfinite(mean).all() and torch.isfinite(var).all() and (var > 0).all()
    assert np.isclose(wsum, float((dw * mean).sum().item()), rtol=1e-12)
    half = M // 2
    mean_b, var_b, _ = m.predict_mc_device(dX[half:], S, None, seed, half)          # second half alone
    assert torch.equal(mean_b, mean[half:]) and torch.equal(var_b, var[half:])
    mean_c, var_c, _ = m.predict_mc_device(dX[:65536], S, None, seed, 0, ws_bytes=200 << 20)   # other chunking
    assert torch.equal(mean_c, mean[:65536]) and torch.equal(var_c, var[:65536])
    # oracle on a subsample, with the normals the in-kernel generator used for those points
    from multifidelity_datafusion_gps_b200 import ops
    o = mo.OracleMFGP(4, 0, 0, util.hf_4d, lf_X=Xl, lf_Y=yl, lf_theta=lf_theta)
    o.fit(Xh, theta=hf_theta)
    first, n = 777216, 256
    eps = ops.fill_normal(seed, first * S, n * S, "cuda:0").cpu().numpy().reshape(n, S, 1)
    mu_ref, var_ref = o.predict_mc(nodes[first:first + n], eps)
    assert util.rel_err(mean[first:first + n].cpu().numpy()[:, None], mu_ref) < 1e-8
    assert util.rel_err(var[first:first + n].cpu().numpy()[:, None], var_ref, 1.1) < 1e-6


# ---- CUDA classes against what the reference's own code computed (tests/golden/reference_runs.npz) ----
_REF_SCENARIOS = {
    "nargp_1d": ("NARGP", dict(dim=1, hf=util.f_high_1d, lf=util.f_low_1d)),
    "gpdf_2d": ("GPDF", dict(dim=2, hf=util.hf_2d, lf=util.lf_2d)),
    "gpdfc_2d": ("GPDFC", dict(dim=2, hf=util.hf_2d, lf=util.lf_2d)),
    "gpdf_2d_add_noise": ("GPDF", dict(dim=2, hf=util.hf_2d, lf=util.lf_2d, add_noise=True)),
    "nargp_2d_adapt": ("NARGP", dict(dim=2, hf=util.hf_2d, lf=util.lf_2d)),
    # LF GP trained by the reference's own constructor (src/abstractMFGP.py:100-104); installed here at the
    # hyper-parameters that run arrived at (its optimiser drove the noise to 5e-17: cond(K_l) = 1.9e10)
    "nargp_2d_data_driven": ("NARGP", dict(dim=2, hf=util.hf_2d, lf=None, data_driven=True)),
}


@pytest.mark.parametrize("name", sorted(_REF_SCENARIOS))
def test_cuda_classes_match_the_executed_reference_at_fixed_theta(pkg, name):
    """The golden file holds predictions of the REFERENCE's classes (src/ executed unmodified over the
    oracle's GP arithmetic) on the training set its own fit / adaptation loop ended with, at fixed
    hyper-parameters.  Same classes, same calls here, on the GPU: augmentation, add_noise and predict."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_runs.npz"))
    cls, sc = _REF_SCENARIOS[name]
    if sc.get("data_driven"):
        X_lf = np.random.RandomState(10).uniform(size=(60, 2))       # make_reference_run_golden.py: X_lf2
        m = pkg.NARGP(sc["dim"], sc["hf"], None, lf_X=X_lf, lf_Y=util.lf_2d(X_lf))
        m.lf_model._set_params(g[name + "/lf_theta"])
    elif cls == "NARGP":
        m = pkg.NARGP(sc["dim"], sc["hf"], sc["lf"], add_noise=sc.get("add_noise", False))
    else:
        m = getattr(pkg, cls)(sc["dim"], 0.001, 2, sc["hf"], sc["lf"], add_noise=sc.get("add_noise", False))
    m.fit(g[name + "/hf_X_final"], theta=g[name + "/theta_fixed"])
    if sc.get("data_driven"):        # augmentation through the LF GP's mean on the GPU: FP64 tolerance, not bits
        assert util.rel_err(m.hf_model.X, g[name + "/aug_X"]) < 1e-8
    else:
        assert np.array_equal(m.hf_model.X, g[name + "/aug_X"])          # the reference's augmentation
    assert np.array_equal(m.hf_Y, g[name + "/hf_Y_final"])
    mean, var = m.predict(g[name + "/X_test"])
    assert util.rel_err(mean, g[name + "/mean_fixed"]) < 1e-8
    assert util.rel_err(var, g[name + "/var_fixed"], 1.2) < 1e-6
    if not sc.get("add_noise"):
        assert np.isclose(m.hf_model.log_likelihood(), float(g[name + "/lml_fixed"]), rtol=1e-6)


def test_predictions_are_bit_invariant_to_batch_size(pkg):
    """A shard of the test points must give the bits the full batch gives for those points, whatever the
    shard size (kernel selection must not depend on it): 4000 points against shards of 37, 1000, 2500."""
    m, _ = _mc_models(pkg)
    Xt = np.random.default_rng(21).uniform(size=(4000, 4))
    mean, var = m.predict(Xt)
    mc_mean, mc_var = m.predict_mc(Xt, n_samples=8, seed=4)
    for lo, hi in ((0, 37), (1000, 2000), (1500, 4000)):
        mu_s, var_s = m.predict(Xt[lo:hi])
        assert np.array_equal(mu_s, mean[lo:hi]) and np.array_equal(var_s, var[lo:hi])
        mc_mu_s, mc_var_s = m.predict_mc(Xt[lo:hi], n_samples=8, seed=4, m0=lo)
        assert np.array_equal(mc_mu_s, mc_mean[lo:hi]) and np.array_equal(mc_var_s, mc_var[lo:hi])


def test_three_level_nargp_recursion_matches_oracle_chain(pkg):
    # SURVEY.md section 8f rank 4: level 1 GP -> level 2 NARGP on [x, mu_1(x)] -> level 3 NARGP on [x, mu_2(x)]
    from multifidelity_datafusion_gps_b200.models import MultiLevelNARGP
    rs = np.random.RandomState(13)
    X1, X2, X3 = rs.uniform(size=(80, 2)), rs.uniform(size=(30, 2)), rs.uniform(size=(12, 2))
    f1 = lambda x: util.lf_2d(x) + 0.3 * np.cos(4 * x[:, :1])
    Y1, Y2, Y3 = f1(X1), util.lf_2d(X2), util.hf_2d(X3)
    lf_theta = np.array([1.5, 0.4, 1e-3])
    ml = MultiLevelNARGP(2, [X1, X2, X3], [Y1, Y2, Y3]).fit(thetas=[THETA_C, THETA_C], lf_theta=lf_theta)
    o2 = mo.OracleMFGP(2, 0, 0, lambda X: Y2, lf_X=X1, lf_Y=Y1, lf_theta=lf_theta)
    o2.fit(X2, theta=THETA_C)
    o3 = mo.OracleMFGP(2, 0, 0, lambda X: Y3, f_low=lambda x: o2.predict(x)[0])
    o3.fit(X3, theta=THETA_C)
    Xt = rs.uniform(size=(500, 2))
    mean, var = ml.predict(Xt)
    mu_ref, var_ref = o3.predict(Xt)
    assert util.rel_err(ml.models[-1].hf_model.X, o3.hf_model.X) < 1e-8     # augmentation through level 2
    assert util.rel_err(mean, mu_ref) < 1e-8 and util.rel_err(var, var_ref, 1.2) < 1e-6
    mean2, _ = ml.predict_level(2, Xt)
    assert util.rel_err(mean2, o2.predict(Xt)[0]) < 1e-8


def test_lockstep_restarts_equal_the_serial_loop(pkg, monkeypatch):
    """optimize_restarts (src/abstractMFGP.py:137) with the six restarts in lock-step on one GPU (one batched
    launch per round of evaluations) must end where the reference's serial loop ends: same runs, same
    objectives, same winner, bit for bit -- for the composite and the plain kernel."""
    from multifidelity_datafusion_gps_b200 import gp
    _, X_hf, _ = _data(2, n_hf=14)
    for cls, args in ((pkg.GPDF, (2, 0.001, 2)), (pkg.NARGP, (2,))):
        out = {}
        for mode in ("0", "1"):      # "0": the serial loop, "1": lock-step
            with monkeypatch.context() as mp:
                if mode == "0":
                    mp.setattr(gp.GPRegression, "_lockstep_ok", lambda self, n: False)
                np.random.seed(3)
                m = cls(*args, util.hf_2d, util.lf_2d)
                m.fit(X_hf)
                out[mode] = (m.hf_model.param_array.copy(), [f for _, f in m.hf_model.optimization_runs],
                             [x.copy() for x, _ in m.hf_model.optimization_runs], m.predict(X_hf[:3]))
        assert np.array_equal(out["0"][0], out["1"][0])
        assert out["0"][1] == out["1"][1] and len(out["1"][1]) == 7
        assert all(np.array_equal(a, b) for a, b in zip(out["0"][2], out["1"][2]))
        assert np.array_equal(out["0"][3][0], out["1"][3][0])


def _three_levels(pkg):
    from multifidelity_datafusion_gps_b200.models import MultiLevelNARGP
    rs = np.random.RandomState(13)
    X1, X2, X3 = rs.uniform(size=(80, 2)), rs.uniform(size=(30, 2)), rs.uniform(size=(12, 2))
    f1 = lambda x: util.lf_2d(x) + 0.3 * np.cos(4 * x[:, :1])
    Y1, Y2, Y3 = f1(X1), util.lf_2d(X2), util.hf_2d(X3)
    lf_theta = np.array([1.5, 0.4, 1e-3])
    ml = MultiLevelNARGP(2, [X1, X2, X3], [Y1, Y2, Y3]).fit(thetas=[THETA_C, THETA_C], lf_theta=lf_theta)
    o2 = mo.OracleMFGP(2, 0, 0, lambda X: Y2, lf_X=X1, lf_Y=Y1, lf_theta=lf_theta)
    o2.fit(X2, theta=THETA_C)
    o3 = mo.OracleMFGP(2, 0, 0, lambda X: Y3, f_low=lambda x: o2.predict(x)[0])
    o3.fit(X3, theta=THETA_C)
    return ml, [o2.lf_model, o2.hf_model, o3.hf_model], rs


def test_mc_propagation_through_three_levels(pkg):
    # SURVEY.md section 8f rank 4: samples (not means) travel up the chain level 1 -> 2 -> 3
    from multifidelity_datafusion_gps_b200 import ops
    ml, levels, rs = _three_levels(pkg)
    M, S = 300, 48
    Xt = rs.uniform(size=(M, 2))
    eps = np.random.default_rng(6).standard_normal((2, M, S))
    mean, var = ml.predict_mc(Xt, n_samples=S, eps=eps)
    mu_ref, var_ref = mo.predict_mc_chain(levels, Xt, eps)
    assert util.rel_err(mean, mu_ref) < 1e-8 and util.rel_err(var, var_ref, 1.2) < 1e-6
    # zero normals collapse every level to its mean: the mean-propagating predict()
    mean0, var0 = ml.predict_mc(Xt, n_samples=1, eps=np.zeros((2, M, 1)))
    mu, v = ml.predict(Xt)
    assert util.rel_err(mean0, mu) < 1e-12 and util.rel_err(var0, v, 1.2) < 1e-10
    # in-kernel Philox: level 1 -> 2 draws the keys of mfgp_predict_mc, level 2 -> 3 its own key; a shard with
    # m0 reproduces the rows of the full batch
    seed = 9
    mean_p, var_p = ml.predict_mc(Xt, n_samples=S, seed=seed)
    e1 = ops.fill_normal(seed, 0, M * S, "cuda:0").cpu().numpy().reshape(M, S)
    e2 = ops.fill_normal((seed + 0x9E3779B97F4A7C15) % (1 << 64), 0, M * S, "cuda:0").cpu().numpy().reshape(M, S)
    mu_ref, var_ref = mo.predict_mc_chain(levels, Xt, np.stack([e1, e2]))
    assert util.rel_err(mean_p, mu_ref) < 1e-8 and util.rel_err(var_p, var_ref, 1.2) < 1e-6
    mean_s, var_s = ml.predict_mc(Xt[100:], n_samples=S, seed=seed, m0=100)
    assert np.array_equal(mean_s, mean_p[100:]) and np.array_equal(var_s, var_p[100:])
    # two levels through the chain entry point == NARGP.predict_mc, bit for bit
    from multifidelity_datafusion_gps_b200.models import MultiLevelNARGP
    two = MultiLevelNARGP(2, ml.level_X[:2], ml.level_Y[:2]).fit(thetas=[THETA_C], lf_theta=np.array([1.5, 0.4, 1e-3]))
    a = two.predict_mc(Xt, n_samples=S, seed=seed)
    b = two.models[0].predict_mc(Xt, n_samples=S, seed=seed)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_mc_with_joint_lf_sampling_across_test_points(pkg):
    # SURVEY.md section 8f rank 4, "full-covariance LF sampling for small M": z_s = mu_l + chol(Sigma_l) eps_s
    # with the M x M low-fidelity predictive covariance; per-path functionals come back too
    m, o = _mc_models(pkg, n_l=100, n_h=30, d=4, seed=4)
    for M, S in ((200, 64), (130, 33)):
        Xt = np.random.default_rng(M).uniform(size=(M, 4))
        w = np.random.default_rng(M + 1).uniform(size=M)
        w /= w.sum()
        eps = np.random.default_rng(M + 2).standard_normal((M, S))
        mean, var = m.predict_mc(Xt, n_samples=S, eps=eps, weights=w, joint=True)
        mu_ref, var_ref, mu_s = o.predict_mc_joint(Xt, eps)
        assert util.rel_err(mean, mu_ref) < 1e-8 and util.rel_err(var, var_ref, 1.1) < 1e-6
        paths_ref = (w[:, None] * mu_s).sum(axis=0)
        assert util.rel_err(m.last_pce_paths, paths_ref) < 1e-8
        assert np.isclose(m.last_pce_mean, paths_ref.mean(), rtol=1e-10)
    # in-kernel Philox (counter m*S + s) and extra jitter
    from multifidelity_datafusion_gps_b200 import ops
    M, S, seed = 150, 40, 12
    Xt = np.random.default_rng(77).uniform(size=(M, 4))
    mean, var = m.predict_mc(Xt, n_samples=S, seed=seed, joint=True, lf_jitter=1e-5)
    eps = ops.fill_normal(seed, 0, M * S, "cuda:0").cpu().numpy().reshape(M, S)
    mu_ref, var_ref, _ = o.predict_mc_joint(Xt, eps, jitter=1e-5)
    assert util.rel_err(mean, mu_ref) < 1e-8 and util.rel_err(var, var_ref, 1.1) < 1e-6
    # the marginal statistics agree with independent-marginal sampling in expectation (same marginals):
    # with S large the two estimates of the mean are close
    S2 = 1000
    a, _ = m.predict_mc(Xt[:40], n_samples=S2, seed=1, joint=True)
    b, _ = m.predict_mc(Xt[:40], n_samples=S2, seed=2)
    assert np.max(np.abs(a - b)) < 0.05 * max(1.0, np.max(np.abs(b)))
    # a joint covariance that is not positive definite is reported, not silently sampled from
    with pytest.raises(np.linalg.LinAlgError):
        m.predict_mc(Xt[:20], n_samples=8, seed=1, joint=True, lf_jitter=-10.0)


def test_predict_point_latency_path_matches_predict(pkg):
    # mfgp_predict_small: what one DIRECT objective evaluation costs (scipydirect_wrapper.py:22-26)
    lf_X, X_hf, _ = _data(2, n_hf=9)
    rs = np.random.RandomState(3)
    models = []
    m = pkg.GPDF(2, 0.001, 2, util.hf_2d, util.lf_2d)                        # callable LF, delays (D = 7)
    m.fit(X_hf, theta=THETA_R)
    models.append(m)
    m = pkg.NARGP(2, util.hf_2d, None, lf_X=lf_X, lf_Y=util.lf_2d(lf_X))     # data-driven LF
    m.lf_model._set_params(np.array([1.5, 0.4, 1e-3]))
    m.fit(X_hf, theta=THETA_C)
    models.append(m)
    m = pkg.GPDFC(2, 0.05, 2, util.hf_2d, None, lf_X=lf_X, lf_Y=util.lf_2d(lf_X))   # data-driven LF with delays
    m.lf_model._set_params(np.array([1.5, 0.4, 1e-3]))
    m.fit(np.vstack([X_hf, rs.uniform(size=(150, 2))]), theta=THETA_C)       # N_h = 159: beyond one 128-tile
    models.append(m)
    for m in models:
        for M in (1, 5, 16):
            Xq = rs.uniform(size=(M, 2))
            mu, var = m.predict(Xq)
            mu_p, var_p = m.predict_point(Xq)
            assert mu_p.shape == (M, 1) and var_p.shape == (M, 1)
            assert util.rel_err(mu_p, mu) < 1e-11 and util.rel_err(var_p, var, 1.2) < 1e-10
        mu_f, var_f = m.predict_point(rs.uniform(size=(40, 2)))               # too many rows: falls back
        assert mu_f.shape == (40, 1)


# ---- point service: the resident single-row predictor behind the default DIRECT maximiser -----------------
def _service_models(pkg):
    lf_X, X_hf, _ = _data(2, n_hf=12)
    callable_lf = pkg.GPDF(2, 0.001, 2, util.hf_2d, util.lf_2d)
    callable_lf.fit(X_hf, theta=THETA_R)
    data_lf = pkg.NARGP(2, util.hf_2d, None, lf_X=lf_X, lf_Y=util.lf_2d(lf_X))
    data_lf.fit(X_hf, theta=THETA_C)
    return callable_lf, data_lf


def test_point_service_equals_the_latency_path_bit_for_bit(pkg):
    import time
    import torch
    for m in _service_models(pkg):
        pts = np.random.default_rng(12).uniform(size=(40, 2))
        ref = [m.predict_point(p[None]) for p in pts]
        assert m.point_service_start(idle_ms=2.0)
        try:
            got = [m.point_service_eval(p) for p in pts[:20]]
            time.sleep(0.05)                               # the kernel leaves on its idle limit ...
            torch.cuda.synchronize()                       # ... so a device-wide synchronisation returns
            got += [m.point_service_eval(p) for p in pts[20:]]   # ... and the next question relaunches it
            h = m._svc_handle
            assert h.lib.mfgp_point_service_relaunches(h.h) >= 1
        finally:
            m.point_service_stop()
        for (mu, v), (mu_r, v_r) in zip(got, ref):
            assert mu == mu_r[0, 0] and v == v_r[0, 0]
        mu2, v2 = m.predict(pts)                           # the ordinary path is untouched afterwards
        assert util.rel_err(np.array([g[0] for g in got]), mu2[:, 0]) < 1e-10


def test_direct_maximiser_through_the_service_finds_the_same_point(pkg):
    callable_lf, _ = _service_models(pkg)
    maxi = pkg.ScipyDirectMaximizer(maxf=600, maxT=200)
    lo, hi = np.zeros(2), np.ones(2)
    x_s, f_s = maxi.maximize(callable_lf.predict, lo, hi)
    orig = callable_lf.point_service_start
    callable_lf.point_service_start = lambda *a, **k: False     # force the latency path
    try:
        x_l, f_l = maxi.maximize(callable_lf.predict, lo, hi)
    finally:
        callable_lf.point_service_start = orig
    assert np.array_equal(x_s, x_l) and f_s == f_l
