"""Predictive gradients on the GPU (mfgp_predictive_gradients, GPRegression / MultifidelityDataFusion
.predictive_gradients) and the multi-start L-BFGS-B acquisition built on them (LBFGSBMaximizer): agreement with the
NumPy gradient oracle, bit-invariance to chunking and batching, the multi-fidelity chain rule against central
differences of predict, the maximizer's guarantees at the config-2 and config-3 shapes, two ranks, argument errors."""
import ctypes
import socket
import types

import numpy as np
import pytest

from multifidelity_datafusion_gps_b200 import _lbfgsb
from tests import util
from tests.gradient_oracle import central_diff, level_gradients

pytestmark = pytest.mark.gpu

THETA_C = np.array([1.0, 0.8, 1.0, 0.5, 0.1, 0.3, 1e-3])
THETA_R = np.array([1.2, 0.9, 1e-3])
THETA_4D = np.array([1.0, 0.3, 1.0, 0.3, 0.1, 0.3, 1e-3])
CASES = ["config2_gpdf_d7", "config3_nargp_4d", "nargp_data_driven_lf", "gpdfc_outside_shapes"]


@pytest.fixture(scope="module")
def pkg(gpu):
    import multifidelity_datafusion_gps_b200 as pkg
    return pkg


def _x_hf(dim, n=30, seed=10):
    return np.random.RandomState(seed).uniform(size=(n, dim))


def _gpdf(pkg, mx=None):
    m = pkg.GPDF(2, 0.001, 2, util.hf_2d, util.lf_2d, adapt_maximizer=mx)      # config 2: GPDF 2-D, D = 7
    m.fit(_x_hf(2), theta=THETA_R)
    return m


def _nargp_4d(pkg, mx=None):
    m = pkg.NARGP(4, util.hf_4d, util.lf_4d, adapt_maximizer=mx)                 # config 3: NARGP 4-D
    m.fit(_x_hf(4, n=5), theta=THETA_4D)
    return m


def _case(pkg, name):
    """The model shapes of tests/test_gpu_batch_acquisition.py."""
    if name == "config2_gpdf_d7":
        return _gpdf(pkg)
    if name == "config3_nargp_4d":
        return _nargp_4d(pkg)
    if name == "nargp_data_driven_lf":
        lf_X = np.random.RandomState(3).uniform(size=(100, 2))
        m = pkg.NARGP(2, util.hf_2d, None, lf_X=lf_X, lf_Y=util.lf_2d(lf_X))
        m.lf_model._set_params(np.array([1.5, 0.4, 1e-3]))
        m.fit(_x_hf(2, n=12), theta=THETA_C)
        return m
    m = pkg.GPDFC(2, 0.001, 1, util.hf_2d, util.lf_2d)          # composite d = 2, E = 3: runtime-width kernel
    m.fit(_x_hf(2, n=20), theta=THETA_C)
    return m


def _normwise(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def _call(level, dX, want_var=True, ws_bytes=None):
    """mfgp_predictive_gradients on a GPRegression: (dmean, dvar, mean, var) as NumPy."""
    import torch
    from multifidelity_datafusion_gps_b200 import _ffi, gp
    h = _ffi.get_handle(level.device)
    lvl = level.level_struct()
    M, D = dX.shape
    new = lambda *s: torch.empty(s, dtype=torch.float64, device=dX.device)
    dmean, mean = new(M, D), new(M)
    dvar = var = ws = None
    if want_var:
        dvar, var = new(M, D), new(M)
        ws = new(((ws_bytes or h.lib.mfgp_predictive_gradients_ws_bytes(level.N, M)) + 7) // 8)
    p = lambda t: t.data_ptr() if t is not None else None
    h.check(h.lib.mfgp_predictive_gradients(h.h, ctypes.byref(lvl), dX.data_ptr(), M, dmean.data_ptr(), p(dvar),
                                            mean.data_ptr(), p(var), 1, p(ws), ws.numel() * 8 if ws is not None else 0))
    c = lambda t: t.cpu().numpy() if t is not None else None
    return c(dmean), c(dvar), c(mean), c(var)


def _large_level(pkg):
    from multifidelity_datafusion_gps_b200 import gp
    rng = np.random.default_rng(4)
    X = rng.uniform(size=(1000, 5))                             # N_h = 1000: not a multiple of 128
    Y = np.sin(3.0 * X.sum(axis=1))[:, None]
    level = gp.GPRegression(X, Y, kernel=gp.NARGPKernel(4, 1))
    level._set_params(np.array([1.3, 0.7, 0.9, 0.5, 0.2, 0.4, 1e-2]))
    return level


def _check_oracle(level, Xq, rows):
    from multifidelity_datafusion_gps_b200 import gp
    dm, dv, _, _ = _call(level, gp.to_device(Xq, level.device))
    rm, rv = level_gradients(level.kern.kind, level.X, level.Y, level.kern.d, level.param_array, Xq[rows])
    assert _normwise(dm[rows], rm) < 1e-8
    assert _normwise(dv[rows], rv) < 1e-6


@pytest.mark.parametrize("name", CASES)
def test_level_gradients_match_the_oracle(pkg, name):
    m = _case(pkg, name)
    Xa = m.augment_data(np.random.default_rng(1).uniform(size=(700, m.input_dim)))
    _check_oracle(m.hf_model, Xa, np.arange(700))


def test_level_gradients_match_the_oracle_at_n1000(pkg):
    level = _large_level(pkg)
    Xq = np.random.default_rng(2).uniform(size=(1 << 16, 5))
    _check_oracle(level, Xq, np.sort(np.random.default_rng(3).choice(1 << 16, 256, replace=False)))


def _bit_invariance(level, Xq):
    from multifidelity_datafusion_gps_b200 import _ffi, gp
    dX = gp.to_device(Xq, level.device)
    full = _call(level, dX)
    h = _ffi.get_handle(level.device)
    small = _call(level, dX, ws_bytes=h.lib.mfgp_predictive_gradients_ws_bytes(level.N, 128))   # several chunks
    for a, b in zip(full, small):
        assert np.array_equal(a, b)
    for r in (0, 1, len(Xq) // 2, len(Xq) - 1):                # one row per call
        one = _call(level, dX[r:r + 1].contiguous())
        for a, b in zip(full, one):
            assert np.array_equal(a[r:r + 1], b)
    mean_only = _call(level, dX, want_var=False)
    assert np.array_equal(mean_only[0], full[0])
    mean, var = level.predict_device(dX, True, True)
    scale = float(level.param_array[0] * level.param_array[2] + level.param_array[4]) \
        if level.kern.kind == 1 else float(level.param_array[0])
    assert np.max(np.abs(full[2] - mean.cpu().numpy())) <= 1e-12 * max(1.0, np.max(np.abs(full[2])))
    assert np.max(np.abs(full[3] - var.cpu().numpy())) <= 1e-12 * scale


@pytest.mark.parametrize("name", ["config2_gpdf_d7", "gpdfc_outside_shapes"])
def test_outputs_are_bit_invariant_to_chunking_and_batching(pkg, name):
    m = _case(pkg, name)
    _bit_invariance(m.hf_model, m.augment_data(np.random.default_rng(5).uniform(size=(300, m.input_dim))))


def test_outputs_are_bit_invariant_at_n1000(pkg):
    level = _large_level(pkg)
    _bit_invariance(level, np.random.default_rng(6).uniform(size=(3000, 5)))


@pytest.mark.parametrize("name", CASES)
def test_mf_gradients_match_central_differences_of_predict(pkg, name):
    m = _case(pkg, name)
    X = np.random.default_rng(8).uniform(0.1, 0.9, size=(16, m.input_dim))
    dmu, dv = m.predictive_gradients(X)
    assert dmu.shape == (16, m.input_dim, 1) and dv.shape == (16, m.input_dim)
    assert np.all(m.predict(X)[1] > 1e-10 + m.hf_model.likelihood.variance)
    assert _normwise(dmu[:, :, 0], central_diff(lambda Z: m.predict(Z)[0].ravel(), X, 1e-5)) < 1e-5
    assert _normwise(dv, central_diff(lambda Z: m.predict(Z)[1].ravel(), X, 1e-5)) < 1e-5
    h = m.hf_model
    gp_dmu, gp_dv = h.predictive_gradients(m.augment_data(X))          # GPy's shapes on the level itself
    assert gp_dmu.shape == (16, h.D, 1) and gp_dv.shape == (16, h.D)


# -- LBFGSBMaximizer --------------------------------------------------------------------------------------------------
def _maximize(pkg, name, n_cands):
    m = _gpdf(pkg) if name == "config2" else _nargp_4d(pkg)
    cands = np.random.default_rng(0).uniform(size=(n_cands, m.input_dim))
    mx = pkg.LBFGSBMaximizer(candidates=cands)
    lb, ub = np.zeros(m.input_dim), np.ones(m.input_dim)
    x, fopt = mx.maximize(m.predict, lb, ub)
    return m, mx, cands, lb, ub, x, fopt


@pytest.mark.parametrize("name,n_cands", [("config2", 100000), ("config3", 1 << 20)])
def test_lbfgsb_maximizer_refines_the_candidate_argmax(pkg, name, n_cands):
    m, mx, cands, lb, ub, x, fopt = _maximize(pkg, name, n_cands)
    assert np.all(x >= lb) and np.all(x <= ub)
    i0, v0 = m.acquisition_argmax(cands)
    assert -fopt >= v0 and fopt == -m.predict(x[None])[1][0, 0]
    _, g = m.variance_and_gradient(x[None])
    on_bound = (x == lb) | (x == ub)
    assert np.all((np.abs(g[0]) <= 1e-4 * v0) | on_bound), (g, x)
    # lock-step equals every start run alone (single-row gradient calls), bit for bit
    fun = lambda z: (lambda v, gg: (-v[0] / v0, -gg[0] / v0))(*m.variance_and_gradient(z[None]))
    for s, (xs, fs, _) in zip(mx.last_starts, mx.last_runs):
        alone = _lbfgsb.minimize(fun, s, maxfun=mx.maxfun, maxiter=mx.maxiter, bounds=list(zip(lb, ub)))
        assert np.array_equal(alone[0], xs) and alone[1] == fs


def test_adapt_with_the_lbfgsb_maximizer(pkg):
    cands = np.random.default_rng(0).uniform(size=(100000, 2))
    m = _gpdf(pkg, pkg.LBFGSBMaximizer(candidates=cands, n_starts=4))
    n0 = len(m.hf_X)
    m.adapt(3)
    assert len(m.hf_X) == n0 + 3 and np.all((m.hf_X >= 0.0) & (m.hf_X <= 1.0))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank(rank, world, port, out):
    import torch
    import torch.distributed as tdist
    import multifidelity_datafusion_gps_b200 as pkg
    torch.cuda.set_device(0)
    tdist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    m = _gpdf(pkg)
    cands = np.random.default_rng(0).uniform(size=(20001, 2))
    x, fopt = pkg.LBFGSBMaximizer(candidates=cands, n_starts=8, distributed=True).maximize(
        m.predict, np.zeros(2), np.ones(2))
    out.put((rank, x.view(np.int64).tolist(), np.float64(fopt).view(np.int64).tolist()))
    tdist.barrier()
    tdist.destroy_process_group()


def test_two_ranks_return_the_single_process_point(pkg):
    import torch.multiprocessing as mp
    m = _gpdf(pkg)
    cands = np.random.default_rng(0).uniform(size=(20001, 2))
    x, fopt = pkg.LBFGSBMaximizer(candidates=cands, n_starts=8).maximize(m.predict, np.zeros(2), np.ones(2))
    ref = (x.view(np.int64).tolist(), np.float64(fopt).view(np.int64).tolist())
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    res = [out.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for _, xr, fr in res:
        assert (xr, fr) == ref


def test_argument_errors_launch_nothing(pkg):
    import torch
    from multifidelity_datafusion_gps_b200 import _ffi, gp, ops
    m = _gpdf(pkg)
    level = m.hf_model
    h = _ffi.get_handle(m.device)
    lvl = level.level_struct()
    M, D = 200, level.D
    dX = gp.to_device(np.random.default_rng(0).uniform(size=(M, D)), m.device)
    t = lambda *s: torch.empty(s, dtype=torch.float64, device=dX.device)
    dm, dv, mean, var = t(M, D), t(M, D), t(M), t(M)
    need = h.lib.mfgp_predictive_gradients_ws_bytes(level.N, 128)
    ws = t(need // 8)
    torch.cuda.synchronize()
    before = h.launches
    bad = [
        (dX.data_ptr(), M, None, dv.data_ptr(), None, None, ws.data_ptr(), need),           # no dmean
        (dX.data_ptr(), -1, dm.data_ptr(), dv.data_ptr(), None, None, ws.data_ptr(), need),   # M < 0
        (dX.data_ptr(), M, dm.data_ptr(), dv.data_ptr(), mean.data_ptr(), var.data_ptr(), ws.data_ptr(), need - 8),
        (dX.data_ptr(), M, dm.data_ptr(), dv.data_ptr(), None, None, None, need),            # no scratch
        (dX.data_ptr(), M, dm.data_ptr(), None, None, var.data_ptr(), None, 0),               # var without W path
        (None, M, dm.data_ptr(), dv.data_ptr(), None, None, ws.data_ptr(), need),             # no queries
    ]
    for X, MM, a, b, c, d, w, n in bad:
        rc = h.lib.mfgp_predictive_gradients(h.h, ctypes.byref(lvl), X, MM, a, b, c, d, 1, w, n)
        assert rc < 0 and h.lib.mfgp_last_error(h.h).decode()
    assert h.launches == before
    with pytest.raises(AssertionError):
        level.predictive_gradients_device(gp.to_device(np.zeros((3, D - 1)), m.device))   # D mismatch
    ref = ops.LevelRef(level._dX, level.kern.kind, level.kern.d, level.param_array,
                       types.SimpleNamespace(W=level._dW, alpha=level._dalpha))
    with pytest.raises(ValueError):
        ops.predictive_gradients(ref, gp.to_device(np.zeros((3, D + 1)), m.device))
    assert h.launches == before
