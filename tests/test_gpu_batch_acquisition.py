"""Greedy batch acquisition on the GPU (MultifidelityDataFusion.acquisition_batch, mfgp_acq_batch_*): the first pick is
acquisition_argmax bit for bit, the batch follows the oracle's definition and the sequential adaptation loop at fixed
hyper-parameters, sharding over ranks changes no bit, and bad batch sizes are refused."""
import ctypes
import socket

import numpy as np
import pytest

from oracle import mfgp_oracle as mo
from tests import util
from tests.batch_oracle import candidate_batch

pytestmark = pytest.mark.gpu

THETA_C = np.array([1.0, 0.8, 1.0, 0.5, 0.1, 0.3, 1e-3])
THETA_R = np.array([1.2, 0.9, 1e-3])
THETA_4D = np.array([1.0, 0.3, 1.0, 0.3, 0.1, 0.3, 1e-3])


@pytest.fixture(scope="module")
def pkg(gpu):
    import multifidelity_datafusion_gps_b200 as pkg
    return pkg


def _x_hf(dim, n=30, seed=10):
    return np.random.RandomState(seed).uniform(size=(n, dim))


def _gpdf(pkg, mx=None):
    # config 2 (tests/test_mfgp_adapt_2d.py:27): GPDF 2-D, two delays, D = 7
    m = pkg.GPDF(2, 0.001, 2, util.hf_2d, util.lf_2d, adapt_maximizer=mx)
    m.fit(_x_hf(2), theta=THETA_R)
    return m


def _case(pkg, name):
    if name == "config2_gpdf_d7":
        return _gpdf(pkg), np.random.default_rng(0).uniform(size=(100000, 2))
    if name == "config3_nargp_4d":
        m = pkg.NARGP(4, util.hf_4d, util.lf_4d)
        m.fit(_x_hf(4, n=5), theta=THETA_4D)
        return m, np.random.default_rng(0).uniform(size=(1 << 20, 4))
    if name == "nargp_data_driven_lf":
        lf_X = np.random.RandomState(3).uniform(size=(100, 2))
        m = pkg.NARGP(2, util.hf_2d, None, lf_X=lf_X, lf_Y=util.lf_2d(lf_X))
        m.lf_model._set_params(np.array([1.5, 0.4, 1e-3]))
        m.fit(_x_hf(2, n=12), theta=THETA_C)
        return m, np.random.default_rng(1).uniform(size=(30000, 2))
    # composite kernel on d = 2, E = 3 (one delay): a width outside MFGP_SHAPES -> one-warp generators
    m = pkg.GPDFC(2, 0.001, 1, util.hf_2d, util.lf_2d)
    m.fit(_x_hf(2, n=20), theta=THETA_C)
    return m, np.random.default_rng(2).uniform(size=(30000, 2))


@pytest.mark.parametrize("name", ["config2_gpdf_d7", "config3_nargp_4d", "nargp_data_driven_lf",
                                  "gpdfc_outside_shapes"])
def test_batch_of_one_is_the_argmax_bit_for_bit(pkg, name):
    m, cands = _case(pkg, name)
    idx, var = m.acquisition_batch(cands, 1)
    i0, v0 = m.acquisition_argmax(cands)
    assert idx.shape == (1,) and idx.dtype == np.int64 and var.shape == (1,)
    assert int(idx[0]) == i0 and float(var[0]) == v0


def _oracle_prefix(idx, var, ref_idx, ref_var, gaps, scale):
    """Compare picks while the oracle's top-2 gap leaves no room for round-off; returns how many were compared."""
    for i in range(len(idx)):
        if gaps[i] <= 1e-9:
            return i
        assert idx[i] == ref_idx[i], (i, idx, ref_idx)
        assert abs(var[i] - ref_var[i]) <= 1e-9 * scale, (i, var[i], ref_var[i])
    return len(idx)


@pytest.mark.parametrize("model", ["GPDF", "GPDFC"])
def test_batch_follows_the_oracle(pkg, model):
    composite = model == "GPDFC"
    theta = THETA_C if composite else THETA_R
    m = getattr(pkg, model)(2, 0.001, 2, util.hf_2d, util.lf_2d)
    m.fit(_x_hf(2), theta=theta)
    o = mo.OracleMFGP(2, 2, 0.001, util.hf_2d, f_low=util.lf_2d, use_composite_kernel=composite, form="direct")
    o.fit(_x_hf(2), theta=theta)
    cands = np.random.default_rng(6).uniform(size=(4000, 2))
    q = 8
    idx, var = m.acquisition_batch(cands, q)
    ref_idx, ref_var, gaps = candidate_batch(o, cands, q)
    kdiag = theta[0] * theta[2] + theta[4] if composite else theta[0]
    assert _oracle_prefix(idx, var, ref_idx, ref_var, gaps, kdiag + theta[-1]) == q


def _sequential_and_batch(pkg, cands, q, eps, seq_steps, batch_steps):
    seq = _gpdf(pkg, pkg.CandidateSetMaximizer(candidates=cands))
    seq.refit_every = q + 1                        # q steps at fixed theta: bordered updates only
    seq.adapt(seq_steps, eps=eps)
    bat = _gpdf(pkg, pkg.CandidateSetMaximizer(candidates=cands))
    bat.adapt_batch_size = q
    bat.refit_every = 2                            # the first step appends its block
    bat.adapt(batch_steps, eps=eps)
    return seq, bat


def test_batch_step_equals_sequential_steps_at_fixed_theta(pkg):
    cands = np.random.default_rng(7).uniform(size=(20000, 2))
    q = 8
    o = mo.OracleMFGP(2, 2, 0.001, util.hf_2d, f_low=util.lf_2d, use_composite_kernel=False, form="direct")
    o.fit(_x_hf(2), theta=THETA_R)
    _, _, gaps = candidate_batch(o, cands, q)
    assert np.all(gaps > 1e-9), "degenerate case: pick other candidates"
    seq, bat = _sequential_and_batch(pkg, cands, q, 0.0, q, 1)
    assert len(seq.acquired_points) == len(bat.acquired_points) == q
    for (xs, fs), (xb, fb) in zip(seq.acquired_points, bat.acquired_points):
        assert np.array_equal(xs, xb)
        assert abs(fs - fb) <= 1e-9 * (THETA_R[0] + THETA_R[-1])
    assert np.array_equal(seq.hf_X, bat.hf_X)
    assert seq.hf_model.N == bat.hf_model.N == 30 + q
    # a host f_low evaluated on a block instead of one row may round differently in the last bit
    assert util.rel_err(bat.hf_model.X, seq.hf_model.X) < 1e-14
    assert util.rel_err(bat.hf_model.Y, seq.hf_model.Y) < 1e-14
    Xt = np.random.default_rng(8).uniform(size=(500, 2))
    assert util.rel_err(bat.predict(Xt)[1], seq.predict(Xt)[1]) < 1e-9


def test_eps_truncates_the_batch_where_the_sequential_loop_stops(pkg):
    cands = np.random.default_rng(7).uniform(size=(20000, 2))
    q = 8
    _, var = _gpdf(pkg).acquisition_batch(cands, q)
    assert np.all(np.diff(var) <= 0.0)
    eps = 0.5 * (var[3] + var[4])                  # |fopt| of pick 4 is the first below eps
    seq, bat = _sequential_and_batch(pkg, cands, q, eps, q, 3)
    assert len(seq.acquired_points) == len(bat.acquired_points) == 5
    assert seq.adapt_steps == 5 and bat.adapt_steps == 1
    assert np.array_equal(seq.hf_X, bat.hf_X)


def test_large_level_batch_equals_sequential_steps(pkg):
    # bench.py's acquisition shape: N_h = 1024, data-driven LF with N_l = 4096, 2^20 candidates (TMA trmm_sumsq)
    import torch
    from multifidelity_datafusion_gps_b200 import gp
    rng = np.random.default_rng(1)
    Xh, Xl = rng.uniform(size=(1024, 4)), rng.uniform(size=(4096, 4))
    yl = util.lf_4d(Xl)
    cands = np.random.default_rng(0).uniform(size=(1 << 20, 4))
    hf_theta = np.array([1.0, 0.3, 1.0, 0.3, 0.1, 0.3, 0.01 * util.hf_4d(Xh).var()])

    def model():
        m = pkg.NARGP(4, util.hf_4d, None, lf_X=Xl[:8], lf_Y=yl[:8])
        m.lf_X, m.lf_Y = Xl, yl
        m.lf_model = gp.GPRegression(Xl, yl)
        m.lf_model._set_params(np.array([1.0, 0.3, 0.01 * yl.var()]))
        m.fit(Xh, theta=hf_theta)
        return m

    q = 4
    bat = model()
    idx, var = bat.acquisition_batch(cands, q)
    seq = model()
    for i in range(q):                             # the sequential steps, with the top-2 gap of every pick
        j, v = seq.acquisition_argmax(cands)
        _, pv = seq.hf_model.predict_device(seq._resident_candidates(cands, 0, len(cands)), True, True)
        top = torch.topk(pv, 2).values.cpu().numpy()
        if (top[0] - top[1]) / top[0] <= 1e-9:
            break
        assert j == idx[i], (i, j, idx)
        assert abs(v - var[i]) <= 1e-9 * (hf_theta[0] * hf_theta[2] + hf_theta[4] + hf_theta[-1])
        seq._append_hf_point(np.vstack([seq.hf_X, cands[j]]))
    else:
        return
    pytest.fail("near-tie at pick %d: choose another case" % i)


# -- two ranks on one GPU (gloo), as tests/test_gpu_dist.py ---------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


SHARD_CASES = ((20001, 8), (2, 2), (1, 1))         # (C, q); with three ranks C = 2 leaves rank 2 empty


def _shard_cands(C):
    return np.random.default_rng(11).uniform(size=(C, 2))


def _rank(rank, world, port, out):
    import torch
    import torch.distributed as tdist
    import multifidelity_datafusion_gps_b200 as pkg
    torch.cuda.set_device(0)
    tdist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    m = _gpdf(pkg)                                 # deterministic fit at fixed theta: the same state on every rank
    res = [m.acquisition_batch(_shard_cands(C), q, distributed=True) for C, q in SHARD_CASES]
    out.put((rank, [(i.tolist(), v.view(np.int64).tolist()) for i, v in res]))
    tdist.barrier()
    tdist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_batch_matches_the_single_process_bit_for_bit(pkg, world):
    import torch.multiprocessing as mp
    m = _gpdf(pkg)
    ref = []
    for C, q in SHARD_CASES:
        i, v = m.acquisition_batch(_shard_cands(C), q)
        ref.append((i.tolist(), v.view(np.int64).tolist()))
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    res = [out.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for _, r in res:
        assert r == ref


def test_bad_batch_sizes_are_refused(pkg):
    from multifidelity_datafusion_gps_b200 import _ffi, gp
    m = _gpdf(pkg)
    cands = np.random.default_rng(0).uniform(size=(100, 2))
    for q in (0, _ffi.ACQ_MAX_Q + 1):
        with pytest.raises(ValueError):
            m.acquisition_batch(cands, q)
    with pytest.raises(ValueError):
        m.acquisition_batch(cands[:5], 6)              # more picks than candidates
    # the C-ABI refuses them too (rc < 0)
    h = _ffi.get_handle(m.device)
    dXa = m._resident_candidates(cands, 0, len(cands))
    lvl = m.hf_model.level_struct()
    ws = gp.workspace(m.device, h.lib.mfgp_acq_batch_ws_bytes(m.hf_model.N, len(cands), 4))
    val, idx, rec = ctypes.c_double(), ctypes.c_longlong(), np.zeros(1 + m.hf_model.D + _ffi.ACQ_MAX_Q + 1)
    for C, q in ((100, 0), (100, _ffi.ACQ_MAX_Q + 1), (0, 1)):
        rc = h.lib.mfgp_acq_batch_begin(h.h, ctypes.byref(lvl), dXa.data_ptr(), C, q, 1, ws.data_ptr(),
                                        ws.numel() * 8, ctypes.byref(val), ctypes.byref(idx), rec.ctypes.data)
        assert rc < 0, (C, q)
    assert h.lib.mfgp_acq_batch_ws_bytes(m.hf_model.N, 100, 0) == 0
