"""Greedy batch acquisition without a GPU: the oracle's definition against an independent pivoted-Cholesky
formulation and against the oracle's own sequential adaptation, the batch adaptation loop on stubs, and the
record exchange of the sharded batch over two gloo ranks."""
import socket

import numpy as np
import pytest

from oracle import gpy_oracle as go
from oracle import mfgp_oracle as mo
from tests import util
from tests.batch_oracle import candidate_batch

THETA_R = np.array([1.2, 0.9, 1e-3])


def _gpdf_oracle(n_hf=12, seed=10):
    X_hf = np.random.RandomState(seed).uniform(size=(n_hf, 2))
    o = mo.OracleMFGP(2, 2, 0.001, util.hf_2d, f_low=util.lf_2d, use_composite_kernel=False, form="direct")
    o.fit(X_hf, theta=THETA_R)
    return o


def _pivoted_cholesky(Sigma, noise, s2, q):
    """Greedy pivoted partial Cholesky of the latent posterior covariance Sigma (C x C) with observation noise s2:
    pick = argmax max(v, 1e-15) + noise, then v -= r^2 with r = (Sigma[:, p] - R^T R[:, p]) / sqrt(v[p] + s2)."""
    v = np.diag(Sigma).copy()
    R = np.zeros((q, Sigma.shape[0]))
    idx, var = [], []
    for i in range(q):
        rep = np.maximum(v, go.VAR_CLIP) + noise
        p = int(np.argmax(rep))
        idx.append(p)
        var.append(rep[p])
        r = (Sigma[:, p] - R[:i].T.dot(R[:i, p])) / np.sqrt(v[p] + s2)
        R[i] = r
        v = v - r * r
    return np.array(idx), np.array(var)


def test_oracle_batch_equals_pivoted_cholesky_of_the_posterior_covariance():
    o = _gpdf_oracle()
    cands = np.random.default_rng(4).uniform(size=(400, 2))
    q = 10
    idx, var, gaps = candidate_batch(o, cands, q)
    hf = o.hf_model
    Xc = o.augment(cands)
    theta_k, noise = go.split_theta(hf.kind, hf.theta)
    L, _ = hf.posterior()
    Kxc = go.kernel_K(hf.kind, hf.X, Xc, hf.d, theta_k, "direct")
    T = np.linalg.solve(L, Kxc)
    Sigma = go.kernel_K(hf.kind, Xc, None, hf.d, theta_k, "direct") - T.T.dot(T)
    ref_idx, ref_var = _pivoted_cholesky(Sigma, noise, noise + go.JITTER_CONST, q)
    scale = theta_k[0] + noise
    for i in range(q):
        if gaps[i] <= 1e-9:                       # a near-tie may legitimately break either way: stop comparing
            break
        assert idx[i] == ref_idx[i], i
        assert abs(var[i] - ref_var[i]) <= 1e-9 * scale, (i, var[i], ref_var[i])
    else:
        assert np.array_equal(idx, ref_idx)
    assert np.all(np.diff(var) <= 1e-12 * scale)   # conditioning never raises a variance
    assert len(set(idx.tolist())) > 1


def test_oracle_batch_equals_sequential_adaptation_at_fixed_theta():
    # the picks do not depend on the targets: q refits on f_exact's values pick what the batch picks without them
    cands = np.random.default_rng(5).uniform(size=(400, 2))
    q = 6
    idx, var, gaps = candidate_batch(_gpdf_oracle(), cands, q)
    assert np.all(gaps > 1e-9), gaps
    seq = _gpdf_oracle()
    acquired = seq.adapt(q, mo.make_candidate_maximizer(cands), eps=0.0, fit_kwargs=dict(theta=THETA_R))
    assert len(acquired) == q
    for i, (x, fopt) in enumerate(acquired):
        assert np.array_equal(x, cands[idx[i]]), i
        assert abs(-fopt - var[i]) <= 1e-9 * (THETA_R[0] + THETA_R[-1]), i


# -- the adaptation loop on stubs -----------------------------------------------------------------------------
class _StubMaximizer:
    """Scripted (X, fopt) per call; records which entry point the loop used."""

    def __init__(self, batches, d=2):
        self.batches = list(batches)
        self.calls = []
        self.d = d

    def maximize(self, model_predict, lower_bound, upper_bound):
        self.calls.append(("maximize",))
        X, f = self.batches.pop(0)
        return X[0], f[0]

    def maximize_batch(self, model_predict, lower_bound, upper_bound, q):
        self.calls.append(("maximize_batch", q))
        X, f = self.batches.pop(0)
        return X[:q], f[:q]


def _stub_model(maximizer, refit_every=1, batch=1):
    from multifidelity_datafusion_gps_b200.abstractMFGP import AbstractMFGP

    class Stub(AbstractMFGP):
        def __init__(self):
            super().__init__(name="stub", input_dim=2, num_derivatives=0, tau=0.0, f_exact=None, lower_bound=None,
                             upper_bound=None, f_low=None, lf_X=None, lf_Y=None, lf_hf_adapt_ratio=1,
                             use_composite_kernel=True, adapt_maximizer=maximizer, eps=1e-8)
            self.log = []
            self.hf_X = np.zeros((3, 2))

        def fit(self, hf_X):
            self.log.append(("fit", len(hf_X)))
            self.hf_X = hf_X

        def _append_hf_point(self, new_hf_X):
            self.log.append(("append", len(new_hf_X)))
            self.hf_X = new_hf_X

        def _append_hf_points(self, new_hf_X, k):
            self.log.append(("append_block", len(new_hf_X), k))
            self.hf_X = new_hf_X

        def adapt(self, adapt_steps, plot_mode=None, X_test=None, Y_test=None, eps=1e-8):
            self.adapt_steps, self.X_test, self.Y_test, self.eps = adapt_steps, X_test, Y_test, eps
            self.adapt_and_plot(plot_error=X_test is not None)

        def predict(self, X_test):
            return np.zeros((len(X_test), 1)), np.ones((len(X_test), 1))

        def get_mse(self, X_test, Y_test):
            self.log.append(("mse",))
            return 0.5

    m = Stub()
    m.refit_every = refit_every
    m.adapt_batch_size = batch
    return m


def _batch(q, fopt=None, seed=0):
    X = np.random.default_rng(seed).uniform(size=(q, 2))
    return X, np.asarray(fopt if fopt is not None else -np.linspace(1.0, 0.5, q))


def test_batch_loop_truncates_after_the_first_point_below_eps():
    X, f = _batch(4, [-1.0, -0.5, -1e-10, -0.3])
    mx = _StubMaximizer([(X, f), _batch(4, seed=1)])
    m = _stub_model(mx, refit_every=5, batch=4)
    m.adapt(3, X_test=np.zeros((2, 2)), Y_test=np.zeros((2, 1)))
    # the point with |fopt| < eps is acquired and the loop stops after it, as the sequential loop does
    assert len(m.acquired_points) == 3 and m.adapt_steps == 1
    assert all(np.array_equal(m.acquired_points[j][0], X[j]) for j in range(3))
    assert [p[1] for p in m.acquired_points] == [-1.0, -0.5, -1e-10]
    assert m.log == [("mse",), ("append_block", 6, 3)]
    assert mx.calls == [("maximize_batch", 4)] and m.hf_X.shape == (6, 2)


def test_batch_loop_refits_on_refit_steps_and_appends_blocks_between():
    batches = [_batch(3, seed=s) for s in range(4)]
    mx = _StubMaximizer(batches)
    m = _stub_model(mx, refit_every=2, batch=3)
    m.adapt(4)
    assert m.log == [("append_block", 6, 3), ("fit", 9), ("append_block", 12, 3), ("fit", 15)]
    assert mx.calls == [("maximize_batch", 3)] * 4
    assert len(m.acquired_points) == 12 and m.adapt_steps == 4
    assert np.array_equal(m.hf_X[3:], np.vstack([b[0] for b in batches]))


def test_batch_size_one_runs_todays_loop():
    batches = [_batch(1, seed=s) for s in range(3)]
    mx = _StubMaximizer(batches)
    m = _stub_model(mx, refit_every=2, batch=1)
    m.adapt(3, X_test=np.zeros((2, 2)), Y_test=np.zeros((2, 1)))
    assert mx.calls == [("maximize",)] * 3
    assert m.log == [("mse",), ("append", 4), ("mse",), ("fit", 5), ("mse",), ("append", 6)]


def test_appended_block_calls_f_exact_once_then_appends_row_by_row():
    # MultifidelityDataFusion._append_hf_points on a host-only instance (no GPU): the high-fidelity GP is a recorder
    from multifidelity_datafusion_gps_b200.MFDataFusion import MultifidelityDataFusion
    from multifidelity_datafusion_gps_b200.augm_iterators import BackwardAugmentation
    calls = []

    def f_exact(X):
        calls.append(np.array(X))
        return util.hf_2d(X)

    class Recorder:
        def __init__(self):
            self.rows = []

        def append_point(self, x_row, y):
            self.rows.append((np.array(x_row), np.array(y)))

    m = MultifidelityDataFusion.__new__(MultifidelityDataFusion)
    m.input_dim, m.tau, m.f_exact, m.f_low = 2, 0.001, f_exact, util.lf_2d
    m.augm_iterator = BackwardAugmentation(2, dim=2)
    m.data_driven_lf_approach = False
    m.hf_X = np.random.default_rng(0).uniform(size=(4, 2))
    m.hf_Y = util.hf_2d(m.hf_X)
    m.hf_model = Recorder()
    X_new = np.random.default_rng(1).uniform(size=(3, 2))
    m._append_hf_points(np.vstack([m.hf_X, X_new]), 3)
    assert len(calls) == 1 and np.array_equal(calls[0], X_new)
    assert m.hf_X.shape == (7, 2) and np.array_equal(m.hf_Y[4:], util.hf_2d(X_new))
    assert len(m.hf_model.rows) == 3
    aug = m.augment_data(X_new)
    for j, (x_row, y) in enumerate(m.hf_model.rows):
        assert x_row.shape == (1, 7) and np.array_equal(x_row[0], aug[j])
        assert y.shape == (1, 1) and y[0, 0] == util.hf_2d(X_new[j:j + 1])[0, 0]


def test_default_maximizer_refuses_batches_it_cannot_condition():
    from multifidelity_datafusion_gps_b200.adaptation_maximizers import ScipyDirectMaximizer
    with pytest.raises(NotImplementedError):
        ScipyDirectMaximizer().maximize_batch(lambda X: None, np.zeros(2), np.ones(2), 2)


# -- record exchange over two gloo ranks ----------------------------------------------------------------------
def test_shard_owner_inverts_shard_range():
    from multifidelity_datafusion_gps_b200 import dist
    for n in (1, 2, 3, 7, 100, 101):
        for world in (1, 2, 3, 4, 8):
            for r in range(world):
                lo, hi = dist.shard_range(n, r, world)
                assert all(dist.shard_owner(i, n, world) == r for i in range(lo, hi))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _record(rank, n=40):
    """Per-rank record with bit patterns a lossy path would disturb: -0.0, a denormal, NaN payloads, inf."""
    bits = np.random.default_rng(100 + rank).integers(0, 2 ** 63, size=n, dtype=np.int64)
    rec = bits.view(np.float64).copy()
    rec[:5] = [-0.0, 5e-324, np.inf, -np.inf, 1.0 + 2.0 ** -52]
    rec[5:7] = np.array([0x7FF8000000000123, 0x7FF0000000000001], dtype=np.int64).view(np.float64)
    return rec


def _rank(rank, world, port, out):
    import torch.distributed as tdist
    from multifidelity_datafusion_gps_b200 import dist
    tdist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    res = []
    for C, winner in ((10, 7), (10, 2), (1, 0)):          # C = 1: rank 1 holds no candidate
        lo, hi = dist.shard_range(C, rank, world)
        val, idx = (float(winner), winner) if lo <= winner < hi else (-np.inf, -1)
        gv, gi = dist.gather_argmax(val, idx)
        owner = dist.shard_owner(gi, C, world)
        rec = dist.broadcast_record(_record(rank), owner)
        res.append((gi, owner, rec.view(np.int64).tolist()))
    out.put((rank, res))
    tdist.barrier()
    tdist.destroy_process_group()


def test_record_exchange_over_two_gloo_ranks_is_bit_exact():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(out.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    expect = [(7, 1), (2, 0), (0, 0)]
    for r in (0, 1):
        for (gi, owner, rec), (w, o) in zip(res[r], expect):
            assert (gi, owner) == (w, o)
            assert rec == _record(o).view(np.int64).tolist()
