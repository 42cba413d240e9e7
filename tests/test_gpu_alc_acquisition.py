"""Integrated-variance (ALC) acquisition on the GPU (GPRegression.alc_device, MultifidelityDataFusion.acquisition_alc,
ALCMaximizer, mfgp_alc): values against the NumPy oracle on five model shapes, the identity with append_point, the
arg-max, bit invariance to batching, scratch size and sharding, the adaptation loop, edge shapes, argument errors and
the two resident cache slots."""
import ctypes
import socket

import numpy as np
import pytest

from tests import alc_oracle, util
from tests.test_gpu_batch_acquisition import THETA_R, _case, _gpdf

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg(gpu):
    import multifidelity_datafusion_gps_b200 as pkg
    return pkg


def _ref(n, dim=2, seed=21):
    return np.random.default_rng(seed).uniform(size=(n, dim))


def _level(m):
    hf = m.hf_model
    return hf.kern.kind, hf.X, hf.kern.d, hf.param_array


def _alc(m, cands, ref, w=None, ws_bytes=None):
    """GPU values for plain candidate and reference rows, plus the augmented rows (host) the oracle takes."""
    import torch
    dXc = m._augment_host_input(cands)
    dXr = m._augment_host_input(ref)
    dw = None if w is None else torch.from_numpy(np.ascontiguousarray(w, dtype=np.float64)).to(dXc.device)
    a = m.hf_model.alc_device(dXc, dXr, dw, ws_bytes=ws_bytes)
    return a, dXc, dXr


def _top2_gap(a):
    s = np.sort(a)
    return (s[-1] - s[-2]) / abs(s[-1])


def _bench_like(pkg):
    # N_h = 1024 (npad 1024: several k tiles), 2^16 candidates and R = 1024: the products take the TMA kernel
    rng = np.random.default_rng(1)
    Xh = rng.uniform(size=(1024, 4))
    m = pkg.NARGP(4, util.hf_4d, util.lf_4d)
    m.fit(Xh, theta=np.array([1.0, 0.3, 1.0, 0.3, 0.1, 0.3, 0.01 * util.hf_4d(Xh).var()]))
    return m, np.random.default_rng(0).uniform(size=(1 << 16, 4))


CASES = ["config2_gpdf_d7", "config3_nargp_4d", "nargp_data_driven_lf", "gpdfc_outside_shapes", "nargp_4d_nh1024"]


@pytest.mark.parametrize("name", CASES)
def test_values_and_argmax_match_the_oracle(pkg, name):
    m, cands = _bench_like(pkg) if name == "nargp_4d_nh1024" else _case(pkg, name)
    dim = cands.shape[1]
    R = 1024 if name == "nargp_4d_nh1024" else 256
    ref = _ref(R, dim)
    a, dXc, dXr = _alc(m, cands, ref)
    a = a.cpu().numpy()
    n_or = min(len(cands), 1 << 16)                # the oracle scores a leading subset of the 2^20 candidates
    kind, X, d, theta = _level(m)
    assert m.hf_model.last_jitter == 0.0
    ref_a = alc_oracle.closed_form(kind, X, d, theta, dXc[:n_or].cpu().numpy(), dXr.cpu().numpy())
    assert np.all(np.isfinite(ref_a)) and np.all(np.isfinite(a))
    scale = np.max(ref_a)
    assert np.max(np.abs(a[:n_or] - ref_a)) <= 1e-9 * scale, (name, np.max(np.abs(a[:n_or] - ref_a)), scale)
    # the arg-max through the model, over the candidates the oracle scored
    sub = cands[:n_or] if n_or < len(cands) else cands
    idx, val = m.acquisition_alc(sub, ref)
    assert val == a[idx]                           # the reported value is the candidate's, bit for bit
    if _top2_gap(ref_a) > 1e-9:
        assert idx == int(np.argmax(ref_a)), (name, idx, int(np.argmax(ref_a)))
    if name == "config2_gpdf_d7":                  # and through the maximizer plug-in
        m.adapt_maximizer = pkg.ALCMaximizer(candidates=cands, reference=ref)
        x, fopt = m.get_input_with_highest_uncertainty(m)
        assert np.array_equal(x, cands[idx]) and fopt == -val


def test_alc_is_the_variance_drop_after_append_point(pkg):
    m = _gpdf(pkg)
    ref = _ref(300)
    w = np.random.default_rng(4).uniform(size=300)
    cands = np.random.default_rng(5).uniform(size=(8, 2))
    a, dXc, dXr = _alc(m, cands, ref, w)
    a = a.cpu().numpy()
    kdiag = THETA_R[0]
    for j in range(8):
        f = _gpdf(pkg)                             # fresh model: the same fit at the same theta
        _, before = f.hf_model.predict_device(dXr, True, False)
        f.hf_model.append_point(dXc[j:j + 1].cpu().numpy(), 0.0)   # any y: the variance does not depend on it
        _, after = f.hf_model.predict_device(dXr, True, False)
        before, after = before.cpu().numpy(), after.cpu().numpy()
        assert np.all(after > 1e-12), "the 1e-15 clip must be inactive"
        drop = float(w @ (before - after))
        assert abs(a[j] - drop) <= 1e-10 * kdiag, (j, a[j], drop)


def test_a_candidate_value_does_not_depend_on_batch_or_scratch(pkg):
    from multifidelity_datafusion_gps_b200 import _ffi
    import torch
    m = _gpdf(pkg)
    cands = np.random.default_rng(0).uniform(size=(200001, 2))
    ref = _ref(300)
    dXc, dXr = m._augment_host_input(cands), m._augment_host_input(ref)
    full = m.hf_model.alc_device(dXc, dXr)
    for j in (0, 1, 127, 128, 12345, 200000):
        assert torch.equal(m.hf_model.alc_device(dXc[j:j + 1], dXr), full[j:j + 1]), j
    h = _ffi.get_handle(m.device)
    least = h.lib.mfgp_alc_ws_bytes(m.hf_model.N, 1, 300)
    assert torch.equal(m.hf_model.alc_device(dXc, dXr, ws_bytes=least), full)


def test_edge_shapes(pkg):
    import torch
    for name in ("config2_gpdf_d7", "gpdfc_outside_shapes"):
        m, cands = _case(pkg, name)
        kind, X, d, theta = _level(m)
        for C, R in ((50, 1), (50, 300), (1, 1), (300, 128), (129, 257)):
            ref = _ref(R, seed=R)
            a, dXc, dXr = _alc(m, cands[:C], ref)
            ref_a = alc_oracle.closed_form(kind, X, d, theta, dXc.cpu().numpy(), dXr.cpu().numpy())
            assert np.max(np.abs(a.cpu().numpy() - ref_a)) <= 1e-9 * np.max(ref_a), (name, C, R)
            b, _, _ = _alc(m, cands[:C], ref, np.full(R, 1.0 / R))
            assert torch.equal(a, b), (name, C, R)      # explicit 1/R weights equal the default bit for bit
            w = np.random.default_rng(R).uniform(size=R)
            c, _, _ = _alc(m, cands[:C], ref, w)
            ref_c = alc_oracle.closed_form(kind, X, d, theta, dXc.cpu().numpy(), dXr.cpu().numpy(), w)
            assert np.max(np.abs(c.cpu().numpy() - ref_c)) <= 1e-9 * np.max(ref_c), (name, C, R)


def test_bad_arguments_are_refused_before_any_launch(pkg):
    import torch
    from multifidelity_datafusion_gps_b200 import _ffi, gp
    m = _gpdf(pkg)
    cands, ref = np.random.default_rng(0).uniform(size=(100, 2)), _ref(20)
    dXc, dXr = m._augment_host_input(cands), m._augment_host_input(ref)
    hf = m.hf_model
    h = _ffi.get_handle(m.device)
    lvl = hf.level_struct()
    torch.cuda.synchronize()
    n0 = h.launches
    with pytest.raises(ValueError):
        hf.alc_device(dXc, dXr[:0])
    with pytest.raises(ValueError):
        m.acquisition_alc(cands, ref[:0])
    with pytest.raises(ValueError):
        hf.alc_device(dXc, dXr, torch.ones(19, dtype=torch.float64, device=dXc.device))
    for w in (np.ones(21), -np.ones(20), np.zeros(20), np.full(20, np.nan)):
        with pytest.raises(ValueError):
            m.acquisition_alc(cands, ref, w)
    least = h.lib.mfgp_alc_ws_bytes(hf.N, 1, 20)
    with pytest.raises(_ffi.MfgpError):
        hf.alc_device(dXc, dXr, ws_bytes=least - 8)
    ws = gp.workspace(m.device, least)
    out = torch.empty(100, dtype=torch.float64, device=dXc.device)
    for C, R, nb in ((100, 0, least), (0, 20, least), (100, -1, least), (100, 20, least - 8), (100, 20, 0)):
        rc = h.lib.mfgp_alc(h.h, ctypes.byref(lvl), dXc.data_ptr(), C, dXr.data_ptr(), R, None, 0.0,
                            out.data_ptr(), ws.data_ptr(), nb)
        assert rc < 0, (C, R, nb)
    assert h.lib.mfgp_alc(h.h, ctypes.byref(lvl), dXc.data_ptr(), 100, dXr.data_ptr(), 20, None, -1.0,
                          out.data_ptr(), ws.data_ptr(), least) < 0
    assert h.launches == n0


def test_both_cache_slots_are_reused_and_rebuilt(pkg):
    m, cands = _case(pkg, "nargp_data_driven_lf")
    ref = _ref(200)
    idx, val = m.acquisition_alc(cands, ref)
    c0, r0 = getattr(m, "candidate_cache_hits", 0), getattr(m, "reference_cache_hits", 0)
    assert (m.acquisition_alc(cands, ref)) == (idx, val)
    assert m.candidate_cache_hits == c0 + 1 and m.reference_cache_hits == r0 + 1
    m.acquisition_argmax(cands)                    # the ALC call left the candidate rows resident
    assert m.candidate_cache_hits == c0 + 2
    m.lf_model._set_params(np.array([1.4, 0.45, 1e-3]))   # a low-fidelity change: both slots are rebuilt
    m.acquisition_alc(cands, ref)
    assert m.candidate_cache_hits == c0 + 2 and m.reference_cache_hits == r0 + 1
    m.acquisition_alc(cands, ref)
    assert m.candidate_cache_hits == c0 + 3 and m.reference_cache_hits == r0 + 2
    m.invalidate_candidate_cache()
    m.acquisition_alc(cands, ref)
    assert m.candidate_cache_hits == c0 + 3 and m.reference_cache_hits == r0 + 2


def test_adapt_follows_the_oracle_sequential_alc_loop(pkg):
    cands, ref = np.random.default_rng(7).uniform(size=(4000, 2)), _ref(200)
    m = _gpdf(pkg, pkg.ALCMaximizer(candidates=cands, reference=ref))
    kind, X, d, theta = _level(m)
    Xc = m._augment_host_input(cands).cpu().numpy()
    Xr = m._augment_host_input(ref).cpu().numpy()
    steps = 5
    ref_idx, ref_val, gaps = alc_oracle.sequential_picks(kind, X, d, theta, Xc, Xr, steps)
    m.refit_every = steps + 1                      # fixed theta: bordered updates only
    m.adapt(steps, eps=0.0)
    assert len(m.acquired_points) == steps and m.hf_model.N == 30 + steps
    for i, (x, fopt) in enumerate(m.acquired_points):
        if gaps[i] <= 1e-9:
            break
        assert np.array_equal(x, cands[ref_idx[i]]), (i, x, cands[ref_idx[i]])
        assert abs(fopt + ref_val[i]) <= 1e-9 * ref_val[0], (i, fopt, ref_val[i])
    else:
        return
    pytest.fail("near-tie at step %d: choose another case" % i)


def test_adapt_with_the_default_refit_runs_end_to_end(pkg):
    m = _gpdf(pkg, pkg.ALCMaximizer(n_candidates=20000, n_reference=256, seed=3))
    Xt = np.random.default_rng(8).uniform(size=(500, 2))
    m.adapt(2, plot_mode="e", X_test=Xt, Y_test=util.hf_2d(Xt))
    assert len(m.acquired_points) == 2 and m.hf_X.shape == (32, 2) and m.hf_model.N == 32
    for x, fopt in m.acquired_points:
        assert np.all((x >= 0.0) & (x <= 1.0)) and fopt < 0.0
    assert len(m.mse_history) == 2 and np.all(np.isfinite(m.mse_history))


# -- two ranks on one GPU (gloo), as tests/test_gpu_dist.py ---------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


SHARD_CASES = (20001, 129, 1)                     # with two ranks C = 1 leaves rank 1 empty


def _shard_inputs(C):
    return np.random.default_rng(11).uniform(size=(C, 2)), _ref(300)


def _rank(rank, world, port, out):
    import torch
    import torch.distributed as tdist
    import multifidelity_datafusion_gps_b200 as pkg
    torch.cuda.set_device(0)
    tdist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    m = _gpdf(pkg)                                 # deterministic fit at fixed theta: the same state on every rank
    res = []
    for C in SHARD_CASES:
        i, v = m.acquisition_alc(*_shard_inputs(C), distributed=True)
        res.append((i, np.float64(v).view(np.int64).item()))
    out.put((rank, res))
    tdist.barrier()
    tdist.destroy_process_group()


def test_sharded_alc_matches_the_single_process_bit_for_bit(pkg):
    import torch.multiprocessing as mp
    m = _gpdf(pkg)
    ref = []
    for C in SHARD_CASES:
        i, v = m.acquisition_alc(*_shard_inputs(C))
        ref.append((i, np.float64(v).view(np.int64).item()))
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
    for _, r in res:
        assert r == ref
