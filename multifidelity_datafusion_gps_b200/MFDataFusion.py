"""MultifidelityDataFusion -- the reference's concrete model (src/MFDataFusion.py:13-208) on the
B200 GP engine.  Same constructor, same ``fit / adapt / predict / get_mse`` contracts (NumPy in,
NumPy out, ``assert``-based validation).  What changes underneath:

* ``__augment_Data`` (:177-208): the reference maps a Python lambda over rows twice; here a callable
  ``f_low`` is evaluated ONCE on all M*E augmented locations (host, vectorised), and a data-driven
  low-fidelity GP is evaluated on the GPU for all locations in one batched kernel (mfgp_augment).
* ``fit`` (:75-100): every LML+gradient of the ARD recipe is one GPU evaluation.
* ``predict`` (:141-156): fused cross-covariance -> mean -> W Kx -> variance on the GPU.

Extensions (keyword-only, defaults reproduce the reference):
* ``predict_mc``  Monte-Carlo propagation of the low-fidelity posterior (README.md:13; absent in the
  reference, which collapses the LF level to its mean, src/abstractMFGP.py:104).
* ``acquisition_argmax``  candidate-set arg-max of the predictive variance (used by
  ``CandidateSetMaximizer``), optionally sharded over ranks.
* ``acquisition_batch``  greedy batch of q candidates per adaptation step (``adapt_batch_size``).
* ``acquisition_alc``  candidate-set arg-max of the integrated-variance reduction over a reference set
  (used by ``ALCMaximizer``), optionally sharded over ranks.
* ``broadcast_state``  NCCL broadcast of the fitted state so that other ranks can predict.
"""
import ctypes
import zlib

import numpy as np
import torch

from . import _ffi, dist, gp
from .abstractMFGP import AbstractMFGP
from .adaptation_maximizers import AbstractMaximizer, ScipyDirectMaximizer
from .adaptation_maximizers.alc_maximizer import alc_weights
from .augm_iterators import BackwardAugmentation


class MultifidelityDataFusion(AbstractMFGP):
    """Regression model for a scarce/precise (high-fidelity) and an abundant/imprecise (low-fidelity)
    data source; see the reference docstring (src/MFDataFusion.py:14-54) for the parameters."""

    def __init__(self, name: str, input_dim: int, num_derivatives: int, tau: float, f_exact: callable,
                 lower_bound: np.ndarray = None, upper_bound: float = None, f_low: callable = None,
                 lf_X: np.ndarray = None, lf_Y: np.ndarray = None, lf_hf_adapt_ratio: int = 1,
                 use_composite_kernel: bool = True, adapt_maximizer: AbstractMaximizer = None,
                 eps: float = 1e-8, add_noise: bool = False, augm_iterator=None):
        if adapt_maximizer is None:
            adapt_maximizer = ScipyDirectMaximizer()      # the reference's default (:59)
        super().__init__(name=name, input_dim=input_dim, num_derivatives=num_derivatives, tau=tau,
                         f_exact=f_exact, lower_bound=lower_bound, upper_bound=upper_bound, f_low=f_low,
                         lf_X=lf_X, lf_Y=lf_Y, lf_hf_adapt_ratio=lf_hf_adapt_ratio,
                         use_composite_kernel=use_composite_kernel, adapt_maximizer=adapt_maximizer,
                         eps=eps)
        # The reference hard-wires BackwardAugmentation here (:67) although it ships EvenAugmentation too
        # (src/augm_iterators/even_augm_iterator.py); `augm_iterator` (extension) selects the delay
        # pattern: None / "backward", "even", an AbstractAugmIterator class or a ready instance.
        if augm_iterator is None or augm_iterator == "backward":
            augm_iterator = BackwardAugmentation
        elif augm_iterator == "even":
            from .augm_iterators import EvenAugmentation
            augm_iterator = EvenAugmentation
        if isinstance(augm_iterator, type):
            augm_iterator = augm_iterator(self.num_derivatives, dim=input_dim)
        assert augm_iterator.dim == input_dim, "delay iterator / input dimension mismatch"
        self.augm_iterator = augm_iterator
        self.initialize_kernel(use_composite_kernel)
        self.initialize_lf_level(f_low, lf_X, lf_Y)
        self.add_noise = add_noise
        self.device = gp.current_device()

    # -- A5 fit -----------------------------------------------------------------------------------
    def fit(self, hf_X, theta=None):
        """Fit the high-fidelity GP on the augmented inputs.  ``theta`` (extension): skip the
        optimiser and install these hyper-parameters (parity tests at fixed theta)."""
        assert hf_X.ndim == 2, "invalid input shape"
        assert hf_X.shape[1] == self.input_dim, "invalid input dim"
        self.hf_X = hf_X
        self.hf_Y = self.f_exact(self.hf_X)
        assert self.hf_Y.shape == (self.hf_X.shape[0], 1)
        self.hf_model = gp.GPRegression(X=self.__augment_Data(self.hf_X), Y=self.hf_Y,
                                        kernel=self.kernel, initialize=True)
        if theta is None:
            self.ARD(self.hf_model, 6)
        else:
            self.hf_model._set_params(np.asarray(theta, dtype=np.float64))

    def _append_hf_point(self, new_hf_X):
        """Last row of new_hf_X joins the high-fidelity GP at fixed hyper-parameters: O(N^2) bordered
        update of (L, L^-1, alpha) on the GPU (gp.GPRegression.append_point) instead of a refit."""
        x = np.atleast_2d(new_hf_X[-1])
        y = np.asarray(self.f_exact(x), dtype=np.float64).reshape(1, 1)
        self.hf_X = new_hf_X
        self.hf_Y = np.vstack((self.hf_Y, y))
        self.hf_model.append_point(self.__augment_Data(x), y)

    def _append_hf_points(self, new_hf_X, k):
        """The last k rows of new_hf_X (one acquired batch) join the high-fidelity GP at fixed hyper-parameters:
        f_exact is called ONCE on the (k, d) block -- the expensive simulations of a batch run together -- and the
        rows then enter by bordered updates, in order."""
        X = np.atleast_2d(new_hf_X[len(new_hf_X) - k:])
        Y = np.asarray(self.f_exact(X), dtype=np.float64).reshape(k, 1)
        self.hf_X = new_hf_X
        self.hf_Y = np.vstack((self.hf_Y, Y))
        Xa = self.__augment_Data(X)
        for j in range(k):
            self.hf_model.append_point(Xa[j:j + 1], Y[j:j + 1])

    # -- A10 adapt --------------------------------------------------------------------------------
    def adapt(self, adapt_steps: int, plot_mode: str = None, X_test: np.ndarray = None,
              Y_test: np.ndarray = None, eps: float = 1e-8):
        """Acquire `adapt_steps` new high-fidelity points where the predictive variance is largest.
        plot_mode is accepted for compatibility ('u','m','e','um','mu',None); nothing is drawn."""
        self.adapt_steps = adapt_steps
        self.X_test = X_test
        self.Y_test = Y_test
        self.eps = eps
        # The reference calls self.__adapt_lf() here for a data-driven LF level, a method that does
        # not exist (AttributeError).  Low-fidelity adaptation is skipped (SURVEY.md section 5).
        modes = {'u': dict(plot_uncertainties=True), 'm': dict(plot_means=True), 'e': dict(plot_error=True),
                 'um': dict(plot_means=True, plot_uncertainties=True),
                 'mu': dict(plot_means=True, plot_uncertainties=True), None: dict()}
        assert plot_mode in modes.keys(), "Invalid plot mode. Select one of these: {}".format(list(modes.keys()))
        self.adapt_and_plot(**modes[plot_mode])

    # -- A6 predict -------------------------------------------------------------------------------
    def predict(self, X_test):
        """(mean (M,1), variance (M,1)); the variance includes the noise variance (GPy semantics)."""
        assert X_test.ndim == 2
        assert X_test.shape[1] == self.input_dim
        self._apply_add_noise()
        mean, var = self.hf_model.predict_device(self._augment_host_input(X_test), True, True)
        return mean.cpu().numpy()[:, None], var.cpu().numpy()[:, None]

    def predict_point(self, X_test):
        """``predict`` for a handful of rows at minimum latency (mfgp_predict_small: one or two launches, one
        synchronisation, inputs and results through mapped host memory) -- what one objective evaluation of
        the reference's default DIRECT acquisition costs (src/adaptation_maximizers/scipydirect_wrapper.py:22-26).
        Same formulas as ``predict``; other summation orders, so equal to round-off, not bit for bit (which is
        why ``predict`` itself never switches kernels with the batch size).  Falls back to ``predict`` for
        shapes the latency kernels do not serve."""
        X_test = np.ascontiguousarray(X_test, dtype=np.float64)
        assert X_test.ndim == 2 and X_test.shape[1] == self.input_dim
        h = _ffi.get_handle(self.device)
        M = X_test.shape[0]
        dev_f = getattr(self.f_low, "device_predict", None)
        E = self.augm_iterator.new_entries_count()
        if (M < 1 or M > h.lib.mfgp_predict_small_max_rows() or self.hf_model.N > 2048 or dev_f is not None
                or M * (self.input_dim + E) > 128 or E * self.input_dim > 96):
            return self.predict(X_test)
        self._apply_add_noise()
        hf = self.hf_model.level_struct()
        mean, var = np.empty(M), np.empty(M)
        vp = ctypes.c_void_p
        if self.data_driven_lf_approach:
            lf = self.lf_model.level_struct()
            offs = np.ascontiguousarray(self.augm_iterator.offset_table(), dtype=np.float64)
            rc = h.lib.mfgp_predict_small(h.h, ctypes.byref(hf), ctypes.byref(lf), X_test.ctypes.data, M,
                                          offs.ctypes.data, E, float(self.tau), 1, mean.ctypes.data, var.ctypes.data)
        else:
            offsets = self.augm_iterator.offset_table()
            Xa = np.ascontiguousarray(np.concatenate(
                [X_test, self._f_low_batched(X_test[:, None, :] + offsets[None, :, :] * self.tau)], axis=1))
            rc = h.lib.mfgp_predict_small(h.h, ctypes.byref(hf), None, Xa.ctypes.data, M, None, 0, 0.0, 1,
                                          mean.ctypes.data, var.ctypes.data)
        h.check(rc)
        return mean[:, None], var[:, None]

    # -- resident form of predict_point: what the default DIRECT maximiser drives ---------------------------
    def point_service_start(self, idle_ms=20.0):
        """Put the single-row predictor on the device as a RESIDENT kernel (mfgp_point_service_start) for a run
        of sequential single-point questions -- the reference's default acquisition asks up to 20 000 of them,
        each depending on the previous answer (src/adaptation_maximizers/scipydirect_wrapper.py:22-26).
        Returns False (nothing started) for shapes the service does not take; pair with point_service_stop()."""
        h = _ffi.get_handle(self.device)
        E = self.augm_iterator.new_entries_count()
        if (getattr(self.f_low, "device_predict", None) is not None or self.hf_model.N > 2048
                or self.input_dim + E > 64 or E * self.input_dim > 96):
            return False
        self._apply_add_noise()
        self.hf_model._ensure_posterior()
        self._svc_levels = [self.hf_model.level_struct()]           # keep the structs alive while the kernel runs
        offs = np.ascontiguousarray(self.augm_iterator.offset_table(), dtype=np.float64)
        if self.data_driven_lf_approach:
            self.lf_model._ensure_posterior()
            self._svc_levels.append(self.lf_model.level_struct())
            h.check(h.lib.mfgp_point_service_start(h.h, ctypes.byref(self._svc_levels[0]),
                                                   ctypes.byref(self._svc_levels[1]), offs.ctypes.data, E,
                                                   float(self.tau), 1, float(idle_ms)))
            self._svc_x = np.empty(self.input_dim)
        else:
            h.check(h.lib.mfgp_point_service_start(h.h, ctypes.byref(self._svc_levels[0]), None, None, 0, 0.0, 1,
                                                   float(idle_ms)))
            self._svc_x = np.empty(self.input_dim + E)
        self._svc_offs_tau = offs * self.tau
        self._svc_out = np.empty(2)
        self._svc_call = (h.lib.mfgp_point_service_eval, h.h, self._svc_x.ctypes.data, self._svc_out.ctypes.data)
        self._svc_handle = h
        return True

    def point_service_eval(self, x):
        """(mean, variance) at ONE input x (input_dim,), through the resident kernel; bit-identical to
        predict_point(x[None])."""
        fn, hh, px, po = self._svc_call
        d = self.input_dim
        if self.data_driven_lf_approach:
            self._svc_x[:] = x
        else:
            self._svc_x[:d] = x
            # one call of the user's low-fidelity function per (E, d) group, as the reference makes it
            # (src/MFDataFusion.py:197)
            self._svc_x[d:] = np.asarray(self.f_low(np.asarray(x)[None, :] + self._svc_offs_tau)).ravel()
        rc = fn(hh, px, po)
        if rc:
            self._svc_handle.check(rc)
        return self._svc_out[0], self._svc_out[1]

    def point_service_stop(self):
        h = getattr(self, "_svc_handle", None)
        if h is not None:
            h.check(h.lib.mfgp_point_service_stop(h.h))
            self._svc_handle = None
            self._svc_levels = None

    def _apply_add_noise(self):
        if self.add_noise:                                  # :154-155: re-inference at noise 1e-6
            if self.hf_model.likelihood.variance != 1e-6:
                self.hf_model.likelihood.variance = 1e-6

    def _predict_device(self, dX):
        dXa = self._augment_device(dX)
        self._apply_add_noise()
        return self.hf_model.predict_device(dXa, True, True)

    # -- predictive gradients (extension) -----------------------------------------------------------
    def _f_low_jacobian(self, locations):
        """d f_low / d x at (n, d) host locations -> (n, d).  A data-driven LF level: its mean-only predictive
        gradients on the device.  A callable: its ``gradient(locations)`` if it has one, otherwise central differences
        (step 1e-6 max(1, |x_i|)) over the 2 d shifted location sets in one vectorised f_low evaluation."""
        n, d = locations.shape
        if self.data_driven_lf_approach:
            dmean, _, _, _ = self.lf_model.predictive_gradients_device(gp.to_device(locations, self.device), False)
            return dmean.cpu().numpy()
        grad = getattr(self.f_low, "gradient", None)
        if grad is not None:
            J = np.asarray(grad(locations), dtype=np.float64)
            assert J.shape == (n, d), "f_low.gradient must return one row of d partial derivatives per location"
            return J
        step = 1e-6 * np.maximum(1.0, np.abs(locations))                       # (n, d)
        shifted = np.empty((2, d, n, d))
        for i in range(d):
            for s, sign in enumerate((1.0, -1.0)):
                shifted[s, i] = locations
                shifted[s, i, :, i] += sign * step[:, i]
        vals = self._f_low_batched(shifted.reshape(2 * d * n, 1, d)).reshape(2, d, n)
        return ((vals[0] - vals[1]) / (2.0 * step.T)).T

    def predictive_gradients_device(self, dX, include_noise=True):
        """dX (M, d) CUDA -> (dmean (M, d), dvar (M, d), mean (M,), var (M,)) CUDA tensors: the gradients of the
        predictive mean and of the latent variance with respect to the plain inputs x, by the chain rule through the
        augmentation [x, f_low(x + o_e tau)]; mean and var are ``predict``'s outputs to round-off."""
        d, E = self.input_dim, self.augm_iterator.new_entries_count()
        self._apply_add_noise()
        dXa = self._augment_device(dX)
        gm, gv, mean, var = self.hf_model.predictive_gradients_device(dXa, True, include_noise)
        offs = torch.from_numpy(np.ascontiguousarray(self.augm_iterator.offset_table() * self.tau)).to(dX.device)
        loc = (dX[:, None, :] + offs[None, :, :]).reshape(-1, d)
        J = torch.from_numpy(np.ascontiguousarray(self._f_low_jacobian(loc.cpu().numpy()))).to(dX.device)
        J = J.reshape(-1, E, d)
        dmean, dvar = gm[:, :d].clone(), gv[:, :d].clone()
        for e in range(E):              # element-wise, in a fixed order: a row's result does not depend on M
            dmean += gm[:, d + e, None] * J[:, e, :]
            dvar += gv[:, d + e, None] * J[:, e, :]
        return dmean, dvar, mean, var

    def predictive_gradients(self, X):
        """GP.predictive_gradients with respect to the plain inputs: (dmu_dX (M, d, 1), dv_dX (M, d)) as NumPy."""
        X = np.ascontiguousarray(X, dtype=np.float64)
        assert X.ndim == 2 and X.shape[1] == self.input_dim
        dmean, dvar, _, _ = self.predictive_gradients_device(gp.to_device(X, self.device))
        return dmean.cpu().numpy()[:, :, None], dvar.cpu().numpy()

    def variance_and_gradient(self, X):
        """(var (M,), dvar (M, d)) as NumPy: the predictive variance as ``predict`` reports it (to round-off) and its
        gradient, which is zero where the clip at 1e-15 holds the latent variance.  What LBFGSBMaximizer asks."""
        X = np.ascontiguousarray(X, dtype=np.float64)
        _, dvar, _, var = self.predictive_gradients_device(gp.to_device(X, self.device), include_noise=False)
        v, g = var.cpu().numpy(), dvar.cpu().numpy()
        g[v <= 1e-15] = 0.0
        return v + self.hf_model.likelihood.variance, g

    def get_mse(self, X_test, Y_test):
        assert len(X_test) == len(Y_test), 'unequal number of X and y values'
        assert X_test.shape[1] == self.input_dim, 'wrong input value dimension'
        assert Y_test.shape[1] == 1, 'target values must be scalars'
        preds, _ = self.predict(X_test)
        return float(np.mean((np.asarray(Y_test) - preds) ** 2))

    # -- A1 augmentation --------------------------------------------------------------------------
    def _f_low_batched(self, locations):
        """Host callable f_low on (M, E, d) locations -> (M, E).  The reference calls f_low once per
        (E, d) group (:197).  Whether the callable is also row-wise on a stack of groups is probed ONCE
        per callable -- the first group through the reference's call, then the first two groups stacked,
        which must return one value per row and reproduce the first group -- and cached; genuine errors
        of f_low propagate from the reference-style call instead of being swallowed."""
        M, E = locations.shape[0], locations.shape[1]
        if M == 0:
            return np.zeros((0, E))
        flat = locations.reshape(M * E, self.input_dim)
        mode = getattr(self, "_f_low_mode", None)
        if mode is None or mode[0] is not self.f_low:
            first = np.asarray(self.f_low(locations[0]), dtype=np.float64)       # errors surface here, as in :197
            assert first.size == E, "f_low must return one value per row"
            n = min(M, 2) * E
            rowwise = False
            try:
                probe = np.asarray(self.f_low(flat[:n]), dtype=np.float64)
                rowwise = probe.shape in ((n,), (n, 1)) and np.allclose(probe.ravel()[:E], first.ravel(),
                                                                        rtol=1e-12, atol=0.0)
            except Exception:
                # the stacked call is speculative -- the reference never makes it -- so whatever it raises
                # (shape errors, the callable's own asserts) only means "not row-wise"; genuine errors of
                # f_low have already surfaced from the reference-style call above
                rowwise = False
            mode = self._f_low_mode = (self.f_low, rowwise)
        if mode[1]:
            vals = np.asarray(self.f_low(flat), dtype=np.float64)
            assert vals.shape in ((M * E,), (M * E, 1)), "f_low must return one value per row"
            return vals.reshape(M, E)
        return np.array([np.asarray(self.f_low(loc), dtype=np.float64).reshape(E) for loc in locations])

    def _augment_host_input(self, X):
        """Host (M, d) inputs -> (M, d+E) CUDA tensor.  A callable low fidelity is evaluated on the host
        array it arrived as and the augmented rows go up in ONE copy (no device round trip); a data-driven
        or device-evaluable low fidelity augments on the GPU."""
        if self.data_driven_lf_approach or getattr(self.f_low, "device_predict", None) is not None:
            return self._augment_device(gp.to_device(X, self.device))
        X = np.ascontiguousarray(X, dtype=np.float64)
        offsets = self.augm_iterator.offset_table()
        locations = X[:, None, :] + offsets[None, :, :] * self.tau
        return gp.to_device(np.concatenate([X, self._f_low_batched(locations)], axis=1), self.device)

    def _augment_device(self, dX):
        """(M, d) CUDA tensor -> (M, d+E) CUDA tensor."""
        M = int(dX.shape[0])
        offsets = self.augm_iterator.offset_table()
        E = offsets.shape[0]
        if self.data_driven_lf_approach:
            h = _ffi.get_handle(self.device)
            lvl = self.lf_model.level_struct()
            out = torch.empty((M, self.input_dim + E), dtype=torch.float64, device=dX.device)
            per_row = E * (self.input_dim + 1) * 8
            ws = gp.workspace(self.device, max(min(M, 1 << 20) * per_row, 4096))
            offs = np.ascontiguousarray(offsets, dtype=np.float64)
            h.check(h.lib.mfgp_augment(h.h, ctypes.byref(lvl), dX.data_ptr(), M,
                                       offs.ctypes.data_as(ctypes.c_void_p), E, float(self.tau),
                                       out.data_ptr(), ws.data_ptr(), ws.numel() * 8))
            return out
        dev_f = getattr(self.f_low, "device_predict", None)
        if dev_f is not None:
            # a callable low fidelity that can evaluate on the device (e.g. the mean of another model of this
            # package, models.MultiLevelNARGP): locations and augmented rows never leave the GPU
            offs = torch.from_numpy(np.ascontiguousarray(offsets * self.tau, dtype=np.float64)).to(dX.device)
            loc = (dX[:, None, :] + offs[None, :, :]).reshape(M * E, self.input_dim).contiguous()
            vals = dev_f(loc).reshape(M, E)
            return torch.cat([dX, vals], dim=1).contiguous()
        # host callable on device-resident inputs (bench / gPC hand in CUDA tensors): the rows have to visit
        # the host, where the callable lives
        return self._augment_host_input(dX.cpu().numpy())

    def __augment_Data(self, X):
        """X (M,d) -> [X, f_low(x + o_0 tau), ..., f_low(x + o_{E-1} tau)]  (M, d+E), NumPy."""
        assert X.shape == (len(X), self.input_dim)
        E = self.augm_iterator.new_entries_count()
        if self.data_driven_lf_approach or getattr(self.f_low, "device_predict", None) is not None:
            Xa = self._augment_device(gp.to_device(X, self.device)).cpu().numpy()
        else:
            offsets = self.augm_iterator.offset_table()
            locations = X[:, None, :] + offsets[None, :, :] * self.tau
            assert locations.shape == (len(X), E, self.input_dim)
            Xa = np.concatenate([X, self._f_low_batched(locations)], axis=1)
        assert Xa.shape == (len(X), E + self.input_dim)
        return Xa

    augment_data = __augment_Data

    # -- A8 Monte-Carlo propagation (extension) ------------------------------------------------------
    def predict_mc_device(self, dX, n_samples=100, d_eps=None, seed=0, m0=0, d_weights=None,
                          include_lf_noise=True, ws_bytes=None, lf_jitter=0.0):
        """dX (M,d) CUDA -> (mean (M,), var (M,), weighted sum or None).  d_eps: optional CUDA standard
        normals, (M, S) for E = 1 and (M, S, E) for models with delays; otherwise Philox keyed by
        (seed, global point index m0+m, sample, column).  E = 1 (NARGP) samples the LF marginal;
        E > 1 (GPDF / GPDFC) samples the JOINT LF posterior at the E augmented locations."""
        assert self.data_driven_lf_approach, "MC propagation needs a data-driven low-fidelity GP"
        E = self.augm_iterator.new_entries_count()
        h = _ffi.get_handle(self.device)
        self._apply_add_noise()
        lf, hf = self.lf_model.level_struct(), self.hf_model.level_struct()
        M, S = int(dX.shape[0]), int(n_samples)
        mean = torch.empty(M, dtype=torch.float64, device=dX.device)
        var = torch.empty(M, dtype=torch.float64, device=dX.device)
        wsum = ctypes.c_double(0.0) if d_weights is not None else None
        npl, nph, d = self.lf_model.npad, self.hf_model.npad, self.input_dim
        if E == 1:
            if ws_bytes is None:
                # ~4 column tiles per SM up to N_h = 16384; three doubles per column for N_h <= 64 (fused kernel)
                ws_bytes = h.lib.mfgp_predict_mc_ws_bytes(self.lf_model.N, self.hf_model.N, d, M, S)
            ws = gp.workspace(self.device, ws_bytes)
            h.check(h.lib.mfgp_predict_mc(
                h.h, ctypes.byref(lf), ctypes.byref(hf), dX.data_ptr(), M, S,
                d_eps.data_ptr() if d_eps is not None else None, int(seed), int(m0),
                int(include_lf_noise), 1, d_weights.data_ptr() if d_weights is not None else None,
                mean.data_ptr(), var.data_ptr(), ctypes.byref(wsum) if wsum is not None else None,
                ws.data_ptr(), ws.numel() * 8))
            return mean, var, (wsum.value if wsum is not None else None)
        assert E <= 8, "joint low-fidelity sampling supports at most 8 augmented columns"
        offs = np.ascontiguousarray(self.augm_iterator.offset_table(), dtype=np.float64)
        if ws_bytes is None:
            keep, lf_pp = E + E * E, E * (d + 2 * npl + 1) + E * (E + 1) // 2
            hf_pp = S * (d + E + nph + 2)
            slack = 256 * (2 * npl + nph + d + E + 4)
            # LF chunk ~2 waves of 128-column tiles, HF chunk ~4 tiles per SM (mfgp_predict_mc_delays)
            p_lf, p_hf = min(M, 2 * 148 * 128 // E), min(M, max(1, 148 * 128 * 4 // S))
            want = 8 * (slack + keep * p_lf + max(lf_pp * p_lf, hf_pp * p_hf))
            ws_bytes = max(min(want, 3 << 30), 8 * (slack + keep + max(lf_pp, hf_pp)))
        ws = gp.workspace(self.device, ws_bytes)
        rc = h.lib.mfgp_predict_mc_delays(
            h.h, ctypes.byref(lf), ctypes.byref(hf), dX.data_ptr(), M,
            offs.ctypes.data_as(ctypes.c_void_p), E, float(self.tau), S,
            d_eps.data_ptr() if d_eps is not None else None, int(seed), int(m0),
            int(include_lf_noise), 1, float(lf_jitter),
            d_weights.data_ptr() if d_weights is not None else None, mean.data_ptr(), var.data_ptr(),
            ctypes.byref(wsum) if wsum is not None else None, ws.data_ptr(), ws.numel() * 8)
        if rc > 0:
            raise np.linalg.LinAlgError(
                "joint low-fidelity covariance of test point %d is not positive definite; pass lf_jitter" % (rc - 1))
        h.check(rc)
        return mean, var, (wsum.value if wsum is not None else None)

    def predict_mc_joint_device(self, dX, n_samples=100, d_eps=None, seed=0, d_weights=None,
                                include_lf_noise=True, lf_jitter=0.0):
        """Monte-Carlo propagation with the low-fidelity posterior sampled JOINTLY across the test points
        (full M x M predictive covariance; E = 1 models, small M): every sample is one coherent low-fidelity
        function draw.  dX (M, d) CUDA -> (mean (M,), var (M,), per-path weighted sums (S,)): path s gives
        sum_m w_m mu_s(x_m), e.g. the PCE mean under that draw (weights None -> plain sums).  d_eps: (M, S)."""
        assert self.data_driven_lf_approach, "MC propagation needs a data-driven low-fidelity GP"
        assert self.augm_iterator.new_entries_count() == 1, "joint sampling across test points serves E = 1 models"
        h = _ffi.get_handle(self.device)
        self._apply_add_noise()
        lf, hf = self.lf_model.level_struct(), self.hf_model.level_struct()
        M, S = int(dX.shape[0]), int(n_samples)
        mean = torch.empty(M, dtype=torch.float64, device=dX.device)
        var = torch.empty(M, dtype=torch.float64, device=dX.device)
        paths = torch.empty(S, dtype=torch.float64, device=dX.device)
        ws = gp.workspace(self.device, h.lib.mfgp_predict_mc_joint_ws_bytes(self.lf_model.N, self.hf_model.N, M, S))
        rc = h.lib.mfgp_predict_mc_joint(
            h.h, ctypes.byref(lf), ctypes.byref(hf), dX.data_ptr(), M, S,
            d_eps.data_ptr() if d_eps is not None else None, int(seed), int(include_lf_noise), 1,
            float(lf_jitter), d_weights.data_ptr() if d_weights is not None else None, mean.data_ptr(),
            var.data_ptr(), paths.data_ptr(), ws.data_ptr(), ws.numel() * 8)
        if rc > 0:
            raise np.linalg.LinAlgError(
                "joint low-fidelity covariance of the test points is not positive definite (pivot %d); "
                "pass lf_jitter" % rc)
        h.check(rc)
        return mean, var, paths

    def predict_mc(self, X_test, n_samples=100, eps=None, seed=0, weights=None, include_lf_noise=True,
                   m0=0, lf_jitter=0.0, joint=False):
        """NumPy front end of predict_mc_device.  eps: optional standard normals, (M, S[, 1]) for E = 1,
        (M, S, E) for models with delays.  m0: global index of the first test point (keys the in-kernel
        generator when eps is None).  lf_jitter: added to the diagonal of the joint LF covariance (E > 1).
        Returns (mean (M,1), var (M,1)); with `weights` also sets ``self.last_pce_mean``."""
        assert X_test.ndim == 2 and X_test.shape[1] == self.input_dim
        E = self.augm_iterator.new_entries_count()
        if joint:
            # joint=True: the LF posterior is sampled jointly ACROSS the test points (predict_mc_joint_device);
            # sets ``self.last_pce_paths`` (S,): the weighted sum of every sample path
            d_eps = None if eps is None else gp.to_device(
                np.asarray(eps, dtype=np.float64).reshape(X_test.shape[0], n_samples), self.device)
            d_w = gp.to_device(np.asarray(weights).ravel(), self.device) if weights is not None else None
            mean, var, paths = self.predict_mc_joint_device(gp.to_device(X_test, self.device), n_samples, d_eps,
                                                            seed, d_w, include_lf_noise, lf_jitter)
            self.last_pce_paths = paths.cpu().numpy()
            self.last_pce_mean = float(self.last_pce_paths.mean()) if weights is not None else None
            return mean.cpu().numpy()[:, None], var.cpu().numpy()[:, None]
        d_eps = None
        if eps is not None:
            eps = np.asarray(eps, dtype=np.float64).reshape(X_test.shape[0], n_samples, E)
            d_eps = gp.to_device(eps, self.device)
        d_w = gp.to_device(np.asarray(weights).ravel(), self.device) if weights is not None else None
        mean, var, wsum = self.predict_mc_device(gp.to_device(X_test, self.device), n_samples, d_eps,
                                                 seed, m0, d_w, include_lf_noise, lf_jitter=lf_jitter)
        self.last_pce_mean = wsum
        return mean.cpu().numpy()[:, None], var.cpu().numpy()[:, None]

    # -- A9 acquisition (extension) ------------------------------------------------------------------
    def _lf_state_key(self):
        """Identity of the low-fidelity level as the augmentation sees it: changes when the LF model is
        replaced, refitted, or its data / hyper-parameters change (gp.GPRegression._version)."""
        if self.data_driven_lf_approach:
            return ("gp", id(self.lf_model), self.lf_model._version)
        return ("callable", id(self.f_low))

    def invalidate_candidate_cache(self):
        """Drop both resident slots: the candidates' and the ALC reference rows'."""
        self._cand_cache = None
        self._ref_cache = None

    def _resident_rows(self, slot, hits, rows, lo, hi):
        """Augmented rows of rows[lo:hi], kept on the device in the cache slot `slot` (hits counted in the attribute
        `hits`).  The key is the array (address, shape, a checksum of a strided sample of rows), the shard and the
        low-fidelity state."""
        c = np.ascontiguousarray(rows, dtype=np.float64)
        step = max(1, c.shape[0] // 4096)
        key = (c.ctypes.data, c.shape, zlib.crc32(np.ascontiguousarray(c[::step]).tobytes()), lo, hi,
               float(self.tau), self.augm_iterator.offset_table().tobytes(), self._lf_state_key())
        cache = getattr(self, slot, None)
        if cache is not None and cache[0] == key:
            setattr(self, hits, getattr(self, hits, 0) + 1)
            return cache[1]
        dXa = self._augment_host_input(c[lo:hi])
        setattr(self, slot, (key, dXa))
        return dXa

    def _resident_candidates(self, candidates, lo, hi):
        """Augmented rows [c, f_low(c + o tau)] of the shard candidates[lo:hi], kept on the device.  The
        candidate set is fixed during an adaptation run (CandidateSetMaximizer) and the low-fidelity level
        does not change while high-fidelity points are acquired (src/abstractMFGP.py:317-359), so after the
        first step an acquisition performs no candidate H2D / D2H and no f_low evaluation.  The cache is
        keyed on the array (address, shape, a checksum of a strided sample of rows), the shard and the
        low-fidelity state; ``invalidate_candidate_cache()`` drops it explicitly."""
        return self._resident_rows("_cand_cache", "candidate_cache_hits", candidates, lo, hi)

    def _resident_reference(self, reference):
        """The ALC reference rows, augmented and resident like the candidates, in a slot of their own (hits counted
        in ``reference_cache_hits``), so that an ALC call never evicts the candidate rows."""
        return self._resident_rows("_ref_cache", "reference_cache_hits", reference, 0, int(reference.shape[0]))

    def acquisition_argmax(self, candidates, distributed=False, cache=True):
        """(index, variance) of the candidate with the largest predictive variance; lowest index on
        ties.  With distributed=True every rank scores a contiguous shard and the winners are combined
        with one all_gather (all ranks must hold the same fitted state, see broadcast_state).
        cache=True keeps the augmented shard resident on the device between calls (_resident_candidates)."""
        C = candidates.shape[0]
        rank, world = dist.rank_world() if distributed else (0, 1)
        lo, hi = dist.shard_range(C, rank, world)
        val, idx = -np.inf, -1
        if hi > lo:
            dXa = self._resident_candidates(candidates, lo, hi) if cache else self._augment_host_input(candidates[lo:hi])
            self._apply_add_noise()
            _, var = self.hf_model.predict_device(dXa, True, True)
            h = _ffi.get_handle(self.device)
            c_val, c_idx = ctypes.c_double(), ctypes.c_longlong()
            h.check(h.lib.mfgp_argmax(h.h, var.data_ptr(), hi - lo, ctypes.byref(c_val), ctypes.byref(c_idx)))
            val, idx = c_val.value, lo + c_idx.value
        if distributed and world > 1:
            val, idx = dist.gather_argmax(val, idx, device="cuda:%d" % self.device)
        return int(idx), float(val)

    def acquisition_batch(self, candidates, q, distributed=False, cache=True):
        """Greedy batch of q candidates for one adaptation step: (indices (q,) int64, variances (q,)).  Pick i is the
        arg-max of the predictive variance given the training set plus picks 0..i-1 as noisy observations at the
        current hyper-parameters -- the points q sequential ``acquisition_argmax`` + ``append_point`` steps pick,
        computed without the targets (mfgp_acq_batch_*, a pivoted partial Cholesky of the posterior covariance over
        the candidates).  variances[i] includes the noise, as GPy reports it; pick 0 is ``acquisition_argmax``.
        distributed / cache: as in acquisition_argmax; per pick the ranks agree on the winner with one all_gather
        and its owner broadcasts the pivot record (1 + D + q doubles)."""
        C = int(candidates.shape[0])
        q = int(q)
        if not 1 <= q <= min(_ffi.ACQ_MAX_Q, C):
            raise ValueError("batch size q = %d must lie in [1, min(%d, number of candidates = %d)]"
                             % (q, _ffi.ACQ_MAX_Q, C))
        rank, world = dist.rank_world() if distributed else (0, 1)
        lo, hi = dist.shard_range(C, rank, world)
        self._apply_add_noise()
        hf = self.hf_model
        lvl = hf.level_struct()
        D = hf.D
        jitter = float(hf.last_jitter)
        h = _ffi.get_handle(self.device)
        if hi > lo:
            dXa = self._resident_candidates(candidates, lo, hi) if cache else self._augment_host_input(candidates[lo:hi])
            ws = gp.workspace(self.device, h.lib.mfgp_acq_batch_ws_bytes(hf.N, hi - lo, q))
        indices = np.empty(q, dtype=np.int64)
        variances = np.empty(q)
        rec = np.zeros(1 + D + q)
        c_val, c_idx = ctypes.c_double(), ctypes.c_longlong()
        for i in range(q):
            val, idx, local = -np.inf, -1, np.zeros(1 + D + q)
            if hi > lo:
                if i == 0:
                    rc = h.lib.mfgp_acq_batch_begin(h.h, ctypes.byref(lvl), dXa.data_ptr(), hi - lo, q, 1,
                                                    ws.data_ptr(), ws.numel() * 8, ctypes.byref(c_val),
                                                    ctypes.byref(c_idx), local.ctypes.data)
                else:
                    rc = h.lib.mfgp_acq_batch_step(h.h, ctypes.byref(lvl), dXa.data_ptr(), hi - lo, q, 1, jitter,
                                                   i - 1, rec.ctypes.data, ws.data_ptr(), ws.numel() * 8,
                                                   ctypes.byref(c_val), ctypes.byref(c_idx), local.ctypes.data)
                h.check(rc)
                val, idx = c_val.value, lo + c_idx.value
            elif i > 0 and not rec[0] + hf.likelihood.variance + 1e-8 + jitter > 0.0:
                raise _ffi.NotPositiveDefinite(i)          # what the ranks holding candidates report for this pick
            if distributed and world > 1:
                val, idx = dist.gather_argmax(val, idx, device="cuda:%d" % self.device)
                rec = dist.broadcast_record(local, dist.shard_owner(idx, C, world), device="cuda:%d" % self.device)
            else:
                rec = local
            indices[i], variances[i] = idx, val
        return indices, variances

    def acquisition_alc(self, candidates, reference, weights=None, distributed=False, cache=True):
        """(index, alc) of the candidate whose acquisition most lowers the weighted mean latent predictive variance
        over the reference rows (integrated variance, "active learning Cohn"); lowest index on ties.
        alc(c) = sum_r w_r k_n(c, r)^2 / (v_n(c) + s^2) with k_n the latent posterior covariance, v_n(c) = k_n(c, c)
        and s^2 = noise + 1e-8 + jitter: in exact arithmetic the drop sum_r w_r (v_n(r) - v_{n+c}(r)) that
        ``hf_model.append_point(c)`` at the current hyper-parameters causes (mfgp_alc).  weights: (R,) >= 0, or None
        for 1/R.  distributed / cache: as in acquisition_argmax; the reference rows are replicated on every rank and
        stay resident in a cache slot of their own."""
        C = int(candidates.shape[0])
        reference = np.asarray(reference, dtype=np.float64)
        if reference.ndim != 2 or reference.shape[1] != self.input_dim or reference.shape[0] < 1:
            raise ValueError("reference must be a non-empty (R, %d) array" % self.input_dim)
        w = None if weights is None else alc_weights(weights, reference.shape[0])
        rank, world = dist.rank_world() if distributed else (0, 1)
        lo, hi = dist.shard_range(C, rank, world)
        val, idx = -np.inf, -1
        if hi > lo:
            dXa = self._resident_candidates(candidates, lo, hi) if cache else self._augment_host_input(candidates[lo:hi])
            dXr = self._resident_reference(reference) if cache else self._augment_host_input(reference)
            self._apply_add_noise()
            dw = None if w is None else torch.from_numpy(w).to(dXr.device)
            alc = self.hf_model.alc_device(dXa, dXr, dw)
            h = _ffi.get_handle(self.device)
            c_val, c_idx = ctypes.c_double(), ctypes.c_longlong()
            h.check(h.lib.mfgp_argmax(h.h, alc.data_ptr(), hi - lo, ctypes.byref(c_val), ctypes.byref(c_idx)))
            if c_val.value > -np.inf:                      # else every candidate of the shard is inadmissible
                val, idx = c_val.value, lo + c_idx.value
        if distributed and world > 1:
            val, idx = dist.gather_argmax(val, idx, device="cuda:%d" % self.device)
        if not val > -np.inf:
            raise _ffi.MfgpError("ALC acquisition: no candidate can be appended (v_n(c) + s^2 <= 0 or NaN everywhere)")
        return int(idx), float(val)

    # -- multi-GPU state ------------------------------------------------------------------------------
    def broadcast_state(self, src=0):
        """Broadcast the fitted state of both levels from rank `src`: training inputs/targets and
        hyper-parameters through the object channel, W = L^-1 and alpha as NCCL tensor broadcasts."""
        import torch.distributed as tdist
        if not dist.is_dist():
            return
        rank = tdist.get_rank()
        levels = ["hf_model"] + (["lf_model"] if self.data_driven_lf_approach else [])
        meta = [None]
        if rank == src:
            for name in levels:
                getattr(self, name)._ensure_posterior()       # settles last_jitter before it is sent
            meta[0] = {name: dict(X=getattr(self, name).X, Y=getattr(self, name).Y,
                                  theta=getattr(self, name).param_array,
                                  jitter=getattr(self, name).last_jitter) for name in levels}
            meta[0]["hf_X"] = self.hf_X
            meta[0]["kernel"] = self.kernel.param_array.copy()
        tdist.broadcast_object_list(meta, src=src)
        m = meta[0]
        for name in levels:
            if rank != src:
                kern = self.kernel if name == "hf_model" else None
                model = gp.GPRegression(m[name]["X"], m[name]["Y"], kernel=kern)
                model._set_params(m[name]["theta"])
                setattr(self, name, model)
                if name == "hf_model":
                    self.hf_X, self.hf_Y = m["hf_X"], m[name]["Y"]
            model = getattr(self, name)
            if rank == src:
                model._ensure_posterior()
            dist.broadcast_tensors([model._dW, model._dalpha], src=src)
            model._dirty = False
            if rank != src:
                # receivers hold W and alpha only: their A buffer is not L (append_point must not read it),
                # and a later bordered update has to use the jitter the broadcast factor was built with
                model.last_jitter = float(m[name]["jitter"])
                model._a_holds_L = False
