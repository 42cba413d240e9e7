"""GP engine on the C-ABI: the slice of ``GPy.models.GPRegression`` the reference uses.

The reference delegates all arithmetic to GPy (``src/MFDataFusion.py:93-100``,
``src/abstractMFGP.py:100-104,131-137``).  This module keeps GPy's *object protocol* for that
slice -- ``GPRegression(X, Y, kernel)``, ``model['.*Gaussian_noise']`` with ``fix / unfix /
constrain_positive``, ``optimize``, ``optimize_restarts``, ``predict``, ``likelihood.variance``,
``Y`` -- and routes every numerical step (covariance assembly, Cholesky, solves, LML, gradient,
prediction) to the sm_100a kernels behind ``include/mfgp_b200.h``.  The optimiser itself is
SciPy's L-BFGS-B on the host, exactly as paramz does it; its objective is one GPU evaluation.

No CPU fallback: constructing a model without a visible B200 raises ``MfgpError``.
"""
import ctypes
import re
import threading

import numpy as np
import torch
from scipy import optimize as _sopt

from . import _ffi, _lbfgsb
from ._ffi import TILE, KIND_COMPOSITE, KIND_RBF, MfgpError, NotPositiveDefinite, padded_n

_LIM_VAL = 36.0
_LOG_LIM_VAL = float(np.log(np.finfo(np.float64).max))


# -- paramz Logexp transformation (paramz/transformations.py) --------------------------------
def logexp_f(x):
    x = np.asarray(x, dtype=np.float64)
    return np.where(x > _LIM_VAL, x, np.log1p(np.exp(np.clip(x, -_LOG_LIM_VAL, _LIM_VAL))))


def logexp_finv(f):
    f = np.asarray(f, dtype=np.float64)
    with np.errstate(over="ignore"):
        return np.where(f > _LIM_VAL, f, np.log(np.expm1(f)))


def logexp_gradfactor(f):
    f = np.asarray(f, dtype=np.float64)
    return np.where(f > _LIM_VAL, 1.0, -np.expm1(-f))


# -- kernels --------------------------------------------------------------------------------
class Kernel:
    """Kernel object with persistent hyper-parameters (the reference re-uses ONE kernel object
    across fits, ``src/MFDataFusion.py:96``, so every fit warm-starts from the previous optimum)."""

    def __init__(self, kind, input_dim, d, names):
        self.kind = kind
        self.input_dim = int(input_dim)     # D: all columns
        self.d = int(d)                     # leading plain-input columns
        self.names = list(names)
        self.param_array = np.ones(len(names), dtype=np.float64)   # GPy defaults: all 1.0

    def to_dict(self):
        p = self.param_array
        if self.kind == KIND_RBF:
            return {"class": "RBF", "variance": [p[0]], "lengthscale": [p[1]]}
        rbf = lambda i: {"class": "RBF", "variance": [p[i]], "lengthscale": [p[i + 1]]}
        return {"class": "Add", "parts": {0: {"class": "Prod", "parts": {0: rbf(0), 1: rbf(2)}},
                                          1: rbf(4)}}


def RBF(input_dim):
    """GPy.kern.RBF(input_dim) (non-ARD: one lengthscale; src/abstractMFGP.py:60)."""
    return Kernel(KIND_RBF, input_dim, input_dim, ["rbf.variance", "rbf.lengthscale"])


def NARGPKernel(input_dim, aug_dim):
    """RBF(aug dims) * RBF(x dims) + RBF(x dims) (src/abstractMFGP.py:62-80)."""
    return Kernel(KIND_COMPOSITE, input_dim + aug_dim, input_dim,
                  ["sum.mul.rbf.variance", "sum.mul.rbf.lengthscale",
                   "sum.mul.rbf_1.variance", "sum.mul.rbf_1.lengthscale",
                   "sum.rbf.variance", "sum.rbf.lengthscale"])


class _Likelihood:
    def __init__(self, model):
        self._m = model

    @property
    def variance(self):
        return self._m._noise

    @variance.setter
    def variance(self, v):   # GPy: assignment triggers parameters_changed -> re-inference
        self._m._noise = float(np.asarray(v).ravel()[0])
        self._m._dirty = True
        self._m._version += 1


class _ParamView:
    """Result of ``model[regex]``: supports fix / unfix / constrain_positive / value access."""

    def __init__(self, model, idx):
        self._m, self._idx = model, idx

    def fix(self):
        self._m._fixed[self._idx] = True

    def unfix(self):
        self._m._fixed[self._idx] = False

    def constrain_positive(self):
        pass   # every parameter of this model is Logexp-constrained already

    @property
    def values(self):
        return self._m.param_array[self._idx]


def current_device():
    """torch's current CUDA device; raises MfgpError when there is none (no CPU fallback)."""
    if not torch.cuda.is_available():
        raise MfgpError("no CUDA device visible: mfgp_b200 runs on B200 only and has no CPU fallback")
    return torch.cuda.current_device()


_ws_pool = {}


def workspace(device, nbytes):
    """Grow-only scratch tensor per (device, Python thread) -- the same ownership as the C-ABI handle
    (_ffi.get_handle): calls of one thread are stream-ordered, so they can share one scratch; two
    threads never alias it."""
    key = (int(device), threading.get_ident())
    n = (int(nbytes) + 7) // 8
    cur = _ws_pool.get(key)
    if cur is None or cur.numel() < n:
        _ws_pool[key] = None
        cur = torch.empty(n, dtype=torch.float64, device="cuda:%d" % key[0])
        _ws_pool[key] = cur
    return cur


def release_workspaces():
    """Drop every cached scratch tensor (bench.py between sections)."""
    _ws_pool.clear()


def to_device(arr, device):
    """numpy (host) -> contiguous float64 CUDA tensor through pinned memory."""
    a = np.ascontiguousarray(arr, dtype=np.float64)
    t = torch.from_numpy(a)
    if a.size >= 1 << 16 and not t.is_pinned():     # callers may hand in views of pinned buffers
        t = t.pin_memory()
    return t.to("cuda:%d" % device, non_blocking=False)


SMALL_BATCH_N = 128      # mfgp_lml_grad_batch: one CTA per hyper-parameter vector


class GPRegression:
    """GPy.models.GPRegression look-alike running on one B200."""

    _opt_handle = None          # the calling thread's handle while optimize() runs (saves a look-up per evaluation)

    def __init__(self, X, Y, kernel=None, initialize=True, device=None):
        X = np.ascontiguousarray(X, dtype=np.float64)
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        assert X.ndim == 2 and Y.ndim == 2 and Y.shape == (X.shape[0], 1)
        if kernel is None:
            kernel = RBF(X.shape[1])                       # GPRegression default kernel
        assert kernel.input_dim == X.shape[1], "kernel/input dimension mismatch"
        self.device = current_device() if device is None else int(device)
        self._handle = _ffi.get_handle(self.device)        # raises without a GPU / library
        self.X, self.Y = X, Y
        self.kern = kernel
        self._noise = 1.0                                   # Gaussian likelihood default
        self.likelihood = _Likelihood(self)
        self.N, self.D = X.shape
        self.npad = padded_n(self.N)
        dev = "cuda:%d" % self.device
        self._dX = to_device(X, self.device)
        self._dy = to_device(Y.ravel(), self.device)
        self._dA = torch.empty((self.npad, self.npad), dtype=torch.float64, device=dev)
        self._dW = torch.empty((self.npad, self.npad), dtype=torch.float64, device=dev)
        self._dalpha = torch.empty(self.npad, dtype=torch.float64, device=dev)
        self._fixed = np.zeros(len(kernel.names) + 1, dtype=bool)
        self._dirty = True
        self._fail_count = 0
        self.n_evals = 0
        self.optimization_runs = []
        self._theta_c = (ctypes.c_double * 8)()
        self.last_jitter = 0.0
        self._a_holds_L = False
        self._version = 0                                   # bumped whenever data or hyper-parameters change

    # -- parameters ------------------------------------------------------------------------
    @property
    def names(self):
        return self.kern.names + ["Gaussian_noise.variance"]

    @property
    def param_array(self):
        return np.concatenate([self.kern.param_array, [self._noise]])

    def _set_params(self, theta):
        self.kern.param_array[:] = theta[:-1]
        self._noise = float(theta[-1])
        self._dirty = True
        self._version += 1

    def _match(self, pattern):
        rx = re.compile(pattern)
        idx = np.array([bool(rx.match(n)) for n in self.names])
        if not idx.any():
            raise KeyError(pattern)
        return idx

    def __getitem__(self, pattern):
        return _ParamView(self, self._match(pattern))

    def __setitem__(self, pattern, value):
        theta = self.param_array
        theta[self._match(pattern)] = float(np.asarray(value).ravel()[0])
        self._set_params(theta)

    # -- inference on the GPU ----------------------------------------------------------------
    def _theta_ptr(self, theta):
        for i, v in enumerate(theta):
            self._theta_c[i] = float(v)
        return ctypes.cast(self._theta_c, ctypes.c_void_p)

    def _jitter_schedule(self, theta):
        """GPy.util.linalg.jitchol: first try without jitter, then mean(diag)*1e-6*10^k, k<5."""
        kdiag = theta[0] * theta[2] + theta[4] if self.kern.kind == KIND_COMPOSITE else theta[0]
        base = (kdiag + theta[-1] + 1e-8) * 1e-6
        return [0.0] + [base * 10.0 ** k for k in range(5)]

    def _call_with_jitter(self, fn, theta):
        last = None
        for jit in self._jitter_schedule(theta):
            rc = fn(jit)
            if rc == 0:
                self.last_jitter = jit
                return
            if rc < 0:
                self._handle.check(rc)
            last = rc
        raise NotPositiveDefinite(last)

    def lml_and_grad(self, theta=None, timings=None):
        """One LML + gradient evaluation (untransformed space).  Leaves the posterior
        (W = L^-1, alpha) of ``theta`` in place."""
        h = _ffi.get_handle(self.device)
        theta = self.param_array if theta is None else np.asarray(theta, dtype=np.float64)
        P = len(theta)
        lml = ctypes.c_double()
        grad = (ctypes.c_double * 8)()
        ms = (ctypes.c_double * 8)() if timings is not None else None
        tp = self._theta_ptr(theta)

        def run(jit):
            return h.lib.mfgp_lml_grad_timed(
                h.h, self.kern.kind, self._dX.data_ptr(), self._dy.data_ptr(), self.N, self.D,
                self.kern.d, tp, P, jit, self._dA.data_ptr(), self._dW.data_ptr(),
                self._dalpha.data_ptr(), ctypes.byref(lml), ctypes.cast(grad, ctypes.c_void_p),
                ctypes.cast(ms, ctypes.c_void_p) if ms is not None else None)

        self._call_with_jitter(run, theta)
        self.n_evals += 1
        if timings is not None:
            timings[:] = [ms[i] for i in range(6)]
        self._post_theta = theta.copy()
        self._dirty = not np.array_equal(theta, self.param_array)
        self._a_holds_L = False                     # d_A now holds K^-1
        return lml.value, np.array([grad[i] for i in range(P)])

    def lml_and_grad_batch(self, thetas, want_grad=True, handle=None):
        """B hyper-parameter vectors (B, P) -> (lml (B,), grad (B, P), info (B,)) in ONE launch, one CTA per
        vector (mfgp_lml_grad_batch; N <= 128).  Nothing but scalars comes back: the posterior of this
        model is NOT updated.  info[b] > 0: the factorisation of vector b met a non-positive pivot
        (evaluate it through ``lml_and_grad``, which replays the jitter schedule)."""
        assert self.N <= SMALL_BATCH_N, "the batched objective serves N <= %d" % SMALL_BATCH_N
        h = handle if handle is not None else _ffi.get_handle(self.device)
        P = len(self.kern.names) + 1
        thetas = np.ascontiguousarray(thetas, dtype=np.float64).reshape(-1, P)
        B = thetas.shape[0]
        lml = np.empty(B)
        grad = np.empty((B, P))
        info = np.zeros(B, dtype=np.int32)
        rc = h.lib.mfgp_lml_grad_batch(
            h.h, self.kern.kind, self._dX.data_ptr(), self._dy.data_ptr(), self.N, self.D, self.kern.d,
            thetas.ctypes.data, P, B, 0.0, lml.ctypes.data, grad.ctypes.data if want_grad else None,
            info.ctypes.data)
        if rc != 0:
            h.check(rc)
        self.n_evals += B
        return lml, grad, info

    def _ensure_posterior(self):
        if not self._dirty:
            return
        h = _ffi.get_handle(self.device)
        theta = self.param_array
        out = (ctypes.c_double * 3)()
        tp = self._theta_ptr(theta)

        def run(jit):
            return h.lib.mfgp_factorize(
                h.h, self.kern.kind, self._dX.data_ptr(), self._dy.data_ptr(), self.N, self.D,
                self.kern.d, tp, len(theta), jit, self._dA.data_ptr(), self._dW.data_ptr(),
                self._dalpha.data_ptr(), ctypes.cast(out, ctypes.c_void_p))

        self._call_with_jitter(run, theta)
        self._lml = out[0]
        self._dirty = False
        self._a_holds_L = True

    def append_point(self, x_row, y):
        """Append one training point at FIXED hyper-parameters with the O(N^2) bordered update
        (mfgp_append_point) instead of refactorising: what one adaptation step adds
        (src/abstractMFGP.py:320,354) when the hyper-parameters are not re-optimised.
        The grown inputs and buffers are built in locals and committed together with N += 1 only after
        the call has been validated; on a failure the model keeps its N-point state."""
        self._ensure_posterior()
        h = _ffi.get_handle(self.device)
        x_row = np.asarray(x_row, dtype=np.float64).reshape(1, self.D)
        X = np.vstack([self.X, x_row])
        Y = np.vstack([self.Y, np.asarray(y, dtype=np.float64).reshape(1, 1)])
        dX = to_device(X, self.device)
        dy = to_device(Y.ravel(), self.device)
        dA, dW, dalpha, npad = self._dA, self._dW, self._dalpha, self.npad
        if self.N % TILE == 0:                       # padded buffers are full: add one 128-tile
            old, npad = self.npad, self.npad + TILE
            dev = self._dA.device
            grown = []
            for src in (self._dA, self._dW):
                buf = torch.zeros((npad, npad), dtype=torch.float64, device=dev)
                buf[:old, :old] = src
                idx = torch.arange(old, npad, device=dev)
                buf[idx, idx] = 1.0                  # identity pad block
                grown.append(buf)
            dA, dW = grown
            dalpha = torch.zeros(npad, dtype=torch.float64, device=dev)
            dalpha[:old] = self._dalpha
        theta = self.param_array
        out = (ctypes.c_double * 4)()
        rc = h.lib.mfgp_append_point(
            h.h, self.kern.kind, dX.data_ptr(), dy.data_ptr(), self.N, self.D, self.kern.d,
            self._theta_ptr(theta), len(theta), float(self.last_jitter), dA.data_ptr(),
            dW.data_ptr(), dalpha.data_ptr(), int(self._a_holds_L), ctypes.cast(out, ctypes.c_void_p))
        if rc < 0:
            # bad argument / CUDA failure: the (possibly half-written) new row sits outside the N-point state
            # when the buffers were grown, inside its pad otherwise -- refactorise lazily either way
            self._dirty = True
            h.check(rc)
        self.X, self.Y, self._dX, self._dy = X, Y, dX, dy
        self._dA, self._dW, self._dalpha, self.npad = dA, dW, dalpha, npad
        self.N += 1
        self._version += 1
        if rc > 0:                                   # new pivot not positive: refactorise (jitter schedule)
            self._dirty = True
            self._ensure_posterior()
            return self
        self._lml = out[0]
        return self

    def log_likelihood(self):
        self._dirty = True
        self._ensure_posterior()
        return self._lml

    # -- paramz optimisation -----------------------------------------------------------------
    @staticmethod
    def _feasible(theta):
        # a line search that left the representable range (NaN, or a softplus that underflowed to 0) is an
        # infeasible point like a failed factorisation (paramz counts both as failures)
        return bool(np.all(np.isfinite(theta)) and np.all(theta[:-1] > 0.0) and theta[-1] >= 0.0)

    def _objective_grads(self, x):
        """paramz Model._objective_grads over the transformed, un-fixed parameters."""
        free = ~self._fixed
        theta = self.param_array
        theta[free] = logexp_f(x)
        self._set_params(theta)
        try:
            if not self._feasible(theta):
                raise NotPositiveDefinite(0)
            if getattr(self, "N", SMALL_BATCH_N + 1) <= SMALL_BATCH_N:
                # the reference's own sizes: scalars-only kernel (no factors written; the posterior is
                # rebuilt once, after the optimiser has finished)
                lml_b, g_b, info = self.lml_and_grad_batch(theta[None, :], handle=self._opt_handle)
                lml, g = (float(lml_b[0]), g_b[0]) if info[0] == 0 else self.lml_and_grad(theta)
            else:
                lml, g = self.lml_and_grad(theta)
            if not (np.isfinite(lml) and np.all(np.isfinite(g))):
                raise NotPositiveDefinite(0)
            self._fail_count = 0
        except NotPositiveDefinite:
            if self._fail_count >= 10:
                raise
            self._fail_count += 1
            return np.inf, np.zeros(int(free.sum()))
        return -lml, -(g[free] * logexp_gradfactor(theta[free]))

    def _minimise(self, fun, x0, max_iters):
        """scipy.optimize.fmin_l_bfgs_b(fun, x0, maxfun=max_iters, maxiter=max_iters) as paramz's opt_lbfgsb
        calls it -- through the stepped driver around the same compiled routine when it reproduces SciPy's
        iterates bit for bit on this installation (_lbfgsb.selfcheck), else through SciPy's own wrapper."""
        if _lbfgsb.selfcheck():
            return _lbfgsb.minimize(fun, x0, maxfun=max_iters, maxiter=max_iters)
        return _sopt.fmin_l_bfgs_b(fun, x0, maxfun=max_iters, maxiter=max_iters)

    def optimize(self, optimizer=None, max_iters=1000, messages=False, **kw):
        free = ~self._fixed
        x0 = logexp_finv(self.param_array[free])
        # one handle look-up (and stream binding) per optimisation instead of one per evaluation
        self._opt_handle = _ffi.get_handle(self.device)
        try:
            x_opt, _, _ = self._minimise(self._objective_grads, x0, max_iters)
            # paramz opt_lbfgsb.opt: self.f_opt = f_fp(self.x_opt)[0] -- the objective is evaluated once more at
            # the returned point (after an abnormal line-search exit SciPy's own f is the last TRIAL point's),
            # and that value is what optimize_restarts compares  [paramz-recall]
            f_opt = self._objective_grads(np.array(x_opt, dtype=np.float64))[0]
        finally:
            self._opt_handle = None
        theta = self.param_array
        theta[free] = logexp_f(x_opt)
        self._set_params(theta)
        self.optimization_runs.append((x_opt, float(f_opt)))
        return self

    def optimize_restarts(self, num_restarts=10, robust=False, verbose=True, parallel=False,
                          num_processes=None, **kwargs):
        """paramz Model.optimize_restarts: run 0 from the current point, runs 1.. from N(0,1) draws
        in the transformed space (global NumPy RNG), keep the best objective."""
        free = ~self._fixed
        kwargs.pop("optimizer", None)      # 'bfgs' resolves to L-BFGS-B in paramz.get_optimizer
        first = len(self.optimization_runs)
        from . import dist
        rank, world = dist.rank_world()
        if parallel and world > 1:
            return self._optimize_restarts_distributed(num_restarts, robust, rank, world, **kwargs)
        if self._lockstep_ok(num_restarts):
            starts = [None] + [np.random.normal(size=int(free.sum())) for _ in range(1, num_restarts)]
            runs = self._optimize_lockstep(list(range(num_restarts)), starts, robust, **kwargs)
            self.optimization_runs.extend((x, f) for _, f, x in runs)
            if runs:
                theta = self.param_array
                theta[free] = logexp_f(dist.best_run(runs)[2])
                self._set_params(theta)
            return self
        for i in range(num_restarts):
            try:
                if i > 0:
                    theta = self.param_array
                    theta[free] = logexp_f(np.random.normal(size=int(free.sum())))
                    self._set_params(theta)
                self.optimize(**kwargs)
            except Exception:
                if robust:
                    continue
                raise
        runs = self.optimization_runs[first:]
        if runs:
            best = int(np.argmin([r[1] for r in runs]))
            theta = self.param_array
            theta[free] = logexp_f(runs[best][0])
            self._set_params(theta)
        return self

    def _optimize_restarts_distributed(self, num_restarts, robust, rank, world, **kwargs):
        """The restarts of optimize_restarts are independent (src/abstractMFGP.py:137): with
        ``parallel=True`` under torch.distributed, rank r runs the restarts i = r (mod world) on its own
        GPU and the best run is agreed on through one all_gather of (index, objective, x_opt).
        Every rank draws ALL starting points from the global NumPy RNG in the serial order, so with the
        same RNG state on every rank the result equals the serial loop's (each L-BFGS-B run is
        deterministic given its start), and every rank ends in the same state."""
        from . import dist
        free = ~self._fixed
        nfree = int(free.sum())
        starts = [None] + [np.random.normal(size=nfree) for _ in range(1, num_restarts)]
        theta0 = self.param_array.copy()
        local = []
        share = dist.restart_share(num_restarts, rank, world)
        if self._lockstep_ok(len(share)):
            local = self._optimize_lockstep(share, starts, robust, **kwargs)     # this rank's share, batched
            share = []
        for i in share:
            try:
                theta = theta0.copy()
                if i > 0:
                    theta[free] = logexp_f(starts[i])
                self._set_params(theta)
                self.optimize(**kwargs)
                x_opt, f_opt = self.optimization_runs.pop()
                local.append((i, float(f_opt), np.asarray(x_opt, dtype=np.float64)))
            except Exception:
                if not robust:
                    raise
        runs = dist.gather_runs(local)
        self.optimization_runs.extend((x, f) for _, f, x in runs)
        theta = theta0.copy()
        if runs:
            theta[free] = logexp_f(dist.best_run(runs)[2])
        self._set_params(theta)
        return self

    def _lockstep_ok(self, n_runs):
        # lock-step drives SciPy's compiled L-BFGS-B step directly; where that does not reproduce SciPy's own
        # iterates (_lbfgsb.selfcheck) the restarts run one after the other, with the same results
        return (n_runs > 1 and getattr(self, "N", SMALL_BATCH_N + 1) <= SMALL_BATCH_N
                and _lbfgsb.selfcheck())

    def _objective_batch(self, thetas, free, handle=None):
        """[(objective, gradient over the free transformed parameters) or None] for full hyper-parameter
        vectors, ONE batched launch for the feasible ones (mfgp_lml_grad_batch, one CTA each).  None =
        infeasible point / failed factorisation (paramz counts both as failures).  A vector whose
        factorisation met a non-positive pivot is re-evaluated through lml_and_grad, which replays GPy's
        jitter schedule."""
        thetas = np.asarray(thetas, dtype=np.float64).reshape(-1, len(self.kern.names) + 1)
        # feasible: finite, kernel parameters > 0, noise >= 0 (see _feasible), for the whole batch at once
        ok = np.isfinite(thetas).all(axis=1) & (thetas[:, :-1] > 0.0).all(axis=1) & (thetas[:, -1] >= 0.0)
        out = [None] * len(thetas)
        if ok.all():
            rows, sel = range(len(thetas)), thetas
        else:
            rows, sel = np.flatnonzero(ok), thetas[ok]
        if len(sel):
            lml, grad, info = self.lml_and_grad_batch(sel, handle=handle)
            # d theta / d x of the Logexp transform, per vector (same reason as in thetas_of)
            chain = np.array([logexp_gradfactor(th[free]) for th in sel])
            obj_grad = -(grad[:, free] * chain)
            fin = np.isfinite(lml) & np.isfinite(obj_grad).all(axis=1)
            for k, b in enumerate(rows):
                if info[k] != 0:
                    try:
                        l, g = self.lml_and_grad(sel[k])
                    except NotPositiveDefinite:
                        continue
                    if np.isfinite(l) and np.all(np.isfinite(g)):
                        out[b] = (-float(l), -(g[free] * logexp_gradfactor(sel[k][free])))
                elif fin[k]:
                    out[b] = (-float(lml[k]), obj_grad[k])
        return out

    def _optimize_lockstep(self, indices, starts, robust, max_iters=1000, **_):
        """The restarts `indices` of optimize_restarts (src/abstractMFGP.py:137) on ONE GPU in lock-step:
        every run is its own L-BFGS-B instance (_lbfgsb.LbfgsbRun: SciPy's compiled step, resumable at
        every objective evaluation); each round, the points at which the still running instances want the
        objective are evaluated by ONE batched launch (one CTA per run).  An evaluation depends on nothing
        but its own hyper-parameters, so every run follows exactly the trajectory it follows in the serial
        loop (same starts: run 0 from the current point, run i > 0 from starts[i], drawn by the caller in the
        serial order).  Returns [(index, objective at x_opt, x_opt)]."""
        free = ~self._fixed
        nfree = int(free.sum())
        base = self.param_array.copy()

        def thetas_of(xs):
            # one Logexp transform PER run, on a vector of the length the serial loop transforms: NumPy's
            # SIMD exp may round the same input differently in the vector body and in the loop tail, so a
            # (runs x parameters) batch would not reproduce the serial loop bit for bit on every CPU
            thetas = np.tile(base, (len(xs), 1))
            for r, x in enumerate(xs):
                thetas[r, free] = logexp_f(x)
            return thetas
        runs = {i: _lbfgsb.LbfgsbRun(logexp_finv(base[free]) if starts[i] is None
                                     else logexp_finv(logexp_f(starts[i])), max_iters, max_iters) for i in indices}
        fails = {i: 0 for i in indices}
        errors = {}
        handle = _ffi.get_handle(self.device)      # one look-up (and stream binding) for the whole optimisation
        while True:
            want = [i for i in indices if i not in errors and runs[i].advance()]
            if not want:
                break
            vals = self._objective_batch(thetas_of([runs[i].x for i in want]), free, handle=handle)
            for i, v in zip(want, vals):
                if v is None:
                    if fails[i] >= 10:                     # paramz: more than ten failures in a row re-raise
                        errors[i] = NotPositiveDefinite(0)
                        continue
                    fails[i] += 1
                    runs[i].supply(np.inf, np.zeros(nfree))
                else:
                    fails[i] = 0
                    runs[i].supply(*v)
        self._dirty = True
        if errors and not robust:
            raise errors[min(errors)]
        done = [i for i in indices if i not in errors]
        # paramz opt_lbfgsb.opt: f_opt = f_fp(x_opt)[0], for all runs in one more batched launch
        final = self._objective_batch(thetas_of([runs[i].x for i in done]), free, handle=handle) if done else []
        return [(i, (v[0] if v is not None else np.inf), np.array(runs[i].x, dtype=np.float64))
                for i, v in zip(done, final)]

    # -- prediction ----------------------------------------------------------------------------
    def level_struct(self):
        """mfgp_level_t view of the fitted state (keeps the ctypes theta buffer alive on self)."""
        self._ensure_posterior()
        theta = self.param_array
        self._level_theta = (ctypes.c_double * 8)(*theta)
        return _ffi.Level(kind=self.kern.kind, N=self.N, D=self.D, d=self.kern.d, P=len(theta),
                          reserved=0, d_X=self._dX.data_ptr(),
                          h_theta=ctypes.cast(self._level_theta, ctypes.c_void_p).value,
                          d_W=self._dW.data_ptr(), d_alpha=self._dalpha.data_ptr())

    def predict_device(self, dXnew, want_var=True, include_noise=True, ws_bytes=None):
        """dXnew: (M, D) CUDA float64 tensor -> (mean (M,), var (M,) or None) CUDA tensors."""
        h = _ffi.get_handle(self.device)
        lvl = self.level_struct()
        M = int(dXnew.shape[0])
        dev = dXnew.device
        mean = torch.empty(M, dtype=torch.float64, device=dev)
        var = torch.empty(M, dtype=torch.float64, device=dev) if want_var else None
        ws_ptr, nbytes = None, 0
        if want_var:
            if ws_bytes is None:
                ws_bytes = min(h.lib.mfgp_predict_ws_bytes(self.N, max(M, 1)), 1 << 30)
                ws_bytes = max(ws_bytes, h.lib.mfgp_predict_ws_bytes(self.N, 128))
            ws = workspace(self.device, ws_bytes)
            ws_ptr, nbytes = ws.data_ptr(), ws.numel() * 8
        h.check(h.lib.mfgp_predict(h.h, ctypes.byref(lvl), dXnew.data_ptr(), M, mean.data_ptr(),
                                   var.data_ptr() if want_var else None, int(include_noise),
                                   ws_ptr, nbytes))
        return mean, var

    def alc_device(self, dXc, dXr, dw=None, ws_bytes=None):
        """Integrated-variance (ALC) acquisition values of the candidate rows dXc (C, D) over the reference rows dXr
        (R, D), CUDA tensors -> (C,) CUDA tensor (mfgp_alc): alc[c] = sum_r w_r k_n(c, r)^2 / (v_n(c) + s^2), the drop
        in the w-weighted latent variance at the references that append_point(c) at the current theta would cause;
        -inf where v_n(c) + s^2 <= 0.  dw: (R,) CUDA weights, or None for 1/R.  ws_bytes: the scratch handed to the
        call (default mfgp_alc_ws_bytes(N, C, R)); a candidate's value does not depend on it."""
        h = _ffi.get_handle(self.device)
        C, R = int(dXc.shape[0]), int(dXr.shape[0])
        if dXc.ndim != 2 or dXr.ndim != 2 or int(dXc.shape[1]) != self.D or int(dXr.shape[1]) != self.D:
            raise ValueError("candidate and reference rows must have the level's input width D = %d" % self.D)
        if R < 1:
            raise ValueError("the reference set is empty")
        if dw is not None and tuple(dw.shape) != (R,):
            raise ValueError("weights must have one entry per reference row (%d), got shape %s"
                             % (R, tuple(dw.shape)))
        lvl = self.level_struct()                           # settles last_jitter
        dXc, dXr = dXc.contiguous(), dXr.contiguous()
        dw = dw.contiguous() if dw is not None else None
        assert dXc.dtype == dXr.dtype == torch.float64 and (dw is None or dw.dtype == torch.float64)
        alc = torch.empty(C, dtype=torch.float64, device=dXc.device)
        if C == 0:
            return alc
        if ws_bytes is None:
            ws_bytes = h.lib.mfgp_alc_ws_bytes(self.N, C, R)
        ws = workspace(self.device, ws_bytes)
        h.check(h.lib.mfgp_alc(h.h, ctypes.byref(lvl), dXc.data_ptr(), C, dXr.data_ptr(), R,
                               dw.data_ptr() if dw is not None else None, float(self.last_jitter),
                               alc.data_ptr(), ws.data_ptr(), int(ws_bytes)))
        return alc

    def predictive_gradients_device(self, dX, want_var=True, include_noise=True):
        """dX (M, D) CUDA -> (dmean (M, D), dvar (M, D) or None, mean (M,), var (M,) or None) CUDA tensors
        (mfgp_predictive_gradients).  dvar: gradient of the unclipped latent variance; mean and var: predict_device's
        outputs to round-off.  want_var=False is the mean-only mode (one generator pass, no W)."""
        h = _ffi.get_handle(self.device)
        lvl = self.level_struct()
        M, D = int(dX.shape[0]), self.D
        assert dX.ndim == 2 and int(dX.shape[1]) == D, "query width must equal the level's input width"
        new = lambda *shape: torch.empty(shape, dtype=torch.float64, device=dX.device)
        dmean, mean = new(M, D), new(M)
        dvar = var = None
        ws_ptr, nbytes = None, 0
        if want_var:
            dvar, var = new(M, D), new(M)
            ws_bytes = max(min(h.lib.mfgp_predictive_gradients_ws_bytes(self.N, max(M, 1)), 1 << 30),
                           h.lib.mfgp_predictive_gradients_ws_bytes(self.N, 128))
            ws = workspace(self.device, ws_bytes)
            ws_ptr, nbytes = ws.data_ptr(), ws.numel() * 8
        h.check(h.lib.mfgp_predictive_gradients(h.h, ctypes.byref(lvl), dX.data_ptr(), M, dmean.data_ptr(),
                                                dvar.data_ptr() if want_var else None, mean.data_ptr(),
                                                var.data_ptr() if want_var else None, int(include_noise),
                                                ws_ptr, nbytes))
        return dmean, dvar, mean, var

    def predictive_gradients(self, Xnew):
        """GP.predictive_gradients (GPy): (dmu_dX (M, D, 1), dv_dX (M, D)) as NumPy; dv_dX is the gradient of the
        latent variance (the noise is a constant)."""
        Xnew = np.ascontiguousarray(Xnew, dtype=np.float64)
        assert Xnew.ndim == 2 and Xnew.shape[1] == self.D
        dmean, dvar, _, _ = self.predictive_gradients_device(to_device(Xnew, self.device))
        return dmean.cpu().numpy()[:, :, None], dvar.cpu().numpy()

    def predict(self, Xnew, full_cov=False, include_likelihood=True):
        """GP.predict: (mean (M,1), var (M,1)) as NumPy; var includes the noise variance."""
        assert not full_cov, "full_cov is not on the reference's path"
        Xnew = np.ascontiguousarray(Xnew, dtype=np.float64)
        assert Xnew.ndim == 2 and Xnew.shape[1] == self.D
        mean, var = self.predict_device(to_device(Xnew, self.device), True, include_likelihood)
        return mean.cpu().numpy()[:, None], var.cpu().numpy()[:, None]
