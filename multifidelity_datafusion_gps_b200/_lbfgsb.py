"""SciPy's L-BFGS-B, stepped one evaluation at a time.

paramz drives GPy's fits with ``scipy.optimize.fmin_l_bfgs_b`` (paramz/optimization/optimization.py,
reached from src/abstractMFGP.py:134,137).  At the reference's own problem sizes (5-30 high-fidelity
points) one GPU evaluation costs ~30 us while the Python layers ``fmin_l_bfgs_b`` puts around SciPy's
compiled ``setulb`` step (ScalarFunction, MemoizeJac, result objects) cost ~45 us per evaluation, and they
hide the step boundary that is needed to evaluate several independent runs in ONE batched launch.

``LbfgsbRun`` is the loop of ``scipy.optimize._lbfgsb_py._minimize_lbfgsb`` around the same compiled
``setulb`` with the same arguments ``fmin_l_bfgs_b`` passes (m = 10, factr = 1e7, pgtol = 1e-5, maxls = 20, and
optional box bounds) and the same termination rules (maxiter, maxfun), turned inside out: ``advance()`` runs until
the algorithm asks for f and g at ``run.x`` (or has finished), ``supply(f, g)`` hands them in.  Same
algorithm, same floating-point operations: the iterates are bit-identical to ``fmin_l_bfgs_b``'s, which
``selfcheck()`` verifies once per process (and tests/test_host.py on several objectives); if the private
``setulb`` is missing or has another signature, callers fall back to ``fmin_l_bfgs_b``.
"""
import numpy as np
from scipy import optimize as _sopt

try:
    from scipy.optimize._constraints import old_bound_to_new as _old_bound_to_new
    from scipy.optimize import _lbfgsb as _core
    from scipy.optimize._lbfgsb_py import HAS_ILP64 as _ILP64
except Exception:          # pragma: no cover - other SciPy layouts
    _core, _ILP64, _old_bound_to_new = None, False, None

M_CORR, FACTR, PGTOL, MAXLS = 10, 1e7, 1e-5, 20       # fmin_l_bfgs_b defaults, as paramz leaves them


class LbfgsbRun:
    """One L-BFGS-B minimisation, resumable at every objective evaluation."""

    def __init__(self, x0, maxfun=15000, maxiter=15000, bounds=None):
        """bounds: None, or one (low, high) pair per coordinate as ``fmin_l_bfgs_b`` takes them (None = unbounded)."""
        x0 = np.asarray(x0, dtype=np.float64).ravel()
        n = x0.shape[0]
        it = np.int64 if _ILP64 else np.int32
        m = M_CORR
        self.n, self.maxfun, self.maxiter = n, int(maxfun), int(maxiter)
        self._nbd = np.zeros(n, dtype=it)
        self._low = np.zeros(n, dtype=np.float64)
        self._up = np.zeros(n, dtype=np.float64)
        if bounds is not None:              # as scipy.optimize._lbfgsb_py._minimize_lbfgsb prepares them
            if len(bounds) != n:
                raise ValueError("length of x0 != length of bounds")
            lu = np.array(_old_bound_to_new(bounds))
            if (lu[0] > lu[1]).any():
                raise ValueError("LBFGSB - one of the lower bounds is greater than an upper bound.")
            x0 = np.clip(x0, lu[0], lu[1])
            for i in range(n):
                lo, up = lu[0, i], lu[1, i]
                if not np.isinf(lo):
                    self._low[i] = lo
                if not np.isinf(up):
                    self._up[i] = up
                self._nbd[i] = {(False, False): 0, (True, False): 1, (True, True): 2, (False, True): 3}[
                    (not np.isinf(lo), not np.isinf(up))]
        self.x = np.array(x0, dtype=np.float64)
        self.f = 0.0
        self.g = np.zeros(n, dtype=np.float64)
        self._wa = np.zeros(2 * m * n + 5 * n + 11 * m * m + 8 * m, np.float64)
        self._iwa = np.zeros(3 * n, dtype=it)
        self._task = np.zeros(2, dtype=it)
        self._ln_task = np.zeros(2, dtype=it)
        self._lsave = np.zeros(4, dtype=it)
        self._isave = np.zeros(44, dtype=it)
        self._dsave = np.zeros(29, dtype=np.float64)
        self.nfev = 0
        self.nit = 0
        self.done = False

    def advance(self):
        """Step until f, g are wanted at ``self.x`` (True) or the minimisation has ended (False)."""
        task = self._task
        while not self.done:
            _core.setulb(M_CORR, self.x, self._low, self._up, self._nbd, self.f, self.g, FACTR, PGTOL, self._wa,
                         self._iwa, task, self._lsave, self._isave, self._dsave, MAXLS, self._ln_task)
            if task[0] == 3:
                return True
            if task[0] == 1:                       # new iteration
                self.nit += 1
                if self.nit >= self.maxiter:
                    task[0], task[1] = 5, 504
                elif self.nfev > self.maxfun:
                    task[0], task[1] = 5, 502
            else:
                self.done = True
        return False

    def supply(self, f, g):
        self.f = float(f)
        self.g = np.asarray(g, dtype=np.float64)
        self.nfev += 1

    @property
    def warnflag(self):
        if self._task[0] == 4:
            return 0
        return 1 if (self.nfev > self.maxfun or self.nit >= self.maxiter) else 2


def minimize(fun, x0, maxfun=15000, maxiter=15000, bounds=None):
    """``fmin_l_bfgs_b(fun, x0, maxfun=, maxiter=, bounds=)`` for fun -> (f, g): (x, f, {funcalls, nit, warnflag})."""
    run = LbfgsbRun(x0, maxfun, maxiter, bounds)
    while run.advance():
        run.supply(*fun(run.x.copy()))
    return run.x, run.f, {"funcalls": run.nfev, "nit": run.nit, "warnflag": run.warnflag}


def minimize_lockstep(batch_fun, x0s, maxfun=15000, maxiter=15000, bounds=None):
    """Several independent minimisations advanced together: every round, the points at which the still
    running ones want (f, g) are handed to ``batch_fun(list of x) -> list of (f, g)`` in one call.  Each run
    sees exactly the evaluations it would see alone, so its iterates equal those of ``minimize``.
    ``bounds`` (as in ``minimize``) apply to every run.  Returns [(x, f, info)] in the order of x0s."""
    runs = [LbfgsbRun(x0, maxfun, maxiter, bounds) for x0 in x0s]
    while True:
        want = [r for r in runs if r.advance()]
        if not want:
            break
        for r, (f, g) in zip(want, batch_fun([r.x.copy() for r in want])):
            r.supply(f, g)
    return [(r.x, r.f, {"funcalls": r.nfev, "nit": r.nit, "warnflag": r.warnflag}) for r in runs]


_checked = None


def selfcheck():
    """True iff the stepped driver reproduces fmin_l_bfgs_b bit for bit on a small problem with a failing
    region (objective +inf), i.e. the private ``setulb`` is the one this module was written against."""
    global _checked
    if _checked is None:
        _checked = False
        if _core is not None:
            def fun(x):
                if x[0] > 2.5:
                    return np.inf, np.zeros_like(x)
                return float(np.sum(np.sin(3.0 * x) + 0.1 * x ** 2)), 3.0 * np.cos(3.0 * x) + 0.2 * x
            try:
                x0 = np.array([0.3, -1.2, 2.0])
                a = _sopt.fmin_l_bfgs_b(fun, x0, maxfun=60, maxiter=60)
                b = minimize(fun, x0, maxfun=60, maxiter=60)
                _checked = bool(np.array_equal(a[0], b[0]) and a[1] == b[1] and a[2]["funcalls"] == b[2]["funcalls"]
                                and a[2]["nit"] == b[2]["nit"] and a[2]["warnflag"] == b[2]["warnflag"])
            except Exception:
                _checked = False
    return _checked
