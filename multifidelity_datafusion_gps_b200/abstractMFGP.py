"""AbstractMFGP -- the reference's public model surface (src/abstractMFGP.py:9-137, 275-359)
re-hosted on the B200 GP engine (``gp.py`` -> ``include/mfgp_b200.h``).

Kept verbatim from the reference: constructor arguments and attributes (:12-33), the abstract
``fit / adapt / predict / get_mse`` (:35-49), ``initialize_kernel`` (:51-60),
``get_NARGP_kernel`` (:62-80), ``initialize_lf_level`` (:82-106),
``get_input_with_highest_uncertainty`` (:124-129), the ``ARD`` fit recipe (:131-137) and the
adaptation loop of ``adapt_and_plot`` (:317-359).  Out of scope: every matplotlib routine
(:139-273, 380-390) and ``adapt_lf`` (:108-122), which is dead code in the reference (it calls the
name-mangled, non-existent ``self.__ARD``; SURVEY.md section 5).
"""
import abc

import numpy as np

from . import gp
from .adaptation_maximizers import AbstractMaximizer


class AbstractMFGP(metaclass=abc.ABCMeta):
    parallel_restarts = False     # set True to spread optimize_restarts over the ranks (SURVEY.md 8f rank 1)
    refit_every = 1               # adaptation steps per hyper-parameter refit (SURVEY.md 8f rank 3)
    adapt_batch_size = 1          # high-fidelity points acquired per adaptation step (adapt_maximizer.maximize_batch)

    def _append_hf_point(self, new_hf_X):
        """One acquired point at fixed hyper-parameters; models without an incremental path refit."""
        self.fit(new_hf_X)

    def _append_hf_points(self, new_hf_X, k):
        """The last k rows of new_hf_X (one acquired batch) at fixed hyper-parameters; models without an
        incremental path refit."""
        self.fit(new_hf_X)

    @abc.abstractmethod
    def __init__(self, name: str, input_dim: int, num_derivatives: int, tau: float, f_exact: callable,
                 lower_bound: np.ndarray, upper_bound: float, f_low: callable, lf_X: np.ndarray,
                 lf_Y: np.ndarray, lf_hf_adapt_ratio: int, use_composite_kernel: bool,
                 adapt_maximizer: AbstractMaximizer, eps: float):
        super().__init__()
        self.name = name
        self.input_dim = input_dim
        self.num_derivatives = num_derivatives
        self.tau = tau
        self.f_exact = f_exact
        self.f_low = f_low
        self.lf_hf_adapt_ratio = lf_hf_adapt_ratio
        self.adapt_maximizer = adapt_maximizer
        self.eps = eps
        if lower_bound is None and upper_bound is None:        # default domain [0,1]^d
            self.lower_bound = np.zeros(input_dim)
            self.upper_bound = np.ones(input_dim)
        else:
            self.lower_bound = lower_bound
            self.upper_bound = upper_bound

    @abc.abstractmethod
    def fit(self, hf_X):
        pass

    @abc.abstractmethod
    def adapt(self, adapt_steps, plot_mode, X_test, Y_test):
        pass

    @abc.abstractmethod
    def predict(self, X_test):
        pass

    @abc.abstractmethod
    def get_mse(self, X_test, Y_test):
        pass

    # -- kernels ---------------------------------------------------------------------------
    def initialize_kernel(self, use_composite_kernel: bool):
        """Composite NARGP kernel, or one RBF over all augmented columns."""
        if use_composite_kernel:
            self.kernel = self.get_NARGP_kernel()
        else:
            self.kernel = gp.RBF(self.input_dim + self.augm_iterator.new_entries_count())

    def get_NARGP_kernel(self):
        """k1(z, z') * k2(x, x') + k3(x, x'): z = augmented columns, x = the first input_dim columns.
        (The reference's kern_class arguments only ever take their RBF defaults.)"""
        return gp.NARGPKernel(self.input_dim, self.augm_iterator.new_entries_count())

    # -- low-fidelity level -------------------------------------------------------------------
    def initialize_lf_level(self, f_low: callable = None, lf_X: np.ndarray = None, lf_Y: np.ndarray = None):
        """Either a low-fidelity callable or low-fidelity data (then a GP is trained on it)."""
        lf_model_params_are_valid = (f_low is not None) ^ (
            (lf_X is not None) and (lf_Y is not None) and (self.lf_hf_adapt_ratio is not None))
        assert lf_model_params_are_valid, 'define low-fidelity model either by predicition function or by data'
        self.data_driven_lf_approach = f_low is None
        if self.data_driven_lf_approach:
            self.lf_X = lf_X
            self.lf_Y = lf_Y
            self.lf_model = gp.GPRegression(X=lf_X, Y=lf_Y, initialize=True)
            self.lf_model.optimize()
            self.f_low = lambda t: self.lf_model.predict(t)[0]
        else:
            self.f_low = f_low

    # -- acquisition ----------------------------------------------------------------------------
    def get_input_with_highest_uncertainty(self, model):
        assert hasattr(model, 'predict')
        x, fopt = self.adapt_maximizer.maximize(self.predict, self.lower_bound, self.upper_bound)
        return x, fopt

    # -- fit recipe -------------------------------------------------------------------------------
    def ARD(self, model, num_restarts):
        """Two-stage optimisation: noise pinned to 1 % of var(Y) for a first L-BFGS-B run, then freed
        for `num_restarts` restarts of which the best is kept."""
        model[".*Gaussian_noise"] = model.Y.var() * 0.01
        model[".*Gaussian_noise"].fix()
        model.optimize(max_iters=500)
        model[".*Gaussian_noise"].unfix()
        model[".*Gaussian_noise"].constrain_positive()
        # parallel_restarts: under torch.distributed every rank calls fit() collectively and takes a
        # share of the independent restarts (gp.GPRegression._optimize_restarts_distributed)
        model.optimize_restarts(num_restarts, optimizer="bfgs", max_iters=1000, verbose=False,
                                parallel=getattr(self, "parallel_restarts", False))

    # -- adaptation loop --------------------------------------------------------------------------
    def adapt_and_plot(self, plot_means: bool = False, plot_uncertainties: bool = False,
                       plot_error: bool = False, eps: float = 1e-8):
        """The loop body of the reference's adapt_and_plot with the drawing removed: acquire the most
        uncertain input, append it, refit; stop early once |fopt| < eps.  With plot_error the test
        MSE before each refit is recorded in ``self.mse_history`` (what the reference plots).
        With ``adapt_batch_size`` > 1 every step acquires a batch instead (_adapt_batches)."""
        self.mse_history = []
        self.acquired_points = []
        if int(getattr(self, "adapt_batch_size", 1)) > 1:
            return self._adapt_batches(plot_error or plot_uncertainties)
        for i in range(self.adapt_steps):
            acquired_x, fopt = self.get_input_with_highest_uncertainty(self)
            self.acquired_points.append((np.array(acquired_x, dtype=np.float64), float(np.ravel(fopt)[0])))
            new_hf_X = np.vstack((self.hf_X, acquired_x))
            if plot_error or plot_uncertainties:
                if self.X_test is not None and self.Y_test is not None:
                    self.mse_history.append(self.get_mse(self.X_test, self.Y_test))
            # refit_every = 1 is the reference's loop (refit after every acquisition, :354); k > 1 keeps
            # the hyper-parameters for k-1 steps and extends the factorisation by a bordered update
            if (i + 1) % max(1, int(getattr(self, "refit_every", 1))) == 0:
                self.fit(new_hf_X)
            else:
                self._append_hf_point(new_hf_X)
            if np.abs(fopt) < self.eps:
                self.adapt_steps = i + 1
                print("Iteration stopped after {} iterations!".format(i + 1)
                      + " minimum uncertainty reached: {:e}".format(float(np.ravel(fopt)[0])))
                break

    def _adapt_batches(self, record_mse):
        """adapt_and_plot with q = adapt_batch_size points per step: the maximiser's greedy batch (the points q
        sequential steps at fixed hyper-parameters would pick), cut after the first point with |fopt| < eps -- the
        sequential loop stops after acquiring that point -- then one refit on a refit step, or else one f_exact
        call on the block and bordered updates.  Every point goes into ``acquired_points``; the test MSE is
        recorded once per step."""
        q = int(self.adapt_batch_size)
        for i in range(self.adapt_steps):
            X_new, fopt = self.adapt_maximizer.maximize_batch(self.predict, self.lower_bound, self.upper_bound, q)
            X_new = np.atleast_2d(np.asarray(X_new, dtype=np.float64))
            fopt = np.ravel(np.asarray(fopt, dtype=np.float64))
            small = np.flatnonzero(np.abs(fopt) < self.eps)
            k = int(small[0]) + 1 if small.size else len(fopt)
            X_new = X_new[:k]
            for j in range(k):
                self.acquired_points.append((X_new[j].copy(), float(fopt[j])))
            new_hf_X = np.vstack((self.hf_X, X_new))
            if record_mse and self.X_test is not None and self.Y_test is not None:
                self.mse_history.append(self.get_mse(self.X_test, self.Y_test))
            if (i + 1) % max(1, int(getattr(self, "refit_every", 1))) == 0:
                self.fit(new_hf_X)
            else:
                self._append_hf_points(new_hf_X, k)
            if small.size:
                self.adapt_steps = i + 1
                print("Iteration stopped after {} iterations!".format(i + 1)
                      + " minimum uncertainty reached: {:e}".format(float(fopt[k - 1])))
                break
