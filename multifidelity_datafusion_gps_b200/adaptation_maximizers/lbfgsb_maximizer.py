"""Multi-start bounded L-BFGS-B on the predictive variance, started from a greedy batch of candidates.

``CandidateSetMaximizer`` can only return a point of its fixed random candidate set, so the acquired point is as good
as the set's resolution (about 0.06 per axis for 10^5 candidates in 4-D).  This maximizer refines: the owner's greedy
batch (``acquisition_batch``) gives ``n_starts`` diverse high-variance starts, start 0 being the candidate arg-max,
and one bounded L-BFGS-B run per start climbs the variance with its analytic gradient
(``variance_and_gradient``, the GPU predictive gradients).  The runs advance in lock-step, so every round of the
optimisation is ONE batched gradient call over the runs that want (f, g)."""
import numpy as np

from .. import _lbfgsb
from .._ffi import ACQ_MAX_Q
from .candidate_set_maximizer import CandidateSetMaximizer


class LBFGSBMaximizer(CandidateSetMaximizer):
    def __init__(self, candidates=None, n_candidates=100000, seed=0, distributed=False, n_starts=16, maxiter=100,
                 maxfun=200):
        super().__init__(candidates=candidates, n_candidates=n_candidates, seed=seed, distributed=distributed)
        if not 1 <= int(n_starts) <= ACQ_MAX_Q:
            raise ValueError("n_starts = %d must lie in [1, %d]" % (n_starts, ACQ_MAX_Q))
        self.n_starts, self.maxiter, self.maxfun = int(n_starts), int(maxiter), int(maxfun)
        self.last_rounds = None
        self.last_starts = None
        self.last_runs = None

    def maximize(self, model_predict: callable, lower_bound: np.ndarray, upper_bound: np.ndarray):
        owner = getattr(model_predict, "__self__", None)
        if owner is None or not (hasattr(owner, "acquisition_batch") and hasattr(owner, "variance_and_gradient")):
            return super().maximize(model_predict, lower_bound, upper_bound)   # foreign predict callable
        lb = np.asarray(lower_bound, dtype=np.float64).ravel()
        ub = np.asarray(upper_bound, dtype=np.float64).ravel()
        cands = self._candidates(lb, ub)
        idx, var = owner.acquisition_batch(cands, min(self.n_starts, len(cands)), distributed=self.distributed)
        starts = cands[idx]
        v0 = float(var[0])              # f = -var / v0: the tolerances mean the same at every variance scale
        rounds = [0]

        def batch_fun(xs):
            rounds[0] += 1
            v, g = owner.variance_and_gradient(np.array(xs))
            return [(-v[i] / v0, -g[i] / v0) for i in range(len(xs))]

        runs = _lbfgsb.minimize_lockstep(batch_fun, starts, maxfun=self.maxfun, maxiter=self.maxiter,
                                         bounds=list(zip(lb, ub)))
        xs = np.array([r[0] for r in runs])
        _, v = owner.predict(xs)        # the variance predict reports: the contract of every maximizer
        v = np.asarray(v, dtype=np.float64).ravel()
        best = int(np.argmax(v))        # lowest start index on ties
        self.last_index = int(idx[0])
        self.last_starts = starts
        self.last_runs = runs
        self.last_rounds = rounds[0]
        if not v[best] >= v0:           # a run never ends below its start; guard round-off between the two paths
            return starts[0].copy(), -v0
        return xs[best].copy(), -float(v[best])
