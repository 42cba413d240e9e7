"""Integrated-variance ("active learning Cohn", ALC) acquisition over a candidate set.

Every other maximizer here picks the input with the largest predictive variance at the input itself ("active learning
MacKay", the reference's rule).  That rule favours the boundary of the box, where the variance is large but a new
point says little about the rest of the domain.  ALC instead picks the candidate whose acquisition most lowers the
weighted mean predictive variance over a reference set (Cohn 1996; Seo et al. 2000), which is what the test MSE of the
adapted model measures.  The scores come from the owner's ``acquisition_alc`` (GPU K8c) in one call per step."""
import numpy as np

from .candidate_set_maximizer import CandidateSetMaximizer


def alc_weights(weights, R):
    """Validated reference weights: R finite entries >= 0, not all zero, as a contiguous float64 array."""
    w = np.ascontiguousarray(weights, dtype=np.float64)
    if w.shape != (int(R),):
        raise ValueError("weights must have one entry per reference row (%d), got shape %s" % (int(R), w.shape))
    if not np.all(np.isfinite(w)) or np.any(w < 0.0):
        raise ValueError("weights must be finite and >= 0")
    if not np.any(w > 0.0):
        raise ValueError("weights must not all be zero")
    return w


class ALCMaximizer(CandidateSetMaximizer):
    """``maximize`` returns ``(x, -alc)``: the candidate whose acquisition lowers the weighted mean latent variance
    over the reference rows the most, and the negated amount.  This differs from the variance contract of
    ``AbstractMaximizer``: ``adapt``'s stop ``|fopt| < eps`` then means "the best point lowers the mean reference
    variance by less than eps".

    candidates / n_candidates / seed / distributed: as in ``CandidateSetMaximizer``.  reference: (R, d) rows over
    which the variance is integrated; when None, n_reference rows are drawn uniformly in the bounds from a random
    stream of their own (deterministic in seed, independent of the candidates' stream).  weights: (R,) non-negative
    weights of the reference rows, or None for 1/R."""

    def __init__(self, candidates=None, n_candidates=100000, reference=None, n_reference=1024, weights=None, seed=0,
                 distributed=False):
        super().__init__(candidates=candidates, n_candidates=n_candidates, seed=seed, distributed=distributed)
        if reference is not None:
            reference = np.ascontiguousarray(reference, dtype=np.float64)
            if reference.ndim != 2 or reference.shape[0] < 1:
                raise ValueError("reference must be a non-empty (R, d) array")
        elif int(n_reference) < 1:
            raise ValueError("n_reference = %d must be >= 1" % int(n_reference))
        self.reference = reference
        self.n_reference = int(n_reference) if reference is None else reference.shape[0]
        self.weights = None if weights is None else alc_weights(weights, self.n_reference)
        self.last_alc = None

    def _reference(self, lower_bound, upper_bound):
        if self.reference is None:
            lb = np.asarray(lower_bound, dtype=np.float64)
            ub = np.asarray(upper_bound, dtype=np.float64)
            # spawn key (1,): a child stream of the seed, unrelated to default_rng(seed) that draws the candidates
            rng = np.random.default_rng(np.random.SeedSequence(self.seed, spawn_key=(1,)))
            self.reference = lb + (ub - lb) * rng.uniform(size=(self.n_reference, len(lb)))
        return self.reference

    def maximize(self, model_predict: callable, lower_bound: np.ndarray, upper_bound: np.ndarray):
        owner = getattr(model_predict, "__self__", None)
        if owner is None or not hasattr(owner, "acquisition_alc"):
            raise TypeError("ALCMaximizer needs the predict method of a model with acquisition_alc: the integrated "
                            "variance reduction cannot be computed from a predict callable's variances")
        cands = self._candidates(lower_bound, upper_bound)
        ref = self._reference(lower_bound, upper_bound)
        idx, alc = owner.acquisition_alc(cands, ref, self.weights, distributed=self.distributed)   # GPU K8c
        self.last_index = idx
        self.last_alc = alc
        return cands[idx].copy(), -alc

    def maximize_batch(self, model_predict: callable, lower_bound: np.ndarray, upper_bound: np.ndarray, q: int):
        """q = 1 is ``maximize``.  q > 1 raises: the inherited greedy batch ranks by variance, not by ALC."""
        if int(q) != 1:
            raise NotImplementedError("ALCMaximizer picks one point per step (q = %d asked); greedy ALC batches are "
                                      "not implemented" % int(q))
        x, fopt = self.maximize(model_predict, lower_bound, upper_bound)
        return np.atleast_2d(np.asarray(x, dtype=np.float64)), np.array([float(fopt)])
