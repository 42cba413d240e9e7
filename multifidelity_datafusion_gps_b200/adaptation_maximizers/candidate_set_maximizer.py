"""Candidate-set acquisition (north-star item (d), SURVEY.md section 8a row A9).

The reference's maximizers run a sequential DIRECT search of up to 20 000 single-point ``predict``
calls (src/adaptation_maximizers/scipydirect_wrapper.py:22-26).  This maximizer scores a whole
candidate set in one batched GPU predict and takes the arg-max on the device (K8); with
``torch.distributed`` initialised the candidates are split contiguously over the ranks and the
per-rank winners are combined with one all_gather (max value, lowest global index).  ``maximize_batch``
takes a greedy batch of q candidates per step through the owner's ``acquisition_batch``."""
import numpy as np

from .abstract_maximizer import AbstractMaximizer


class CandidateSetMaximizer(AbstractMaximizer):
    def __init__(self, candidates=None, n_candidates=100000, seed=0, distributed=False):
        super().__init__()
        self.candidates = None if candidates is None else np.ascontiguousarray(candidates, dtype=np.float64)
        self.n_candidates = int(n_candidates)
        self.seed = seed
        self.distributed = distributed
        self.last_index = None
        self.last_indices = None
        self.last_gap = None

    def _candidates(self, lower_bound, upper_bound):
        if self.candidates is None:
            lb = np.asarray(lower_bound, dtype=np.float64)
            ub = np.asarray(upper_bound, dtype=np.float64)
            u = np.random.default_rng(self.seed).uniform(size=(self.n_candidates, len(lb)))
            self.candidates = lb + (ub - lb) * u
        return self.candidates

    def maximize(self, model_predict: callable, lower_bound: np.ndarray, upper_bound: np.ndarray):
        cands = self._candidates(lower_bound, upper_bound)
        owner = getattr(model_predict, "__self__", None)
        if owner is not None and hasattr(owner, "acquisition_argmax"):
            idx, val = owner.acquisition_argmax(cands, distributed=self.distributed)   # GPU K6 + K8
        else:   # foreign predict callable: honour the plug-in contract
            _, var = model_predict(cands)
            var = np.asarray(var).ravel()
            idx = int(np.argmax(var))
            val = float(var[idx])
        self.last_index = idx
        return cands[idx].copy(), -val

    def maximize_batch(self, model_predict: callable, lower_bound: np.ndarray, upper_bound: np.ndarray, q: int):
        owner = getattr(model_predict, "__self__", None)
        if int(q) == 1 or owner is None or not hasattr(owner, "acquisition_batch"):
            return super().maximize_batch(model_predict, lower_bound, upper_bound, q)
        cands = self._candidates(lower_bound, upper_bound)
        idx, var = owner.acquisition_batch(cands, int(q), distributed=self.distributed)   # GPU K6 + K8b
        self.last_indices = idx
        self.last_index = int(idx[-1])
        return cands[idx].copy(), -var
