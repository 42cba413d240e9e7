"""Plug-in point of the acquisition step (reference src/adaptation_maximizers/abstract_maximizer.py:5-28)."""
from abc import ABCMeta, abstractmethod

import numpy as np


class AbstractMaximizer(metaclass=ABCMeta):
    """Wrapper for the uncertainty maximisation of the adaptation process."""

    @abstractmethod
    def __init__(self):
        super().__init__()

    @abstractmethod
    def maximize(self, model_predict: callable, lower_bound: np.ndarray, upper_bound: np.ndarray):
        """Return ``(x, fopt)``: the input in [lower_bound, upper_bound] with the largest predictive
        variance and the NEGATED variance there (the reference minimises ``-variance``,
        src/adaptation_maximizers/scipydirect_wrapper.py:22-31)."""

    def maximize_batch(self, model_predict: callable, lower_bound: np.ndarray, upper_bound: np.ndarray, q: int):
        """Return ``(X (q, d), fopt (q,))``: q inputs for one adaptation step, point i being the most uncertain
        input given the training set plus points 0..i-1 at the current hyper-parameters, and the negated
        variances.  q = 1 is ``maximize``; choosing q > 1 needs a maximiser that can condition the model on its
        own picks (CandidateSetMaximizer), so the default raises."""
        if int(q) == 1:
            x, fopt = self.maximize(model_predict, lower_bound, upper_bound)
            return np.atleast_2d(np.asarray(x, dtype=np.float64)), np.array([float(np.ravel(fopt)[0])])
        raise NotImplementedError("%s cannot choose a batch of q = %d points: it searches a predict callable "
                                  "that it cannot condition on its own picks (use CandidateSetMaximizer)"
                                  % (type(self).__name__, int(q)))
