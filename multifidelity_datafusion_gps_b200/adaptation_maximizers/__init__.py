"""Acquisition maximizers: plug-ins that return the input with the largest predictive variance
(reference: src/adaptation_maximizers/; ``CandidateSetMaximizer`` is the GPU candidate-set arg-max)."""
from .abstract_maximizer import AbstractMaximizer
from .alc_maximizer import ALCMaximizer
from .candidate_set_maximizer import CandidateSetMaximizer
from .lbfgsb_maximizer import LBFGSBMaximizer
from .scipydirect_wrapper import ScipyDirectMaximizer

__all__ = ["AbstractMaximizer", "ALCMaximizer", "CandidateSetMaximizer", "LBFGSBMaximizer", "ScipyDirectMaximizer"]
