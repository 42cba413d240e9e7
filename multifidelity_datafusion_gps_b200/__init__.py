"""mfgp-b200: the multi-fidelity GP hot path of MartinKlapacz/multifidelity-datafusion-GPs on B200.

Public surface mirrors the reference's ``src`` package (src/__init__.py:1-6):
``MultifidelityDataFusion``, ``NARGP``, ``GPDF``, ``GPDFC``, the maximizer and delay-iterator plug-ins.
Importing the package does not touch the GPU; constructing a model does (no CPU fallback).
"""
from .MFDataFusion import MultifidelityDataFusion
from .abstractMFGP import AbstractMFGP
from .adaptation_maximizers import (AbstractMaximizer, ALCMaximizer, CandidateSetMaximizer, LBFGSBMaximizer,
                                    ScipyDirectMaximizer)
from .augm_iterators import AbstractAugmIterator, BackwardAugmentation, EvenAugmentation
from .models import GPDF, GPDFC, NARGP
from . import gpc

__all__ = ["MultifidelityDataFusion", "AbstractMFGP", "NARGP", "GPDF", "GPDFC", "AbstractMaximizer",
           "ALCMaximizer", "CandidateSetMaximizer", "LBFGSBMaximizer", "ScipyDirectMaximizer", "AbstractAugmIterator",
           "BackwardAugmentation", "EvenAugmentation"]
