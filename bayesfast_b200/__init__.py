"""
bayesfast_b200 -- B200 (sm_100a) implementation of BayesFast's hot path: PolyModel surrogate fit and
value/gradient evaluation inside lock-step NUTS/HMC for thousands of chains.  See DESIGN.md.

Public interface mirrors the reference (h3jia/bayesfast): PolyConfig, PolyModel, Density, sample,
NTrace / HTrace / TraceTuple.  All numerics run in libbfb200.so (hand-written CUDA, C ABI in
include/bfb200.h); there is no CPU fallback.
"""
from .poly import PolyConfig, PolyModel
from .density import Density, GaussianLikelihood, GaussianPrior
from .sample_trace import NTrace, HTrace, TNTrace, THTrace, TraceTuple, SampleTrace
from .sample import sample
from .diag import diagnostics
from . import random

__all__ = ['PolyConfig', 'PolyModel', 'Density', 'GaussianLikelihood', 'GaussianPrior', 'NTrace', 'HTrace', 'TNTrace', 'THTrace', 'TraceTuple', 'SampleTrace', 'sample',
           'diagnostics', 'random']
__version__ = '0.1.0'
