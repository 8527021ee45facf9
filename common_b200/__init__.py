"""common_b200 -- B200-native hot path of microscopes-common.

Batched posterior-predictive scoring of rows against every group's sufficient
statistics, the categorical draw and the suffstat update that follow, behind
the reference's model / dataview / state interface.  All arithmetic runs in
hand-written sm_100a kernels (common_b200/csrc) reached through the C ABI of
include/mscope_b200.h; this package is the thin host mirror of the reference's
Python layer (microscopes/models.pyx, microscopes/common/recarray/dataview.pyx).
"""
from . import _lib
from ._lib import Context, MsbError
from .models import bb, bbnc, bnb, gp, nich, dd, dm, niw, model_descriptor
from .dataview import numpy_dataview
from .state import state, sample_discrete_log, philox_uniforms
from .hyperprior import log_exponential, log_normal, log_flat, log_noninformative_beta_prior
from . import synth

__all__ = ["Context", "MsbError", "bb", "bbnc", "bnb", "gp", "nich", "dd", "dm", "niw", "model_descriptor",
           "numpy_dataview", "state", "sample_discrete_log", "philox_uniforms", "log_exponential", "log_normal", "log_flat",
           "log_noninformative_beta_prior"]
