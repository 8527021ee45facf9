"""Hyperpriors for state.slice_hp: the reference's in-tree log densities (scalar_functions.hpp:34-74) and a flat interval.

Each prior is a callable that evaluates its log density in numpy, so the same object can also give a grid's log_prior
for state.set_hp_grid, and it carries (kind, a, b), the enum msb_hprior form the device evaluates:

    log_exponential(rate)           log(rate) - rate x for x >= 0, -inf below
    log_normal(mu, sigmasq)         -0.5 log(2 pi sigmasq) - (x - mu)^2 / (2 sigmasq)
    log_flat(lo, hi)                0 on (lo, hi), -inf outside
    log_noninformative_beta_prior   -2.5 log(alpha + beta), a prior on a pair: called as f(alpha, beta), and on the device
                                    each of the pair is updated with its partner at its current value
"""
import numpy as np

FLAT, EXPONENTIAL, NORMAL, NONINFORMATIVE_BETA = range(4)     # enum msb_hprior


class _prior(object):
    kind = None

    def __init__(self, a=0.0, b=0.0):
        self.a, self.b = float(a), float(b)

    def __repr__(self):
        return "%s(%r, %r)" % (type(self).__name__, self.a, self.b)


class log_exponential(_prior):
    kind = EXPONENTIAL

    def __init__(self, rate):
        super().__init__(rate)

    def __call__(self, x):
        x = np.asarray(x, np.float64)
        return np.where(x >= 0.0, np.log(self.a) - self.a * x, -np.inf)


class log_normal(_prior):
    kind = NORMAL

    def __init__(self, mu, sigmasq):
        super().__init__(mu, sigmasq)

    def __call__(self, x):
        t = np.asarray(x, np.float64) - self.a
        return -0.5 * np.log(2.0 * np.pi * self.b) - t * t / (2.0 * self.b)


class log_flat(_prior):
    kind = FLAT

    def __init__(self, lo, hi):
        super().__init__(lo, hi)

    def __call__(self, x):
        x = np.asarray(x, np.float64)
        return np.where((x > self.a) & (x < self.b), 0.0, -np.inf)


class _noninformative_beta(_prior):
    kind = NONINFORMATIVE_BETA

    def __call__(self, alpha, beta):
        with np.errstate(invalid="ignore", divide="ignore"):
            return -2.5 * np.log(np.asarray(alpha, np.float64) + np.asarray(beta, np.float64))

    def __repr__(self):
        return "log_noninformative_beta_prior"


log_noninformative_beta_prior = _noninformative_beta()
