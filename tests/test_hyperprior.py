"""CPU: the hyperpriors of common_b200.hyperprior against scipy, and the flattening of slice_hp's arguments into the
msb_slice_hp_spec array."""
import math

import numpy as np
import pytest
from scipy import stats

from common_b200 import hyperprior as hp
from common_b200.state import slice_hp_specs

X = np.array([-3.0, -1e-300, 0.0, 1e-300, 0.01, 0.5, 1.0, 2.0, 7.5, 30.0, 1e3])


def close(got, want):
    got, want = np.asarray(got), np.asarray(want)
    assert np.array_equal(np.isneginf(got), np.isneginf(want))
    fin = np.isfinite(want)
    assert np.all(np.abs(got[fin] - want[fin]) <= 1e-14 * np.maximum(1.0, np.abs(want[fin])))


@pytest.mark.parametrize("rate", [0.1, 1.0, 3.5])
def test_log_exponential_is_scipy_expon(rate):
    p = hp.log_exponential(rate)
    close(p(X), stats.expon(scale=1.0 / rate).logpdf(X))
    assert (p.kind, p.a) == (hp.EXPONENTIAL, rate)


@pytest.mark.parametrize("mu,s2", [(0.0, 1.0), (-2.0, 0.25), (5.0, 40.0)])
def test_log_normal_is_scipy_norm(mu, s2):
    p = hp.log_normal(mu, s2)
    close(p(X), stats.norm(mu, math.sqrt(s2)).logpdf(X))
    assert (p.kind, p.a, p.b) == (hp.NORMAL, mu, s2)


@pytest.mark.parametrize("lo,hi", [(0.0, 1.0), (-2.0, 7.5), (0.5, 30.0)])
def test_log_flat_is_scipy_uniform_inside_and_minus_inf_outside(lo, hi):
    p = hp.log_flat(lo, hi)
    x = np.concatenate([X, [lo, hi, np.nextafter(lo, np.inf), np.nextafter(hi, -np.inf)]])
    want = stats.uniform(lo, hi - lo).logpdf(x) + math.log(hi - lo)     # 0 inside; the open interval at the ends
    want[(x <= lo) | (x >= hi)] = -np.inf
    close(p(x), want)
    assert (p.kind, p.a, p.b) == (hp.FLAT, lo, hi)


def test_noninformative_beta_prior_formula():
    a = np.array([0.1, 1.0, 3.0, 100.0])
    b = np.array([2.0, 1.0, 0.5, 1e-3])
    close(hp.log_noninformative_beta_prior(a, b), [-2.5 * math.log(x + y) for x, y in zip(a, b)])
    assert hp.log_noninformative_beta_prior.kind == hp.NONINFORMATIVE_BETA


def test_a_prior_gives_a_grid_log_prior():
    pts = np.array([0.5, 1.0, 2.0])
    close(hp.log_exponential(2.0)(pts), [math.log(2.0) - 2.0 * x for x in pts])


def test_specs_flatten_in_order_with_tuple_keys_expanded():
    e, n = hp.log_exponential(1.5), hp.log_normal(0.0, 2.0)
    specs = slice_hp_specs({2: {"mu": (n, 0.5), "kappa": (e, 1.0)},
                            0: {("alpha", "beta"): (hp.log_noninformative_beta_prior, 2.0)},
                            1: {("beta", "alpha"): (e, 0.1)}},
                           {"alpha": (hp.log_flat(0.1, 9.0), 3.0)}, 5)
    assert specs == [(2, "mu", 0.5, hp.NORMAL, 0.0, 2.0), (2, "kappa", 1.0, hp.EXPONENTIAL, 1.5, 0.0),
                     (0, "alpha", 2.0, hp.NONINFORMATIVE_BETA, 0.0, 0.0), (0, "beta", 2.0, hp.NONINFORMATIVE_BETA, 0.0, 0.0),
                     (1, "beta", 0.1, hp.EXPONENTIAL, 1.5, 0.0), (1, "alpha", 0.1, hp.EXPONENTIAL, 1.5, 0.0),
                     (5, "alpha", 3.0, hp.FLAT, 0.1, 9.0)]
    assert slice_hp_specs(None, None, 3) == []
    with pytest.raises(TypeError, match="common_b200.hyperprior"):
        slice_hp_specs({0: {"alpha": (lambda x: 0.0, 1.0)}}, None, 1)
