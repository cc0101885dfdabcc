"""CPU checks of the host side of the device MAP fit (boss_gp_map_multistart): the numpy log-space prior of its host
twin against central differences and the mirror's densities, and the prior-table encoding of a GaussianProcess."""
import math

import numpy as np
import pytest

from tests.map_multistart_oracle import logprior_z, raw_of, z_of

CASES = [
    (0, (0.25, 0.0)),
    (1, (0.3, 0.7)),
    (2, (-0.4, 0.6)),
    (3, (0.05, 4.0)),
]


@pytest.mark.parametrize("kind,par", CASES, ids=["dirac", "normal", "lognormal", "uniform"])
def test_logprior_z_matches_central_differences(kind, par):
    rng = np.random.default_rng(3)
    z = rng.uniform(-1.5, 1.3, 40)
    k = np.array([kind]); p = np.array([par])
    v, g = logprior_z(k, p, raw_of(k, p, z[:, None]))
    h = 1e-6
    vp, _ = logprior_z(k, p, raw_of(k, p, (z + h)[:, None]))
    vm, _ = logprior_z(k, p, raw_of(k, p, (z - h)[:, None]))
    fd = (vp - vm) / (2 * h)
    assert np.all(np.isfinite(v))
    np.testing.assert_allclose(g[:, 0], fd, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("kind,par", CASES[1:], ids=["normal", "lognormal", "uniform"])
def test_logprior_value_is_the_mirror_density(kind, par):
    from boss_b200.types import LogNormal, Normal, Uniform
    prior = {1: Normal, 2: LogNormal, 3: Uniform}[kind](*par)
    raw = np.array([0.01, 0.3, 1.0, 2.5, 3.9])
    v, _ = logprior_z(np.array([kind]), np.array([par]), raw[:, None])
    ref = np.array([prior.logpdf(x) for x in raw])
    np.testing.assert_allclose(v, ref, rtol=1e-13, atol=1e-13)


def test_uniform_outside_support_is_minus_inf():
    v, g = logprior_z(np.array([3]), np.array([(0.5, 2.0)]), np.array([[0.4], [0.5], [2.0], [2.1]]))
    assert v[0] == -math.inf and v[3] == -math.inf and np.isfinite(v[1:3]).all()
    assert np.all(g == 0.0)


def test_pinned_entries_stay_at_zero_in_z():
    kind = np.array([2, 0, 1])
    z = z_of(kind, np.array([[0.5, 123.0, 2.0]]))
    assert z[0, 1] == 0.0 and z[0, 0] == math.log(0.5)
    assert raw_of(kind, np.array([[0, 0], [0.7, 0], [0, 1]]), z)[0, 1] == 0.7


def _gp(ls_priors, amp=None, noise=None, y_dim=1):
    import boss_b200 as B
    return B.GaussianProcess(lengthscale_priors=ls_priors, amplitude_priors=amp or [B.LogNormal(0.0, 0.5)] * y_dim,
                             noise_std_priors=noise or [B.Dirac(0.1)] * y_dim)


def test_prior_tables_decompose_products_and_pin_diracs():
    import boss_b200 as B
    from boss_b200.model_fitters import gp_prior_tables
    ls = [B.Product([B.LogNormal(0.1, 0.2), B.Normal(1.0, 0.5), B.Uniform(0.1, 3.0)]),
          B.Product([B.Dirac(0.4), B.LogNormal(0.0, 1.0), B.LogNormal(0.5, 0.25)])]
    model = _gp(ls, amp=[B.LogNormal(0.0, 0.5), B.Uniform(0.5, 2.0)], noise=[B.Dirac(0.1), B.Dirac(0.0)], y_dim=2)
    kind, par = gp_prior_tables(model, 3, 2)
    assert kind.dtype == np.int32 and kind.shape == (2, 5) and par.shape == (2, 5, 2)
    assert kind.tolist() == [[2, 1, 3, 2, 0], [0, 2, 2, 3, 0]]
    assert par[0, 0].tolist() == [0.1, 0.2] and par[0, 2].tolist() == [0.1, 3.0] and par[0, 4, 0] == 0.1
    assert par[1, 0, 0] == 0.4 and par[1, 3].tolist() == [0.5, 2.0] and par[1, 4, 0] == 0.0
    # mvlognormal is a Product of LogNormals; a single univariate prior is the one lengthscale of a 1-D input
    kind, _ = gp_prior_tables(_gp([B.mvlognormal([0.5, 0.5], [0.5, 0.5])]), 2, 1)
    assert kind.tolist() == [[2, 2, 2, 0]]
    kind, _ = gp_prior_tables(_gp([B.LogNormal(0.0, 1.0)]), 1, 1)
    assert kind.tolist() == [[2, 2, 0]]


def test_prior_tables_fall_back_on_unsupported_priors_and_models():
    import boss_b200 as B
    from boss_b200.model_fitters import gp_prior_tables
    from boss_b200.types import Prior

    class HalfCauchy(Prior):
        def logpdf(self, x):
            return math.log(2 / math.pi) - math.log1p(x * x) if x >= 0 else -math.inf

    assert gp_prior_tables(_gp([B.Product([B.LogNormal(), HalfCauchy()])]), 2, 1) is None
    assert gp_prior_tables(_gp([B.mvlognormal([0, 0], [1, 1])], amp=[HalfCauchy()]), 2, 1) is None
    assert gp_prior_tables(_gp([B.mvlognormal([0, 0, 0], [1, 1, 1])]), 2, 1) is None      # wrong number of parts
    assert gp_prior_tables(_gp([B.LogNormal()]), 2, 1) is None                             # univariate for d = 2
    semi = B.Semiparametric(B.Parametric(lambda x, th: np.array([th[0]]), [B.Uniform(-1, 1)]),
                            _gp([B.mvlognormal([0, 0], [1, 1])]))
    assert gp_prior_tables(semi, 2, 1) is None
