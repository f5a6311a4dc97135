"""CPU: the numpy restatement of the root noise (tests/noise_oracle.py) draws what it claims to draw.  Gamma(alpha, 1)
against scipy by a Kolmogorov-Smirnov test, the Dirichlet mixture's moments against the closed forms, the counter-based
draws' determinism, and the Marsaglia-Tsang fallback after 64 rejections."""
import numpy as np
import pytest
from scipy import stats

import tests.noise_oracle as no

SEED = 0x5EED


def test_mix64_matches_a_python_integer_restatement():
    M = (1 << 64) - 1

    def ref(seed, key, ctr):
        z = seed ^ ((key * 0x9E3779B97F4A7C15) & M) ^ ((ctr * 0xBF58476D1CE4E5B9) & M)
        z = (z + 0x9E3779B97F4A7C15) & M
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
        return z ^ (z >> 31)

    for seed, key, ctr in [(0, 0, 0), (SEED, 12345, (7 << 32) | 3), (M, M, M), (1, (1 << 63) + 5, 1 << 40)]:
        assert int(no.mix64(seed, key, ctr)) == ref(seed, key, ctr)
    u = no.uniform(SEED, np.arange(100000), 0, 0)
    assert (u > 0).all() and (u <= 1).all() and abs(u.mean() - 0.5) < 0.005


@pytest.mark.parametrize("alpha", [0.03, 0.2, 0.3, 1.0, 2.5])
def test_gamma_matches_scipy(alpha):
    n = 20000
    keys = np.arange(n, dtype=np.int64) * 7 + 3
    g = no.gamma(SEED, keys, np.arange(n) % 300, alpha)
    assert np.isfinite(g).all() and (g >= 0).all()
    ks = stats.kstest(g, stats.gamma(alpha).cdf)
    assert ks.pvalue > 1e-3, (alpha, ks)
    assert abs(g.mean() - alpha) < 5 * np.sqrt(alpha / n)


@pytest.mark.parametrize("alpha,k", [(0.3, 2), (0.3, 19), (0.03, 38), (1.0, 38), (0.3, 300)])
def test_dirichlet_moments(alpha, k):
    n = 4000 if k < 300 else 800
    eta = np.stack([no.dirichlet(SEED, key, k, alpha) for key in range(n)])
    assert np.allclose(eta.sum(axis=1), 1.0, rtol=0, atol=1e-12)
    a0 = k * alpha
    mean, var = 1.0 / k, alpha * (a0 - alpha) / (a0 * a0 * (a0 + 1.0))
    # every component has the same marginal Beta(alpha, a0 - alpha): pool them, but judge with the per-component
    # sample size n (the components of one draw are dependent)
    x = eta.reshape(-1)
    se_mean = np.sqrt(var / n)
    assert abs(eta.mean(axis=0) - mean).max() < 6 * se_mean * np.sqrt(2 * np.log(k) + 1)
    m4 = ((x - mean) ** 4).mean()
    se_var = np.sqrt(max(m4 - var * var, 0.0) / n)
    assert abs(x.var() - var) < 6 * se_var, (x.var(), var, se_var)


def test_draws_are_counter_based():
    a = no.noised(np.full(38, 1 / 38, np.float32), SEED, 77, 0.3, 0.25)
    b = no.noised(np.full(38, 1 / 38, np.float32), SEED, 77, 0.3, 0.25)
    assert np.array_equal(a.view(np.int32), b.view(np.int32))
    assert not np.array_equal(a, no.noised(np.full(38, 1 / 38, np.float32), SEED, 78, 0.3, 0.25))
    assert not np.array_equal(a, no.noised(np.full(38, 1 / 38, np.float32), SEED + 1, 77, 0.3, 0.25))
    # child i's draw does not depend on how many siblings it has, and a negative key is its uint64 bit pattern
    assert np.array_equal(no.gamma(SEED, 5, np.arange(19), 0.3), no.gamma(SEED, 5, np.arange(38), 0.3)[:19])
    assert np.array_equal(no.gamma(SEED, -1, np.arange(4), 0.3), no.gamma(SEED, np.uint64(2**64 - 1), np.arange(4), 0.3))


@pytest.mark.parametrize("alpha", [0.3, 1.0, 2.5])
def test_fallback_after_64_rejections(monkeypatch, alpha):
    """Uniforms that put every attempt's v at or below 0 (x = -sqrt(-2 ln 1e-6) < -1/c): the draw is d = a - 1/3,
    times U(i, 192)^(1/alpha) for alpha < 1."""
    def fake(seed, key, i, j):
        return np.where(np.asarray(j) % 3 == 1, 0.5, 1e-6) + np.zeros(np.shape(key))

    monkeypatch.setattr(no, "uniform", fake)
    a = alpha + 1.0 if alpha < 1.0 else alpha
    want = (a - 1.0 / 3.0) * (1e-6 ** (1.0 / alpha) if alpha < 1.0 else 1.0)
    assert np.array_equal(no.gamma(SEED, np.arange(3), np.arange(3), alpha), np.full(3, want))
