"""The numpy restatement of fpc_tree_sample_root (tests/sample_oracle.py) against the distribution the reference's
self-play samples from (alphazero.py:108-118: visits / sum raised to 1 / temperature, renormalised), and the properties
of its keyed uniform: a choice is a function of (seed, key), and distinct keys draw independently."""
import numpy as np
import pytest
from scipy import stats

from tests.sample_oracle import SAMPLE_J, sample_index, sample_many, weights
from tests.noise_oracle import uniform

VISITS = np.array([1, 9, 3, 0, 27, 5, 1, 14, 2, 40, 7, 1], np.int64)
N_KEYS = 200_000


@pytest.mark.parametrize("temperature", [0.5, 1.0, 1.7])
def test_frequencies_follow_the_tempered_visit_distribution(temperature):
    keys = np.arange(N_KEYS, dtype=np.int64) * 977 + 12345
    picks = sample_many(VISITS, temperature, 0x5EED, keys)
    counts = np.bincount(picks, minlength=len(VISITS))
    p = (VISITS / VISITS.sum()) ** (1.0 / temperature)
    p = p / p.sum()
    assert counts[VISITS == 0].sum() == 0  # a child without visits is never drawn
    live = p > 0
    _, pval = stats.chisquare(counts[live], p[live] * N_KEYS)
    assert pval > 1e-4, (temperature, counts, p * N_KEYS)


@pytest.mark.parametrize("temperature", [0.5, 1.0, 1.7])
def test_vectorised_and_scalar_restatements_agree(temperature):
    keys = np.arange(-500, 500, dtype=np.int64) * 7919
    many = sample_many(VISITS, temperature, 99, keys)
    one = [sample_index(VISITS, temperature, 99, int(k))[0] for k in keys]
    assert many.tolist() == one


def test_the_choice_is_a_function_of_seed_and_key():
    keys = np.arange(4096, dtype=np.int64)
    a = sample_many(VISITS, 1.0, 7, keys)
    assert np.array_equal(a, sample_many(VISITS, 1.0, 7, keys))
    assert np.array_equal(a[::-1], sample_many(VISITS, 1.0, 7, keys[::-1]))  # order of the batch does not matter
    assert np.array_equal(a[100:101], sample_many(VISITS, 1.0, 7, keys[100:101]))
    assert not np.array_equal(a, sample_many(VISITS, 1.0, 8, keys))  # another seed, other draws


def test_draws_of_distinct_keys_are_independent():
    # the uniforms of keys k and k + 1 (consecutive plies of one game) and of k and k + T (one ply of two games)
    keys = np.arange(N_KEYS, dtype=np.int64) * 3
    u = uniform(0x5EED, keys, 0, SAMPLE_J)
    assert stats.kstest(u, "uniform").pvalue > 1e-4
    for step in (1, 200):
        v = uniform(0x5EED, keys + step, 0, SAMPLE_J)
        table = np.histogram2d(u, v, bins=8, range=[[0, 1], [0, 1]])[0]
        assert stats.chi2_contingency(table)[1] > 1e-4, step
        assert abs(np.corrcoef(u, v)[0, 1]) < 0.02
    # and the stream is disjoint from the root noise's (j <= 192) and Gumbel's (j = 2^31) at the same key
    for j in (0, 1, 192, 2**31):
        assert not np.any(u == uniform(0x5EED, keys, 0, j))


def test_degenerate_roots():
    assert sample_index([], 1.0, 0, 0)[0] == -1
    assert sample_index([0, 0, 0], 1.0, 0, 0)[0] == -1
    assert sample_index([0, 0, 0], 0.5, 0, 0)[0] == -1
    assert sample_index([0, 5, 0], 1.3, 0, 11)[0] == 1
    assert sample_index([-3, 0, 2], 1.0, 0, 11)[0] == 2  # a negative count weighs 0
    assert np.array_equal(weights([2, 6], 1.0), [2.0, 6.0])
    np.testing.assert_allclose(weights([2, 6], 0.5), [1 / 16, 9 / 16], rtol=1e-15)
