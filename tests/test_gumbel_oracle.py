"""CPU: the numpy restatement of the Gumbel root search (tests/gumbel_oracle.py) -- its halving schedule against a literal
transcription of mctx's, sequential halving on a one-level bandit, Gumbel-max sampling from the prior, policy
improvement, and the draws' determinism."""
import math

import numpy as np
from scipy import stats

from tests.gumbel_oracle import considered_visits, gumbels, result, root_choice

SEED = 0xFEED


def mctx_sequence(m, n_sims):
    """mctx/_src/seq_halving.py get_sequence_of_considered_visits, transcribed literally."""
    if m <= 1:
        return tuple(range(n_sims))
    log2max = int(math.ceil(math.log2(m)))
    sequence = []
    visits = [0] * m
    num_considered = m
    while len(sequence) < n_sims:
        num_extra_visits = max(1, int(n_sims / (log2max * num_considered)))
        for _ in range(num_extra_visits):
            sequence.extend(visits[:num_considered])
            for i in range(num_considered):
                visits[i] += 1
        num_considered = max(2, int(num_considered / 2))
    return tuple(sequence[:n_sims])


def issue_loop(s, m, n_sims):
    """The schedule's loop as include/fpc.h states it, phase by phase (no closed-form tail)."""
    if m <= 1:
        return s
    l2, c, v = math.ceil(math.log2(m)), m, 0
    while True:
        e = max(1, n_sims // (l2 * c))
        if s < e * c:
            return v + s // c
        s, v, c = s - e * c, v + e, max(2, c // 2)


def test_schedule_equals_mctx_and_extends_past_n_sims():
    for m in range(1, 33):
        for n in range(0, 513):
            want = mctx_sequence(m, n)
            assert tuple(considered_visits(s, m, n) for s in range(n)) == want, (m, n)
        for n in (0, 1, 7, 50, 199):
            for s in range(0, 2 * n + 40):
                assert considered_visits(s, m, n) == issue_loop(s, m, n), (m, n, s)


def bandit(k, m, n_sims, q, prior, key, scale=1.0, root_v=0.0):
    """n_sims root visits on a one-level bandit whose arm i always backs up q[i] (in the frame of the root's q_i):
    returns (N, order of choices, action index, improved policy)."""
    N, vs, picks = np.zeros(k, np.int64), np.zeros(k), []
    root = -root_v
    for _ in range(n_sims):
        i, _ = root_choice(N, vs, prior, root, SEED, key, m, n_sims, scale)
        assert i >= 0
        picks.append(i)
        N[i] += 1
        vs[i] += q[i]
    a, pol = result(N, vs, prior, root, SEED, key, scale)
    return N, picks, a, pol


def random_bandit(rng, k):
    prior = rng.dirichlet(np.full(k, 0.7)).astype(np.float32)
    q = rng.uniform(-1.0, 1.0, k)
    return prior, q


def test_bandit_visits_follow_sequential_halving():
    rng = np.random.default_rng(1)
    for k, m, n_sims in [(20, 16, 63), (20, 16, 200), (38, 16, 47), (5, 4, 32), (300, 300, 299), (3, 16, 10), (7, 1, 9)]:
        prior, q = random_bandit(rng, k)
        for key in range(3):
            N, picks, a, _ = bandit(k, m, n_sims, q, prior, key)
            cv = [considered_visits(s, min(m, k), n_sims) for s in range(n_sims)]
            # every visit went to an arm at the considered count, so the arms at or above v + 1 visits are the
            # simulations that considered v
            for v in range(max(cv) + 1):
                assert int((N >= v + 1).sum()) == cv.count(v), (k, m, n_sims, v)
            assert int((N > 0).sum()) == min(min(m, k), n_sims)
            assert N[a] == N.max()


def test_no_visits_samples_the_prior_and_the_first_choices_are_the_top_m():
    rng = np.random.default_rng(2)
    k = 20
    prior, q = random_bandit(rng, k)
    keys = np.arange(20_000)
    logits = np.log(prior.astype(np.float64))
    first = np.argmax(gumbels(SEED, keys, k, 1.0) + (logits - logits.max()), axis=1)
    # the kernel's first choice is this argmax (sigma is 0 while nothing is visited)
    for key in range(0, 20_000, 2_000):
        assert root_choice(np.zeros(k), np.zeros(k), prior, 0.3, SEED, key, 16, 31, 1.0)[0] == first[key]
    counts = np.bincount(first, minlength=k)
    expected = prior.astype(np.float64) / prior.astype(np.float64).sum() * len(keys)
    big = expected >= 5.0
    obs, exp = counts[big], expected[big]
    if not big.all():  # the rare arms pooled into one bin
        obs, exp = np.append(obs, counts[~big].sum()), np.append(exp, expected[~big].sum())
    assert stats.chisquare(obs, exp * obs.sum() / exp.sum()).pvalue > 0.001
    for key in range(5):
        _, picks, _, _ = bandit(k, 16, 64, q, prior, key)
        top = np.argsort(-(gumbels(SEED, key, k, 1.0) + logits - logits.max()), kind="stable")[:16]
        assert picks[:16] == top.tolist()


def test_policy_improvement_on_the_bandit():
    rng = np.random.default_rng(3)
    k = 20
    prior, q = random_bandit(rng, k)
    p = prior.astype(np.float64) / prior.astype(np.float64).sum()
    played, best_mass = [], []
    for key in range(200):
        N, _, a, pol = bandit(k, 16, 32, q, prior, key, root_v=float(p @ q))
        played.append(q[a])
        best_mass.append(pol[np.argmax(q)])
        assert abs(float(pol.astype(np.float64).sum()) - 1.0) < 1e-6
    assert np.mean(played) >= float(p @ q)
    assert np.mean(best_mass) > p[np.argmax(q)]


def test_draws_are_deterministic_key_dependent_and_vanish_at_scale_zero():
    rng = np.random.default_rng(4)
    k = 38
    prior, q = random_bandit(rng, k)
    a = bandit(k, 16, 40, q, prior, key=7)
    b = bandit(k, 16, 40, q, prior, key=7)
    assert a[1] == b[1] and a[2] == b[2] and np.array_equal(a[3], b[3])
    assert len({tuple(bandit(k, 16, 40, q, prior, key=key)[1]) for key in range(8)}) > 1
    assert np.array_equal(gumbels(SEED, 7, k, 1.0), gumbels(SEED, np.array([3, 7]), k, 1.0)[1])
    zero = {tuple(bandit(k, 16, 40, q, prior, key=key, scale=0.0)[1]) for key in range(8)}
    assert len(zero) == 1
