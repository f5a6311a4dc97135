"""CPU: the numpy restatement of Gumbel MuZero's interior selection (tests/gumbel_interior_oracle.py) -- its choice
against a literal transcription of mctx's gumbel_muzero_interior_action_selection, the unvisited node, the visit bound
of the deterministic rule, policy improvement on a fixed-q bandit, and the node_value cache's lifecycle."""
import numpy as np

from tests.gumbel_interior_oracle import TIE, GumbelInteriorTree, improved_policy, interior_choice


# ---- mctx, transcribed literally (mctx/_src/qtransforms.py and mctx/_src/action_selection.py) -----------------------
def softmax(x):
    e = np.exp(x - np.max(x))
    return e / np.sum(e)


def mctx_qtransform_completed_by_mix_value(qvalues, visit_counts, raw_value, prior_logits, value_scale=0.1,
                                           maxvisit_init=50.0, rescale_values=True, use_mixed_value=True,
                                           epsilon=1e-8):
    prior_probs = softmax(prior_logits)
    if use_mixed_value:
        sum_visit_counts = np.sum(visit_counts, axis=-1)
        prior_probs_ = np.maximum(np.finfo(prior_probs.dtype).tiny, prior_probs)
        sum_probs = np.sum(np.where(visit_counts > 0, prior_probs_, 0.0), axis=-1)
        weighted_q = np.sum(np.where(visit_counts > 0,
                                     prior_probs_ * qvalues / np.where(visit_counts > 0, sum_probs, 1.0), 0.0), axis=-1)
        value = (raw_value + sum_visit_counts * weighted_q) / (sum_visit_counts + 1)
    else:
        value = raw_value
    completed_qvalues = np.where(visit_counts > 0, qvalues, value)
    if rescale_values:
        min_value = np.min(completed_qvalues, axis=-1, keepdims=True)
        max_value = np.max(completed_qvalues, axis=-1, keepdims=True)
        completed_qvalues = (completed_qvalues - min_value) / np.maximum(max_value - min_value, epsilon)
    maxvisit = np.max(visit_counts, axis=-1)
    visit_scale = maxvisit_init + maxvisit
    return visit_scale * value_scale * completed_qvalues


def mctx_prepare_argmax_input(probs, visit_counts):
    return probs - visit_counts / (1 + np.sum(visit_counts, keepdims=True, axis=-1))


def mctx_interior_action(visit_counts, prior_logits, qvalues, raw_value):
    completed_qvalues = mctx_qtransform_completed_by_mix_value(qvalues, visit_counts, raw_value, prior_logits)
    to_argmax = mctx_prepare_argmax_input(probs=softmax(prior_logits + completed_qvalues), visit_counts=visit_counts)
    return int(np.argmax(to_argmax, axis=-1))


def random_node(rng, k):
    """(N, value sums, f32 priors, u) with some children unvisited and, for k > 1, an unvisited zero prior."""
    prior = rng.dirichlet(np.full(k, 0.5)).astype(np.float32)
    N = np.where(rng.random(k) < 0.6, rng.integers(1, 12, k), 0)
    if k > 1:
        z = int(rng.integers(0, k))
        prior[z], N[z] = 0.0, 0
    vs = rng.uniform(-1.0, 1.0, k) * N
    return N.astype(np.int64), vs, prior, float(rng.uniform(-1.0, 1.0))


def test_choice_equals_mctx_up_to_near_ties():
    rng = np.random.default_rng(11)
    ties = 0
    for k in (1, 2, 20, 38, 300):
        for _ in range(300):
            N, vs, prior, u = random_node(rng, k)
            if rng.random() < 0.1:
                N[:] = 0
                vs[:] = 0.0
            i, sc = interior_choice(N, vs, prior, u)
            q = np.where(N > 0, vs / np.maximum(N, 1), 0.0)
            with np.errstate(divide="ignore"):
                logits = np.log(prior.astype(np.float64))
            j = mctx_interior_action(N, logits, q, -u)
            assert i >= 0
            if i != j:
                assert abs(sc[i] - sc[j]) <= TIE, (k, i, j, sc[i], sc[j])
                ties += 1
            assert prior[i] > 0.0
    assert ties <= 3, ties


def test_unvisited_node_takes_the_largest_prior():
    rng = np.random.default_rng(12)
    for k in (1, 2, 20, 38, 300):
        prior = rng.dirichlet(np.full(k, 0.5)).astype(np.float32)
        prior[rng.integers(0, k)] = prior.max()  # a tie: the first index wins
        i, _ = interior_choice(np.zeros(k, np.int64), np.zeros(k), prior, float(rng.normal()))
        assert i == int(np.argmax(prior))


def test_visit_counts_stay_within_the_improved_policy():
    """c_scale = 0: sigma = 0, pi' is the normalised prior, and after n visits every N_i < n * pi'_i + 1."""
    rng = np.random.default_rng(13)
    for k in (2, 5, 20, 38):
        prior = rng.dirichlet(np.full(k, 0.4)).astype(np.float32)
        prior[0] = 0.0
        N, vs = np.zeros(k, np.int64), rng.normal(size=k)
        pi, _ = improved_policy(N, vs, prior, 0.0, c_scale=0.0)
        for n in range(1, 513):
            i, _ = interior_choice(N, vs, prior, 0.0, c_scale=0.0)
            assert i != 0  # the zero prior
            N[i] += 1
            assert np.all(N < n * pi + 1), (k, n, N, n * pi + 1)


def test_improved_policy_improves_on_a_fixed_q_bandit():
    """sigma is monotone in the completed Q, so sum pi'_i cq_i >= sum p_i cq_i at every step; once every arm is
    visited cq is the bandit's q itself."""
    rng = np.random.default_rng(14)
    for k in (2, 20, 38):
        prior = rng.dirichlet(np.full(k, 0.7)).astype(np.float32)
        p = prior.astype(np.float64) / prior.astype(np.float64).sum()
        q = rng.uniform(-1.0, 1.0, k)
        u = float(rng.uniform(-1.0, 1.0))
        N, vs = np.zeros(k, np.int64), np.zeros(k)
        for step in range(200):
            pi, s = improved_policy(N, vs, prior, u)
            vis = N > 0
            qn = np.where(vis, vs / np.maximum(N, 1), 0.0)
            w = np.maximum(prior.astype(np.float64), 2.0 ** -126)
            v_mix = (-u + s * (np.sum(w[vis] * qn[vis]) / np.sum(w[vis]) if vis.any() else 0.0)) / (1.0 + s)
            cq = np.where(vis, qn, v_mix)
            assert pi @ cq >= p @ cq - 1e-12, (k, step)
            if vis.all():
                assert pi @ q >= p @ q - 1e-12, (k, step)
            i, _ = interior_choice(N, vs, prior, u)
            N[i] += 1
            vs[i] += q[i]


class _Rules:
    """No terminal positions and boards that never change: a synthetic tree."""

    def game_result(self, rec):
        return 0, None, None

    def make_index(self, rec, flat):
        return rec


def test_node_value_is_written_once_at_the_first_pass_and_read_after():
    rng = np.random.default_rng(15)
    t = GumbelInteriorTree(_Rules(), 3.0, np.zeros(4, np.uint8)).setup_gumbel(7, 3, 4, 119, 1.0).setup_interior()
    own = {}  # each node's network value as its expansion backed it up
    for _ in range(120):
        leaf = t.choose_leaf()
        value = float(np.float32(rng.uniform(-1.0, 1.0)))
        t.backpropagate(leaf, value)
        own[leaf] = value
        b = int(rng.integers(1, 5))
        t.expand(leaf, range(b), rng.dirichlet(np.ones(b)).astype(np.float32).tolist())
    passes = {}
    for kind, node, sel in t.log:
        passes.setdefault(node, []).append((kind, sel))
    assert len(passes) > 10
    for node, ev in passes.items():
        assert ev[0][0] == "w" and all(kind == "r" for kind, _ in ev[1:]), (node, ev)
        assert [sel for _, sel in ev] == sorted(sel for _, sel in ev)
        assert t.node_value[node] == own[node]  # value_sum at the first pass is the node's own network value
    assert sum(len(ev) for ev in passes.values()) > 2 * len(passes)
