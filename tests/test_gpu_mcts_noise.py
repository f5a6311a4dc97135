"""-m gpu: BatchedMCTS(root_noise=True) and SelfPlay(root_noise=True).  The network outputs are recorded on the device
and replayed on the MCTS restatement (one leaf: oracle/mcts_port.search through tests/reuse_oracle.search_on; L leaves:
tests/leaves_oracle.search_leaves), whose trees noise their roots through tests/noise_oracle.NoisedTree.  The network's
f32 priors are pinned to the device's after an rtol check (prior_source), the root's pre-noise priors taken from a
noise-off twin that shares the first batch; the noised root priors are checked against the restatement within rtol 1e-6
and pinned the same way.  Integer state and f64 value sums must then be identical."""
import functools

import numpy as np
import pytest
import torch

import tests.test_gpu_selfplay as selfplay_test
from alphazero_4_player_chess_b200._lib import FpcError
from alphazero_4_player_chess_b200.mcts import BatchedMCTS
from alphazero_4_player_chess_b200.selfplay import SelfPlay
from tests.golden.fake_net import FakeNet
from tests.leaves_oracle import search_leaves
from tests.noise_oracle import NoisedTree, noised, noised_tree
from tests.reuse_oracle import search_on
from tests.test_gpu_mcts import assert_trees_equal, search_roots
from tests.test_gpu_mcts_reuse import expected_reroot, next_boards
from tests.util import mixed_positions, oracle_for

pytestmark = pytest.mark.gpu
C_PUCT = 3
ALPHA, EPS, SEED = 0.3, 0.25, 0xC0FFEE
TREE = ("parent", "first_child", "n_children", "visits", "move_flat", "board_idx", "value_sum", "prior", "n_nodes",
        "n_boards", "leaf", "dropped", "error", "boards")


def make(R, n, sims, L=1, noise=True, eps=EPS, **kw):
    args = {"C": C_PUCT, "num_searches": sims, "dirichlet_alpha": ALPHA, "dirichlet_epsilon": eps}
    return BatchedMCTS(R, n, FakeNet(R, device="cuda"), args, leaves_per_game=L, root_noise=noise, noise_seed=SEED,
                       **kw)


def recorded(m, roots):
    """m.search with every batch's network outputs kept on the host; returns replay(batch, items) for the restatements
    (items: game indices at L = 1, (game, slot) pairs at L > 1)."""
    rec = []
    m.search(roots, record=lambda b, logits, value: rec.append((logits.cpu(), value.reshape(-1, 1).cpu())))
    torch.cuda.synchronize()

    def replay(batch, items):
        rows = [gi * m.leaves + j for gi, j in items] if m.leaves > 1 else list(items)
        return rec[batch][0][rows], rec[batch][1][rows]

    return replay


def root_priors(m):
    fc, k, prior = m.first_child[:, 0].cpu().numpy(), m.n_children[:, 0].cpu().numpy(), m.prior.cpu().numpy()
    return [prior[g, fc[g]: fc[g] + k[g]].copy() if k[g] > 0 else np.zeros(0, np.float32) for g in range(m.n)]


def pinned_priors(m, twin):
    """The device's priors with every root's children replaced by the noise-off twin's (the network's own priors)."""
    out = m.prior.cpu().numpy().copy()
    fc, k = m.first_child[:, 0].cpu().numpy(), m.n_children[:, 0].cpu().numpy()
    for g, p in enumerate(root_priors(twin)):
        assert len(p) == k[g]
        out[g, fc[g]: fc[g] + k[g]] = p
    return out


def twin_of(m, R, sims, L):
    """A noise-off instance holding m's trees (after an advance)."""
    t = make(R, m.n, sims, L, noise=False, reuse_tree=True)
    for name in TREE:
        getattr(t, name).copy_(getattr(m, name))
    t._has_tree = True
    return t


def replay_on_oracle(o, trees, sims, L, replay, prior_source):
    if L == 1:
        return search_on(o, None, trees, C_PUCT, sims, batch_rotation=False, replay=replay, prior_source=prior_source)
    return search_leaves(o, None, None, C_PUCT, sims, L, 1, batch_rotation=False, replay=replay,
                         prior_source=prior_source, trees=trees)


def best_moves(m):
    flat, visits, _, _ = m.root_children()
    return torch.gather(flat, 1, visits.argmax(dim=1, keepdim=True)).squeeze(1)


def same_trees(a, b):
    assert torch.equal(a.n_nodes, b.n_nodes) and torch.equal(a.n_boards, b.n_boards)
    nn = int(a.n_nodes.max())
    used = torch.arange(nn, device="cuda")[None, :] < a.n_nodes[:, None]
    for name in ("parent", "move_flat", "visits", "value_sum", "prior", "first_child", "n_children", "board_idx"):
        assert torch.equal(getattr(a, name)[:, :nn][used], getattr(b, name)[:, :nn][used]), name


def check(m, trees):
    assert_trees_equal(m, trees)
    if m.leaves > 1:
        assert not m.in_flight.any() and m.collisions.cpu().tolist() == [t.collisions for t in trees]


@pytest.mark.parametrize("name,R,n_games,sims", [("STANDARD", 14, 16, 48), ("EIGHT_SIMPLE", 8, 24, 48)])
@pytest.mark.parametrize("L", [1, 4])
def test_noised_search_and_reused_search_replay_on_the_oracle(name, R, n_games, sims, L):
    o = oracle_for(R)
    roots = search_roots(name, R, n_games)
    n = len(roots)
    roots_t = torch.from_numpy(roots)
    # 1. fresh roots: noised after the first batch, keys arange(n)
    off = make(R, n, sims, L, noise=False, reuse_tree=True)
    off.search(roots_t)
    m = make(R, n, sims, L, reuse_tree=True)
    replay = recorded(m, roots_t)
    pre, post = root_priors(off), root_priors(m)
    for g in range(n):
        assert len(pre[g]) == len(post[g]) > 0
        np.testing.assert_allclose(post[g], noised(pre[g], SEED, g, ALPHA, EPS), rtol=1e-6, atol=0, err_msg=str(g))
    assert m.noise_done.cpu().tolist() == [1] * n
    trees = [NoisedTree(o, C_PUCT, r).setup_noise(SEED, g, ALPHA, EPS, adopt=post[g]) for g, r in enumerate(roots)]
    trees = replay_on_oracle(o, trees, sims, L, replay, pinned_priors(m, off))
    assert all(t.noised_root for t in trees)
    check(m, trees)
    assert not torch.equal(m.visits[:, 0:64], off.visits[:, 0:64])  # the noise moved visits
    # 2. advance on the most visited child, search(None): kept roots noised before the first batch, fresh ones after
    actions = best_moves(m)
    boards = next_boards(R, roots, actions.cpu().numpy())
    kept = m.advance(actions, boards).cpu().numpy()
    want = [expected_reroot(o, m, t, int(a)) for t, a in zip(trees, actions.cpu().numpy())]
    assert kept.tolist() == [k for _, k in want]
    assert (kept > 1).sum() >= n // 2
    assert not m.noise_done.any()
    twin = twin_of(m, R, sims, L)
    twin.search(None)
    replay = recorded(m, None)
    post = root_priors(m)
    trees = [noised_tree(t, SEED, n + g, ALPHA, EPS, adopt=post[g]) for g, (t, _) in enumerate(want)]
    trees = replay_on_oracle(o, trees, sims, L, replay, pinned_priors(m, twin))
    assert [t.noised_root for t in trees] == m.noise_done.bool().tolist()  # all but roots without children
    check(m, trees)
    print(f"{name} L={L}: {n} games, {int((kept > 1).sum())} kept subtrees, {int(m.n_nodes.sum())} nodes, root noise "
          f"replayed on the restatement over two searches")


@pytest.mark.parametrize("L", [1, 4])
def test_graph_replay_and_eager_search_give_the_same_noised_trees(L):
    """The noise calls sit outside the captured graph: before and after its first batch, whether that batch is an eager
    warm-up (first search) or a graph replay (search(None) after an advance)."""
    R, sims = 14, 48
    roots = torch.from_numpy(np.ascontiguousarray(mixed_positions("STANDARD", 64)))
    out = []
    for graph in (False, True):
        m = make(R, 64, sims, L, cuda_graph=graph, reuse_tree=True)
        m.search(roots)
        actions = best_moves(m)
        kept = m.advance(actions, next_boards(R, roots.numpy(), actions.cpu().numpy()))
        m.search(None)
        torch.cuda.synchronize()
        out.append((m, kept))
    (a, ka), (b, kb) = out
    assert b._graph is not None and torch.equal(ka, kb) and int((ka > 1).sum()) > 32
    assert torch.equal(a.noise_done, b.noise_done) and int(a.noise_done.sum()) > 32
    same_trees(a, b)


def test_noise_off_changes_nothing(monkeypatch):
    """root_noise=False never calls the kernel and grows the trees of the parent's loop (select -> network ->
    expand_backup by hand) over a search, an advance and a search(None); root_noise=True with epsilon 0 calls it twice
    per search and changes no prior, so its trees are the same too."""
    R, sims = 14, 40
    roots = torch.from_numpy(search_roots("STANDARD", R, 24))
    n = len(roots)
    off = make(R, n, sims, noise=False, reuse_tree=True)
    by_hand = make(R, n, sims, noise=False, reuse_tree=True)
    eps0 = make(R, n, sims, eps=0.0, reuse_tree=True)
    calls = []
    kernel = off.L.fpc_tree_root_noise
    monkeypatch.setattr(off.L, "fpc_tree_root_noise", lambda *a: calls.append(1) or kernel(*a))

    def hand(m):
        for _ in range(sims):
            logits, value = m.net(m.select())
            m.expand_backup(logits, value)

    off.search(roots)
    by_hand.reset(roots)
    hand(by_hand)
    actions = best_moves(off)
    assert torch.equal(actions, best_moves(by_hand))
    boards = next_boards(R, roots.numpy(), actions.cpu().numpy())
    for m in (off, by_hand):
        m.advance(actions, boards)
    off.search(None)
    hand(by_hand)
    torch.cuda.synchronize()
    assert not calls
    same_trees(off, by_hand)
    eps0.search(roots)
    eps0.advance(actions, boards)
    eps0.search(None)
    torch.cuda.synchronize()
    assert len(calls) == 4 and int(eps0.noise_done.sum()) > n // 2
    same_trees(off, eps0)


def test_arguments():
    R = 8
    with pytest.raises(ValueError, match="dirichlet_alpha"):
        BatchedMCTS(R, 2, None, {"C": 3, "num_searches": 4, "dirichlet_epsilon": 0.25}, root_noise=True)
    with pytest.raises(ValueError, match="dirichlet_epsilon"):
        BatchedMCTS(R, 2, None, {"C": 3, "num_searches": 4, "dirichlet_alpha": 0.3}, root_noise=True)
    with pytest.raises(FpcError, match="root_noise=True"):
        make(R, 2, 4, noise=False).add_root_noise(torch.arange(2))
    with pytest.raises(FpcError, match="alpha"):
        BatchedMCTS(R, 2, None, {"C": 3, "num_searches": 4, "dirichlet_alpha": 0.0, "dirichlet_epsilon": 0.25},
                    root_noise=True).add_root_noise(torch.arange(2))


@pytest.mark.parametrize("name,R,n,T,reuse,L", [("EIGHT_SIMPLE", 8, 24, 40, False, 1), ("EIGHT_SIMPLE", 8, 24, 40, True, 4),
                                               ("STANDARD", 14, 8, 6, True, 1)])
def test_noised_selfplay_replays_on_the_oracle_and_repeats(monkeypatch, name, R, n, T, reuse, L):
    """The self-play replay check of tests/test_gpu_selfplay.py (boards, legality, results, rewards) with
    SelfPlay(root_noise=True), run twice: the same torch seed and noise seed give the same games.  A noise-off run from
    the same torch seed searches differently."""
    made = []

    def factory(noise, R_, n_, net, args, start, **kw):
        args = {**args, "dirichlet_alpha": ALPHA, "dirichlet_epsilon": EPS}
        sp = SelfPlay(R_, n_, net, args, start, reuse_tree=reuse, leaves_per_game=L, root_noise=noise, noise_seed=SEED,
                      **kw)
        made.append(sp)
        return sp

    monkeypatch.setattr(selfplay_test, "SelfPlay", functools.partial(factory, True))
    selfplay_test.test_selfplay_replays_on_the_oracle(name, R, n, T)
    selfplay_test.test_selfplay_replays_on_the_oracle(name, R, n, T)
    monkeypatch.setattr(selfplay_test, "SelfPlay", functools.partial(factory, False))
    selfplay_test.test_selfplay_replays_on_the_oracle(name, R, n, T)
    a, b, off = made
    for attr in ("hist_boards", "hist_flat", "hist_visits", "hist_valid", "hist_action"):
        assert torch.equal(getattr(a, attr), getattr(b, attr)), attr
    assert torch.equal(a.env.boards, b.env.boards)
    assert not torch.equal(a.hist_visits[0], off.hist_visits[0])
