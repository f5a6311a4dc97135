"""-m gpu: BatchedMCTS(leaves_per_game=L) and SelfPlay(leaves_per_game=L) against the leaf-parallel restatement
(tests/leaves_oracle.py).  The network outputs are recorded on the device and replayed on the restatement, the device's
f32 priors pinned after an rtol check; integer state and f64 value sums bit-exact."""
import functools

import numpy as np
import pytest
import torch

import tests.test_gpu_selfplay as selfplay_test
from alphazero_4_player_chess_b200.mcts import BatchedMCTS
from alphazero_4_player_chess_b200.selfplay import SelfPlay
from tests.golden.fake_net import FakeNet
from tests.leaves_oracle import search_leaves
from tests.reuse_oracle import reroot
from tests.test_gpu_mcts import assert_trees_equal, search_roots
from tests.test_gpu_mcts_reuse import expected_reroot, next_boards
from tests.util import mixed_positions, oracle_for

pytestmark = pytest.mark.gpu
C_PUCT = 3


def recorded_search(m, roots):
    """m.search with every batch's network outputs kept on the host; returns replay(batch, slots) for the
    restatement."""
    rec = []

    def record(batch, logits, value):
        rec.append((logits.cpu(), value.reshape(-1, 1).cpu()))

    m.search(roots, record=record)
    torch.cuda.synchronize()
    L = m.leaves

    def replay(batch, slots):
        rows = [gi * L + j for gi, j in slots]
        return rec[batch][0][rows], rec[batch][1][rows]

    return replay


def check_batch_state(m, trees):
    assert_trees_equal(m, trees)
    assert not m.in_flight.any()
    assert m.collisions.cpu().tolist() == [t.collisions for t in trees]


@pytest.mark.parametrize("name,R,n_games,sims,L", [("STANDARD", 14, 24, 48, 8), ("EIGHT_SIMPLE", 8, 4, 256, 64)])
@pytest.mark.parametrize("batch_rotation", [True, False])
def test_leaf_parallel_search_replays_on_the_restatement(name, R, n_games, sims, L, batch_rotation):
    o = oracle_for(R)
    roots = search_roots(name, R, n_games)
    m = BatchedMCTS(R, len(roots), FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims},
                    batch_rotation=batch_rotation, leaves_per_game=L)
    replay = recorded_search(m, torch.from_numpy(roots))
    trees = search_leaves(o, None, roots, C_PUCT, sims, L, 1, batch_rotation=batch_rotation, replay=replay,
                          prior_source=m.prior.cpu().numpy())
    check_batch_state(m, trees)
    n_coll = int(m.collisions.sum())
    print(f"{name} L={L} rot={batch_rotation}: {len(trees)} games, {int(m.n_nodes.sum())} nodes, {n_coll} collisions "
          f"of {len(trees) * sims} slots, {int(m.dropped.sum())} dropped roots")


def test_leaf_parallel_cuda_graph_search_equals_eager_search():
    R, sims, L = 14, 48, 8
    roots = torch.from_numpy(np.ascontiguousarray(mixed_positions("STANDARD", 64)))
    out = []
    for graph in (False, True):
        m = BatchedMCTS(R, 64, FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims}, cuda_graph=graph,
                        leaves_per_game=L, virtual_loss=2)
        m.search(roots)
        m.search(roots)  # a second search replays the captured graph from the start
        torch.cuda.synchronize()
        out.append(m)
    a, b = out
    assert b._graph is not None
    assert torch.equal(a.n_nodes, b.n_nodes) and torch.equal(a.n_boards, b.n_boards)
    assert torch.equal(a.collisions, b.collisions) and not b.in_flight.any()
    nn = int(a.n_nodes.max())
    used = torch.arange(nn, device="cuda")[None, :] < a.n_nodes[:, None]
    for name in ("parent", "move_flat", "visits", "value_sum", "prior", "first_child", "n_children", "board_idx"):
        assert torch.equal(getattr(a, name)[:, :nn][used], getattr(b, name)[:, :nn][used]), name


@pytest.mark.parametrize("batch_rotation", [True, False])
def test_leaf_parallel_search_advance_search_with_reuse(batch_rotation):
    R, sims, L = 14, 48, 8
    o = oracle_for(R)
    roots = search_roots("STANDARD", R, 16)
    m = BatchedMCTS(R, len(roots), FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims},
                    batch_rotation=batch_rotation, reuse_tree=True, leaves_per_game=L)
    replay = recorded_search(m, torch.from_numpy(roots))
    trees = search_leaves(o, None, roots, C_PUCT, sims, L, 1, batch_rotation=batch_rotation, replay=replay,
                          prior_source=m.prior.cpu().numpy())
    check_batch_state(m, trees)
    flat, visits, _, _ = m.root_children()
    actions = torch.gather(flat, 1, visits.argmax(dim=1, keepdim=True)).squeeze(1)
    boards = next_boards(R, m._roots, actions.cpu().numpy())
    kept = m.advance(actions, boards).cpu().numpy()
    want = [expected_reroot(o, m, t, int(a)) for t, a in zip(trees, actions.cpu().numpy())]
    assert kept.tolist() == [k for _, k in want]
    trees = [t for t, _ in want]
    assert (kept > 1).sum() >= len(roots) // 2
    replay = recorded_search(m, None)
    trees = search_leaves(o, None, None, C_PUCT, sims, L, 1, batch_rotation=batch_rotation, replay=replay,
                          prior_source=m.prior.cpu().numpy(), trees=trees)
    check_batch_state(m, trees)
    assert reroot  # the restatement's re-rooting is the one tests/test_gpu_mcts_reuse.py checks


@pytest.mark.parametrize("name,R,n,T", [("EIGHT_SIMPLE", 8, 24, 40), ("STANDARD", 14, 8, 6)])
def test_selfplay_with_four_leaves_per_game_replays_on_the_oracle(monkeypatch, name, R, n, T):
    """The self-play replay check of tests/test_gpu_selfplay.py with SelfPlay(leaves_per_game=4): 12 simulations are
    three batches of four leaf slots per game."""
    batches = []
    expand = BatchedMCTS.expand_backup

    def counted(self, logits, values):
        batches.append(int(logits.shape[0]))
        return expand(self, logits, values)

    monkeypatch.setattr(BatchedMCTS, "expand_backup", counted)
    monkeypatch.setattr(selfplay_test, "SelfPlay", functools.partial(SelfPlay, leaves_per_game=4, virtual_loss=1))
    selfplay_test.test_selfplay_replays_on_the_oracle(name, R, n, T)
    assert batches and set(batches) == {4 * n}
    assert len(batches) % 3 == 0  # num_searches 12 / L 4 per move
