"""-m gpu: BatchedMCTS(gumbel=True, gumbel_interior=True) and SelfPlay with the same pair.  The network outputs of a
search are recorded on the device and replayed on the MCTS restatement through
tests/gumbel_interior_oracle.GumbelInteriorTree, the f32 priors pinned to the device's (prior_source).  node_value is
filled with NaN before every search, so a read before a write shows up as a mismatch.  Integer state and f64 value sums
must then be identical, node_value must equal the restatement's cache on every node it wrote, and the result must
match.  A choice where the device and the restatement differ is adopted only on a near-tie, and counted."""

import numpy as np
import pytest
import torch

import tests.test_gpu_selfplay as selfplay_test
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.mcts import BatchedMCTS
from alphazero_4_player_chess_b200.selfplay import SelfPlay
from tests.golden.fake_net import FakeNet
from tests.gumbel_interior_oracle import GumbelInteriorTree
from tests.reuse_oracle import search_on
from tests.test_gpu_mcts import assert_trees_equal, search_roots
from tests.test_gpu_mcts_gumbel import SEED, check_result, device_roots
from tests.test_gpu_mcts_noise import same_trees
from tests.util import mixed_positions, oracle_for

pytestmark = pytest.mark.gpu
C_PUCT = 3


def make(R, n, sims, considered=16, **kw):
    return BatchedMCTS(R, n, FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims}, gumbel=True,
                       gumbel_seed=SEED, gumbel_considered=considered, gumbel_interior=True, **kw)


@pytest.mark.parametrize("name,R,n_games", [("STANDARD", 14, 16), ("EIGHT_SIMPLE", 8, 24)])
@pytest.mark.parametrize("batch_rotation", [True, False])
@pytest.mark.parametrize("considered", [4, 16])
def test_search_replays_on_the_restatement(name, R, n_games, batch_rotation, considered):
    sims = 48
    o = oracle_for(R)
    roots = search_roots(name, R, n_games)
    n = len(roots)
    m = make(R, n, sims, considered, batch_rotation=batch_rotation)
    m.node_value.fill_(float("nan"))
    rec, leaves = [], []

    def record(b, logits, value):
        rec.append((logits.cpu(), value.reshape(-1, 1).cpu()))
        leaves.append(m.leaf.cpu().numpy().copy())

    m.search(torch.from_numpy(roots), record=record)
    torch.cuda.synchronize()
    dev = device_roots(m, leaves)
    trees = [GumbelInteriorTree(o, C_PUCT, r).setup_gumbel(SEED, g, considered, sims - 1, 1.0, dev[g])
             .setup_interior([lv[g] for lv in leaves]) for g, r in enumerate(roots)]
    trees = search_on(o, None, trees, C_PUCT, sims, batch_rotation=batch_rotation,
                      replay=lambda b, games: (rec[b][0][games], rec[b][1][games]), prior_source=m.prior.cpu().numpy())
    assert_trees_equal(m, trees)
    adopted = sum(t.adopted + t.adopted_interior for t in trees)
    assert adopted <= 2, adopted
    root_value, node_value = m.root_value.cpu().numpy(), m.node_value.cpu().numpy()
    written = 0
    for g, t in enumerate(trees):
        if t.root_value is not None:
            assert root_value[g] == t.root_value, g
        for x, v in t.node_value.items():
            assert node_value[g, x] == v, (g, x)
        written += len(t.node_value)
    check_result(m, trees)
    interior = sum(sum(1 for kind, _, _ in t.log if kind == "r") for t in trees)
    print(f"{name} rot={batch_rotation} m={considered}: {n} games, {int(m.n_nodes.sum())} nodes, {written} node values "
          f"written, {interior} cached reads, {int(m.dropped.sum())} dropped, {adopted} near-tie choices adopted")
    assert written > n and interior > n


def test_graph_replay_and_eager_search_give_the_same_trees():
    roots = torch.from_numpy(np.ascontiguousarray(mixed_positions("STANDARD", 64)))
    out = []
    for graph in (False, True):
        m = make(14, 64, 32, cuda_graph=graph)
        m.search(roots)
        first = m.gumbel_result()
        m.search(roots.flip(0).contiguous(), gumbel_keys=torch.arange(64) * 7 + 1)
        torch.cuda.synchronize()
        out.append((m, first, m.gumbel_result()))
    (a, a1, a2), (b, b1, b2) = out
    assert b._graph is not None
    same_trees(a, b)
    assert torch.equal(a.root_value, b.root_value) and torch.equal(a.gumbel_keys, b.gumbel_keys)
    for x, y in ((a1, b1), (a2, b2)):
        assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1])


def test_interior_off_never_calls_the_new_function(monkeypatch):
    calls = []
    m = BatchedMCTS(8, 8, FakeNet(8, device="cuda"), {"C": C_PUCT, "num_searches": 12}, gumbel=True)
    fn = m.L.fpc_tree_select_gumbel_interior
    monkeypatch.setattr(m.L, "fpc_tree_select_gumbel_interior", lambda *a: calls.append(1) or fn(*a))
    m.search(torch.from_numpy(np.repeat(start_record("EIGHT_SIMPLE")[None], 8, axis=0)))
    args = {"C": C_PUCT, "num_searches": 8, "temperature": 1.1, "max_game_length": 6, "heuristic_weight": 0.02}
    for gumbel in (False, True):
        SelfPlay(8, 8, FakeNet(8, device="cuda"), args, start_record("EIGHT_SIMPLE"), gumbel=gumbel).play()
    torch.cuda.synchronize()
    assert not calls and not hasattr(m, "node_value")


def test_refused_combinations():
    args = {"C": C_PUCT, "num_searches": 8, "dirichlet_alpha": 0.3, "dirichlet_epsilon": 0.25}
    with pytest.raises(ValueError, match="gumbel_interior"):
        BatchedMCTS(8, 2, None, args, gumbel_interior=True)
    for kw, what in (({"reuse_tree": True}, "reuse_tree"), ({"root_noise": True}, "root_noise"),
                     ({"leaves_per_game": 2}, "leaves_per_game")):
        with pytest.raises(ValueError, match=what):
            BatchedMCTS(8, 2, None, args, gumbel=True, gumbel_interior=True, **kw)
    m = make(8, 2, 8)
    m.search(torch.from_numpy(np.repeat(start_record("EIGHT_SIMPLE")[None], 2, axis=0)))
    with pytest.raises(Exception, match="search"):
        m.search(None)


@pytest.mark.parametrize("name,R,n,T", [("EIGHT_SIMPLE", 8, 24, 40), ("STANDARD", 14, 8, 6)])
def test_selfplay_replays_on_the_oracle_and_repeats(monkeypatch, name, R, n, T):
    """The self-play replay check of tests/test_gpu_selfplay.py with SelfPlay(gumbel=True, gumbel_interior=True), run
    twice: the same seeds give the same games, and every ply plays its gumbel_result's action."""
    made, results = [], []

    def factory(R_, n_, net, args, start, **kw):
        sp = SelfPlay(R_, n_, net, args, start, gumbel=True, gumbel_seed=SEED, gumbel_considered=8,
                      gumbel_interior=True, **kw)
        fn = sp.mcts.gumbel_result

        def recorded():
            out = fn()
            results.append((len(made) - 1, out[0].clone(), out[1].clone()))
            return out

        sp.mcts.gumbel_result = recorded
        made.append(sp)
        return sp

    monkeypatch.setattr(selfplay_test, "SelfPlay", factory)
    selfplay_test.test_selfplay_replays_on_the_oracle(name, R, n, T)
    selfplay_test.test_selfplay_replays_on_the_oracle(name, R, n, T)
    a, b = made
    assert a.mcts.gumbel_interior
    for attr in ("hist_boards", "hist_flat", "hist_visits", "hist_valid", "hist_action", "hist_policy"):
        assert torch.equal(getattr(a, attr), getattr(b, attr)), attr
    plies = [(a_, p) for run, a_, p in results if run == 0]
    for t, (action, policy) in enumerate(plies):
        valid = a.hist_valid[t]
        assert torch.equal(a.hist_action[t][valid], action[valid]), t
        assert torch.equal(a.hist_policy[t], policy), t
