"""-m gpu: BatchedMCTS(gumbel=True) and SelfPlay(gumbel=True).  The network outputs of a search are recorded on the
device and replayed on the MCTS restatement through tests/gumbel_oracle.GumbelTree (oracle/mcts_port.search through
tests/reuse_oracle.search_on), the f32 priors pinned to the device's after an rtol check (prior_source).  Integer state
and f64 value sums must then be identical, and the actions and improved policies of the result must match.  A root
choice where the device and the restatement differ is adopted only on a last-ulp near-tie (GumbelTree), and counted."""

import numpy as np
import pytest
import torch

import tests.test_gpu_selfplay as selfplay_test
from alphazero_4_player_chess_b200._lib import FpcError
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.mcts import BatchedMCTS
from alphazero_4_player_chess_b200.net import AutocastNet, PolicyValueNet
from alphazero_4_player_chess_b200.selfplay import SelfPlay
from alphazero_4_player_chess_b200.train import Learner
from tests.golden.fake_net import FakeNet
from tests.gumbel_oracle import GumbelTree
from tests.reuse_oracle import search_on
from tests.test_gpu_mcts import assert_trees_equal, search_roots
from tests.test_gpu_mcts_noise import same_trees
from tests.test_gpu_puct_kernels import rot_index
from tests.util import mixed_positions, oracle_for

pytestmark = pytest.mark.gpu
C_PUCT = 3
SEED = 0xB0A7


def make(R, n, sims, considered=16, **kw):
    return BatchedMCTS(R, n, FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims}, gumbel=True,
                       gumbel_seed=SEED, gumbel_considered=considered, **kw)


def device_roots(m, leaves):
    """[game][batch] the root child above each batch's leaf (-1 where the leaf was the root or none)."""
    parent = m.parent.cpu().numpy()
    out = []
    for g in range(m.n):
        row = []
        for lv in leaves:
            x = int(lv[g])
            while x > 0 and parent[g, x] != 0:
                x = int(parent[g, x])
            row.append(x if x > 0 else -1)
        out.append(row)
    return out


def check_result(m, trees):
    action, policy = (x.cpu().numpy() for x in m.gumbel_result())
    for g, t in enumerate(trees):
        flat, pol = t.result()
        k = len(pol)
        assert action[g] == flat, g
        np.testing.assert_allclose(policy[g, :k], pol, rtol=1e-6, atol=0, err_msg=str(g))
        assert not policy[g, k:].any()


@pytest.mark.parametrize("name,R,n_games", [("STANDARD", 14, 16), ("EIGHT_SIMPLE", 8, 24)])
@pytest.mark.parametrize("batch_rotation", [True, False])
@pytest.mark.parametrize("considered", [4, 16])
def test_search_replays_on_the_restatement(name, R, n_games, batch_rotation, considered):
    sims = 48
    o = oracle_for(R)
    roots = search_roots(name, R, n_games)
    n = len(roots)
    m = make(R, n, sims, considered, batch_rotation=batch_rotation)
    rec, leaves = [], []

    def record(b, logits, value):
        rec.append((logits.cpu(), value.reshape(-1, 1).cpu()))
        leaves.append(m.leaf.cpu().numpy().copy())

    m.search(torch.from_numpy(roots), record=record)
    torch.cuda.synchronize()
    dev = device_roots(m, leaves)
    trees = [GumbelTree(o, C_PUCT, r).setup_gumbel(SEED, g, considered, sims - 1, 1.0, dev[g])
             for g, r in enumerate(roots)]
    trees = search_on(o, None, trees, C_PUCT, sims, batch_rotation=batch_rotation,
                      replay=lambda b, games: (rec[b][0][games], rec[b][1][games]), prior_source=m.prior.cpu().numpy())
    assert_trees_equal(m, trees)
    adopted = sum(t.adopted for t in trees)
    assert adopted <= 2, adopted
    root_value = m.root_value.cpu().numpy()
    for g, t in enumerate(trees):
        if t.root_value is not None:
            assert root_value[g] == t.root_value, g
    check_result(m, trees)
    visited = (m.visits[:, 0] > 1).sum().item()
    print(f"{name} rot={batch_rotation} m={considered}: {n} games, {int(m.n_nodes.sum())} nodes, {visited} searched "
          f"roots, {int(m.dropped.sum())} dropped, {adopted} near-tie choices adopted")


def test_graph_replay_and_eager_search_give_the_same_trees():
    """The graph reads the keys and writes root_value at fixed addresses: the second search (new keys) replays the
    graph captured in the first and must still equal eager searches."""
    roots = torch.from_numpy(np.ascontiguousarray(mixed_positions("STANDARD", 64)))
    out = []
    for graph in (False, True):
        m = make(14, 64, 32, cuda_graph=graph)
        m.search(roots)
        first = m.gumbel_result()
        m.search(roots.flip(0).contiguous())
        torch.cuda.synchronize()
        out.append((m, first, m.gumbel_result()))
    (a, a1, a2), (b, b1, b2) = out
    assert b._graph is not None
    same_trees(a, b)
    assert torch.equal(a.root_value, b.root_value) and torch.equal(a.gumbel_keys, b.gumbel_keys)
    for x, y in ((a1, b1), (a2, b2)):
        assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1])


def test_gumbel_off_never_calls_the_new_functions(monkeypatch):
    calls = []
    m = BatchedMCTS(8, 8, FakeNet(8, device="cuda"), {"C": C_PUCT, "num_searches": 12})
    for name in ("fpc_tree_select_gumbel", "fpc_tree_gumbel_result"):
        fn = getattr(m.L, name)
        monkeypatch.setattr(m.L, name, lambda *a, _fn=fn: calls.append(1) or _fn(*a))
    m.search(torch.from_numpy(np.repeat(start_record("EIGHT_SIMPLE")[None], 8, axis=0)))
    args = {"C": C_PUCT, "num_searches": 8, "temperature": 1.1, "max_game_length": 6, "heuristic_weight": 0.02}
    SelfPlay(8, 8, FakeNet(8, device="cuda"), args, start_record("EIGHT_SIMPLE")).play()
    torch.cuda.synchronize()
    assert not calls
    with pytest.raises(FpcError, match="gumbel=True"):
        m.gumbel_result()


def test_refused_combinations_and_arguments():
    args = {"C": C_PUCT, "num_searches": 8, "dirichlet_alpha": 0.3, "dirichlet_epsilon": 0.25}
    for kw, what in (({"reuse_tree": True}, "reuse_tree"), ({"root_noise": True}, "root_noise"),
                     ({"leaves_per_game": 2}, "leaves_per_game")):
        with pytest.raises(ValueError, match=what):
            BatchedMCTS(8, 2, None, args, gumbel=True, **kw)
    roots = torch.from_numpy(np.repeat(start_record("EIGHT_SIMPLE")[None], 2, axis=0))
    m = make(8, 2, 8)
    m.search(roots)
    with pytest.raises(FpcError, match="search"):
        m.search(None)
    for kw, what in (({"considered": 0}, "max_considered"), ({"gumbel_scale": -1.0}, "scale")):
        bad = make(8, 2, 8, **kw)
        with pytest.raises(FpcError, match=what):
            bad.search(roots)


@pytest.mark.parametrize("name,R,n,T", [("EIGHT_SIMPLE", 8, 24, 40), ("STANDARD", 14, 8, 6)])
def test_gumbel_selfplay_replays_on_the_oracle_and_targets_the_networks_frame(monkeypatch, name, R, n, T):
    """The self-play replay check of tests/test_gpu_selfplay.py (boards, legality, results, rewards, policy targets
    summing to 1) with SelfPlay(gumbel=True), run twice: the same seeds give the same games.  Every ply plays the action
    of that ply's gumbel_result, its improved policy is the replay's policy target, placed in the network's frame: child
    `flat` of a position with colour k to move at rot_index(k)[flat]."""
    made, results = [], []

    def factory(R_, n_, net, args, start, **kw):
        sp = SelfPlay(R_, n_, net, args, start, gumbel=True, gumbel_seed=SEED, gumbel_considered=8, **kw)
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
    for attr in ("hist_boards", "hist_flat", "hist_visits", "hist_valid", "hist_action", "hist_policy"):
        assert torch.equal(getattr(a, attr), getattr(b, attr)), attr
    plies = [(a_, p) for run, a_, p in results if run == 0]
    for t, (action, policy) in enumerate(plies):
        valid = a.hist_valid[t]
        assert torch.equal(a.hist_action[t][valid], action[valid]), t
        assert torch.equal(a.hist_policy[t], policy), t
    replay = a.finish(torch.zeros(n, dtype=torch.bool, device="cuda"), torch.full((n,), -1, device="cuda"))
    pol = a.policy_targets(replay)
    cp, flat = replay["child_policy"], replay["child_flat"].long()
    assert torch.allclose(pol.sum(dim=1), torch.ones(len(pol), device="cuda"), atol=1e-5)
    mask = cp > 0  # the root's children (padding columns are zero)
    assert bool(mask.any(dim=1).all())
    # the targets are in the network's frame: the search reads child `flat` of a position with colour k to move at
    # rot_index(k)[flat] of the row
    A, ks = a.geom.num_action_channels, replay["boards"][:, a.geom.off_turn].long()
    rot = torch.stack([torch.from_numpy(rot_index(R, A, k)) for k in range(4)]).cuda()
    at = rot[ks[:, None], flat]
    assert torch.allclose(torch.gather(pol, 1, at)[mask], cp[mask], rtol=1e-5, atol=1e-7)


def test_learner_trains_on_a_gumbel_replay():
    torch.manual_seed(0)
    R = 8
    model = PolicyValueNet(R, blocks=1, hidden=16, device="cuda")
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    args = {"C": 3, "num_searches": 8, "temperature": 1.1, "max_game_length": 10, "heuristic_weight": 0.02,
            "batch_size": 16, "replay_buffer_capacity": 4096, "validation_buffer_capacity": 1024}
    sp = SelfPlay(R, 16, AutocastNet(model), args, start_record("EIGHT_SIMPLE"), gumbel=True, gumbel_considered=4)
    learner = Learner(sp, model, opt, args)
    assert learner.train_buf.child_policy is not None
    learner.store(sp.play())
    used = learner.train_buf.child_policy[:len(learner.train_buf)]
    assert torch.allclose(used.sum(dim=1), torch.ones(len(used), device="cuda"), atol=1e-5)
    assert learner.train() >= 1
    assert all(np.isfinite(e["policy_loss"]) and np.isfinite(e["value_loss"]) for e in learner.log)
