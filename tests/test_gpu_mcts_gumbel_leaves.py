"""-m gpu: BatchedMCTS(gumbel=True, gumbel_leaves=L), root-only and interior, with SelfPlay and Arena.  The network
outputs of a search are recorded on the device with every batch's slot endpoints and replayed on the leaf-parallel
Gumbel restatement (tests/gumbel_leaves_oracle.py), the f32 priors pinned to the device's (prior_source).  Integer state
and f64 value sums must then be identical node for node, issued and the collision counts equal, node_value equal on
every node the restatement cached, and the result's actions and improved policies match.  A choice where the device and
the restatement differ is adopted only on a near-tie, and counted."""
import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200.arena import Arena, Player
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.geometry import GEOMETRIES
from alphazero_4_player_chess_b200.mcts import BatchedMCTS
from alphazero_4_player_chess_b200.selfplay import SelfPlay
from tests.golden.fake_net import FakeNet
from tests.gumbel_leaves_oracle import make_trees, search
from tests.test_gpu_arena import host as arena_host
from tests.test_gpu_arena import replay as arena_replay
from tests.test_gpu_mcts import assert_trees_equal, search_roots
from tests.test_gpu_mcts_gumbel import SEED
from tests.test_gpu_mcts_noise import same_trees
from tests.util import mixed_positions, oracle_for

pytestmark = pytest.mark.gpu
C_PUCT = 3


def make(R, n, sims, L, considered=8, interior=False, **kw):
    return BatchedMCTS(R, n, FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims}, gumbel=True,
                       gumbel_seed=SEED, gumbel_considered=considered, gumbel_interior=interior, gumbel_leaves=L, **kw)


@pytest.mark.parametrize("name,R,n_games,batch_rotation", [("STANDARD", 14, 12, False), ("EIGHT_SIMPLE", 8, 16, True)])
@pytest.mark.parametrize("L", [2, 4, 8])
@pytest.mark.parametrize("interior", [False, True])
@pytest.mark.parametrize("considered", [4, 16])
def test_search_replays_on_the_restatement(name, R, n_games, batch_rotation, L, interior, considered):
    sims = 32
    o = oracle_for(R)
    roots = search_roots(name, R, n_games)
    n = len(roots)
    m = make(R, n, sims, L, considered, interior, batch_rotation=batch_rotation)
    if interior:
        m.node_value.fill_(float("nan"))  # a read before a write shows up as a mismatch
    rec, slots = [], []

    def record(b, logits, value):
        rec.append((logits.cpu(), value.reshape(-1, 1).cpu()))
        slots.append(m.slot_node.cpu().numpy().reshape(n, L).copy())

    m.search(torch.from_numpy(roots), record=record)
    torch.cuda.synchronize()
    dev = [[s[g] for s in slots] for g in range(n)]
    trees = make_trees(o, C_PUCT, roots, SEED, range(n), considered, sims - L, 1.0, L, 1, interior, dev)

    def replay(b, evals):
        rows = [g * L + j for g, j in evals]
        return rec[b][0][rows], rec[b][1][rows]

    trees = search(o, None, trees, sims, batch_rotation=batch_rotation, replay=replay,
                   prior_source=m.prior.cpu().numpy())
    assert_trees_equal(m, trees)
    assert not m.in_flight.any()
    assert m.collisions.cpu().tolist() == [t.collisions for t in trees]
    issued = m.issued.cpu().numpy()
    root_value, adopted = m.root_value.cpu().numpy(), 0
    node_value = m.node_value.cpu().numpy() if interior else None
    action, policy = (x.cpu().numpy() for x in m.gumbel_result())
    for g, t in enumerate(trees):
        adopted += t.adopted + t.adopted_interior
        k = len(t.children[0])
        if t.issued is not None:
            assert issued[g, :k].tolist() == t.issued.tolist(), g
        if t.root_value is not None:
            assert root_value[g] == t.root_value, g
        for x, v in t.node_value.items():
            assert node_value[g, x] == v, (g, x)
        flat, pol = t.result_leaves()
        assert action[g] == flat, g
        np.testing.assert_allclose(policy[g, :k], pol, rtol=1e-6, atol=0, err_msg=str(g))
        assert not policy[g, k:].any()
    assert adopted <= 2, adopted
    lost = sum(int(t.issued.sum()) - int(sum(t.visits[c] - 1 for c in t.children[0]))
               for t in trees if t.issued is not None)
    print(f"{name} L={L} interior={interior} m={considered}: {n} games, {int(m.n_nodes.sum())} nodes, "
          f"{int(m.collisions.sum())} collisions, {lost} root visits lost, {int(m.dropped.sum())} dropped, "
          f"{adopted} near-tie choices adopted")


@pytest.mark.parametrize("interior", [False, True])
def test_graph_replay_and_eager_search_give_the_same_trees(interior):
    roots = torch.from_numpy(np.ascontiguousarray(mixed_positions("STANDARD", 64)))
    out = []
    for graph in (False, True):
        m = make(14, 64, 32, 8, 16, interior, cuda_graph=graph, virtual_loss=2)
        m.search(roots)
        first = m.gumbel_result()
        m.search(roots.flip(0).contiguous(), gumbel_keys=torch.arange(64) * 7 + 1)
        torch.cuda.synchronize()
        out.append((m, first, m.gumbel_result()))
    (a, a1, a2), (b, b1, b2) = out
    assert b._graph is not None
    same_trees(a, b)
    assert torch.equal(a.root_value, b.root_value) and torch.equal(a.issued, b.issued)
    assert torch.equal(a.collisions, b.collisions) and not b.in_flight.any()
    for x, y in ((a1, b1), (a2, b2)):
        assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1])


def test_one_leaf_is_the_sequential_search_and_l_batches_are_counted(monkeypatch):
    """gumbel_leaves=1 makes the sequential Gumbel calls only; L = 4 makes num_searches / 4 batches of 4 rows per game
    through the new select and result, and SelfPlay passes the option through."""
    calls = []
    for name in ("fpc_tree_select_gumbel_leaves", "fpc_tree_gumbel_result_leaves", "fpc_tree_select_gumbel"):
        m0 = make(8, 2, 8, 1)
        fn = getattr(m0.L, name)
        monkeypatch.setattr(m0.L, name, lambda *a, _fn=fn, _n=name: calls.append(_n) or _fn(*a))
    roots = torch.from_numpy(np.repeat(start_record("EIGHT_SIMPLE")[None], 2, axis=0))
    m = make(8, 2, 8, 1)
    assert m.batch is None and not hasattr(m, "issued")
    m.search(roots)
    m.gumbel_result()
    assert set(calls) == {"fpc_tree_select_gumbel"}
    calls.clear()
    batches = []
    fwd = FakeNet(8, device="cuda")
    net = lambda planes: batches.append(int(planes.shape[0])) or fwd(planes)  # noqa: E731
    args = {"C": C_PUCT, "num_searches": 12, "temperature": 1.1, "max_game_length": 4, "heuristic_weight": 0.02}
    sp = SelfPlay(8, 3, net, args, start_record("EIGHT_SIMPLE"), gumbel=True, gumbel_leaves=4)
    assert sp.mcts.leaves == 4 and sp.mcts.gumbel_desc.n_sims == 8
    sp.play()
    assert batches and set(batches) == {12} and len(batches) % 3 == 0
    assert "fpc_tree_select_gumbel" not in calls and "fpc_tree_gumbel_result_leaves" in calls


@pytest.mark.parametrize("interior", [False, True])
def test_selfplay_plays_the_same_games_on_any_number_of_slots(interior):
    R, G, T = 8, 20, 40
    args = {"C": C_PUCT, "num_searches": 16, "temperature": 1.1, "max_game_length": T, "heuristic_weight": 0.02}
    runs = []
    for n in (3, 8, 20):
        sp = SelfPlay(R, n, FakeNet(R, device="cuda"), args, start_record("EIGHT_SIMPLE"), gumbel=True,
                      gumbel_seed=5, gumbel_considered=8, gumbel_interior=interior, gumbel_leaves=4, virtual_loss=2)
        out = sp.play_games(G)
        torch.cuda.synchronize()
        runs.append({k: v.cpu().numpy() if torch.is_tensor(v) else v for k, v in out.items()})
    for other in runs[1:]:
        for key in ("boards", "child_flat", "child_visits", "child_policy", "value", "action", "game", "ply",
                    "finished", "losing_team", "result", "plies"):
            assert np.array_equal(runs[0][key], other[key]), key
    assert len(runs[0]["action"]) > G


def test_arena_match_with_a_gumbel_leaves_player_replays_move_by_move():
    R, P, T = 8, 3, 24
    off_turn = GEOMETRIES[R].off_turn
    a = Player(FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": 16}, name="gl",
               gumbel=True, gumbel_seed=SEED, gumbel_considered=8, gumbel_leaves=4)
    b = Player(FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": 8}, name="puct")
    res = Arena(R, P, a, b, start_record("EIGHT_SIMPLE"), opening_plies=4, max_game_length=T, seed=2).play()
    torch.cuda.synchronize()
    moves = arena_replay(R, res)  # legality, result codes and plies on the oracle
    h = arena_host(res)
    mine = [(t, g, rec) for t, g, rec in moves if (int(rec[off_turn]) & 1) == h["a_team"][g]]
    assert mine
    roots = np.stack([rec for _, _, rec in mine])
    keys = torch.tensor([(g // 2) * T + t for t, g, _ in mine], dtype=torch.int64)
    m = make(R, len(mine), 16, 4, 8)
    m.search(torch.from_numpy(roots), gumbel_keys=keys)
    action = m.gumbel_result()[0].cpu().numpy()
    assert [int(h["actions"][t, g]) for t, g, _ in mine] == action.tolist()
    print(res.summary(), f"{len(mine)} moves of the gumbel_leaves player re-derived")


def test_argument_errors():
    args = {"C": C_PUCT, "num_searches": 8}
    with pytest.raises(ValueError, match="gumbel_leaves"):
        BatchedMCTS(8, 2, None, args, gumbel_leaves=2)
    for L in (0, 257, 3):
        with pytest.raises(ValueError, match="gumbel_leaves"):
            BatchedMCTS(8, 2, None, args, gumbel=True, gumbel_leaves=L)
    with pytest.raises(ValueError, match="leaves_per_game"):
        BatchedMCTS(8, 2, None, args, gumbel=True, gumbel_leaves=2, leaves_per_game=2)
    for kw, what in (({"reuse_tree": True}, "reuse_tree"), ({"root_noise": True}, "root_noise")):
        with pytest.raises(ValueError, match=what):
            BatchedMCTS(8, 2, None, dict(args, dirichlet_alpha=0.3, dirichlet_epsilon=0.25), gumbel=True,
                        gumbel_leaves=2, **kw)
    m = make(8, 2, 8, 2)
    m.search(torch.from_numpy(np.repeat(start_record("EIGHT_SIMPLE")[None], 2, axis=0)))
    with pytest.raises(Exception, match="search"):
        m.search(None)
    with pytest.raises(ValueError, match="gumbel_leaves"):
        SelfPlay(8, 2, None, dict(args, max_game_length=4), start_record("EIGHT_SIMPLE"), gumbel_leaves=2)
