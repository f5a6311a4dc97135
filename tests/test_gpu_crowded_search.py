"""-m gpu: the search kernels on crowded roots (tests/util.crowded_bands at 14x14: 129-300 legal moves, promotion groups
across list index 31/32 and 255/256), whole trees against the restatements; and a leaf past 300 legal moves, which the
search reports as error bit 4 without touching the other games.

The default node arena (96 nodes per simulation, mcts.py NODES_PER_SIM) is too small for trees whose nodes have a few
hundred children: every search here passes node_cap."""
import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200.mcts import ERR_NODE_CAP, ERR_OVERFLOW, BatchedMCTS
from oracle.mcts_port import search as oracle_search
from tests.golden.fake_net import FakeNet
from tests.leaves_oracle import search_leaves
from tests.test_gpu_mcts import assert_trees_equal
from tests.test_gpu_mcts_leaves import check_batch_state, recorded_search
from tests.util import crowded_bands, oracle_for

pytestmark = pytest.mark.gpu
R, C_PUCT = 14, 3


def crowded_roots():
    """Roots with 129-300 legal moves and at most 300 pseudo-legal ones (the restatement's rules abort above that, as
    the reference does), the promotion groups across 31/32 and 255/256 among them."""
    o = oracle_for(R)
    bands = crowded_bands(R)
    roots = []
    for band in ("promotion at 255/256", "promotion at 31/32", "129-256", "257-299", "300"):
        for rec in bands[band]:
            moves, n_pseudo = o.legal_moves_wide(rec)
            if 129 <= len(moves) <= 300 and n_pseudo <= 300:
                roots.append(rec)
    flats = [[o.move_flat_index(m) for m in o.legal_moves_wide(r)[0]] for r in roots]
    assert any(len(f) > 256 and f[255] == f[256] for f in flats)
    assert any(f[31] == f[32] for f in flats)
    return np.stack(roots)


@pytest.mark.parametrize("batch_rotation", [True, False])
def test_crowded_whole_trees_match_the_oracle(batch_rotation):
    o = oracle_for(R)
    roots = crowded_roots()
    sims = 16
    trees = oracle_search(o, FakeNet(R), roots, C_PUCT, sims, batch_rotation=batch_rotation)
    m = BatchedMCTS(R, len(roots), FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims},
                    batch_rotation=batch_rotation, node_cap=1 + 300 * sims)
    m.search(torch.from_numpy(roots))
    torch.cuda.synchronize()
    assert_trees_equal(m, trees)
    assert int(m.n_children[:, 0].max()) > 256
    print(f"rot={batch_rotation}: {len(trees)} games, {int(m.n_nodes.sum())} nodes")


@pytest.mark.parametrize("batch_rotation", [True, False])
def test_crowded_leaf_parallel_trees_match_the_restatement(batch_rotation):
    o = oracle_for(R)
    roots = crowded_roots()
    sims, L = 32, 8
    m = BatchedMCTS(R, len(roots), FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims},
                    batch_rotation=batch_rotation, leaves_per_game=L, node_cap=1 + 300 * sims)
    replay = recorded_search(m, torch.from_numpy(roots))
    trees = search_leaves(o, None, roots, C_PUCT, sims, L, 1, batch_rotation=batch_rotation, replay=replay,
                          prior_source=m.prior.cpu().numpy())
    check_batch_state(m, trees)


def test_crowded_node_cap_overflow_leaves_other_games_alone():
    """A node arena too small for one crowded root's children: error bit 0 there, and the other games (sparse roots
    that fit) grow the trees they grow in an arena large enough for everyone."""
    from alphazero_4_player_chess_b200.fen import start_record
    roots = np.stack([crowded_roots()[0]] + [start_record("STANDARD")] * 3)
    sims = 6
    small = BatchedMCTS(R, 4, FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims}, node_cap=200)
    small.search(torch.from_numpy(roots), check=False)
    big = BatchedMCTS(R, 4, FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims}, node_cap=1 + 300 * sims)
    big.search(torch.from_numpy(roots))
    torch.cuda.synchronize()
    assert small.error.cpu().tolist() == [ERR_NODE_CAP, 0, 0, 0]
    assert int(small.n_nodes[0]) == 1 and int(small.n_nodes[1:].max()) <= 200
    nn = int(big.n_nodes[1:].max())
    for name in ("parent", "move_flat", "visits", "value_sum", "prior", "first_child", "n_children"):
        a, b = getattr(small, name)[1:], getattr(big, name)[1:]
        used = torch.arange(nn, device="cuda")[None, :] < big.n_nodes[1:, None]
        assert torch.equal(small.n_nodes[1:], big.n_nodes[1:]) and torch.equal(a[:, :nn][used], b[:, :nn][used]), name


def overflow_root():
    return crowded_bands(R)[">300"][0]


@pytest.mark.parametrize("L", [1, 8])
@pytest.mark.parametrize("batch_rotation", [True, False])
def test_overflowing_leaf_is_error_bit_4(L, batch_rotation):
    """A root with more than 300 legal moves in game 0: error bit 4, no children, the game dropped.  Every other game is
    bit-exact the game of the same batch run without game 0 (batch_rotation included: the overflowing leaf is not the
    rotation's leaf)."""
    roots = crowded_roots()[:7]
    with_over = np.concatenate([overflow_root()[None], roots])
    sims = 16
    runs = []
    for batch in (with_over, roots):
        m = BatchedMCTS(R, len(batch), FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims},
                        batch_rotation=batch_rotation, leaves_per_game=L, node_cap=1 + 300 * sims)
        m.search(torch.from_numpy(np.ascontiguousarray(batch)), check=False)
        torch.cuda.synchronize()
        runs.append(m)
    a, b = runs
    assert int(a.error[0]) == ERR_OVERFLOW and int(a.dropped[0]) == 1
    assert int(a.n_children[0, 0]) == 0 and int(a.n_nodes[0]) == 1 and int(a.visits[0, 0]) == 1
    assert not b.error.any() and not a.error[1:].any()
    assert torch.equal(a.n_nodes[1:], b.n_nodes) and torch.equal(a.dropped[1:], b.dropped)
    nn = int(b.n_nodes.max())
    used = torch.arange(nn, device="cuda")[None, :] < b.n_nodes[:, None]
    for name in ("parent", "move_flat", "visits", "value_sum", "prior", "first_child", "n_children"):
        assert torch.equal(getattr(a, name)[1:, :nn][used], getattr(b, name)[:, :nn][used]), name
    with pytest.raises(Exception, match="tree error bits 0x10"):
        a.check_errors()


@pytest.mark.parametrize("interior", [False, True])
@pytest.mark.parametrize("considered", [16, 300])
def test_crowded_gumbel_search_replays_on_the_restatement(interior, considered):
    """Gumbel root search (and Gumbel MuZero interior selection) over roots with a few hundred children, k = 16 and
    k = 300 (every child considered), replayed on the restatements as in test_gpu_mcts_gumbel*.py."""
    from tests.gumbel_interior_oracle import GumbelInteriorTree
    from tests.gumbel_oracle import GumbelTree
    from tests.reuse_oracle import search_on
    from tests.test_gpu_mcts_gumbel import SEED, check_result, device_roots
    o = oracle_for(R)
    roots = crowded_roots()
    n, sims = len(roots), 32
    m = BatchedMCTS(R, n, FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims}, gumbel=True, gumbel_seed=SEED,
                    gumbel_considered=considered, gumbel_interior=interior, node_cap=1 + 300 * sims)
    if interior:
        m.node_value.fill_(float("nan"))
    rec, leaves = [], []

    def record(b, logits, value):
        rec.append((logits.cpu(), value.reshape(-1, 1).cpu()))
        leaves.append(m.leaf.cpu().numpy().copy())

    m.search(torch.from_numpy(roots), record=record)
    torch.cuda.synchronize()
    dev = device_roots(m, leaves)
    if interior:
        trees = [GumbelInteriorTree(o, C_PUCT, r).setup_gumbel(SEED, g, considered, sims - 1, 1.0, dev[g])
                 .setup_interior([lv[g] for lv in leaves]) for g, r in enumerate(roots)]
    else:
        trees = [GumbelTree(o, C_PUCT, r).setup_gumbel(SEED, g, considered, sims - 1, 1.0, dev[g])
                 for g, r in enumerate(roots)]
    trees = search_on(o, None, trees, C_PUCT, sims, batch_rotation=False,
                      replay=lambda b, games: (rec[b][0][games], rec[b][1][games]), prior_source=m.prior.cpu().numpy())
    assert_trees_equal(m, trees)
    adopted = sum(t.adopted + getattr(t, "adopted_interior", 0) for t in trees)
    assert adopted <= 2, adopted
    root_value = m.root_value.cpu().numpy()
    for g, t in enumerate(trees):
        if t.root_value is not None:
            assert root_value[g] == t.root_value, g
    if interior:
        node_value = m.node_value.cpu().numpy()
        for g, t in enumerate(trees):
            for x, v in t.node_value.items():
                assert node_value[g, x] == v, (g, x)
    check_result(m, trees)
    assert not m.error.any()
    print(f"interior={interior} k={considered}: {n} games, {int(m.n_nodes.sum())} nodes, {adopted} near-ties adopted")
