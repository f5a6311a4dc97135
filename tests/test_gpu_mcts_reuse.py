"""-m gpu: searches that continue a kept subtree (BatchedMCTS(reuse_tree=True): search -> advance -> search(None), and
SelfPlay(reuse_tree=True)) against the MCTS restatement, re-rooted and continued by tests/reuse_oracle.py.  Integer
state and f64 value sums bit-exact, f32 priors within the rtol of tests/test_gpu_mcts.py."""
import functools

import numpy as np
import pytest
import torch

import tests.test_gpu_selfplay as selfplay_test
from alphazero_4_player_chess_b200.env import BatchedEnv
from alphazero_4_player_chess_b200.mcts import NODES_PER_SIM, BatchedMCTS
from alphazero_4_player_chess_b200.selfplay import SelfPlay
from oracle.mcts_port import Tree
from oracle.mcts_port import search as oracle_search
from tests.golden.fake_net import FakeNet
from tests.reuse_oracle import reroot, search_on
from tests.test_gpu_mcts import assert_trees_equal, search_roots
from tests.util import mixed_positions, oracle_for

pytestmark = pytest.mark.gpu
C_PUCT = 3


def pick_actions(trees, move):
    """One root child per game: the most visited, the least visited or one never visited (visit count 1), by game."""
    out = []
    for gi, t in enumerate(trees):
        ch = t.children[0]
        if not ch:
            out.append(-1)
            continue
        v = [t.visits[c] for c in ch]
        rule = (gi + move) % 3
        if rule == 0:
            c = ch[int(np.argmax(v))]
        elif rule == 1:
            c = ch[int(np.argmin(v))]
        else:
            never = [c for c in ch if t.visits[c] == 1]
            c = never[len(never) // 2] if never else ch[-1]
        out.append(t.move_flat[c])
    return np.array(out, np.int32)


def expected_reroot(o, m, t, flat):
    """The oracle's tree after the move, and the node count the device keeps (0: a fresh root).  The device keeps the
    subtree within max_keep_nodes = node_cap - 96 sims nodes and max_keep_boards = board_cap - sims boards; its
    materialised boards are those of the nodes that were ever reached by a simulation, i.e. visit count > 1."""
    if flat < 0:
        return Tree(o, C_PUCT, t.rec[0]), 0
    sims = int(m.args["num_searches"])
    kept = reroot(t, int(flat))
    n_boards = sum(v > 1 for v in kept.visits)
    if len(kept.parent) <= m.node_cap - NODES_PER_SIM * sims and n_boards <= m.board_cap - sims:
        return kept, len(kept.parent)
    return Tree(o, C_PUCT, kept.rec[0]), 0


def next_boards(R, boards, actions):
    env = BatchedEnv(R, len(boards), device="cuda")
    env.load(boards)
    env.make_index(torch.from_numpy(actions).cuda())  # action -1: the record stays as it is
    return env.boards.clone()


@pytest.mark.parametrize("name,R,n_games,sims", [("STANDARD", 14, 24, 48), ("EIGHT_SIMPLE", 8, 32, 80)])
@pytest.mark.parametrize("batch_rotation", [True, False])
def test_three_moves_with_reuse_match_the_oracle(name, R, n_games, sims, batch_rotation):
    o = oracle_for(R)
    roots = search_roots(name, R, n_games)
    m = BatchedMCTS(R, len(roots), FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims},
                    batch_rotation=batch_rotation, reuse_tree=True)
    m.search(torch.from_numpy(roots))
    trees = oracle_search(o, FakeNet(R), roots, C_PUCT, sims, batch_rotation=batch_rotation)
    assert_trees_equal(m, trees)
    boards = m._roots
    n_kept = n_fresh = 0
    for move in range(3):
        actions = pick_actions(trees, move)
        boards = next_boards(R, boards, actions)
        kept = m.advance(torch.from_numpy(actions), boards).cpu().numpy()
        want = [expected_reroot(o, m, t, a) for t, a in zip(trees, actions)]
        trees = [t for t, _ in want]
        assert kept.tolist() == [k for _, k in want], move
        for gi, t in enumerate(trees):
            assert np.array_equal(boards[gi].cpu().numpy(), t.rec[0]), (move, gi)
        n_kept += int((kept > 1).sum())
        n_fresh += int((kept == 0).sum())
        m.search(None)
        trees = search_on(o, FakeNet(R), trees, C_PUCT, sims, batch_rotation=batch_rotation)
        assert_trees_equal(m, trees)
    assert n_kept >= len(roots)  # most moves carried a searched subtree
    print(f"{name} rot={batch_rotation}: {len(roots)} games x 3 moves: {n_kept} subtrees of more than one node kept, "
          f"{n_fresh} fresh roots, {int(m.n_nodes.sum())} nodes at the end, root visits {m.visits[:, 0].tolist()[:6]}...")


def test_continued_cuda_graph_search_equals_eager_search():
    """search(None) replays the graph captured by the first search, across an advance (which moves no pointer)."""
    R, sims = 14, 40
    roots = torch.from_numpy(np.ascontiguousarray(mixed_positions("STANDARD", 64)))
    out = []
    for graph in (False, True):
        m = BatchedMCTS(R, 64, FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims}, cuda_graph=graph,
                        reuse_tree=True)
        m.search(roots)
        flat, visits, _, _ = m.root_children()
        actions = torch.gather(flat, 1, visits.argmax(dim=1, keepdim=True)).squeeze(1)
        kept = m.advance(actions, next_boards(R, roots.numpy(), actions.cpu().numpy()))
        m.search(None)
        torch.cuda.synchronize()
        out.append((m, kept))
    (a, ka), (b, kb) = out
    assert b._graph is not None and torch.equal(ka, kb) and int((ka > 1).sum()) > 32
    assert torch.equal(a.n_nodes, b.n_nodes) and torch.equal(a.n_boards, b.n_boards)
    nn = int(a.n_nodes.max())
    used = torch.arange(nn, device="cuda")[None, :] < a.n_nodes[:, None]
    for name in ("parent", "move_flat", "visits", "value_sum", "prior", "first_child", "n_children", "board_idx"):
        assert torch.equal(getattr(a, name)[:, :nn][used], getattr(b, name)[:, :nn][used]), name


def test_configs3_two_moves_with_reuse_replayed_on_the_oracle():
    """BASELINE.json configs[3] at its stated size with reuse: 1,024 games x 400 simulations per move, fp32 ResNet
    10 x 128, two moves (search, advance on the most visited child, search(None)).  The network outputs and the priors
    of a sample of games are recorded per move and the games replayed on the oracle (as
    test_configs3_search_replayed_on_the_oracle does for one move)."""
    from alphazero_4_player_chess_b200.fen import start_record
    from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet
    R, n, sims = 14, 1024, 400
    o = oracle_for(R)
    torch.manual_seed(0)
    net = InferenceNet(PolicyValueNet(R, 10, 128, device="cuda"), bf16=False)
    pool = mixed_positions("STANDARD", 256)
    roots = np.ascontiguousarray(np.concatenate([pool] * (n // len(pool)))[:n])
    roots[::2] = start_record("STANDARD")
    sample = torch.tensor([0, 1, 2, 3, 101, 255, 256, 511, 640, 777, 901, 1023], device="cuda")
    idx = sample.cpu().numpy()
    m = BatchedMCTS(R, n, net, {"C": C_PUCT, "num_searches": sims}, reuse_tree=True)
    trees, boards, kept_all = None, torch.from_numpy(roots), None
    for move in range(2):
        rec_logits, rec_values = [], []

        def record(sim, logits, value):
            rec_logits.append(logits[sample].cpu())
            rec_values.append(value[sample].reshape(-1, 1).cpu())

        def replay(sim, games):
            return rec_logits[sim][list(games)], rec_values[sim][list(games)]

        if move == 0:
            m.search(boards, record=record)
        else:
            flat, visits, _, _ = m.root_children()
            actions = torch.gather(flat, 1, visits.argmax(dim=1, keepdim=True)).squeeze(1)
            boards = next_boards(R, boards.cpu().numpy(), actions.cpu().numpy())
            kept_all = m.advance(actions, boards)
            want = [expected_reroot(o, m, t, int(a)) for t, a in zip(trees, actions[sample].cpu().numpy())]
            trees = [t for t, _ in want]
            assert kept_all[sample].cpu().numpy().tolist() == [k for _, k in want]
            m.search(None, record=record)
        torch.cuda.synchronize()
        prior = m.prior[sample].cpu().numpy()
        if move == 0:
            trees = oracle_search(o, None, roots[idx], C_PUCT, sims, batch_rotation=False, replay=replay,
                                  prior_source=prior)
        else:
            trees = search_on(o, None, trees, C_PUCT, sims, batch_rotation=False, replay=replay, prior_source=prior)
        n_nodes, visits = m.n_nodes[sample].cpu().numpy(), m.visits[sample].cpu().numpy()
        move_flat, value_sum = m.move_flat[sample].cpu().numpy(), m.value_sum[sample].cpu().numpy()
        parent = m.parent[sample].cpu().numpy()
        for i, t in enumerate(trees):
            nn = len(t.parent)
            assert n_nodes[i] == nn, (move, i, n_nodes[i], nn)
            assert parent[i, :nn].tolist() == t.parent
            assert move_flat[i, :nn].tolist() == t.move_flat
            assert visits[i, :nn].tolist() == t.visits
            assert value_sum[i, :nn].tolist() == t.value_sum
    root_visits = m.visits[:, 0]
    assert int((kept_all > 1).sum()) > n // 2 and int((root_visits > sims + 1).sum()) > n // 2
    print(f"configs[3] with reuse: kept {float(kept_all.float().mean()):.0f} nodes per game on average, "
          f"{int((kept_all == 0).sum())} fresh roots; root visits after the second search: mean "
          f"{float(root_visits.float().mean()):.0f}; {sum(len(t.parent) for t in trees)} sampled nodes identical")


@pytest.mark.parametrize("name,R,n,T", [("EIGHT_SIMPLE", 8, 24, 40), ("STANDARD", 14, 8, 6)])
def test_selfplay_with_reuse_replays_on_the_oracle(monkeypatch, name, R, n, T):
    """The self-play replay check of tests/test_gpu_selfplay.py (boards, legality, results, rewards) with
    SelfPlay(reuse_tree=True); every ply after the first continues the played move's subtree."""
    log = []
    advance = BatchedMCTS.advance

    def logged(self, actions, root_boards):
        kept = advance(self, actions, root_boards)
        log.append((actions.cpu().numpy().copy(), kept.cpu().numpy().copy()))
        return kept

    monkeypatch.setattr(BatchedMCTS, "advance", logged)
    monkeypatch.setattr(selfplay_test, "SelfPlay", functools.partial(SelfPlay, reuse_tree=True))
    selfplay_test.test_selfplay_replays_on_the_oracle(name, R, n, T)
    assert log
    moved = np.concatenate([k[a >= 0] for a, k in log])
    assert (moved > 0).mean() > 0.5 and (moved > 1).any(), moved
    assert all((k[a < 0] == 0).all() for a, k in log)  # finished games get a fresh root
    print(f"{name}: {len(log)} plies continued a subtree; kept > 0 on {(moved > 0).mean():.0%} of the moves of running "
          f"games, {moved.mean():.1f} nodes on average")
