"""-m gpu: Arena matches between FakeNet players (outputs exact per row), checked game by game.

* Mirror: equal players play both games of every pair identically, so every pair scores exactly 1.
* Routing: every recorded action is legal on the oracle, and is the move a standalone BatchedMCTS with the mover's
  settings picks for that position; those searches' root visits equal oracle/mcts_port.search's (priors pinned to the
  device's), and the result codes and plies equal the oracle's game_result along the replay.
* Openings follow the oracle's playouts, with a forced replacement; games do not depend on n_pairs.
* Scoring: wins, draws, unfinished games and pentanomial counts from the oracle replay.
* CUDA graphs and one stream play the same actions as eager search on two streams."""
import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200.arena import Arena, Player
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.geometry import GEOMETRIES
from alphazero_4_player_chess_b200.mcts import BatchedMCTS
from oracle.mcts_port import search as oracle_search
from tests.golden.fake_net import FakeNet
from tests.util import oracle_for

pytestmark = pytest.mark.gpu

START = {8: "EIGHT_SIMPLE", 14: "STANDARD"}


def player(R, sims, C=3.0, name="", **search):
    return Player(FakeNet(R, device="cuda"), {"C": C, "num_searches": sims}, name=name, **search)


def play(R, n_pairs, a, b, opening_plies, T, seed=0, one_stream=False):
    arena = Arena(R, n_pairs, a, b, start_record(START[R]), opening_plies=opening_plies, max_game_length=T, seed=seed)
    if one_stream:
        arena._streams = [None, None]
    res = arena.play()
    torch.cuda.synchronize()
    return res


def host(res):
    return {k: getattr(res, k).cpu().numpy() for k in ("openings", "actions", "result", "plies", "a_team")}


def replay(R, res):
    """Replays every game on the oracle from its recorded opening; checks legality, the result codes and the plies.
    Returns [(t, g, position before the move)] for every move played."""
    o, h = oracle_for(R), host(res)
    T, n = h["actions"].shape
    moves = []
    for g in range(n):
        rec, code, played = h["openings"][g], 0, 0
        assert o.game_result(rec)[0] == 0
        for t in range(T):
            a = int(h["actions"][t, g])
            if a < 0:
                break
            assert a in {o.move_flat_index(m) for m in o.legal_moves(rec)}, (g, t)
            moves.append((t, g, rec))
            rec = o.make_index(rec, a)
            played += 1
            code = o.game_result(rec)[0]
            if code:
                break
        assert code != 0 or played == T, g
        assert (h["actions"][played:, g] == -1).all(), g
        assert h["result"][g] == code and h["plies"][g] == played, g
    return moves


def standalone_moves(R, roots, sims, C):
    """The move a standalone BatchedMCTS with these settings picks for each root (most visited child, first in slab
    order), with the instance for the oracle comparison."""
    m = BatchedMCTS(R, len(roots), FakeNet(R, device="cuda"), {"C": C, "num_searches": sims})
    m.search(torch.from_numpy(np.ascontiguousarray(roots)))
    m.check_errors()
    flat, visits, _, cnt = (t.cpu().numpy() for t in m.root_children())
    return np.array([flat[i, int(np.argmax(visits[i, :cnt[i]]))] for i in range(len(roots))]), m


@pytest.mark.parametrize("mode", ["puct", "gumbel"])
def test_mirror_match_plays_both_games_of_a_pair_alike(mode):
    search = {"gumbel": True, "gumbel_scale": 1.0} if mode == "gumbel" else {}
    p = player(8, 12, **search)
    res = play(8, 8, p, p, opening_plies=6, T=40)
    h = host(res)
    assert (h["actions"][:, 0::2] == h["actions"][:, 1::2]).all()
    assert (h["openings"][0::2] == h["openings"][1::2]).all()
    assert (h["plies"] > 0).all()
    assert res.pentanomial == (0, 0, 8, 0, 0) and res.score == 0.5 and res.elo == 0.0 and res.sigma == 0.0
    print(res.summary())


@pytest.mark.parametrize("R,n_pairs,T", [(8, 4, 30), (14, 2, 6)])
def test_moves_route_to_the_mover_and_match_the_oracle(R, n_pairs, T):
    o, off_turn = oracle_for(R), GEOMETRIES[R].off_turn
    settings = [(16, 3.0), (4, 1.5)]  # A, B
    res = play(R, n_pairs, player(R, 16, 3.0), player(R, 4, 1.5), opening_plies=4, T=T, seed=3)
    moves = replay(R, res)
    h = host(res)
    differs = 0
    for who in (0, 1):
        mine = [(t, g, rec) for t, g, rec in moves if ((int(rec[off_turn]) & 1) == h["a_team"][g]) == (who == 0)]
        assert mine
        roots = np.stack([rec for _, _, rec in mine])
        sims, C = settings[who]
        picks, m = standalone_moves(R, roots, sims, C)
        assert [int(h["actions"][t, g]) for t, g, _ in mine] == picks.tolist()
        other, _ = standalone_moves(R, roots, *settings[1 - who])
        differs += int((other != picks).sum())
        trees = oracle_search(o, FakeNet(R), roots, C, sims, batch_rotation=False, prior_source=m.prior.cpu().numpy())
        _, visits, _, cnt = (t.cpu().numpy() for t in m.root_children())
        for i, tree in enumerate(trees):
            assert visits[i, :cnt[i]].tolist() == [tree.visits[c] for c in tree.children[0]], i
    assert differs > 0  # the test tells the two players apart
    print(res.summary(), f"{len(moves)} moves, {differs} would differ under the other player's settings")


def oracle_opening(R, start, seed, pair, plies):
    o = oracle_for(R)
    for j in range(16):
        p = o.playout(start, seed, pair + (j << 32), plies + 1)
        if p["n"] > plies and p["result"][plies] == 0:
            return j, p["recs"][plies]
    raise AssertionError(pair)


def test_openings_follow_the_playouts_with_a_forced_replacement():
    start = start_record("EIGHT_SIMPLE")
    p = player(8, 4)
    arena = Arena(8, 12, p, p, start, opening_plies=10, max_game_length=4, seed=2)
    got = arena.openings().cpu().numpy()
    tries = []
    for pair in range(12):
        j, want = oracle_opening(8, start, 2, pair, 10)
        tries.append(j)
        assert (got[pair] == want).all(), pair
    assert tries[9] >= 1  # the playout of game id 9 under seed 2 ends within 10 plies
    start_only = Arena(8, 3, p, p, start, opening_plies=0, max_game_length=4).openings().cpu().numpy()
    assert (start_only == start).all()


def test_games_do_not_depend_on_the_number_of_pairs():
    a, b = player(8, 8), player(8, 8, gumbel=True, gumbel_considered=4)
    small = host(play(8, 4, a, b, opening_plies=6, T=30, seed=1))
    large = host(play(8, 12, a, b, opening_plies=6, T=30, seed=1))
    for k in ("openings", "result", "plies", "a_team"):
        assert (small[k] == large[k][:8]).all(), k
    assert (small["actions"] == large["actions"][:, :8]).all()


def test_scoring_counts_checkmates_stalemates_and_unfinished_games():
    res = play(8, 16, player(8, 4, 3.0), player(8, 2, 1.5), opening_plies=8, T=100, seed=0)
    replay(8, res)  # the result codes and plies are the oracle's
    h = host(res)
    code, team = h["result"], h["a_team"]
    assert {0, 3} <= set(code.tolist()) and ({1, 2} & set(code.tolist()))
    win = ((code == 1) & (team == 0)) | ((code == 2) & (team == 1))
    loss = ((code == 1) & (team == 1)) | ((code == 2) & (team == 0))
    for name, mask in (("wins", win), ("losses", loss), ("draws", code == 3), ("unfinished", code == 0)):
        assert getattr(res, name) == (int((mask & (team == 0)).sum()), int((mask & (team == 1)).sum())), name
    pair = (win + 0.5 * ((code == 3) | (code == 0))).reshape(-1, 2).sum(axis=1)
    assert res.pentanomial == tuple(int((pair == i / 2).sum()) for i in range(5))
    assert res.score == pair.sum() / 32
    print(res.summary())


def test_cuda_graphs_and_one_stream_play_the_eager_games():
    def pair_of_players(graph):
        return player(8, 16, cuda_graph=graph), player(8, 8, gumbel=True, gumbel_considered=4, cuda_graph=graph)

    eager = host(play(8, 4, *pair_of_players(False), opening_plies=6, T=30))
    graphed = host(play(8, 4, *pair_of_players(True), opening_plies=6, T=30))
    one_stream = host(play(8, 4, *pair_of_players(True), opening_plies=6, T=30, one_stream=True))
    for k in ("actions", "result", "plies"):
        assert (eager[k] == graphed[k]).all() and (eager[k] == one_stream[k]).all(), k
