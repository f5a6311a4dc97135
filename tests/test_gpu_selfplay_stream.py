"""-m gpu: continuous self-play (SelfPlay.play_games) and the Learner's continuous option.

Every emitted game is replayed from the start record on the oracle: boards, legality, result codes, plies, the losing
team and each entry's value, for games that ended and games cut off at max_game_length.  Because the moves are keyed by
(game, ply) and FakeNet's rows are exact functions of their own planes, a game's trajectory must be bit for bit the same
whatever slot it plays in and whatever games share its batches: play_games(20) on 3, 8 and 20 slots must agree for
every search option, which is what shows that refilling a slot leaves nothing of the previous game behind (tree,
noise marks, collisions, node values or the incremental planes)."""
import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200 import _lib
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.geometry import GEOMETRIES
from alphazero_4_player_chess_b200.selfplay import SelfPlay
from alphazero_4_player_chess_b200.train import Learner
from tests.golden.fake_net import FakeNet
from tests.util import oracle_for

pytestmark = pytest.mark.gpu

HW = 0.02
ENTRY_KEYS = ("boards", "child_flat", "child_visits", "value", "action", "game", "ply")
GAME_KEYS = ("finished", "losing_team", "result", "plies")


def make(R, n, T, sims=8, temperature=1.1, **kw):
    args = {"C": 3, "num_searches": sims, "temperature": temperature, "max_game_length": T, "heuristic_weight": HW,
            "dirichlet_alpha": 0.3, "dirichlet_epsilon": 0.25}
    name = "EIGHT_SIMPLE" if R == 8 else "STANDARD"
    return SelfPlay(R, n, FakeNet(R, device="cuda"), args, start_record(name), **kw)


def host(out):
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def replay_on_the_oracle(R, out, first, G, T):
    """Every game of a play_games output re-played from the start record on the oracle."""
    g, o = GEOMETRIES[R], oracle_for(R)
    name = "EIGHT_SIMPLE" if R == 8 else "STANDARD"
    h = host(out)
    games, plies_e = h["game"], h["ply"]
    assert np.all(np.diff(games * T + plies_e) > 0)  # (game, ply) order, each entry once
    assert set(games.tolist()) == set(range(first, first + G))
    for key in GAME_KEYS:
        assert len(h[key]) == G, key
    for j in range(first, first + G):
        rows = np.flatnonzero(games == j)
        assert np.array_equal(plies_e[rows], np.arange(len(rows))), j
        assert h["plies"][j - first] == len(rows), j
        rec = start_record(name)
        teams, ended, mover_team = [], 0, -1
        for i, row in enumerate(rows):
            assert not ended, (j, i)
            assert np.array_equal(h["boards"][row], rec), (j, i)
            legal = set(o.move_flat_index(m) for m in o.legal_moves(rec))
            kids = [f for f, v in zip(h["child_flat"][row], h["child_visits"][row]) if v > 0]
            action = int(h["action"][row])
            assert set(kids) <= legal and action in legal, (j, i)
            mover_team = int(rec[g.off_turn]) & 1
            teams.append(mover_team)
            rec = o.make_index(rec, action)
            ended, _, _ = o.game_result(rec)
        k = j - first
        if ended:
            assert h["finished"][k] and h["result"][k] == ended and h["losing_team"][k] == mover_team, j
            want = [1.0 if team != mover_team else -1.0 for team in teams]
        else:
            assert len(rows) == T and not h["finished"][k] and h["result"][k] == 0 and h["losing_team"][k] == -1, j
            cur = int(rec[g.off_turn]) & 1
            heur = float(np.float32(o.heuristic(rec, cur)) * np.float32(HW))
            want = [heur if team == cur else -heur for team in teams]
        np.testing.assert_allclose(h["value"][rows], want, rtol=0, atol=1e-6, err_msg=str(j))
    return h


@pytest.mark.parametrize("R,n,G,T,first", [(8, 8, 40, 120, 0), (14, 5, 12, 6, 1000)])
def test_the_stream_replays_on_the_oracle(R, n, G, T, first):
    sp = make(R, n, T)
    out = sp.play_games(G, first_game=first)
    h = replay_on_the_oracle(R, out, first, G, T)
    assert sp.next_game == first + G
    assert G > n  # every game was played, so slots were refilled
    if R == 8:
        assert (h["finished"] & (h["plies"] < T)).any()  # some games ended early: their slots took the next game early
    pol = sp.policy_targets(out)
    assert torch.allclose(pol.sum(dim=1), torch.ones(pol.shape[0], device="cuda"), atol=1e-5)
    # successive calls continue the ids
    out2 = sp.play_games(3)
    assert set(out2["game"].cpu().tolist()) == {first + G, first + G + 1, first + G + 2}


OPTIONS = {
    "puct": {},
    "root_noise": {"root_noise": True, "noise_seed": 17},
    "reuse_tree": {"reuse_tree": True},
    "leaves": {"leaves_per_game": 4, "virtual_loss": 2},
    "gumbel": {"gumbel": True, "gumbel_seed": 5, "gumbel_considered": 8},
    "gumbel_interior": {"gumbel": True, "gumbel_seed": 5, "gumbel_considered": 8, "gumbel_interior": True},
}


@pytest.mark.parametrize("option", list(OPTIONS))
def test_a_game_does_not_depend_on_its_slot_or_its_neighbours(option):
    R, G, T = 8, 20, 60
    runs = []
    for n in (3, 8, 20):
        sp = make(R, n, T, sample_seed=99, **OPTIONS[option])
        runs.append(host(sp.play_games(G)))
    base = runs[0]
    for other in runs[1:]:
        keys = ENTRY_KEYS + GAME_KEYS + (("child_policy",) if "gumbel" in OPTIONS[option] else ())
        for key in keys:
            assert np.array_equal(base[key], other[key]), (option, key)


def test_play_games_on_n_slots_plays_the_games_of_play():
    R, n, T = 8, 8, 40
    kw = {"gumbel": True, "gumbel_seed": 3, "gumbel_considered": 8}
    a = make(R, n, T, **kw)
    ref = a.play()
    torch.cuda.synchronize()
    valid = a.hist_valid.cpu().numpy()
    t_idx, g_idx = np.nonzero(valid)  # the (ply, game) order of play()'s entries
    order = np.lexsort((t_idx, g_idx))
    out = host(make(R, n, T, **kw).play_games(n, first_game=0))
    assert np.array_equal(out["game"], g_idx[order]) and np.array_equal(out["ply"], t_idx[order])
    assert np.array_equal(out["action"], a.hist_action.cpu().numpy()[t_idx, g_idx][order])
    for key in ("boards", "child_flat", "child_visits", "child_policy", "value"):
        assert np.array_equal(out[key], ref[key].cpu().numpy()[order]), key
    assert np.array_equal(out["finished"], ref["finished"].cpu().numpy())
    assert np.array_equal(out["losing_team"], ref["losing_team"].cpu().numpy())


@pytest.mark.parametrize("continuous", [True, False])
def test_learner_continuous(monkeypatch, continuous):
    R, n, T = 8, 4, 16
    sp = make(R, n, T)
    calls = []
    for method in ("play", "play_games"):
        fn = getattr(sp, method)

        def recorded(*a, _fn=fn, _method=method, **kw):
            out = _fn(*a, **kw)
            calls.append((_method, out))
            return out

        monkeypatch.setattr(sp, method, recorded)
    args = {"batch_size": 10**9, "replay_buffer_capacity": 10**5, "validation_buffer_capacity": 10**5,
            "num_iterations": 2, "num_games": 10, "num_parallel_games": n}
    learner = Learner(sp, torch.nn.Linear(1, 1), torch.optim.SGD([torch.zeros(1, requires_grad=True)], lr=0.0), args,
                      continuous=continuous)
    learner.learn(2)
    stored = len(learner.train_buf) + len(learner.valid_buf)
    assert stored == sum(out["boards"].shape[0] for _, out in calls)
    if continuous:
        assert [m for m, _ in calls] == ["play_games"] * 4
        assert stored == sum(int(out["plies"].sum()) for _, out in calls)
        ids = [sorted(set(out["game"].cpu().tolist())) for _, out in calls]
        sizes = [10, n, 10, n]
        assert ids == [list(range(s, s + k)) for s, k in zip(np.cumsum([0] + sizes[:-1]), sizes)]
    else:
        assert [m for m, _ in calls] == (["play"] * (10 // n) + ["play"]) * 2


def test_play_makes_no_sample_root_call(monkeypatch):
    sp = make(8, 6, 12)

    def refuse(*a, **kw):
        raise AssertionError("play() called fpc_tree_sample_root")

    monkeypatch.setattr(_lib.lib(), "fpc_tree_sample_root", refuse)
    out = sp.play()
    assert out["boards"].shape[0] > 0
