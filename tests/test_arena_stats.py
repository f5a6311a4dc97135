"""The arena's match statistics (score, σ, Elo and its interval, counts from result codes) against hand-computed values
and scipy / numpy, and the refusals of Player and Arena, which come before any device work.  No GPU needed."""
import math

import numpy as np
import pytest
import torch
from scipy import special

from alphazero_4_player_chess_b200.arena import Arena, MatchResult, Player, elo, pair_statistics
from alphazero_4_player_chess_b200.fen import start_record
from tests.golden.fake_net import FakeNet


def test_all_draws_give_zero_elo_and_a_zero_width_interval():
    st = pair_statistics([1.0] * 12)
    assert st == {"score": 0.5, "sigma": 0.0, "elo": 0.0, "elo_low": 0.0, "elo_high": 0.0}


def test_all_wins_give_plus_infinity_and_all_losses_minus_infinity():
    st = pair_statistics([2.0] * 5)
    assert st["score"] == 1.0 and st["sigma"] == 0.0
    assert st["elo"] == st["elo_low"] == st["elo_high"] == math.inf
    st = pair_statistics([0.0] * 5)
    assert st["elo"] == st["elo_low"] == st["elo_high"] == -math.inf
    assert elo(0.0) == -math.inf and elo(1.0) == math.inf and elo(0.5) == 0.0


def test_mixed_pentanomial_against_hand_values_and_scipy():
    x = [0.0, 0.5, 1.0, 1.0, 1.5, 2.0, 2.0, 2.0]
    st = pair_statistics(x)
    # by hand: s = 10/16; the squared deviations of x/2 from s sum to 1, so σ = sqrt(1/8)/sqrt(8) = 1/8
    assert st["score"] == 0.625 and abs(st["sigma"] - 0.125) < 1e-15
    assert abs(st["elo"] - (-400 * math.log10(0.6))) < 1e-12
    assert abs(st["elo_low"] - (-400 * math.log10(1 / 0.38 - 1))) < 1e-12
    assert abs(st["elo_high"] - (-400 * math.log10(1 / 0.87 - 1))) < 1e-12
    # independently: numpy's population standard deviation and scipy's logit (Elo = 400 logit(s) / ln 10)
    half = np.asarray(x) / 2
    sigma = np.std(half) / math.sqrt(len(x))
    assert abs(st["sigma"] - sigma) < 1e-12
    for key, s in (("elo", half.mean()), ("elo_low", half.mean() - 1.96 * sigma), ("elo_high", half.mean() + 1.96 * sigma)):
        assert abs(st[key] - 400 * special.logit(s) / math.log(10)) < 1e-12, key


def test_interval_ends_are_clamped_before_conversion():
    st = pair_statistics([2.0, 2.0, 2.0, 1.5])  # s = 7/8, s + 1.96σ > 1
    assert st["elo_high"] == math.inf and math.isfinite(st["elo_low"])
    st = pair_statistics([0.0, 0.0, 0.0, 0.5])
    assert st["elo_low"] == -math.inf and math.isfinite(st["elo_high"])


@pytest.mark.parametrize("x", [[0.0, 0.5, 1.0, 1.0, 1.5, 2.0, 2.0, 2.0], [0.5, 1.5, 1.5, 2.0, 1.0, 0.5, 1.5], [1.0, 2.0]])
def test_elo_is_antisymmetric_in_the_players(x):
    st = pair_statistics(x)
    sw = pair_statistics([2.0 - v for v in x])
    assert abs(st["score"] + sw["score"] - 1.0) < 1e-15 and st["sigma"] == pytest.approx(sw["sigma"], abs=1e-15)
    for k, k_swapped in (("elo", "elo"), ("elo_low", "elo_high"), ("elo_high", "elo_low")):
        assert sw[k_swapped] == pytest.approx(-st[k], abs=1e-9), k


def test_counts_from_result_codes():
    # pairs (game 2p: A is team 0, game 2p+1: A is team 1); codes 1 WIN_RY, 2 WIN_BG, 3 stalemate, 0 unfinished
    code = torch.tensor([1, 2,   # A wins both: 2
                         2, 1,   # A loses both: 0
                         1, 1,   # 1
                         3, 0,   # stalemate + unfinished: 1
                         1, 3,   # 1.5
                         0, 1],  # 0.5
                        dtype=torch.int32)
    team = torch.arange(12, dtype=torch.int32) & 1
    r = MatchResult.from_games("a", "b", code, team, openings=None, actions=None, plies=None)
    assert r.wins == (3, 1) and r.losses == (1, 3) and r.draws == (1, 1) and r.unfinished == (1, 1)
    assert r.pentanomial == (1, 1, 2, 1, 1)
    st = pair_statistics([2, 0, 1, 1, 1.5, 0.5])
    assert (r.score, r.sigma, r.elo, r.elo_low, r.elo_high) == (st["score"], st["sigma"], st["elo"], st["elo_low"],
                                                                st["elo_high"])
    assert "+4 =2 -4 unfinished 2" in r.summary()


def test_player_refuses_tree_reuse_root_noise_and_unknown_arguments():
    args = {"C": 3, "num_searches": 8}
    for key in ("reuse_tree", "root_noise"):
        with pytest.raises(ValueError, match=key):
            Player(FakeNet(8), args, **{key: True})
    with pytest.raises(ValueError, match="noise_seed"):
        Player(FakeNet(8), args, noise_seed=1)
    p = Player(FakeNet(8), args, gumbel=True, gumbel_scale=0.0, cuda_graph=True)
    assert p.gumbel and p.R == 8


def test_arena_refuses_bad_arguments_before_any_search():
    args = {"C": 3, "num_searches": 8}
    a = Player(FakeNet(8), args)
    start = start_record("EIGHT_SIMPLE")
    for kw, what in (({"n_pairs": 0}, "n_pairs"), ({"opening_plies": -1}, "opening_plies"),
                     ({"max_game_length": 0}, "max_game_length")):
        call = dict(n_pairs=2, opening_plies=2, max_game_length=10) | kw
        with pytest.raises(ValueError, match=what):
            Arena(8, call.pop("n_pairs"), a, a, start, **call)
    with pytest.raises(ValueError, match="R = 14"):
        Arena(8, 2, a, Player(FakeNet(14), args), start)
