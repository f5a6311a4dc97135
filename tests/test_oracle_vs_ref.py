"""CPU: pin the restatement oracle (oracle/fpc_oracle.c) against the UNMODIFIED reference engine
compiled into oracle/_ref/ (oracle/Makefile) -- perft tables, legal-move sets, post-move boards,
results, attack tests and heuristics over deterministic random playouts at all four geometries.

The reference ships no tests or golden vectors (SURVEY 4), so the known answers are the reference
itself run here.  Skipped when oracle/_ref was not built (the reference sources are not part of this
repository), except for the perft tables, whose known answers are stored here.  The committed fixtures in
tests/golden/ (tests/test_golden.py) hold the reference's playouts, legal lists, results and encodings, but
not the pseudo-move sets, check and attack tests, per-move boards, move-index map, random positions or
castling cases compared here: without oracle/_ref those comparisons do not run."""
import numpy as np
import pytest

from alphazero_4_player_chess_b200.fen import START_FENS, start_record
from alphazero_4_player_chess_b200.geometry import GEOMETRIES
from oracle import ref_engine
from tests.util import SEED, oracle_for

PERFT = {  # SURVEY 8c
    "STANDARD": [20, 395, 7800, 152050],
    "EIGHT_SIMPLE": [14, 66, 887, 4086, 58416],
    "EIGHT": [10, 83, 677, 4828, 41693],
    "TEN": [14, 215, 2856, 41416],
}
GAMES = {"STANDARD": (6, 400), "THIRTEEN": (4, 300), "TEN": (6, 300), "EIGHT": (8, 300), "EIGHT_SIMPLE": (8, 300)}


def ref_for(R):
    if not ref_engine.available(R):
        pytest.skip("oracle/_ref not built")
    return ref_engine.RefEngine(R)


def sort_canonical(o, moves):
    return sorted((int(m) for m in moves), key=lambda m: (o.move_flat_index(m), (m >> 24) & 0xff))


@pytest.mark.parametrize("name", list(PERFT))
@pytest.mark.parametrize("castling", [False, True])
def test_perft_tables(name, castling):
    """The oracle against the reference's perft counts stored above, and the unmodified engine too where it is built."""
    _, R = START_FENS[name]
    ref = ref_engine.RefEngine(R) if ref_engine.available(R) else None
    o = oracle_for(R)
    rec = start_record(name, castling=castling)
    for depth, want in enumerate(PERFT[name], start=1):
        if ref is not None:
            assert ref.perft(rec, depth) == want, (name, depth)
        assert o.perft(rec, depth) == want, (name, depth)


@pytest.mark.parametrize("name", list(GAMES))
@pytest.mark.parametrize("castling", [True, False])
def test_playouts_agree(name, castling):
    """Same games move for move; per position: pseudo sets, legal lists (canonical order), result,
    post-move boards for every legal move (full and index-built), check and attack tests."""
    _, R = START_FENS[name]
    g = GEOMETRIES[R]
    ref, o = ref_for(R), oracle_for(R)
    start = start_record(name, castling=castling)
    n_games, max_plies = GAMES[name]
    early_out = 0
    for game in range(n_games):
        a = ref.playout(start, SEED, game, max_plies)
        b = o.playout(start, SEED, game, max_plies)
        assert a["n"] == b["n"]
        assert np.array_equal(a["recs"], b["recs"])
        assert np.array_equal(a["n_legal"], b["n_legal"])
        assert np.array_equal(a["result"], b["result"])
        assert np.array_equal(a["moves"], b["moves"])
        for p in range(0, a["n"], 5):
            rec = a["recs"][p]
            assert sorted(int(m) for m in ref.pseudo_moves(rec)) == sorted(int(m) for m in o.pseudo_moves(rec))
            legal_ref = sort_canonical(o, ref.legal_moves(rec))
            legal = [int(m) for m in o.legal_moves(rec)]
            assert legal == legal_ref
            res, nl, kc = o.game_result(rec)
            rr = ref.game_result(rec)
            if rr != res:  # SURVEY 8a row 8: order-dependent early-out
                assert res == 0 and kc and nl > 0
                early_out += 1
            for m in legal[:: max(1, len(legal) // 6)]:
                assert np.array_equal(ref.make_move(rec, m), o.make_move(rec, m))
                fi = o.move_flat_index(m)
                assert fi == ref.move_flat_index(m)
                assert np.array_equal(ref.make_index(rec, fi), o.make_index(rec, fi))
            for color in range(4):
                assert ref.king_in_check(rec, color) == o.king_in_check(rec, color)
            for team in range(2):
                assert ref.heuristic(rec, team) == o.heuristic(rec, team)
            if p % 25 == 0:
                for sq in range(g.nsq):
                    if g.is_legal_location(sq // R, sq % R):
                        for team in range(2):
                            assert ref.is_attacked_by_team(rec, team, sq) == o.is_attacked_by_team(rec, team, sq)
    # informational: how often the reference's early-out fired on these games
    print(f"{name} castling={castling}: GetGameResult early-out cases = {early_out}")


@pytest.mark.parametrize("R", [14, 13, 10, 8])
def test_move_index_map(R):
    ref, o = ref_for(R), oracle_for(R)
    g = GEOMETRIES[R]
    # planes >= 8(R-1)+8 index past the reference's 8-entry knight table (move.cpp:56-58, undefined
    # behaviour); no generated move maps there, so they are outside the parity contract
    for flat in range(0, (8 * (R - 1) + 8) * g.nsq, 11):
        m = ref.move_from_flat(flat)
        assert m == o.move_from_flat(flat)
        assert ref.move_flat_index(m) == o.move_flat_index(m)
    for a, b, c in [(0, 0, 0), (SEED, 5, 9), (2**63, 2**40, 2047)]:
        assert ref.mix(a, b, c) == o.mix(a, b, c)


def test_hand_made_castling_cases():
    """Castling details on the 14x14 board, oracle vs the unmodified engine: sets of pseudo and legal moves, and
    the boards after every legal move (rook relocation, rights update)."""
    from tests.util import castling_positions
    ref, o = ref_for(14), oracle_for(14)
    recs = castling_positions(14)
    n_castles = 0
    for rec in recs:
        assert sorted(int(m) for m in ref.pseudo_moves(rec)) == sorted(int(m) for m in o.pseudo_moves(rec))
        legal = [int(m) for m in o.legal_moves(rec)]
        assert legal == sort_canonical(o, ref.legal_moves(rec))
        for m in legal:
            assert np.array_equal(ref.make_move(rec, m), o.make_move(rec, m))
            n_castles += ((m >> 32) & 0xff) != 196
    assert n_castles >= 16  # every colour castles both ways in several of the cases


@pytest.mark.parametrize("R", [14, 13, 10, 8])
def test_random_positions(R):
    """Random, mostly unreachable positions (tests/util.random_positions): pseudo and legal sets, the canonical
    result, check tests and the board after every legal move, oracle vs the unmodified engine."""
    from tests.util import random_positions
    ref, o = ref_for(R), oracle_for(R)
    early = 0
    for rec in random_positions(R, 250):
        assert sorted(int(m) for m in ref.pseudo_moves(rec)) == sorted(int(m) for m in o.pseudo_moves(rec))
        legal = [int(m) for m in o.legal_moves(rec)]
        assert legal == sort_canonical(o, ref.legal_moves(rec))
        res, nl, kc = o.game_result(rec)
        rr = ref.game_result(rec)
        if rr != res:
            assert res == 0 and kc and nl > 0
            early += 1
        for color in range(4):
            assert ref.king_in_check(rec, color) == o.king_in_check(rec, color)
        for m in legal[::3]:
            assert np.array_equal(ref.make_move(rec, m), o.make_move(rec, m))
            fi = o.move_flat_index(m)
            assert np.array_equal(ref.make_index(rec, fi), o.make_index(rec, fi))
    print(f"R={R}: GetGameResult early-out cases = {early}")
