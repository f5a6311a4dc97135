"""The oracle's no-abort legal-move entry (Oracle.legal_moves_wide) against the reference-bound one (legal_moves) wherever
both apply, and the crowded position bands the -m gpu crowded tests draw from.  No GPU needed."""
import numpy as np
import pytest

from tests.util import (CROWDED_BANDS, castling_positions, crowded_bands, crowded_positions, mixed_positions, oracle_for,
                        random_positions)


@pytest.mark.parametrize("R,recs", [(14, lambda: random_positions(14, 3000, seed=11)),
                                    (8, lambda: random_positions(8, 1500, seed=11)),
                                    (14, lambda: mixed_positions("STANDARD", 4096)),
                                    (10, lambda: mixed_positions("TEN", 1024)),
                                    (14, lambda: castling_positions(14)),
                                    (14, lambda: crowded_positions(14, 2000, seed=3)),
                                    (13, lambda: crowded_positions(13, 2000, seed=3))])
def test_wide_entry_equals_legal_moves(R, recs):
    o = oracle_for(R)
    n_pseudo_max, n_legal_max, compared = 0, 0, 0
    for rec in recs():
        wide, n_pseudo = o.legal_moves_wide(rec)
        n_pseudo_max, n_legal_max = max(n_pseudo_max, n_pseudo), max(n_legal_max, len(wide))
        if n_pseudo > 300:  # legal_moves aborts there, as the reference does
            continue
        assert n_pseudo == len(o.pseudo_moves(rec))
        assert np.array_equal(wide, o.legal_moves(rec))
        compared += 1
    assert compared > 0
    print(f"R={R}: {compared} positions compared, largest pseudo-legal / legal count {n_pseudo_max} / {n_legal_max}")


def test_wide_entry_sorts_past_300_moves():
    """Past 300 legal moves the wide list stays canonical: strictly ascending (flat index, promotion type) keys, every
    move legal (the mover's king is safe after it)."""
    R = 14
    o = oracle_for(R)
    bands = crowded_bands(R)
    assert len(bands[">300"])
    for rec in bands[">300"]:
        wide, n_pseudo = o.legal_moves_wide(rec)
        assert len(wide) > 300 and n_pseudo >= len(wide)
        keys = [o.move_flat_index(m) * 8 + ((int(m) >> 24) & 0xff) for m in wide]
        assert all(a < b for a, b in zip(keys, keys[1:]))
        turn = int(rec[R * R]) & 3
        for m in wide[::17]:
            assert not o.king_in_check(o.make_move(rec, m), turn)


@pytest.mark.parametrize("R", [14, 13])
def test_crowded_band_counts(R):
    """Every band the crowded tests use is populated at 14x14 (13x13 lacks two: no list long enough for a promotion group
    at 255/256 in this sample, and no hand-built late king capture past 300 moves)."""
    bands = crowded_bands(R)
    counts = {b: len(bands[b]) for b in CROWDED_BANDS}
    print(f"R={R} band counts:", counts)
    empty = [b for b, c in counts.items() if c == 0]
    assert empty == ([] if R == 14 else ["late king capture", "promotion at 255/256"]), counts
