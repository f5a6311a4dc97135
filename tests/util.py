"""Shared helpers for the test-suite (test infrastructure)."""
from __future__ import annotations

import functools

import numpy as np

from alphazero_4_player_chess_b200.fen import START_FENS, start_record
from alphazero_4_player_chess_b200.geometry import GEOMETRIES
from oracle.port import Oracle

SEED = 0x5EED


@functools.lru_cache(maxsize=None)
def oracle_for(R: int) -> Oracle:
    return Oracle(R, GEOMETRIES[R].IA)


@functools.lru_cache(maxsize=None)
def playout_positions(name: str, castling: bool, n_games: int, max_plies: int, first_game: int = 0):
    """Positions visited by the oracle's deterministic playouts: dict of stacked arrays."""
    _, R = START_FENS[name]
    o = oracle_for(R)
    start = start_record(name, castling=castling)
    recs, games, plies = [], [], []
    for g in range(first_game, first_game + n_games):
        p = o.playout(start, SEED, g, max_plies)
        recs.append(p["recs"])
        games.append(np.full(p["n"], g))
        plies.append(np.arange(p["n"]))
    return dict(R=R, recs=np.concatenate(recs), game=np.concatenate(games), ply=np.concatenate(plies))


def mixed_positions(name: str, n_positions: int, max_plies: int = 400):
    """At least n_positions positions, half from castling-on and half from castling-off games."""
    out = []
    per = 0
    g = 8
    while per < n_positions:
        a = playout_positions(name, True, g, max_plies)
        b = playout_positions(name, False, g, max_plies, first_game=100000)
        per = len(a["recs"]) + len(b["recs"])
        out = [a, b]
        g *= 2
    recs = np.concatenate([x["recs"] for x in out])[:n_positions]
    return np.ascontiguousarray(recs)


def oracle_legal_lists(R: int, recs: np.ndarray):
    o = oracle_for(R)
    return [o.legal_moves(r) for r in recs]


def castling_positions(R: int = 14):
    """Hand-made castling cases on the 14x14 board (engine/board.cpp:343-465), every colour to move: clean
    castling both sides, a piece in between, the king in check, the crossed square attacked, the destination
    attacked (pseudo-legal, rejected by the legal filter), the partner's rook on the rook square, rights off."""
    g = GEOMETRIES[R]
    base = start_record("STANDARD", castling=True)
    out = []
    for color in range(4):
        rec = base.copy()
        rec[g.off_turn] = color
        # strip every knight, bishop, queen and pawn: kings and rooks only
        for sq in range(g.nsq):
            p = int(rec[sq])
            if p & 0x80 and ((p >> 2) & 7) not in (3, 5):
                rec[sq] = 0x18
        out.append(rec.copy())                                   # clean: both castles available
        ksq = int(rec[g.off_king + color])
        kr, kc = divmod(ksq, R)
        # unit step along the back rank towards the kingside rook
        step = {0: (0, 1), 1: (1, 0), 2: (0, -1), 3: (-1, 0)}[color]
        inward = {0: (-1, 0), 1: (0, 1), 2: (1, 0), 3: (0, -1)}[color]  # away from the own edge

        def sq_at(k, depth=0):
            return (kr + step[0] * k + inward[0] * depth) * R + (kc + step[1] * k + inward[1] * depth)

        enemy_rook = 0x80 | (((color + 1) & 3) << 5) | (3 << 2)
        partner_rook = 0x80 | (((color + 2) & 3) << 5) | (3 << 2)
        for k in (1, 2, -1, -2, -3):                               # a blocker on each between square
            r2 = rec.copy()
            r2[sq_at(k)] = 0x80 | (color << 5) | (1 << 2)
            out.append(r2)
        for k in (0, 1, 2, -1, -2):                                # an enemy rook staring down the file at from / crossed / dest
            r2 = rec.copy()
            r2[sq_at(k, 5)] = enemy_rook
            out.append(r2)
        r2 = rec.copy()                                            # partner's rook on the kingside rook square
        r2[sq_at(3)] = partner_rook
        out.append(r2)
        r2 = rec.copy()                                            # enemy rook there instead
        r2[sq_at(3)] = enemy_rook
        out.append(r2)
        for bits in (0x80, 0x80 | 0x40, 0x80 | 0x20):              # rights: none, kingside only, queenside only
            r2 = rec.copy()
            r2[g.off_rights + color] = bits
            out.append(r2)
    return np.stack(out)


def random_positions(R: int, n: int, seed: int = 7):
    """Random (mostly unreachable) positions: all four kings (one of them missing now and then), up to 10 random
    pieces per colour on random on-board squares, pawns only on squares before their promotion line, random side to
    move and random castling rights.  A differential test bed that does not depend on what playouts reach."""
    g = GEOMETRIES[R]
    rng = np.random.default_rng(seed)
    squares = [sq for sq in range(g.nsq) if g.is_legal_location(sq // R, sq % R)]
    out = []

    def pawn_ok(color, r, c):  # strictly before the promotion line, in the pawn's direction of travel
        return {0: r > R // 4, 2: r < 3 * R // 4, 1: c < 3 * R // 4, 3: c > R // 4}[color]

    for _ in range(n):
        rec = g.empty_record()
        rec[g.off_turn] = rng.integers(0, 4)
        free = list(rng.permutation(squares))
        for color in range(4):
            if rng.random() > 0.1:
                sq = int(free.pop())
                rec[sq] = 0x80 | (color << 5) | (5 << 2)
                rec[g.off_king + color] = sq
            for _ in range(int(rng.integers(0, 11))):
                ptype = int(rng.choice([0, 0, 0, 1, 2, 3, 4]))
                sq = int(free.pop())
                if ptype == 0 and not pawn_ok(color, sq // R, sq % R):
                    ptype = 1
                rec[sq] = 0x80 | (color << 5) | (ptype << 2)
            rec[g.off_rights + color] = 0x80 | (int(rng.integers(0, 2)) << 6) | (int(rng.integers(0, 2)) << 5)
        out.append(rec)
    return np.stack(out)


def crowded_positions(R: int, n: int, seed: int = 0):
    """Crowded random positions, where the legal list runs to hundreds of moves: all four kings, a queen-heavy army for
    the side to move (1-14 queens at 13x13 and 14x14, 1-6 on smaller boards, a few rooks, bishops and knights), 1-3 of
    its pawns one step before their promotion line (promotion groups: four moves sharing one flat index inside a long
    list) and 0-3 pieces for each other colour, so that checks and pins still occur.  No castling rights."""
    g = GEOMETRIES[R]
    rng = np.random.default_rng(seed)
    squares = [sq for sq in range(g.nsq) if g.is_legal_location(sq // R, sq % R)]

    def before_promotion(color, r, c):  # one step before the promotion line, in the pawn's direction of travel
        return {0: r == R // 4 + 1, 1: c == 3 * R // 4 - 1, 2: r == 3 * R // 4 - 1, 3: c == R // 4 + 1}[color]

    q_hi = 14 if R >= 13 else 6
    out = []
    for _ in range(n):
        rec = g.empty_record()
        turn = int(rng.integers(0, 4))
        rec[g.off_turn] = turn
        free = [int(x) for x in rng.permutation(squares)]
        for color in range(4):
            sq = free.pop()
            rec[sq] = 0x80 | (color << 5) | (5 << 2)
            rec[g.off_king + color] = sq
        army = [4] * int(rng.integers(1, q_hi + 1)) + [3] * int(rng.integers(0, 4)) + \
            [2] * int(rng.integers(0, 3)) + [1] * int(rng.integers(0, 3))
        for ptype in army:
            sq = free.pop()
            rec[sq] = 0x80 | (turn << 5) | (ptype << 2)
        lanes = [sq for sq in free if before_promotion(turn, sq // R, sq % R)]
        for sq in rng.permutation(lanes)[: int(rng.integers(1, 4))]:
            free.remove(int(sq))
            rec[int(sq)] = 0x80 | (turn << 5)
        for color in range(4):
            if color != turn:
                for _ in range(int(rng.integers(0, 4))):
                    rec[free.pop()] = 0x80 | (color << 5) | (int(rng.choice([1, 2, 3, 4])) << 2)
        out.append(rec)
    return np.stack(out)


def checkers(R: int, rec) -> int:
    """The number of enemy pieces giving check to the side to move: each enemy piece is tested alone, the other enemy
    pieces recoloured to the mover's colour so that every ray is blocked as before."""
    g = GEOMETRIES[R]
    o = oracle_for(R)
    turn = int(rec[g.off_turn]) & 3
    enemy = [sq for sq in range(g.nsq) if rec[sq] & 0x80 and ((rec[sq] >> 5) & 1) != (turn & 1)]
    n = 0
    for e in enemy:
        r2 = rec.copy()
        for sq in enemy:
            if sq != e:
                r2[sq] = (int(r2[sq]) & 0x9f) | (turn << 5)
        n += o.king_in_check(r2, turn)
    return n


def _king_takers(rec, moves):
    """From-squares of the legal moves that capture a king."""
    return {int(m) & 0xff for m in moves if (int(m) >> 16) & 0x80 and ((int(m) >> 18) & 7) == 5}


def _late_king_capture(R: int, rec):
    """rec with the next colour's king moved next to the mover's last sliding piece in square order, on one of its rays,
    so that only the last two pieces capture a king (None where no such square is found).  In a list past 300 moves
    that capture sits in the rules kernel's last generation round, which the buffer may no longer take."""
    g = GEOMETRIES[R]
    o = oracle_for(R)
    turn = int(rec[g.off_turn]) & 3
    own = [sq for sq in range(g.nsq) if rec[sq] & 0x80 and ((rec[sq] >> 5) & 3) == turn]
    victim = (turn + 1) & 3
    for src in reversed(own[-2:]):
        if ((rec[src] >> 2) & 7) not in (2, 3, 4):
            continue
        for dr in (-1, 0, 1):
            for dc in (-1, 0, 1):
                r, c = src // R + dr, src % R + dc
                if (dr or dc) and g.is_legal_location(r, c) and rec[r * R + c] == 0x18:
                    out = rec.copy()
                    out[int(rec[g.off_king + victim])] = 0x18
                    out[r * R + c] = 0x80 | (victim << 5) | (5 << 2)
                    out[g.off_king + victim] = r * R + c
                    moves, _ = o.legal_moves_wide(out)
                    takers = _king_takers(out, moves)
                    if len(moves) > 300 and takers and takers <= set(own[-2:]):
                        return out
    return None


CROWDED_BANDS = ("33-64", "65-128", "129-256", "257-299", "300", "pseudo>300", ">300", "check", "double check",
                 "late king capture", "promotion at 31/32", "promotion at 255/256")


@functools.lru_cache(maxsize=None)
def crowded_bands(R: int, per_band: int = 12, n: int = 6000, seed: int = 1):
    """A fixed selection of crowded_positions(R, n, seed) by the oracle's full legal list (Oracle.legal_moves_wide):
    {band: [record, ...]}, at most per_band records per band (twice that above 300 legal moves), in generation order.
    Bands: legal count 33-64, 65-128, 129-256, 257-299, exactly 300; more than 300 pseudo-legal but at most 300 legal
    moves; more than 300 legal moves; in check (one checker) with at least 20 legal moves; double check; past 300 legal moves, a king capture
    only by the mover's last pieces in square order (the last generation round of the rules kernel); a promotion group
    (four moves, one flat index) across list index 31/32 and across 255/256 (a warp and a thread-slot boundary of the
    search's expansion)."""
    g = GEOMETRIES[R]
    o = oracle_for(R)
    bands = {b: [] for b in CROWDED_BANDS}

    def take(band, rec, cap=per_band):
        if len(bands[band]) < cap:
            bands[band].append(rec)

    for rec in crowded_positions(R, n, seed):
        moves, n_pseudo = o.legal_moves_wide(rec)
        nl = len(moves)
        for lo, hi in ((33, 64), (65, 128), (129, 256), (257, 299)):
            if lo <= nl <= hi:
                take(f"{lo}-{hi}", rec)
        if nl == 300:
            take("300", rec)
        if nl <= 300 < n_pseudo:
            take("pseudo>300", rec)
        if nl > 300:
            take(">300", rec, 2 * per_band)
        turn = int(rec[g.off_turn]) & 3
        if nl >= 20 and o.king_in_check(rec, turn):
            take("check", rec)
        elif len(bands["double check"]) < per_band:
            # an enemy knight and an enemy rook next to the king (random double checks are rare)
            kr, kc = divmod(int(rec[g.off_king + turn]), R)
            dbl = rec.copy()
            for (dr, dc), ptype in (((2, 1), 1), ((1, 0), 3)):
                for sr, sc in ((1, 1), (-1, -1), (1, -1), (-1, 1)):
                    r, c = kr + sr * dr, kc + sc * dc
                    if g.is_legal_location(r, c) and dbl[r * R + c] == 0x18:
                        dbl[r * R + c] = 0x80 | (((turn + 1) & 3) << 5) | (ptype << 2)
                        break
            if checkers(R, dbl) == 2 and len(o.legal_moves_wide(dbl)[0]):
                take("double check", dbl)
        if nl > 300 and len(bands["late king capture"]) < per_band:
            late = _late_king_capture(R, rec)
            if late is not None:
                take("late king capture", late)
        flats = [o.move_flat_index(m) for m in moves]
        if nl > 32 and flats[31] == flats[32]:
            take("promotion at 31/32", rec)
        if nl > 256 and flats[255] == flats[256]:
            take("promotion at 255/256", rec)
    return {b: np.stack(v) if v else np.zeros((0, g.record_bytes), np.uint8) for b, v in bands.items()}
