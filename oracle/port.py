"""TEST INFRASTRUCTURE.  ctypes view of oracle/libfpc_oracle.so (oracle/fpc_oracle.c), the CPU
restatement of the reference hot path.  Import only from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline leg."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
_u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")

_LIB = None


def build() -> str:
    path = os.path.join(_HERE, "libfpc_oracle.so")
    src = os.path.join(_HERE, "fpc_oracle.c")
    if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "oracle"], stdout=subprocess.DEVNULL)
    return path


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.fpo_pseudo_moves.argtypes = [C.c_int, C.c_int, _u8p, _u64p, C.c_int]
        L.fpo_legal_moves.argtypes = [C.c_int, C.c_int, _u8p, _u64p, C.c_int]
        L.fpo_legal_moves_wide.argtypes = [C.c_int, C.c_int, _u8p, _u64p, C.c_int, C.POINTER(C.c_int)]
        L.fpo_is_attacked_by_team.argtypes = [C.c_int, C.c_int, _u8p, C.c_int, C.c_int]
        L.fpo_king_in_check.argtypes = [C.c_int, C.c_int, _u8p, C.c_int]
        L.fpo_is_attacked_by_player.argtypes = [C.c_int, C.c_int, _u8p, C.c_int, C.c_int]
        L.fpo_attack_map.argtypes = [C.c_int, C.c_int, _u8p, _u8p]
        L.fpo_make_move.argtypes = [C.c_int, C.c_int, _u8p, C.c_uint64, _u8p]
        L.fpo_make_index.argtypes = [C.c_int, C.c_int, _u8p, C.c_int, _u8p]
        L.fpo_move_from_flat.argtypes = [C.c_int, C.c_int]
        L.fpo_move_from_flat.restype = C.c_uint64
        L.fpo_move_flat_index.argtypes = [C.c_int, C.c_uint64]
        L.fpo_game_result.argtypes = [C.c_int, C.c_int, _u8p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.fpo_heuristic.argtypes = [C.c_int, C.c_int, _u8p, C.c_int]
        L.fpo_perft.argtypes = [C.c_int, C.c_int, _u8p, C.c_int]
        L.fpo_perft.restype = C.c_uint64
        L.fpo_mix.argtypes = [C.c_uint64] * 3
        L.fpo_mix.restype = C.c_uint64
        L.fpo_encode.argtypes = [C.c_int, _u8p, C.c_int, _i32p, _f32p]
        L.fpo_mask.argtypes = [C.c_int, C.c_int, _u8p, C.c_int, _f32p]
        L.fpo_playout_step.argtypes = [C.c_int, C.c_int, _u8p, C.c_uint64, C.c_uint64, C.c_uint64, _u8p,
                                       C.POINTER(C.c_int), C.POINTER(C.c_uint64)]
        L.fpo_bench_playout.argtypes = [C.c_int, C.c_int, _u8p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int,
                                        C.POINTER(C.c_uint64)]
        L.fpo_bench_playout.restype = C.c_uint64
        L.fpo_playout_checksum.argtypes = [C.c_int, C.c_int, _u8p, C.c_uint64, C.c_uint64, C.c_int, C.c_int,
                                           C.POINTER(C.c_uint64)]
        L.fpo_playout_checksum.restype = C.c_uint64
        L.fpo_select_child.argtypes = [_i32p, _i32p, _i32p, _f64p, _f64p, C.c_int, C.c_double]
        L.fpo_backpropagate.argtypes = [_i32p, _i32p, _f64p, C.c_int, C.c_float]
        _LIB = L
    return _LIB


class Oracle:
    """The restatement bound to one geometry."""

    def __init__(self, R: int, IA: int):
        self.R, self.IA = R, IA
        self.L = lib()
        self.record_bytes = ((R * R + 12 + 15) // 16) * 16
        self.nsq = R * R
        self.A = 8 * R + 8

    def pseudo_moves(self, rec):
        out = np.zeros(300, dtype=np.uint64)
        n = self.L.fpo_pseudo_moves(self.R, self.IA, np.ascontiguousarray(rec), out, 300)
        return out[:n].copy()

    def legal_moves(self, rec):
        out = np.zeros(300, dtype=np.uint64)
        n = self.L.fpo_legal_moves(self.R, self.IA, np.ascontiguousarray(rec), out, 300)
        return out[:n].copy()

    def legal_moves_wide(self, rec):
        """(moves, n_pseudo): the full canonical legal list, also where the position has more than 300 pseudo-legal
        or legal moves (legal_moves aborts there, as the reference does)."""
        out = np.zeros(1024, dtype=np.uint64)
        n_pseudo = C.c_int(0)
        n = self.L.fpo_legal_moves_wide(self.R, self.IA, np.ascontiguousarray(rec), out, len(out), C.byref(n_pseudo))
        if n < 0:
            raise ValueError(f"more than {len(out)} pseudo-legal moves ({n_pseudo.value})")
        return out[:n].copy(), n_pseudo.value

    def is_attacked_by_team(self, rec, team, sq) -> bool:
        return bool(self.L.fpo_is_attacked_by_team(self.R, self.IA, np.ascontiguousarray(rec), team, sq))

    def is_attacked_by_player(self, rec, sq, color) -> bool:
        """fpchess::Board::IsAttackedByPlayer (src/cpp/board.cpp:142-209)."""
        return bool(self.L.fpo_is_attacked_by_player(self.R, self.IA, np.ascontiguousarray(rec), sq, color))

    def attack_map(self, rec) -> np.ndarray:
        """[R*R] u8: bit c = IsAttackedByPlayer(colour c), bit 4+t = IsAttackedByTeam(team t)."""
        out = np.zeros(self.R * self.R, dtype=np.uint8)
        self.L.fpo_attack_map(self.R, self.IA, np.ascontiguousarray(rec), out)
        return out

    def king_in_check(self, rec, color) -> bool:
        return bool(self.L.fpo_king_in_check(self.R, self.IA, np.ascontiguousarray(rec), color))

    def make_move(self, rec, move):
        out = np.zeros(self.record_bytes, dtype=np.uint8)
        rc = self.L.fpo_make_move(self.R, self.IA, np.ascontiguousarray(rec), int(move), out)
        if rc != 0:
            raise RuntimeError("piece missing for move")
        return out

    def make_index(self, rec, flat):
        out = np.zeros(self.record_bytes, dtype=np.uint8)
        rc = self.L.fpo_make_index(self.R, self.IA, np.ascontiguousarray(rec), int(flat), out)
        if rc != 0:
            raise RuntimeError("piece missing for move")
        return out

    def move_from_flat(self, flat) -> int:
        return int(self.L.fpo_move_from_flat(self.R, int(flat)))

    def move_flat_index(self, move) -> int:
        return self.L.fpo_move_flat_index(self.R, int(move))

    def game_result(self, rec):
        n, kc = C.c_int(0), C.c_int(0)
        res = self.L.fpo_game_result(self.R, self.IA, np.ascontiguousarray(rec), C.byref(n), C.byref(kc))
        return res, n.value, bool(kc.value)

    def heuristic(self, rec, team) -> int:
        return self.L.fpo_heuristic(self.R, self.IA, np.ascontiguousarray(rec), team)

    def perft(self, rec, depth) -> int:
        return int(self.L.fpo_perft(self.R, self.IA, np.ascontiguousarray(rec), depth))

    def mix(self, seed, game, ply) -> int:
        return int(self.L.fpo_mix(seed, game, ply))

    def encode(self, recs, k):
        recs = np.ascontiguousarray(recs, dtype=np.uint8).reshape(-1, self.record_bytes)
        n = recs.shape[0]
        k = np.ascontiguousarray(np.broadcast_to(np.asarray(k, dtype=np.int32), (n,)))
        out = np.zeros((n, 24, self.R, self.R), dtype=np.float32)
        self.L.fpo_encode(self.R, recs, n, k, out)
        return out

    def mask(self, recs):
        recs = np.ascontiguousarray(recs, dtype=np.uint8).reshape(-1, self.record_bytes)
        n = recs.shape[0]
        out = np.zeros((n, self.A, self.R, self.R), dtype=np.float32)
        self.L.fpo_mask(self.R, self.IA, recs, n, out)
        return out

    def playout_step(self, rec, seed, game, ply):
        out = np.zeros(self.record_bytes, dtype=np.uint8)
        n, mv = C.c_int(0), C.c_uint64(0)
        res = self.L.fpo_playout_step(self.R, self.IA, np.ascontiguousarray(rec), seed, game, ply, out,
                                      C.byref(n), C.byref(mv))
        return res, out, n.value, mv.value

    def playout(self, start, seed, game, max_plies):
        """Positions (before each move), n_legal, result and move per ply, like RefEngine.playout."""
        recs, nl, rs, mv = [], [], [], []
        cur = np.ascontiguousarray(start).copy()
        for p in range(max_plies):
            res, nxt, n, m = self.playout_step(cur, seed, game, p)
            recs.append(cur)
            nl.append(n)
            rs.append(res)
            mv.append(m)
            if res != 0:
                break
            cur = nxt
        return dict(n=len(recs), recs=np.stack(recs), n_legal=np.array(nl, dtype=np.int32),
                    result=np.array(rs, dtype=np.int32), moves=np.array(mv, dtype=np.uint64))

    def playout_checksum(self, start, seed, first_game, n_games, max_plies):
        pos = C.c_uint64(0)
        chk = self.L.fpo_playout_checksum(self.R, self.IA, np.ascontiguousarray(start), seed, first_game, n_games,
                                          max_plies, C.byref(pos))
        return int(chk), int(pos.value)

    def bench_playout(self, start, seed, first_game, min_positions, max_plies):
        chk = C.c_uint64(0)
        n = self.L.fpo_bench_playout(self.R, self.IA, np.ascontiguousarray(start), seed, first_game,
                                     min_positions, max_plies, C.byref(chk))
        return int(n), int(chk.value)
