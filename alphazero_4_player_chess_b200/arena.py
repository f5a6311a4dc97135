"""Arena: a match between two players, every game resident on the device, scored with its uncertainty.

A player is a network plus search settings (`Player`); `Arena(...).play()` returns a `MatchResult`.  Nothing here is
new device code: every ply is one `BatchedMCTS.search` per player (the sm_100a select / expand kernels and the
network) plus one index-built make-move and one observe of `BatchedEnv`.

Semantics
---------
* Pairs and teams.  There are 2·n_pairs games.  Game 2p has A playing team 0 (Red + Yellow, colour & 1 == 0) and B
  team 1; game 2p+1 swaps them.  Both games of pair p start from the same opening.
* Openings.  The opening of pair p is the first `opening_plies` plies of the random playout the playout kernel plays
  for game id p under `seed` (`BatchedEnv.playout_step`; the oracle's `playout_step(rec, seed, game, ply)` restates
  it).  If a position after plies 1 .. opening_plies of that playout is terminal, the pair uses game id p + j·2^32 for
  the smallest j >= 1 whose playout has none; after 16 tries the match is refused.  An opening depends only on
  (seed, p, opening_plies, start_record), never on n_pairs.  opening_plies = 0 is the start position.
* Turns.  Every running game makes one move per ply and all openings have the same length, so at arena ply t the
  same colour is to move in every running game.  Each player owns one `BatchedMCTS` of n_pairs games: with team τ to
  move, A's slot p is game 2p + τ and B's slot p is game 2p + 1 − τ, so slot p is always pair p.  Every move is a
  fresh root (`reset`); finished games are marked dropped after the reset.
* Move choice.  A PUCT player plays its most visited root child, ties to the first in slab order (the smallest flat
  index).  A Gumbel player plays `gumbel_result()`'s action; its keys are p·max_game_length + t for both games of pair
  p at ply t, so the two games of a pair draw the same noise at the same ply.  There is no temperature: given its
  inputs a game is deterministic, and the openings provide the variety.
* End and score.  After each move `observe` gives the result code: 1 (WIN_RY) is a win for team 0, 2 (WIN_BG) for
  team 1, 3 (stalemate) a draw.  A game still running after max_game_length arena plies (the opening not counted) is
  scored as a draw and counted as unfinished, apart from the stalemates.
* Statistics.  x_p ∈ {0, ½, 1, 3/2, 2} is A's points over the two games of pair p; s = Σ x_p / (2P),
  σ = sqrt(Σ_p (x_p/2 − s)² / P) / sqrt(P), Elo = −400·log10(1/s − 1) (∓inf at s = 0 / 1), and the 95 % interval
  [Elo(s − 1.96σ), Elo(s + 1.96σ)] with both ends clamped to [0, 1] first.

The two searches of a ply run on two streams and are joined before the move is made (DESIGN.md §6 has the measured
effect).  Inside the ply loop the host reads one small vector per ply: the two players' error flags and whether any
game is still running."""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .env import BatchedEnv
from .geometry import GEOMETRIES
from .mcts import BatchedMCTS

SEARCH_ARGS = ("cuda_graph", "leaves_per_game", "virtual_loss", "batch_rotation", "gumbel", "gumbel_seed",
               "gumbel_considered", "gumbel_scale", "gumbel_interior", "gumbel_leaves", "node_cap")
OPENING_TRIES = 16
Z95 = 1.96


class Player:
    def __init__(self, net, args: dict, name: str = "", **search):
        """net: the search's network callable (InferenceNet, AutocastNet, ...); args: the reference's dict (C,
        num_searches); search: BatchedMCTS keyword arguments, passed through unchanged (SEARCH_ARGS).  Evaluation play
        starts every move from a fresh root without exploration noise, so reuse_tree and root_noise are refused."""
        for key in ("reuse_tree", "root_noise"):
            if key in search:
                raise ValueError(f"Player: {key} is not supported in evaluation play (every move is a fresh, "
                                 f"noise-free root)")
        unknown = sorted(set(search) - set(SEARCH_ARGS))
        if unknown:
            raise ValueError(f"Player: unknown search arguments {unknown} (allowed: {', '.join(SEARCH_ARGS)})")
        self.net, self.args, self.name, self.search = net, args, str(name), dict(search)
        self.R = getattr(net, "R", None)  # the board size the network was built for, when it says so

    @property
    def gumbel(self) -> bool:
        return bool(self.search.get("gumbel", False))

    def __repr__(self) -> str:
        return f"Player({self.name!r}, num_searches={self.args.get('num_searches')}, {self.search})"


def elo(s: float) -> float:
    """Elo difference of an expected score s in [0, 1]: −400·log10(1/s − 1), −inf at 0 and +inf at 1."""
    if s <= 0.0:
        return -math.inf
    if s >= 1.0:
        return math.inf
    return -400.0 * math.log10(1.0 / s - 1.0)


def pair_statistics(pair_points) -> dict:
    """Score, σ, Elo and its 95 % interval from A's points per pair x_p ∈ {0, ½, 1, 3/2, 2} (module docstring)."""
    x = np.asarray(pair_points, dtype=np.float64)
    P = x.size
    if P < 1:
        raise ValueError("pair_statistics needs at least one pair")
    s = float(x.sum() / (2 * P))
    sigma = math.sqrt(float(((x / 2 - s) ** 2).sum()) / P) / math.sqrt(P)
    lo, hi = (min(1.0, max(0.0, v)) for v in (s - Z95 * sigma, s + Z95 * sigma))
    return {"score": s, "sigma": sigma, "elo": elo(s), "elo_low": elo(lo), "elo_high": elo(hi)}


@dataclass
class MatchResult:
    """A match from A's side.  wins / draws / losses / unfinished are (A as team 0, A as team 1) pairs of counts;
    draws are stalemates, unfinished games (still running after max_game_length plies) are scored ½ and counted apart,
    so the four add up to 2·n_pairs.  pentanomial[i] counts the pairs in which A scored i/2 points.  The per-game
    records are device tensors: openings [2P, record] u8 (each game's start position), actions [max_game_length, 2P]
    i32 (flat action index, −1 once the game has ended), result [2P] i32 (result code, 0 for unfinished), plies [2P]
    i32 (moves played after the opening) and a_team [2P] i32 (A's team)."""
    a: str
    b: str
    n_pairs: int
    wins: tuple
    draws: tuple
    losses: tuple
    unfinished: tuple
    pentanomial: tuple
    score: float
    sigma: float
    elo: float
    elo_low: float
    elo_high: float
    openings: torch.Tensor
    actions: torch.Tensor
    result: torch.Tensor
    plies: torch.Tensor
    a_team: torch.Tensor

    @classmethod
    def from_games(cls, a: str, b: str, result: torch.Tensor, a_team: torch.Tensor, **records) -> "MatchResult":
        """Counts and statistics of the games' result codes (0 = unfinished) with A's team per game."""
        code = result.cpu().numpy().astype(np.int64)
        team = a_team.cpu().numpy().astype(np.int64)
        win = ((code == 1) & (team == 0)) | ((code == 2) & (team == 1))
        loss = ((code == 1) & (team == 1)) | ((code == 2) & (team == 0))
        points = np.where(win, 1.0, np.where(loss, 0.0, 0.5))
        pair = points.reshape(-1, 2).sum(axis=1)

        def split(mask):
            return tuple(int((mask & (team == t)).sum()) for t in (0, 1))

        penta = tuple(int((np.rint(pair * 2) == i).sum()) for i in range(5))
        return cls(a=a, b=b, n_pairs=pair.size, wins=split(win), draws=split(code == 3), losses=split(loss),
                   unfinished=split(code == 0), pentanomial=penta, result=result, a_team=a_team, **records,
                   **pair_statistics(pair))

    def summary(self) -> str:
        w, d, l, u = (sum(c) for c in (self.wins, self.draws, self.losses, self.unfinished))
        return (f"{self.a} vs {self.b}: {2 * self.n_pairs} games, +{w} ={d} -{l} unfinished {u} "
                f"(A as team 0: +{self.wins[0]} ={self.draws[0]} -{self.losses[0]} ~{self.unfinished[0]}), "
                f"pentanomial {list(self.pentanomial)}, score {self.score:.4f} ± {self.sigma:.4f}, "
                f"Elo {self.elo:+.1f} [{self.elo_low:+.1f}, {self.elo_high:+.1f}]")

    def to_json(self) -> dict:
        keys = ("a", "b", "n_pairs", "wins", "draws", "losses", "unfinished", "pentanomial", "score", "sigma", "elo",
                "elo_low", "elo_high")
        return {k: (list(v) if isinstance(v, tuple) else v) for k, v in ((k, getattr(self, k)) for k in keys)}


class Arena:
    def __init__(self, R: int, n_pairs: int, a: Player, b: Player, start_record, opening_plies: int = 8,
                 max_game_length: int = 200, seed: int = 0, device: str | torch.device = "cuda"):
        """A match of 2·n_pairs games between a and b from start_record (module docstring).  Both players' search
        instances are built here; bad arguments raise ValueError before any search runs."""
        if int(n_pairs) < 1:
            raise ValueError(f"n_pairs must be at least 1, got {n_pairs}")
        if int(opening_plies) < 0:
            raise ValueError(f"opening_plies must be non-negative, got {opening_plies}")
        if int(max_game_length) < 1:
            raise ValueError(f"max_game_length must be at least 1, got {max_game_length}")
        for side, p in (("a", a), ("b", b)):
            if p.R is not None and p.R != R:
                raise ValueError(f"player {side} ({p.name or p}) is built for R = {p.R}, the arena plays R = {R}")
        self.geom = GEOMETRIES[R]
        self.R, self.P = R, int(n_pairs)
        self.a, self.b = a, b
        self.opening_plies, self.T, self.seed = int(opening_plies), int(max_game_length), int(seed) & (2**64 - 1)
        self.device = torch.device(device)
        self.start = np.ascontiguousarray(start_record, dtype=np.uint8).reshape(self.geom.record_bytes)
        self.mcts = [BatchedMCTS(R, self.P, p.net, p.args, device=self.device, **p.search) for p in (a, b)]
        self.env = BatchedEnv(R, 2 * self.P, device=self.device)
        pairs = torch.arange(self.P, dtype=torch.int64, device=self.device)
        # games[τ] = (A's games, B's games) with team τ to move: slot p -> game 2p + τ for A, 2p + 1 − τ for B
        self.games = [(2 * pairs + tau, 2 * pairs + 1 - tau) for tau in (0, 1)]
        self.key_base = pairs * self.T  # Gumbel keys p·T + t
        self._streams = [torch.cuda.Stream(self.device) for _ in self.mcts]

    # ---- openings ----------------------------------------------------------------------------------
    def openings(self) -> torch.Tensor:
        """[n_pairs, record] u8: each pair's opening position (module docstring)."""
        op, dev = self.opening_plies, self.device
        env = BatchedEnv(self.R, self.P, device=dev)
        pairs = torch.arange(self.P, dtype=torch.int64, device=dev)
        out = torch.from_numpy(self.start).to(dev).expand(self.P, -1).clone()
        todo = torch.ones(self.P, dtype=torch.bool, device=dev)
        for j in range(OPENING_TRIES):
            ids = pairs + (j << 32)
            env.reset_playout(self.start)
            env.game.copy_(ids)
            for _ in range(op):  # a slot whose position turns terminal is re-seeded: its game id changes
                env.playout_step(self.seed, max_plies=op + 1, planes=False, mask=False)
            env.observe(planes=False, mask=False)
            ok = (env.game == ids) & ((env.status & 3) == 0)
            out = torch.where((todo & ok)[:, None], env.boards, out)
            todo &= ~ok
            if not bool(todo.any()):
                return out
        bad = torch.nonzero(todo).flatten()[:8].tolist()
        raise _lib.FpcError(f"no opening of {op} plies without a terminal position after {OPENING_TRIES} tries for "
                            f"pairs {bad} (seed {self.seed})")

    # ---- play ----------------------------------------------------------------------------------------
    def _begin(self) -> None:
        n, dev = 2 * self.P, self.device
        self.opening_boards = self.openings().repeat_interleave(2, dim=0)
        self.env.load(self.opening_boards)
        self.running = torch.ones(n, dtype=torch.bool, device=dev)
        self.result = torch.zeros(n, dtype=torch.int32, device=dev)
        self.plies = torch.zeros(n, dtype=torch.int32, device=dev)
        self.actions = torch.full((self.T, n), -1, dtype=torch.int32, device=dev)
        self.a_team = (torch.arange(n, device=dev) & 1).to(torch.int32)
        self._turn0 = int(self.start[self.geom.off_turn]) + self.opening_plies

    def _choose(self, m: BatchedMCTS) -> torch.Tensor:
        """[n_pairs] i32: the move m's search picks, −1 for a root without children."""
        if m.gumbel:
            return m.gumbel_result()[0]
        flat, visits, _, cnt = m.root_children()
        best = torch.gather(flat, 1, visits.argmax(dim=1, keepdim=True)).squeeze(1)  # argmax: the first maximum
        return torch.where(cnt > 0, best, torch.full_like(best, -1))

    def _ply(self, t: int) -> bool:
        """One move in every running game; returns whether any game is still running."""
        games = self.games[(self._turn0 + t) & 1]
        cur = torch.cuda.current_stream(self.device)
        chosen = []
        for m, g, stream in zip(self.mcts, games, self._streams):
            if stream is not None:
                stream.wait_stream(cur)
            with torch.cuda.stream(stream):
                m.search(self.env.boards[g], check=False, dropped=~self.running[g], gumbel_keys=self.key_base + t)
                action = self._choose(m)
            if stream is not None:
                action.record_stream(cur)
            chosen.append(action)
        for stream in self._streams:
            if stream is not None:
                cur.wait_stream(stream)
        action = torch.empty(2 * self.P, dtype=torch.int32, device=self.device)
        for g, act in zip(games, chosen):
            action[g] = act
        action = torch.where(self.running, action, torch.full_like(action, -1))
        self.actions[t] = action
        self.env.make_index(action)  # action −1: the record is left untouched
        self.env.observe(planes=False, mask=False)
        code = self.env.status & 3
        moved = self.running & (action >= 0)
        ended = moved & (code != 0)
        self.result = torch.where(ended, code, self.result)
        self.plies += moved.int()
        self.running &= moved & ~ended
        err_a, err_b, running = torch.stack([self.mcts[0].error.amax(), self.mcts[1].error.amax(),
                                             self.running.any().int()]).tolist()
        if err_a or err_b:
            for m in self.mcts:
                m.check_errors()
        return bool(running)

    @torch.no_grad()
    def play(self) -> MatchResult:
        """Play the match to the end (every game finished or max_game_length plies) and score it."""
        with torch.cuda.device(self.device):
            self._begin()
            for t in range(self.T):
                if not self._ply(t):
                    break
        return MatchResult.from_games(self.a.name or "A", self.b.name or "B", self.result, self.a_team,
                                      openings=self.opening_boards, actions=self.actions, plies=self.plies)
