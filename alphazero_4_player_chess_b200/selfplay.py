"""SelfPlay: the reference's self-play loop `AlphaZero.play` (`src/py/alphazero.py:81-178`) with every
game, tree and replay entry resident on the device.

Per move, for all games at once: `BatchedMCTS.search` -> visit counts of the root's children
(`alphazero.py:104-110`) -> temperature + multinomial sampling (`:114-118`) -> index-built make-move
(`state.TakeAction(Move(action_index))`, `:119-121`) -> `GetGameResult` (`:123`) -> terminal rewards by
team (`:128-137`, `handle_terminal_state :53-79`); games still running at `max_game_length` are scored
by `CalculateHeuristic * heuristic_weight` (`:161-175`).  Replay entries are device tensors (board
record + sparse visit distribution + value) instead of `MemoryEntry` copies of whole boards; the
training-side encoding `GetEncodedState(entry.state)` is produced on demand by `encoded_states()`.

This is the caller of the hot path (SURVEY 8f rank 2), not part of the bit-exact contract: play() samples with
torch's device RNG.  The deterministic pieces (advance, rewards) are checked against the oracle in
tests/test_gpu_selfplay.py.  play_games() is continuous self-play: a slot takes the next game as soon as its game ends,
and moves are drawn on the device by a counter-based uniform keyed by (game, ply), so every game can be re-derived on its
own (tests/test_gpu_selfplay_stream.py)."""
from __future__ import annotations

import functools

import torch

from ._lib import FPC_MAX_MOVES
from .env import BatchedEnv
from .geometry import GEOMETRIES, Geometry
from .mcts import BatchedMCTS


@functools.lru_cache(maxsize=None)
def _network_index(R: int, device: torch.device) -> torch.Tensor:
    """[4, A*R*R] i64: row k maps a board-frame flat action index to the entry of the network's policy row that the
    search reads for it when the network sees the position rotated by colour k (torch.rot90(., -k) over [A, R, R], as
    tree_expand_backup_kernel un-rotates)."""
    g = GEOMETRIES[R]
    idx = torch.arange(g.action_space_size, dtype=torch.int64).view(g.num_action_channels, R, R)
    return torch.stack([torch.rot90(idx, -k, (1, 2)).reshape(-1) for k in range(4)]).to(device)


def policy_targets(geom: Geometry, boards: torch.Tensor, child_flat: torch.Tensor, weights: torch.Tensor) -> torch.Tensor:
    """Dense [M, A*R*R] f32 policy targets in the network's frame: row i is weights[i] normalised, with the weight of
    child child_flat[i, j] (a board-frame flat index) placed where the search reads that move in the network's row
    when the position is encoded rotated by its own side to move k = boards[i, off_turn] (`BatchedEnv.encode(k=-1)`,
    `BatchedMCTS(batch_rotation=False)`).  That is torch.rot90 of the board-frame target over [A, R, R] by +k.
    Padding columns carry weight 0; a row whose weights are all zero stays zero."""
    k = boards[:, geom.off_turn].long()
    dest = _network_index(geom.R, child_flat.device)[k[:, None], child_flat.long()]
    probs = torch.zeros((child_flat.shape[0], geom.action_space_size), dtype=torch.float32, device=child_flat.device)
    probs.scatter_add_(1, dest, weights.to(torch.float32))
    return probs / probs.sum(dim=1, keepdim=True).clamp_min(1e-30)


class SelfPlay:
    def __init__(self, R: int, n_games: int, neural_net, args: dict, start_record, device="cuda",
                 batch_rotation: bool = False, reuse_tree: bool = False, leaves_per_game: int = 1,
                 virtual_loss: int = 1, root_noise: bool = False, noise_seed: int = 0, gumbel: bool = False,
                 gumbel_seed: int = 0, gumbel_considered: int = 16, gumbel_scale: float = 1.0,
                 gumbel_interior: bool = False, gumbel_leaves: int = 1, sample_seed: int = 0):
        """args: the reference's dict (`alphazero.py:291-306`); uses C, num_searches, temperature,
        max_game_length, heuristic_weight.  reuse_tree=True keeps the played move's subtree for the next move's search
        (`BatchedMCTS.advance`) where the reference starts every move from a fresh root: num_searches simulations are
        still added per move, on top of the visits carried over, and the policy targets are the root children's visit
        counts including those.  leaves_per_game / virtual_loss: leaf-parallel search (BatchedMCTS), num_searches / L
        network batches of n_games * L leaf slots per move.  root_noise / noise_seed: Dirichlet noise on every move's
        root priors (BatchedMCTS; args then needs dirichlet_alpha and dirichlet_epsilon), keyed by g * max_game_length + t
        for game g at ply t, so the noise of a game does not depend on the batch it plays in; play() with the same
        noise_seed draws the same noise again.  gumbel / gumbel_seed / gumbel_considered / gumbel_scale: Gumbel root
        search (BatchedMCTS), keyed like the noise by g * max_game_length + t; every move plays the action of
        `gumbel_result` (temperature is then unused) and the replay's policy targets are its improved policy, kept in
        `hist_policy` and returned as replay["child_policy"].  gumbel_interior: Gumbel MuZero's interior selection below
        the Gumbel root (BatchedMCTS); keys, actions and policy targets are as with gumbel alone.  gumbel_leaves: the
        leaf-parallel Gumbel search (BatchedMCTS), num_searches / L network batches of n_games * L rows per move, with
        `virtual_loss` below the root.  sample_seed: the seed of
        play_games' keyed move sampling (`BatchedMCTS.sample_root`); play() samples with torch's RNG and ignores it."""
        self.geom = GEOMETRIES[R]
        self.R, self.n, self.args = R, int(n_games), args
        self.device = torch.device(device)
        self.env = BatchedEnv(R, self.n, device=self.device)
        self.reuse_tree = bool(reuse_tree)
        self.mcts = BatchedMCTS(R, self.n, neural_net, args, device=self.device, batch_rotation=batch_rotation,
                                reuse_tree=self.reuse_tree, leaves_per_game=leaves_per_game,
                                virtual_loss=virtual_loss, root_noise=root_noise, noise_seed=noise_seed, gumbel=gumbel,
                                gumbel_seed=gumbel_seed, gumbel_considered=gumbel_considered, gumbel_scale=gumbel_scale,
                                gumbel_interior=gumbel_interior, gumbel_leaves=gumbel_leaves)
        self.start = torch.as_tensor(start_record, dtype=torch.uint8)
        self.sample_seed = int(sample_seed)
        self.next_game = 0  # the first game id of the next play_games(first_game=None)
        T = int(args["max_game_length"])
        i32 = dict(dtype=torch.int32, device=self.device)
        self.hist_boards = torch.zeros((T, self.n, self.geom.record_bytes), dtype=torch.uint8, device=self.device)
        self.hist_flat = torch.zeros((T, self.n, FPC_MAX_MOVES), **i32)
        self.hist_visits = torch.zeros((T, self.n, FPC_MAX_MOVES), **i32)
        self.hist_valid = torch.zeros((T, self.n), dtype=torch.bool, device=self.device)
        self.hist_action = torch.full((T, self.n), -1, **i32)
        if self.mcts.gumbel:
            self.hist_policy = torch.zeros((T, self.n, FPC_MAX_MOVES), dtype=torch.float32, device=self.device)

    # ---- one move for every running game -----------------------------------------------------------
    def sample_actions(self, flat: torch.Tensor, visits: torch.Tensor, running: torch.Tensor) -> torch.Tensor:
        """`alphazero.py:108-118`: probs = visits / sum; probs ** (1/temperature), renormalised; multinomial."""
        w = visits.float()
        w = w / w.sum(dim=1, keepdim=True).clamp_min(1e-30)
        w = torch.pow(w, 1.0 / float(self.args["temperature"]))
        has = (w.sum(dim=1) > 0) & running
        w = torch.where(has[:, None], w, torch.ones_like(w))  # multinomial needs a non-zero row
        pick = torch.multinomial(w, 1).squeeze(1)
        action = torch.gather(flat, 1, pick[:, None]).squeeze(1)
        return torch.where(has, action, torch.full_like(action, -1))

    def advance(self, actions: torch.Tensor) -> torch.Tensor:
        """TakeAction(Move(action_index)) for every game with action >= 0 (the others keep their board), then
        GetGameResult of the new positions.  Returns the result codes [n] (0 = IN_PROGRESS)."""
        self.env.make_index(actions.to(torch.int32).contiguous())  # action -1: FPC_ERR_MOVE, record untouched
        self.env.observe(planes=False, mask=False)
        return self.env.status & 3

    def _search(self, keys: torch.Tensor, running: torch.Tensor, actions: torch.Tensor | None) -> None:
        """One move's search in every slot: fresh trees at the current boards (actions None), or each tree re-rooted on
        the move its slot played (`BatchedMCTS.advance`; action -1 gives the slot a fresh root, as reset() makes it).
        Slots not running sit the search out (`dropped`); keys [n] i64 select the root noise and the Gumbel draws."""
        if actions is not None:
            self.mcts.advance(actions, self.env.boards)
        else:
            self.mcts.reset(self.env.boards)
        self.mcts.dropped.copy_((~running).int())  # finished games take no part in the search
        if self.mcts.gumbel:
            self.mcts.gumbel_keys.copy_(keys)
        if self.mcts.root_noise:
            self.mcts.add_root_noise(keys)  # the roots a kept subtree brought
        for b in range(int(self.args["num_searches"]) // self.mcts.leaves):
            planes = self.mcts.select()
            logits, value = self.mcts.net(planes)
            self.mcts.expand_backup(logits, value)
            if b == 0 and self.mcts.root_noise:
                self.mcts.add_root_noise(keys)  # the roots the first batch expanded

    @torch.no_grad()
    def play(self) -> dict:
        n, T = self.n, int(self.args["max_game_length"])
        off_turn = self.geom.off_turn
        self.env.load(self.start.numpy())
        running = torch.ones(n, dtype=torch.bool, device=self.device)
        losing_team = torch.full((n,), -1, dtype=torch.int64, device=self.device)
        self.hist_valid.zero_()
        for t in range(T):
            keys = torch.arange(n, dtype=torch.int64, device=self.device) * T + t
            self._search(keys, running, actions if self.reuse_tree and t > 0 else None)
            flat, visits, _, _ = self.mcts.root_children()
            self.hist_boards[t].copy_(self.env.boards)
            self.hist_flat[t].copy_(flat)
            self.hist_visits[t].copy_(visits)
            if self.mcts.gumbel:
                actions, policy = self.mcts.gumbel_result()
                self.hist_policy[t].copy_(policy)
                actions = torch.where(running, actions, torch.full_like(actions, -1))
            else:
                actions = self.sample_actions(flat, visits, running)
            moved = running & (actions >= 0)
            self.hist_valid[t].copy_(moved)
            self.hist_action[t].copy_(actions)
            mover_team = (self.env.boards[:, off_turn] & 1).long()
            result = self.advance(actions)
            ended = moved & (result != 0)
            # alphazero.py:128: losing_team = state.GetTurn().GetTeam() of the state the move was made FROM
            losing_team = torch.where(ended, mover_team, losing_team)
            running = running & ~ended & moved
            if not bool(running.any()):
                break
        self.mcts.check_errors()
        return self.finish(running, losing_team)

    @torch.no_grad()
    def play_games(self, num_games: int, first_game: int | None = None) -> dict:
        """Continuous self-play: games first_game .. first_game + num_games - 1 on the n slots, each slot taking the next
        game as soon as its own ends.  first_game=None continues from the previous call's next id (`self.next_game`), so
        successive calls never reuse keys.

        Slots start with the lowest ids.  Whenever a slot's game ends or reaches max_game_length plies, the slot takes the
        next id that has not started yet, if one remains, and its board is loaded with the start record; otherwise it
        stays idle, dropped from the search.  The call returns when every game has ended or been cut off; games in
        progress never carry over to the next call.  Each slot has its own ply counter p: the game's history rows are
        hist_*[p, slot], and game j at its ply p searches and samples with key j * max_game_length + p -- for j < n the
        keys play() gives slot j -- for the root noise, the Gumbel draws and the move.  The move is gumbel_result()'s
        action with gumbel=True, else `BatchedMCTS.sample_root(sample_seed, keys, temperature)`: a game's moves depend on
        its key and its own tree only, so its trajectory does not depend on its slot or on the games beside it (except
        with batch_rotation=True, where a leaf is read in the colour of its batch's first leaf).  With reuse_tree=True a
        refilled slot re-roots with action -1, a fresh root; without, every move starts from a fresh root anyway.  The
        value rule is play()'s (`_values`); a cut-off game's heuristic is read from its slot's final board before the
        slot is refilled.  The host reads two numbers per ply (games that ended, whether a slot still runs), and gathers
        the replay entries only on plies where some game ended.

        Returns play()'s replay keys (boards, child_flat, child_visits, value, child_policy with Gumbel), ordered by
        (game, ply) whatever the slots, plus per entry: game [M] i64, ply [M] i32, action [M] i32 (the move played); and
        per game, indexed by id - first_game: finished [G] bool (ended by a result, not cut off), losing_team [G] i64
        (-1 when none), result [G] i32 (the result code that ended it, 0 when cut off) and plies [G] i32."""
        n, T, dev = self.n, int(self.args["max_game_length"]), self.device
        G = int(num_games)
        if G < 1:
            raise ValueError(f"num_games must be at least 1, got {G}")
        first = self.next_game if first_game is None else int(first_game)
        end = first + G
        self.next_game = end
        off_turn, gumbel = self.geom.off_turn, self.mcts.gumbel
        i64 = dict(dtype=torch.int64, device=dev)
        slots = torch.arange(n, **i64)
        rows = torch.arange(T, **i64)[:, None]
        start = self.start.to(dev)
        self.env.load(self.start.numpy())
        game = first + slots
        active = slots < G
        ply = torch.zeros(n, **i64)
        next_id = first + min(n, G)
        finished = torch.zeros(G, dtype=torch.bool, device=dev)
        losing_team = torch.full((G,), -1, **i64)
        result = torch.zeros(G, dtype=torch.int32, device=dev)
        plies = torch.zeros(G, dtype=torch.int32, device=dev)
        parts = []
        actions = None
        while True:
            keys = game * T + ply
            self._search(keys, active, actions if self.reuse_tree else None)
            flat, visits, _, _ = self.mcts.root_children()
            self.hist_boards[ply, slots] = self.env.boards
            self.hist_flat[ply, slots] = flat
            self.hist_visits[ply, slots] = visits
            if gumbel:
                actions, policy = self.mcts.gumbel_result()
                self.hist_policy[ply, slots] = policy
            else:
                # a descent that reached a terminal leaf dropped its game for the rest of the search; the move is still
                # drawn from the visits it has, as play() draws it, so only idle slots stay dropped for the sampler
                self.mcts.dropped.copy_((~active).int())
                actions = self.mcts.sample_root(self.sample_seed, keys, float(self.args["temperature"]))
            actions = torch.where(active, actions, torch.full_like(actions, -1))
            self.hist_action[ply, slots] = actions
            moved = active & (actions >= 0)
            mover_team = (self.env.boards[:, off_turn] & 1).long()
            code = self.advance(actions)
            ended = moved & (code != 0)
            ply = ply + moved.long()
            cut = moved & ~ended & (ply >= T)
            done = active & (ended | cut | ~moved)  # ~moved: a root without a move stops its game, as in play()
            active = active & ~done
            n_done, left = torch.stack([done.sum(), active.any().long()]).tolist()
            if n_done:
                sel = done[None, :] & (rows < ply[None, :])  # [T, n]: the entries of the games that ended
                lost = torch.where(ended, mover_team, torch.full_like(mover_team, -1))
                value = self._values((self.hist_boards[:, :, off_turn] & 1).long(), lost, cut)
                parts.append({"boards": self.hist_boards[sel], "child_flat": self.hist_flat[sel],
                              "child_visits": self.hist_visits[sel], "value": value[sel],
                              "action": self.hist_action[sel], "game": game[None, :].expand(T, n)[sel],
                              "ply": rows.expand(T, n)[sel].int(),
                              **({"child_policy": self.hist_policy[sel]} if gumbel else {})})
                idx = game[done] - first
                finished[idx] = ~cut[done]
                losing_team[idx] = lost[done]
                result[idx] = torch.where(ended, code, torch.zeros_like(code))[done]
                plies[idx] = ply[done].int()
                # refill: the slots that ended, in ascending order, take the next ids that have not started
                new = next_id + torch.cumsum(done.long(), 0) - 1
                take = done & (new < end)
                game = torch.where(take, new, game)
                ply = torch.where(done, torch.zeros_like(ply), ply)
                active = active | take
                self.env.boards.copy_(torch.where(take[:, None], start[None, :], self.env.boards))
                actions = torch.where(take, torch.full_like(actions, -1), actions)  # a fresh root for a new game
                refilled = max(0, min(n_done, end - next_id))
                next_id += n_done
                left = left or refilled
            if not left:
                break
        self.mcts.check_errors()
        out = {key: torch.cat([p[key] for p in parts]) for key in parts[0]}
        order = torch.argsort(out["game"] * T + out["ply"])
        out = {key: v[order] for key, v in out.items()}
        return {**out, "finished": finished, "losing_team": losing_team, "result": result, "plies": plies}

    # ---- rewards (handle_terminal_state, alphazero.py:53-79,128-137,161-175) ------------------------
    def _values(self, entry_team: torch.Tensor, losing_team: torch.Tensor, cut: torch.Tensor) -> torch.Tensor:
        """[T, n] f32: the value of every history entry of every slot.  entry_team [T, n]: the team to move at the entry;
        losing_team [n]: the team that lost the slot's finished game; cut [n]: games cut off at max_game_length, valued
        by the heuristic of the slot's current position (self.env.boards) times heuristic_weight, for the team to move
        there, and its negation for the other team."""
        # finished games: +1 for the team that is not the losing team, GetOpponentValue(1) = -1 otherwise
        win = torch.where(entry_team != losing_team[None, :], 1.0, -1.0)
        # games cut off at max_game_length: heuristic of the team to move in the final position
        curr_team = (self.env.boards[:, self.geom.off_turn] & 1).long()
        heur = self.env.heuristic().float() * float(self.args["heuristic_weight"])
        cut_value = torch.where(entry_team == curr_team[None, :], heur[None, :], -heur[None, :])
        return torch.where(cut[None, :], cut_value, win)

    def finish(self, running: torch.Tensor, losing_team: torch.Tensor) -> dict:
        entry_team = (self.hist_boards[:, :, self.geom.off_turn] & 1).long()  # [T, n] team of the side to move
        value = self._values(entry_team, losing_team, running)
        sel = self.hist_valid
        extra = {"child_policy": self.hist_policy[sel]} if self.mcts.gumbel else {}  # [M, FPC_MAX_MOVES] improved policy
        return {
            "boards": self.hist_boards[sel],        # [M, record] the replay states
            "child_flat": self.hist_flat[sel],      # [M, FPC_MAX_MOVES] board-frame flat indices of the root's children
            "child_visits": self.hist_visits[sel],  # [M, FPC_MAX_MOVES] their visit counts (targets: policy_targets)
            "value": value[sel],                    # [M]
            "finished": ~running,
            "losing_team": losing_team,
            **extra,
        }

    def policy_targets(self, replay: dict) -> torch.Tensor:
        """Dense [M, A*R*R] action-probability targets in the network's frame, the frame of `encoded_states`
        (module-level `policy_targets`): the normalised visit counts (`alphazero.py:104-110`), or the Gumbel search's
        improved policy when the replay has child_policy.  The reference scatters the visits at the board-frame index
        (`alphazero.py:109`) while its network sees rotated planes; here the targets follow the rotation.  A self-play
        run with batch_rotation=True read its leaves in the colour of each batch's first state, so these own-colour
        targets match what its search read only for Red-led batches."""
        weights = replay["child_policy"] if "child_policy" in replay else replay["child_visits"]
        return policy_targets(self.geom, replay["boards"], replay["child_flat"], weights)

    def encoded_states(self, replay: dict) -> torch.Tensor:
        """`GetEncodedState(entry.state)` for every replay entry (`alphazero.py:71-75`): each state rotated by its
        own side to move, [M,24,R,R] f32, the network's frame of `policy_targets`."""
        boards = replay["boards"].contiguous()
        env = BatchedEnv(self.R, boards.shape[0], device=self.device)
        env.load(boards)
        return env.encode(k=-1)
