"""BatchedMCTS: the reference's `MCTS.search` (`src/py/mcts.py:17-43`) over `fpchess::Node`
(`src/cpp/node.{h,cpp}`) for N games at once, every tree resident in HBM.

Host-side mirror of the reference interface: `MCTS(gameType, neural_net, args).search(games)` becomes
`BatchedMCTS(R, n_games, neural_net, args).search(root_boards)`.  Per simulation the host issues
`fpc_tree_select` (descend + leaf rules + planes), the network forward (PyTorch, untouched) and
`fpc_tree_expand_backup` (softmax -> un-rotate -> mask -> renormalise -> backup -> expand); nothing
crosses to the host inside the loop, where the reference moves the dense policy to the CPU every
simulation (`mcts.py:83-87`).  PyTorch owns the device arrays; all tree logic runs in libfpc.so."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import FPC_MAX_MOVES, MAX_LEAVES_PER_GAME, GumbelDesc, LeafBatchDesc, TreeDesc, check
from .geometry import GEOMETRIES, NUM_STATE_CHANNELS

ERR_NODE_CAP, ERR_BOARD_CAP, ERR_NO_CHILD, ERR_MOVE = 1, 2, 4, 8
# node slots per simulation: a leaf adds at most FPC_MAX_MOVES children; the legal-move average is ~19-38 at 14x14
NODES_PER_SIM = 96
# sigma(q) = (GUMBEL_C_VISIT + max N) * GUMBEL_C_SCALE * q: the constants of Danihelka et al. (ICLR 2022) and mctx
GUMBEL_C_VISIT, GUMBEL_C_SCALE = 50.0, 0.1


class BatchedMCTS:
    def __init__(self, R: int, n_games: int, neural_net, args: dict, device: str | torch.device = "cuda",
                 batch_rotation: bool = False, node_cap: int | None = None, cuda_graph: bool = False,
                 reuse_tree: bool = False, leaves_per_game: int = 1, virtual_loss: int = 1, root_noise: bool = False,
                 noise_seed: int = 0, gumbel: bool = False, gumbel_seed: int = 0, gumbel_considered: int = 16,
                 gumbel_scale: float = 1.0, gumbel_interior: bool = False, gumbel_leaves: int = 1):
        """args: the reference's dict (`alphazero.py:291-306`): uses "C" and "num_searches".
        batch_rotation=True reproduces the reference bit for bit (a whole leaf batch is rotated by the
        colour of its first expandable state); False rotates every leaf by its own side to move.
        cuda_graph=True captures one whole simulation (select -> network -> expand/backup) in a CUDA graph after
        three eager ones and replays it: the ~70 launches of a simulation become one.
        reuse_tree=True sizes the default capacities for `advance` (keeping the played move's subtree between moves):
        room for a kept subtree plus a full new search.  It changes nothing else; `advance` works either way, it only
        keeps less with the smaller default arenas.
        leaves_per_game=L > 1 evaluates L leaf slots per game in every network call (leaf parallelism, outside the
        reference): each game descends L times per batch, every pending descent adding `virtual_loss` lost visits along
        its path so that later descents of the batch pick other leaves; a descent that ends on a leaf already taken in
        the batch is a collision and spends its slot without a visit (counted in `self.collisions`).  A search is then
        num_searches / L batches of n_games * L network rows; L must divide num_searches.  The first batch after a
        reset reaches the unexpanded root in every slot: one leaf and L - 1 collisions.  L = 1 is the one-leaf path.
        root_noise=True mixes AlphaZero's exploration noise into the root's children priors (outside the reference):
        prior <- (1 - eps) * prior + eps * Dir(alpha) with alpha = args["dirichlet_alpha"] and eps =
        args["dirichlet_epsilon"], both required then; once per root, i.e. per reset / advance (`add_root_noise`,
        `search`).  A game's draws depend only on (noise_seed, its key).  root_noise=False changes nothing.
        gumbel=True replaces the root's step by Gumbel AlphaZero's (Danihelka et al., ICLR 2022; outside the reference):
        gumbel_considered root moves sampled without replacement by Gumbel-top-k on the prior logits, the simulations
        spent on them by sequential halving, and `gumbel_result` gives the surviving move and the improved policy
        softmax(logits + sigma(completed Q)) (include/fpc.h states the recipe).  Below the root the descent is the
        reference's SelectChild.  A game's draws depend only on (gumbel_seed, its key); gumbel_scale=0 makes the search
        deterministic.  The schedule is planned for num_searches - 1 root visits (the first batch expands the root) and
        indexed by the root's own visits, so gumbel=True refuses reuse_tree, root_noise and leaves_per_game > 1, and
        search(None) cannot continue a finished search.  gumbel=False changes nothing.
        gumbel_interior=True (with gumbel=True) completes Gumbel MuZero: below the root the descent takes at every node
        the child maximising pi'_i - N_i / (1 + sum_j N_j), pi' = softmax(logits + sigma(completed Q)) computed at that
        node with its own network value (`fpc_tree_select_gumbel_interior`), instead of SelectChild.  It costs one f64
        per node slot (`node_value`, n_games x node_cap): 25 MB at 1,024 games x 32 simulations, 403 MB at 8,192 x 64.
        gumbel_interior=False changes nothing.
        gumbel_leaves=L > 1 (with gumbel=True, root-only or interior) runs the Gumbel search leaf-parallel
        (`fpc_tree_select_gumbel_leaves`): num_searches / L batches of n_games * L network rows, the L slots of a game
        taking the halving schedule's next L root visits, each continued below its root child with `virtual_loss` (or
        the interior step over the same effective statistics).  The schedule is indexed by `issued`, the visits it
        handed out per root child, so a collision (counted in `collisions`) costs that child a visit but never derails
        the schedule, and `gumbel_result` keeps the children with the most issued visits.  The first batch expands the
        root (one leaf, L - 1 collisions), so the schedule is planned for num_searches - L root visits: at 32
        simulations and L = 8 the root gets at most 24, against 31 at L = 1.  L must divide num_searches.
        gumbel_leaves=1 is the sequential Gumbel search, call for call."""
        self.geom = GEOMETRIES[R]
        self.R, self.n = R, int(n_games)
        self.net = neural_net
        self.args = args
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.FpcError("BatchedMCTS needs a CUDA device (there is no CPU fallback)")
        self.batch_rotation = bool(batch_rotation)
        self.cuda_graph = bool(cuda_graph)
        self._graph = None
        self.L = _lib.lib()
        sims = int(args["num_searches"])
        self.gumbel_leaves = int(gumbel_leaves)
        if not 1 <= self.gumbel_leaves <= MAX_LEAVES_PER_GAME:
            raise ValueError(f"gumbel_leaves must be in 1 .. {MAX_LEAVES_PER_GAME}, got {self.gumbel_leaves}")
        if self.gumbel_leaves > 1 and not gumbel:
            raise ValueError("gumbel_leaves > 1 needs gumbel=True")
        if sims % self.gumbel_leaves:
            raise ValueError(f"gumbel_leaves={self.gumbel_leaves} does not divide num_searches={sims}")
        self.leaves, self.virtual_loss = int(leaves_per_game), int(virtual_loss)
        if not 1 <= self.leaves <= MAX_LEAVES_PER_GAME:
            raise ValueError(f"leaves_per_game must be in 1 .. {MAX_LEAVES_PER_GAME}, got {self.leaves}")
        if self.virtual_loss < 1:
            raise ValueError(f"virtual_loss must be at least 1, got {self.virtual_loss}")
        if sims % self.leaves:
            raise ValueError(f"leaves_per_game={self.leaves} does not divide num_searches={sims}")
        gumbel_refused = ((reuse_tree, "reuse_tree=True"), (root_noise, "root_noise=True"),
                          (self.leaves > 1, "leaves_per_game > 1"))
        if self.gumbel_leaves > 1:
            self.leaves = self.gumbel_leaves  # the leaf batch below, with the Gumbel select (`select`)
        self._open = False  # a leaf batch was selected and not yet expanded: its in_flight marks are still set
        reuse = 2 if reuse_tree else 1
        self.node_cap = int(node_cap) if node_cap else 1 + reuse * NODES_PER_SIM * sims
        self.board_cap = reuse * sims + 2
        self._has_tree = False
        n, nc, dev = self.n, self.node_cap, self.device
        i32 = dict(dtype=torch.int32, device=dev)
        self.parent = torch.empty((n, nc), **i32)
        self.first_child = torch.empty((n, nc), **i32)
        self.n_children = torch.empty((n, nc), **i32)
        self.visits = torch.empty((n, nc), **i32)
        self.move_flat = torch.empty((n, nc), **i32)
        self.board_idx = torch.empty((n, nc), **i32)
        self.value_sum = torch.empty((n, nc), dtype=torch.float64, device=dev)
        self.prior = torch.empty((n, nc), dtype=torch.float32, device=dev)
        self.n_nodes = torch.zeros(n, **i32)
        self.n_boards = torch.zeros(n, **i32)
        self.leaf = torch.full((n,), -1, **i32)
        self.dropped = torch.zeros(n, **i32)
        self.error = torch.zeros(n, **i32)
        rec = self.geom.record_bytes
        self.boards = torch.empty((n, self.board_cap, rec), dtype=torch.uint8, device=dev)
        self.leaf_boards = torch.zeros((n, rec), dtype=torch.uint8, device=dev)
        self.leaf_flat = torch.zeros((n, FPC_MAX_MOVES), **i32)
        self.leaf_counts = torch.zeros(n, **i32)
        self.leaf_status = torch.zeros(n, **i32)
        self.k = torch.zeros(n, **i32)
        slots = n * self.leaves
        self.planes = torch.empty((slots, NUM_STATE_CHANNELS, R, R), dtype=torch.float32, device=dev)
        with torch.cuda.device(self.device):
            self._track = self.L.fpc_dense_track_create(R, slots)  # lets select() update self.planes in place
        if not self._track:
            raise _lib.FpcError(self.L.fpc_last_error().decode())
        d = TreeDesc()
        d.R, d.n_games, d.node_cap, d.board_cap, d.C = R, n, self.node_cap, self.board_cap, float(args["C"])
        for name in ("parent", "first_child", "n_children", "visits", "move_flat", "board_idx", "value_sum", "prior",
                     "n_nodes", "n_boards", "leaf", "dropped", "error", "boards", "leaf_boards", "leaf_flat",
                     "leaf_counts", "leaf_status", "k"):
            setattr(d, name, getattr(self, name).data_ptr())
        self.desc = d
        self.batch = None
        self.collisions = torch.zeros(n, **i32)  # collision slots since the last reset / advance (none at L = 1)
        if self.leaves > 1:
            # the leaf batch (struct fpc_leaf_batch): per-slot arrays for n * L slots, slot s = g * L + j
            self.in_flight = torch.zeros((n, nc), **i32)  # zero between batches; the two leaf calls keep it so
            self.slot_node = torch.full((slots,), -1, **i32)
            self.slot_kind = torch.zeros(slots, **i32)
            self.slot_boards = torch.zeros((slots, rec), dtype=torch.uint8, device=dev)
            self.slot_flat = torch.zeros((slots, FPC_MAX_MOVES), **i32)
            self.slot_counts = torch.zeros(slots, **i32)
            self.slot_status = torch.zeros(slots, **i32)
            self.slot_k = torch.zeros(slots, **i32)
            self.slot_priors = torch.zeros((slots, FPC_MAX_MOVES), dtype=torch.float32, device=dev)
            b = LeafBatchDesc()
            b.L, b.virtual_loss = self.leaves, self.virtual_loss
            for field, name in (("in_flight", "in_flight"), ("slot_node", "slot_node"), ("slot_kind", "slot_kind"),
                                ("leaf_boards", "slot_boards"), ("leaf_flat", "slot_flat"),
                                ("leaf_counts", "slot_counts"), ("leaf_status", "slot_status"), ("k", "slot_k"),
                                ("priors", "slot_priors"), ("collisions", "collisions")):
                setattr(b, field, getattr(self, name).data_ptr())
            self.batch = b
        self.gumbel = bool(gumbel)
        self.gumbel_interior = bool(gumbel_interior)
        if self.gumbel_interior and not self.gumbel:
            raise ValueError("gumbel_interior=True needs gumbel=True")
        if self.gumbel:
            for refused, what in gumbel_refused:
                if refused:
                    raise ValueError(f"gumbel=True does not combine with {what}")
            # fixed addresses: a captured CUDA graph of simulate() reads the keys and writes root_value in place
            self.gumbel_keys = torch.zeros(n, dtype=torch.int64, device=dev)
            self.root_value = torch.zeros(n, dtype=torch.float64, device=dev)
            gd = GumbelDesc()
            gd.seed = int(gumbel_seed) & (2**64 - 1)
            gd.keys, gd.root_value = self.gumbel_keys.data_ptr(), self.root_value.data_ptr()
            # the schedule's root visits: the first batch expands the root and spends all its L slots there
            gd.max_considered, gd.n_sims = int(gumbel_considered), max(0, sims - self.leaves)
            gd.scale, gd.c_visit, gd.c_scale = float(gumbel_scale), GUMBEL_C_VISIT, GUMBEL_C_SCALE
            self.gumbel_desc = gd
            if self.gumbel_interior:
                # each node's network value, cached by the select at the node's first pass; every entry is written
                # before it is read, so it needs no initialisation (fixed address, like root_value)
                self.node_value = torch.empty((n, nc), dtype=torch.float64, device=dev)
            if self.batch is not None:
                # I_i: the root visits the halving schedule issued to child i since the reset (fixed address)
                self.issued = torch.zeros((n, FPC_MAX_MOVES), **i32)
            self._gumbel_searches = 0
        self.root_noise = bool(root_noise)
        if self.root_noise:
            missing = [key for key in ("dirichlet_alpha", "dirichlet_epsilon") if key not in args]
            if missing:
                raise ValueError(f"root_noise=True needs args {missing}")
            self.noise_alpha, self.noise_eps = float(args["dirichlet_alpha"]), float(args["dirichlet_epsilon"])
            self.noise_seed = int(noise_seed) & (2**64 - 1)
            self.noise_done = torch.zeros(n, **i32)  # 1 once the current root was noised; zeroed by reset / advance
            self._searches = 0

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _close_batch(self) -> None:
        """Before the trees are replaced or re-rooted: clear the marks of a leaf batch that was selected and never
        expanded, and restart the collision count and the root-noise marks."""
        if self._open:
            self.in_flight.zero_()
            self._open = False
        if self.batch is not None:
            self.collisions.zero_()
            if self.gumbel:
                self.issued.zero_()  # a new root: the schedule starts again
        if self.root_noise:
            self.noise_done.zero_()  # a new root: noised again by the next add_root_noise

    # ---- the three device steps ----------------------------------------------------------------
    def reset(self, root_boards: torch.Tensor) -> None:
        self._close_batch()
        roots = root_boards.to(self.device, torch.uint8).contiguous()
        assert roots.shape == (self.n, self.geom.record_bytes)
        with torch.cuda.device(self.device):
            check(self.L.fpc_tree_reset(C.byref(self.desc), roots.data_ptr(), self._stream()))
        self._roots = roots  # keep alive until the kernel has run
        self._has_tree = True

    def advance(self, actions: torch.Tensor, root_boards: torch.Tensor) -> torch.Tensor:
        """Re-root every game's tree on the root child that played actions[g] (i32 flat index; -1 = none), keeping
        that child's subtree -- its visits, value sums, priors and boards -- for the next search.  root_boards = the
        positions after the move, made with the index-built move (`BatchedEnv.make_index`).  A game whose child is
        missing, whose subtree would leave less headroom than a fresh tree has (more than node_cap - 96 * sims nodes or
        board_cap - sims boards) or whose child's board differs from root_boards[g] gets a fresh root instead, as
        reset() makes it.  Returns kept [n] i32: the nodes carried over per game, 0 for a fresh root."""
        if not self._has_tree:
            raise _lib.FpcError("advance() needs a tree: call reset() or search(root_boards) first")
        acts = actions.to(self.device, torch.int32).contiguous()
        roots = root_boards.to(self.device, torch.uint8).contiguous()
        assert acts.shape == (self.n,) and roots.shape == (self.n, self.geom.record_bytes)
        sims = int(self.args["num_searches"])
        max_nodes = max(0, self.node_cap - NODES_PER_SIM * sims)
        max_boards = max(0, self.board_cap - sims)
        kept = torch.empty(self.n, dtype=torch.int32, device=self.device)
        self._close_batch()
        with torch.cuda.device(self.device):
            check(self.L.fpc_tree_advance(C.byref(self.desc), acts.data_ptr(), roots.data_ptr(), max_nodes, max_boards,
                                          kept.data_ptr(), self._stream()))
        self._roots, self._acts = roots, acts  # keep alive until the kernel has run
        return kept

    def select(self) -> torch.Tensor:
        """Node.ChooseLeaf for every live game; returns the encoded leaf batch [n,24,R,R] ([n*L,24,R,R] with L leaf slots
        per game, slot s = g*L + j; the rows of collision and empty slots are evaluated and ignored)."""
        # the planes tensor is resident and only read by the network between selects: after the first full encode
        # through this instance's handle it is updated in place (FPC_FLAG_INCREMENTAL)
        with torch.cuda.device(self.device):
            if self.gumbel and self.batch is not None:
                node_value = self.node_value.data_ptr() if self.gumbel_interior else None
                check(self.L.fpc_tree_select_gumbel_leaves(C.byref(self.desc), C.byref(self.gumbel_desc), C.byref(self.batch),
                                                           self.issued.data_ptr(), node_value, int(self.batch_rotation),
                                                           self.planes.data_ptr(), _lib.FLAG_INCREMENTAL, self._track,
                                                           self._stream()))
                self._open = True
            elif self.gumbel_interior:
                check(self.L.fpc_tree_select_gumbel_interior(C.byref(self.desc), C.byref(self.gumbel_desc),
                                                             self.node_value.data_ptr(), int(self.batch_rotation),
                                                             self.planes.data_ptr(), _lib.FLAG_INCREMENTAL,
                                                             self._track, self._stream()))
            elif self.gumbel:
                check(self.L.fpc_tree_select_gumbel(C.byref(self.desc), C.byref(self.gumbel_desc), int(self.batch_rotation),
                                                    self.planes.data_ptr(), _lib.FLAG_INCREMENTAL, self._track,
                                                    self._stream()))
            elif self.batch is None:
                check(self.L.fpc_tree_select(C.byref(self.desc), int(self.batch_rotation), self.planes.data_ptr(),
                                             _lib.FLAG_INCREMENTAL, self._track, self._stream()))
            else:
                check(self.L.fpc_tree_select_leaves(C.byref(self.desc), C.byref(self.batch), int(self.batch_rotation),
                                                    self.planes.data_ptr(), _lib.FLAG_INCREMENTAL, self._track,
                                                    self._stream()))
                self._open = True
        return self.planes

    def add_root_noise(self, keys) -> None:
        """Dirichlet noise on the root's children priors of every game whose root is expanded, not dropped and not yet
        noised since the last reset / advance (`fpc_tree_root_noise`); keys [n] i64 select the games' draws.  A caller
        that drives select / expand_backup itself calls it before its first batch and again right after it: the second
        call reaches the roots that the first batch expanded."""
        if not self.root_noise:
            raise _lib.FpcError("add_root_noise() needs BatchedMCTS(..., root_noise=True)")
        keys = torch.as_tensor(keys, dtype=torch.int64).to(self.device).contiguous()
        assert keys.shape == (self.n,)
        with torch.cuda.device(self.device):
            check(self.L.fpc_tree_root_noise(C.byref(self.desc), self.noise_seed, keys.data_ptr(), self.noise_alpha,
                                             self.noise_eps, self.noise_done.data_ptr(), self._stream()))
        self._noise_keys = keys  # keep alive until the kernel has run

    def gumbel_result(self):
        """(action [n] i32, policy [n, FPC_MAX_MOVES] f32) of the current search (`fpc_tree_gumbel_result`): the flat
        action of the root child the halving leaves standing, and the improved policy softmax(logits + sigma(completed
        Q)) with its columns aligned with root_children().  A root without children gets action -1 and a zero row; a
        dropped game's result comes from the visits it has.  With gumbel_leaves > 1 the survivors are the children with
        the most issued visits (`fpc_tree_gumbel_result_leaves`)."""
        if not self.gumbel:
            raise _lib.FpcError("gumbel_result() needs BatchedMCTS(..., gumbel=True)")
        action = torch.empty(self.n, dtype=torch.int32, device=self.device)
        policy = torch.empty((self.n, FPC_MAX_MOVES), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            if self.batch is not None:
                check(self.L.fpc_tree_gumbel_result_leaves(C.byref(self.desc), C.byref(self.gumbel_desc),
                                                           self.issued.data_ptr(), action.data_ptr(), policy.data_ptr(),
                                                           self._stream()))
            else:
                check(self.L.fpc_tree_gumbel_result(C.byref(self.desc), C.byref(self.gumbel_desc), action.data_ptr(),
                                                    policy.data_ptr(), self._stream()))
        return action, policy

    def sample_root(self, seed: int, keys, temperature: float) -> torch.Tensor:
        """[n] i32: a move drawn from every game's root visit counts with the reference's distribution (visits / sum
        raised to 1 / temperature, `alphazero.py:108-118`), by one counter-based uniform per (seed, keys[g])
        (`fpc_tree_sample_root`), so that a game's move does not depend on the games it shares the batch with.  -1 for a
        dropped game and for a root without children or visits.  A search drops a game whose descent reached a terminal
        leaf, so a caller that wants a move for such a game sets `dropped` back first."""
        keys = torch.as_tensor(keys, dtype=torch.int64).to(self.device).contiguous()
        assert keys.shape == (self.n,)
        action = torch.empty(self.n, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            check(self.L.fpc_tree_sample_root(C.byref(self.desc), int(seed) & (2**64 - 1), keys.data_ptr(),
                                              float(temperature), action.data_ptr(), self._stream()))
        self._sample_keys = keys  # keep alive until the kernel has run
        return action

    def close(self) -> None:
        if getattr(self, "_track", None):
            self.L.fpc_dense_track_destroy(self._track)
            self._track = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def expand_backup(self, logits: torch.Tensor, values: torch.Tensor) -> None:
        logits = logits.to(torch.float32).contiguous()
        values = values.to(torch.float32).reshape(-1).contiguous()
        rows = self.n * self.leaves
        assert logits.shape == (rows, self.geom.action_space_size) and values.shape == (rows,)
        with torch.cuda.device(self.device):
            if self.batch is None:
                check(self.L.fpc_tree_expand_backup(C.byref(self.desc), logits.data_ptr(), values.data_ptr(),
                                                    self._stream()))
            else:
                check(self.L.fpc_tree_expand_backup_leaves(C.byref(self.desc), C.byref(self.batch), logits.data_ptr(),
                                                           values.data_ptr(), self._stream()))
                self._open = False

    # ---- MCTS.search (mcts.py:17-43) -------------------------------------------------------------
    def simulate(self) -> None:
        """One simulation for every live game (`MCTS.step` + `MCTS.expand`, mcts.py:59-89); with L leaf slots per game,
        one batch of L slots per game."""
        planes = self.select()
        logits, value = self.net(planes)
        self.expand_backup(logits, value)

    @torch.no_grad()
    def search(self, root_boards: torch.Tensor | None = None, record=None, check: bool = True,
               noise_keys=None, gumbel_keys=None, dropped=None) -> "BatchedMCTS":
        """num_searches simulations from fresh roots at root_boards, or, with root_boards=None, on top of the current
        trees (after advance(), or to add simulations to a finished search).
        record: optional callable(sim, logits, value) called after every network forward (eager mode only), e.g.
        to keep the outputs of some games for a replay on the CPU oracle (with L leaf slots per game: sim = the batch,
        rows g*L + j).  check: raise on tree errors (arena full ...)
        instead of leaving them in `self.error`.
        noise_keys: with root_noise=True, the [n] i64 keys of this search's root noise (default arange(n) + n * s for
        this instance's s-th search).  add_root_noise runs before the first batch (roots that already have children:
        a kept subtree) and right after it (roots the first batch expanded), outside the CUDA graph; a root noised since
        the last reset / advance is not noised again.
        gumbel_keys: with gumbel=True, the [n] i64 keys of this search's Gumbel draws, copied into `self.gumbel_keys`
        (default arange(n) + n * s for this instance's s-th search).
        dropped: optional [n] bool mask of games that sit this search out (finished games), set after the reset as a
        caller driving select / expand_backup itself would set `self.dropped`."""
        if self.gumbel and root_boards is None:
            raise _lib.FpcError("search(None) with gumbel=True: a finished halving schedule cannot be continued")
        if root_boards is not None:
            self.reset(root_boards)
        elif not self._has_tree:
            raise _lib.FpcError("search(None) continues the current trees, but there are none: pass root_boards")
        if dropped is not None:
            self.dropped.copy_(torch.as_tensor(dropped).reshape(self.n))
        sims = int(self.args["num_searches"])
        if sims % self.leaves:
            raise ValueError(f"leaves_per_game={self.leaves} does not divide num_searches={sims}")
        sims //= self.leaves  # network batches
        if self.gumbel:
            if gumbel_keys is None:
                gumbel_keys = torch.arange(self.n, dtype=torch.int64, device=self.device) + self.n * self._gumbel_searches
            self._gumbel_searches += 1
            self.gumbel_keys.copy_(torch.as_tensor(gumbel_keys, dtype=torch.int64).reshape(self.n))
        keys = None
        if self.root_noise:
            keys = noise_keys
            if keys is None:
                keys = torch.arange(self.n, dtype=torch.int64, device=self.device) + self.n * self._searches
            self._searches += 1
            self.add_root_noise(keys)

        def after_batch(done):
            if done == 1 and keys is not None:
                self.add_root_noise(keys)

        done = 0
        if self.cuda_graph and record is None:
            # eager warm-up (the first select writes the planes in full; cuDNN / cuBLAS pick their kernels), then capture
            while self._graph is None and done < min(3, sims):
                self.simulate()
                done += 1
                after_batch(done)
            if self._graph is None and done < sims:
                torch.cuda.synchronize(self.device)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self.simulate()
                self._graph = g  # capturing runs nothing: the simulation count is unchanged
            while done < sims:
                self._graph.replay()
                done += 1
                after_batch(done)
        else:
            for sim in range(sims):
                planes = self.select()
                logits, value = self.net(planes)
                if record is not None:
                    record(sim, logits, value)
                self.expand_backup(logits, value)
                after_batch(sim + 1)
        if check:
            self.check_errors()
        return self

    # ---- results -----------------------------------------------------------------------------------
    def check_errors(self) -> None:
        e = int(self.error.max().item())
        if e:
            raise _lib.FpcError(f"tree error bits {e:#x} (1 node_cap, 2 board_cap, 4 no child selectable, 8 move)")

    def root_children(self):
        """(flat [n,FPC_MAX_MOVES] i32, visits [n,FPC_MAX_MOVES] i32, prior f32, count [n]) of the root's
        children, zero-padded: what `AlphaZero.play` reads through GetChildren / GetVisitCount /
        GetMoveMade (`alphazero.py:104-110`)."""
        cnt = self.n_children[:, 0]
        fc = self.first_child[:, 0].long()
        idx = fc[:, None] + torch.arange(FPC_MAX_MOVES, device=self.device)[None, :]
        valid = torch.arange(FPC_MAX_MOVES, device=self.device)[None, :] < cnt[:, None]
        idx = torch.where(valid, idx, torch.zeros_like(idx))
        zero = torch.zeros((), dtype=torch.int32, device=self.device)
        flat = torch.where(valid, torch.gather(self.move_flat, 1, idx), zero)
        visits = torch.where(valid, torch.gather(self.visits, 1, idx), zero)
        prior = torch.where(valid, torch.gather(self.prior, 1, idx), torch.zeros((), device=self.device))
        return flat, visits, prior, cnt

    def action_probs(self) -> torch.Tensor:
        """`alphazero.py:104-110`: visit counts of the root's children scattered over the action space and
        normalised, [n, A*R*R] f32."""
        flat, visits, _, _ = self.root_children()
        probs = torch.zeros((self.n, self.geom.action_space_size), dtype=torch.float32, device=self.device)
        probs.scatter_add_(1, flat.long(), visits.float())
        return probs / probs.sum(dim=1, keepdim=True).clamp_min(1e-30)
