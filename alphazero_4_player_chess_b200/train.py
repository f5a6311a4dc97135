"""Learner: the reference's outer loop `AlphaZero.learn / train / validate` (`src/py/alphazero.py:181-276`)
around the device-resident self-play of selfplay.py.

This is the last ring around the hot path (SURVEY 8f rank 4): replay tensors stay on the device
(board records + sparse visit distributions + values; the dense targets and the encoded planes are
expanded per mini-batch by the CUDA encoder), the optimiser step is plain PyTorch, and with more
than one GPU each rank plays its own shard of games and gradients are averaged by
`DistributedDataParallel` (NCCL all-reduce) -- the only bulk cross-GPU traffic of the whole system.
The loss is the reference's: cross-entropy(policy logits, visit distribution) + MSE(value, outcome),
Adam + StepLR(1000, 0.1).  Planes and policy targets are both in the network's frame, each entry rotated by its own
side to move (`SelfPlay.encoded_states`, `SelfPlay.policy_targets`), where the reference trains on board-frame targets."""
from __future__ import annotations

import torch
import torch.distributed as dist
import torch.nn.functional as F

from .geometry import GEOMETRIES


class ReplayStore:
    """Ring buffer of replay entries as device tensors (`src/py/replay_buffer.py:4-20` keeps Python tuples): board
    records, the root children's board-frame flat indices and visit counts, and values."""

    def __init__(self, capacity: int, record_bytes: int, max_children: int, device, child_policy: bool = False):
        """child_policy=True also keeps an f32 policy weight per child (the Gumbel search's improved policy)."""
        self.capacity, self.size, self.head = int(capacity), 0, 0
        self.boards = torch.zeros((self.capacity, record_bytes), dtype=torch.uint8, device=device)
        self.child_flat = torch.zeros((self.capacity, max_children), dtype=torch.int32, device=device)
        self.child_visits = torch.zeros((self.capacity, max_children), dtype=torch.int32, device=device)
        self.value = torch.zeros(self.capacity, dtype=torch.float32, device=device)
        self.child_policy = (torch.zeros((self.capacity, max_children), dtype=torch.float32, device=device)
                             if child_policy else None)

    def add(self, boards, child_flat, child_visits, value, child_policy=None) -> None:
        m = boards.shape[0]
        if m == 0:
            return
        if m >= self.capacity:
            boards, child_flat, child_visits, value = (t[-self.capacity:] for t in (boards, child_flat, child_visits, value))
            child_policy = child_policy[-self.capacity:] if child_policy is not None else None
            m = self.capacity
        idx = (self.head + torch.arange(m, device=self.boards.device)) % self.capacity
        self.boards[idx], self.child_flat[idx], self.child_visits[idx], self.value[idx] = boards, child_flat, child_visits, value
        if self.child_policy is not None:
            self.child_policy[idx] = child_policy
        self.head = (self.head + m) % self.capacity
        self.size = min(self.capacity, self.size + m)

    def sample(self, batch: int):
        """(boards, child_flat, child_visits, value) of `batch` entries drawn with replacement, and child_policy after
        them when the store keeps it."""
        idx = torch.randint(0, self.size, (batch,), device=self.boards.device)
        out = (self.boards[idx], self.child_flat[idx], self.child_visits[idx], self.value[idx])
        return out if self.child_policy is None else out + (self.child_policy[idx],)

    def __len__(self) -> int:
        return self.size


class Learner:
    def __init__(self, selfplay, model: torch.nn.Module, optimizer: torch.optim.Optimizer, args: dict,
                 continuous: bool = False):
        """selfplay: a SelfPlay whose network wraps `model` for inference; args: the reference's dict
        (`alphazero.py:291-306`): batch_size, replay_buffer_capacity, validation_buffer_capacity, num_iterations,
        num_games, num_parallel_games.  continuous=True plays each iteration's games with `SelfPlay.play_games`
        (a slot takes the next game as soon as its own ends): num_games games for training, then num_parallel_games for
        validation, the game ids continuing across iterations.  continuous=False plays rounds of `SelfPlay.play`, as the
        reference does."""
        self.sp, self.model, self.opt, self.args = selfplay, model, optimizer, args
        self.continuous = bool(continuous)
        self.sched = torch.optim.lr_scheduler.StepLR(optimizer, step_size=1000, gamma=0.1)  # alphazero.py:25-27
        g = selfplay.geom
        dev = selfplay.device
        self.geom = GEOMETRIES[g.R]
        # a self-play that records an improved policy (Gumbel search) trains on it: the stores keep it beside the visits
        pol = hasattr(selfplay, "hist_policy")
        self.train_buf = ReplayStore(args["replay_buffer_capacity"], g.record_bytes, selfplay.hist_flat.shape[-1], dev, pol)
        self.valid_buf = ReplayStore(args["validation_buffer_capacity"], g.record_bytes, selfplay.hist_flat.shape[-1], dev,
                                     pol)
        self.ddp = None
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            ids = [dev.index] if dev.type == "cuda" else None
            self.ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=ids)
        self.log: list[dict] = []

    # ---- replay (handle_terminal_state, alphazero.py:53-79) ------------------------------------------
    def store(self, replay: dict) -> None:
        m = replay["boards"].shape[0]
        cap_t, cap_v = self.args["replay_buffer_capacity"], self.args["validation_buffer_capacity"]
        to_train = torch.rand(m, device=replay["boards"].device) < cap_t / (cap_t + cap_v)
        for buf, sel in ((self.train_buf, to_train), (self.valid_buf, ~to_train)):
            policy = replay["child_policy"][sel] if buf.child_policy is not None else None
            buf.add(replay["boards"][sel], replay["child_flat"][sel], replay["child_visits"][sel], replay["value"][sel], policy)

    def _batch(self, buf: ReplayStore):
        """(planes, policy targets, values) of one drawn mini-batch; planes and targets in the network's frame."""
        boards, flat, visits, value, *policy = buf.sample(int(self.args["batch_size"]))
        fake = {"boards": boards, "child_flat": flat, "child_visits": visits}
        if policy:
            fake["child_policy"] = policy[0]
        return self.sp.encoded_states(fake), self.sp.policy_targets(fake), value

    def _loss(self, net, planes, policy_t, value_t):
        out_policy, out_value = net(planes)
        policy_loss = F.cross_entropy(out_policy, policy_t)          # alphazero.py:201
        value_loss = F.mse_loss(out_value.squeeze(-1), value_t)       # alphazero.py:202
        return policy_loss + value_loss, policy_loss, value_loss

    # ---- train / validate (alphazero.py:181-258) ------------------------------------------------------
    def train(self) -> int:
        bs = int(self.args["batch_size"])
        # alphazero.py:185-186: one mini-batch per batch_size entries of the replay buffer.  Under DDP every rank must run
        # the SAME number of steps (each backward is a collective): ranks play games of different lengths and split
        # train / validation with their own draws, so the count is agreed on first -- the minimum over the ranks, and
        # nobody trains while some rank has less than one batch.
        n_steps = -(-len(self.train_buf) // bs) if len(self.train_buf) >= bs else 0
        if self.ddp is not None:
            t = torch.tensor([n_steps], dtype=torch.int64, device=self.train_buf.boards.device)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            n_steps = int(t.item())
        if n_steps == 0:
            return 0
        net = self.ddp if self.ddp is not None else self.model
        self.model.train()
        steps = 0
        for _ in range(n_steps):
            planes, policy_t, value_t = self._batch(self.train_buf)
            loss, pl, vl = self._loss(net, planes, policy_t, value_t)
            self.opt.zero_grad(set_to_none=True)
            loss.backward()  # DistributedDataParallel averages the gradients over the ranks here
            self.opt.step()
            self.sched.step()
            self.log.append({"policy_loss": float(pl.detach()), "value_loss": float(vl.detach()), "lr": self.opt.param_groups[0]["lr"]})
            steps += 1
        return steps

    @torch.no_grad()
    def validate(self):
        if len(self.valid_buf) < int(self.args["batch_size"]):
            return None
        self.model.eval()
        planes, policy_t, value_t = self._batch(self.valid_buf)
        loss, pl, vl = self._loss(self.model, planes, policy_t, value_t)
        return {"validation_policy_loss": float(pl), "validation_value_loss": float(vl), "validation_loss": float(loss)}

    # ---- learn (alphazero.py:260-276) --------------------------------------------------------------------
    def learn(self, iterations: int | None = None) -> list[dict]:
        out = []
        for _ in range(int(iterations if iterations is not None else self.args["num_iterations"])):
            self.model.eval()
            if self.continuous:
                self.store(self.sp.play_games(int(self.args["num_games"])))
            else:
                for _ in range(max(1, int(self.args["num_games"]) // int(self.args["num_parallel_games"]))):
                    self.store(self.sp.play())
            steps = self.train()
            self.model.eval()
            self.store(self.sp.play_games(int(self.args["num_parallel_games"])) if self.continuous else self.sp.play())
            out.append({"train_steps": steps, "replay": len(self.train_buf), "validation": self.validate()})
        return out
