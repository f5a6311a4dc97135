"""CPU: the learner's side of self-play.  The dense policy targets (selfplay.policy_targets) against an f64 restatement
on oracle positions, read back the way tree_expand_backup_kernel reads the network's row (rot_index); Learner._loss
against an f64 restatement of the reference's loss; ReplayStore against a plain Python ring."""
import functools
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200._lib import FPC_MAX_MOVES
from alphazero_4_player_chess_b200.geometry import GEOMETRIES
from alphazero_4_player_chess_b200.selfplay import SelfPlay, policy_targets
from alphazero_4_player_chess_b200.train import Learner, ReplayStore
from tests.test_gpu_puct_kernels import START, rot_index
from tests.util import oracle_for, playout_positions, random_positions


# ---- the f64 restatement of the targets -----------------------------------------------------------------------------

def legal_flats(R, rec):
    o = oracle_for(R)
    return np.unique(np.array([o.move_flat_index(m) for m in o.legal_moves(rec)], dtype=np.int64))


def normalised(weights):
    w = np.asarray(weights, dtype=np.float64)
    s = w.sum()
    return w / s if s > 0 else w


def targets_f64(R, recs, child_flat, weights):
    """[M, A*R*R] f64: each row's normalised weights scattered at the board-frame flats, then np.rot90 by +k over
    [A, R, R], k the row's side to move -- the network's frame when the planes are encoded rotated by k."""
    g = GEOMETRIES[R]
    A = g.num_action_channels
    out = np.zeros((len(recs), g.action_space_size))
    for i, rec in enumerate(recs):
        t = np.zeros(g.action_space_size)
        np.add.at(t, child_flat[i], normalised(weights[i]))
        out[i] = np.rot90(t.reshape(A, R, R), int(rec[g.off_turn]), axes=(1, 2)).reshape(-1)
    return out


def synthetic_children(R, recs, rng, source):
    """child_flat [M, FPC_MAX_MOVES] i32 (each position's legal flats in random order, zero padded) and weights:
    random visit counts 0..5 as i32 ("visits"), or an f32 soft-max row like the Gumbel improved policy ("gumbel")."""
    flat = np.zeros((len(recs), FPC_MAX_MOVES), np.int32)
    w = np.zeros((len(recs), FPC_MAX_MOVES), np.int32 if source == "visits" else np.float32)
    for i, rec in enumerate(recs):
        legal = rng.permutation(legal_flats(R, rec))
        n = len(legal)
        flat[i, :n] = legal
        if source == "visits":
            w[i, :n] = rng.integers(0, 6, n)
        else:
            x = rng.normal(0.0, 3.0, n)
            e = np.exp(x - x.max()) if n else x
            w[i, :n] = (e / e.sum()).astype(np.float32)
    return flat, w


@functools.lru_cache(maxsize=None)
def positions(R):
    """Oracle playout positions (castling on and off) and random positions at R."""
    play = [playout_positions(START[R], c, 4, 24)["recs"] for c in (True, False)]
    return np.concatenate(play + [random_positions(R, 96, seed=R)])


def check_targets(R, recs, flat, w, got):
    """got [M, A*R*R] against the restatement to f32 rounding (zero where the restatement is zero), and read back
    through rot_index(k): the legal moves hold all the mass, each move its own normalised weight."""
    g = GEOMETRIES[R]
    A = g.num_action_channels
    want = targets_f64(R, recs, flat, w)
    np.testing.assert_allclose(got, want, rtol=2e-6, atol=0)
    for i, rec in enumerate(recs):
        share = normalised(w[i])
        if not share.any():
            assert not got[i].any(), i
            continue
        read = got[i][rot_index(R, A, int(rec[g.off_turn]))].astype(np.float64)  # the prior the kernel gives each flat
        assert read[legal_flats(R, rec)].sum() >= 1 - 1e-6, i
        live = share > 0
        np.testing.assert_allclose(read[flat[i][live]], share[live], rtol=2e-6, atol=0, err_msg=str(i))


@pytest.mark.parametrize("source", ["visits", "gumbel"])
@pytest.mark.parametrize("colour", [0, 1, 2, 3])
@pytest.mark.parametrize("R", [8, 10, 13, 14])
def test_targets_match_the_f64_restatement(R, colour, source):
    g = GEOMETRIES[R]
    recs = positions(R)
    recs = recs[recs[:, g.off_turn] == colour]
    assert len(recs) >= 20
    rng = np.random.default_rng(1000 * R + 10 * colour + (source == "gumbel"))
    flat, w = synthetic_children(R, recs, rng, source)
    w[0] = 0  # an all-zero row stays all zero
    got = policy_targets(g, torch.from_numpy(recs), torch.from_numpy(flat), torch.from_numpy(w)).numpy()
    check_targets(R, recs, flat, w, got)


@pytest.mark.parametrize("R", [8, 14])
def test_selfplay_sends_both_sources_through_the_placement(R):
    """SelfPlay.policy_targets trains on child_policy when the replay has it, on the visits otherwise, both placed by
    policy_targets (the method only reads self.geom)."""
    g = GEOMETRIES[R]
    recs = positions(R)
    rng = np.random.default_rng(R)
    flat, visits = synthetic_children(R, recs, rng, "visits")
    _, policy = synthetic_children(R, recs, np.random.default_rng(R), "gumbel")  # the same flats, other weights
    replay = {"boards": torch.from_numpy(recs), "child_flat": torch.from_numpy(flat),
              "child_visits": torch.from_numpy(visits)}
    sp = SimpleNamespace(geom=g)
    check_targets(R, recs, flat, visits, SelfPlay.policy_targets(sp, replay).numpy())
    replay["child_policy"] = torch.from_numpy(policy)
    check_targets(R, recs, flat, policy, SelfPlay.policy_targets(sp, replay).numpy())


# ---- Learner._loss ------------------------------------------------------------------------------------------------

class Given(torch.nn.Module):
    """A network stub that returns fixed outputs."""

    def __init__(self, logits, value):
        super().__init__()
        self.logits, self.value = logits, value

    def forward(self, planes):
        assert planes.shape[0] == self.logits.shape[0]
        return self.logits, self.value


def stub_learner(R):
    sp = SimpleNamespace(geom=GEOMETRIES[R], device=torch.device("cpu"),
                         hist_flat=torch.zeros((1, 1, FPC_MAX_MOVES), dtype=torch.int32))
    w = torch.zeros(1, requires_grad=True)
    return Learner(sp, torch.nn.Linear(1, 1), torch.optim.SGD([w], lr=0.0),
                   {"replay_buffer_capacity": 8, "validation_buffer_capacity": 8, "batch_size": 4})


@pytest.mark.parametrize("target", ["spread", "one_move"])
@pytest.mark.parametrize("sigma,offset", [(0.01, 0.0), (1.0, 0.0), (20.0, 0.0), (1.0, 1e4), (20.0, 1e4)])
def test_loss_matches_the_f64_restatement(sigma, offset, target):
    R, B = 14, 12
    g = GEOMETRIES[R]
    rng = np.random.default_rng(int(sigma * 100) + int(offset) + (target == "one_move"))
    logits = (offset + sigma * rng.standard_normal((B, g.action_space_size))).astype(np.float32)
    t = np.zeros((B, g.action_space_size), np.float32)
    for i in range(B):
        cols = rng.choice(g.action_space_size, 1 if target == "one_move" else int(rng.integers(2, 300)), replace=False)
        x = rng.uniform(0.0, 1.0, len(cols))
        t[i, cols] = (x / x.sum()).astype(np.float32)
    v = rng.uniform(-1.0, 1.0, (B, 1)).astype(np.float32)
    z = rng.choice(np.array([-1.0, 1.0, 0.02 * 37, -0.02 * 5], np.float32), B)
    learner = stub_learner(R)
    net = Given(torch.from_numpy(logits), torch.from_numpy(v))
    planes = torch.zeros((B, 24, R, R))
    loss, pl, vl = (float(x) for x in learner._loss(net, planes, torch.from_numpy(t), torch.from_numpy(z)))

    l64 = logits.astype(np.float64)
    m = l64.max(axis=1, keepdims=True)
    log_softmax = l64 - m - np.log(np.exp(l64 - m).sum(axis=1, keepdims=True))
    want_pl = float(np.mean(-(t.astype(np.float64) * log_softmax).sum(axis=1)))
    want_vl = float(np.mean((v[:, 0].astype(np.float64) - z.astype(np.float64)) ** 2))
    assert pl == pytest.approx(want_pl, rel=2e-6), (pl, want_pl)
    assert vl == pytest.approx(want_vl, rel=2e-6), (vl, want_vl)
    assert loss == pytest.approx(want_pl + want_vl, rel=2e-6), (loss, want_pl + want_vl)


# ---- ReplayStore against a plain ring ------------------------------------------------------------------------------

CAP, REC, KIDS = 7, 16, 5


def entry(i):
    """Replay entry number i (from 1): every field a distinct function of i, exact in its dtype."""
    board = np.zeros(REC, np.uint8)
    board[0], board[1], board[2:] = i & 0xFF, i >> 8, (i * 7) & 0xFF
    return (board, np.arange(KIDS, dtype=np.int32) + 10 * i, np.arange(KIDS, dtype=np.int32) + i, np.float32(0.5 * i),
            np.arange(KIDS, dtype=np.float32) * 0.25 + i)


class Ring:
    """A ring of CAP slots: a batch writes its entries one at a time at head, head advancing by one; of a batch longer
    than the ring only the last CAP entries are written."""

    def __init__(self):
        self.slots, self.head, self.size = [None] * CAP, 0, 0

    def add(self, entries):
        for e in entries[-CAP:]:
            self.slots[self.head] = e
            self.head = (self.head + 1) % CAP
            self.size = min(CAP, self.size + 1)


@pytest.mark.parametrize("sizes", [[0, 1, CAP - 1, 3, 5, 0, CAP, CAP + 4, 2, 3 * CAP + 1, 1], [CAP + 2, 1, CAP - 1],
                                   [CAP, CAP - 1, 2]])
@pytest.mark.parametrize("with_policy", [False, True])
def test_replay_store_against_a_ring(sizes, with_policy):
    torch.manual_seed(0)
    store = ReplayStore(CAP, REC, KIDS, "cpu", child_policy=with_policy)
    ring, history, n = Ring(), [], 0
    for m in sizes:
        batch = [entry(n + j + 1) for j in range(m)]
        n += m
        history += batch
        cols = [np.stack([e[f] for e in batch]) if m else np.zeros((0,) + np.shape(entry(1)[f]), entry(1)[f].dtype)
                for f in range(5)]
        store.add(*(torch.from_numpy(c) for c in cols[:4]), torch.from_numpy(cols[4]) if with_policy else None)
        ring.add(batch)
        assert (store.size, store.head, len(store)) == (ring.size, ring.head, ring.size), m
        fields = [store.boards, store.child_flat, store.child_visits, store.value]
        fields += [store.child_policy] if with_policy else []
        for s, e in enumerate(ring.slots):
            for f, t in enumerate(fields):
                want = e[f] if e is not None else np.zeros_like(entry(1)[f])
                assert np.array_equal(t[s].numpy(), want), (m, s, f)
        # the live slots, oldest first from head - size, are the last `size` entries added
        for j, e in enumerate(history[len(history) - ring.size:]):
            assert np.array_equal(store.boards[(ring.head - ring.size + j) % CAP].numpy(), e[0])
        if ring.size == 0:
            continue
        out = store.sample(400)
        assert len(out) == (5 if with_policy else 4)
        live = {int(e[0][0]) | int(e[0][1]) << 8: e for e in ring.slots if e is not None}
        drawn = set()
        for r in range(400):
            i = int(out[0][r, 0]) | int(out[0][r, 1]) << 8
            assert i in live, (m, i)
            drawn.add(i)
            for f in range(len(out)):
                assert np.array_equal(out[f][r].numpy(), live[i][f]), (m, r, f)
        assert drawn == set(live), (m, sorted(drawn), sorted(live))
