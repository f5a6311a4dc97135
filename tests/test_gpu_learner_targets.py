"""-m gpu: the training data self-play produces, end to end.  SelfPlay's replays (plain, tree reuse, Gumbel) pass
through Learner.store / _batch, and each drawn mini-batch must hold the oracle's planes, the f64 restatement of the
targets (tests/test_learner_targets.py) and the replay's values.  Then the frame check through the CUDA kernels: a
network that has learned its targets exactly, searched by BatchedMCTS on the same positions, must give every root
child the prior the target meant for it -- which holds only if the encoder's rotation, tree_expand_backup_kernel's
un-rotation and the learner's placement agree.  Last, heuristic_kernel (the value of games cut off at
max_game_length) against the oracle on random positions."""
import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200._lib import FPC_MAX_MOVES
from alphazero_4_player_chess_b200.env import BatchedEnv
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.geometry import GEOMETRIES, KING, PAWN
from alphazero_4_player_chess_b200.mcts import BatchedMCTS
from alphazero_4_player_chess_b200.selfplay import SelfPlay
from alphazero_4_player_chess_b200.train import Learner
from tests.golden.fake_net import FakeNet
from tests.test_gpu_puct_kernels import START
from tests.test_learner_targets import legal_flats, normalised, synthetic_children, targets_f64
from tests.util import oracle_for, random_positions

pytestmark = pytest.mark.gpu

# the configurations of tests/test_gpu_selfplay.py: name -> (R, games, max_game_length)
CONFIGS = {"EIGHT_SIMPLE": (8, 24, 40), "STANDARD": (14, 8, 6)}
MODES = {"plain": {}, "reuse": {"reuse_tree": True},
         "gumbel": {"gumbel": True, "gumbel_seed": 0xB0A7, "gumbel_considered": 8}}
ARGS = {"C": 3, "num_searches": 12, "temperature": 1.1, "heuristic_weight": 0.02, "batch_size": 64,
        "replay_buffer_capacity": 4096, "validation_buffer_capacity": 1024}
FIELDS = ("boards", "child_flat", "child_visits", "value", "child_policy")
PRIOR_RTOL = 4e-6  # the logits are log(f32 target) rounded to f32: half an ulp of |log t| <= 70 is 3.8e-6 relative


@pytest.fixture(scope="module")
def runs():
    """(SelfPlay, replay) per (name, mode), played once for the module."""
    cache = {}

    def get(name, mode):
        if (name, mode) not in cache:
            R, n, T = CONFIGS[name]
            torch.manual_seed(1234)
            sp = SelfPlay(R, n, FakeNet(R, device="cuda"), dict(ARGS, max_game_length=T), start_record(name),
                          **MODES[mode])
            cache[name, mode] = (sp, sp.play())
        return cache[name, mode]

    yield get
    cache.clear()


def host_rows(d):
    """Each row of a replay-like dict of tensors / arrays as one bytes key over every field it has."""
    cols = [np.asarray(d[f].cpu() if torch.is_tensor(d[f]) else d[f]) for f in FIELDS if f in d]
    return [b"".join(c[i].tobytes() for c in cols) for i in range(len(cols[0]))]


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("name", list(CONFIGS))
def test_learner_batches_are_the_replay_in_the_networks_frame(runs, name, mode):
    sp, replay = runs(name, mode)
    R, g = sp.R, sp.geom
    o = oracle_for(R)
    gumbel = mode == "gumbel"
    m = replay["boards"].shape[0]
    assert m > 0 and ("child_policy" in replay) == gumbel
    recs = replay["boards"].cpu().numpy()
    assert set(recs[:, g.off_turn]) == {0, 1, 2, 3}
    flat = replay["child_flat"].cpu().numpy()
    weights = replay["child_policy" if gumbel else "child_visits"].cpu().numpy()
    np.testing.assert_allclose(sp.policy_targets(replay).cpu().numpy(), targets_f64(R, recs, flat, weights),
                               rtol=2e-6, atol=0)

    learner = Learner(sp, torch.nn.Linear(1, 1), torch.optim.SGD([torch.zeros(1, requires_grad=True)], lr=0.0), ARGS)
    assert (learner.train_buf.child_policy is not None) == gumbel
    torch.manual_seed(5)
    learner.store(replay)
    assert len(learner.train_buf) + len(learner.valid_buf) == m
    rows = set(host_rows(replay))
    drawn_any = 0
    for buf in (learner.train_buf, learner.valid_buf):
        if len(buf) == 0:
            continue
        drawn = []
        sample = buf.sample

        def recorded(batch, _sample=sample):
            out = _sample(batch)
            drawn.append([t.cpu().numpy() for t in out])
            return out

        buf.sample = recorded
        planes, targets, value = learner._batch(buf)
        torch.cuda.synchronize()
        (d,) = drawn
        got = dict(zip(FIELDS, d))
        assert all(r in rows for r in host_rows(got)), "a drawn entry is not a replay entry"
        boards = got["boards"]
        assert np.array_equal(planes.cpu().numpy(), o.encode(boards, boards[:, g.off_turn].astype(np.int32)))
        w = got["child_policy" if gumbel else "child_visits"]
        np.testing.assert_allclose(targets.cpu().numpy(), targets_f64(R, boards, got["child_flat"], w), rtol=2e-6,
                                   atol=0)
        assert np.array_equal(value.cpu().numpy(), got["value"])
        drawn_any += len(boards)
    assert drawn_any >= ARGS["batch_size"]


class LearnedNet:
    """A network that has learned its targets exactly: asserts that it is shown `planes`, and returns
    log(max(target, 1e-30)) per row and value 0."""

    def __init__(self, planes, targets):
        self.planes, self.logits = planes, torch.log(targets.clamp_min(1e-30))
        self.calls = 0

    def __call__(self, planes):
        assert torch.equal(planes, self.planes), "the search's planes are not the learner's"
        self.calls += 1
        return self.logits, torch.zeros((planes.shape[0], 1), device=planes.device)


def check_frame(sp, replay):
    """One simulation of BatchedMCTS(batch_rotation=False) on the replay's positions, with the network that returns
    the learner's targets: every root child with non-zero weight gets its normalised weight as prior.  Returns the
    largest relative error."""
    R, g = sp.R, sp.geom
    recs = replay["boards"].cpu().numpy()
    n = len(recs)
    planes = sp.encoded_states(replay).clone()
    net = LearnedNet(planes, sp.policy_targets(replay))
    m = BatchedMCTS(R, n, net, {"C": 3, "num_searches": 1}, node_cap=1 + FPC_MAX_MOVES)
    m.search(replay["boards"])
    torch.cuda.synchronize()
    assert net.calls == 1
    flat, _, prior, cnt = (x.cpu().numpy() for x in m.root_children())
    cflat = replay["child_flat"].cpu().numpy()
    weights = replay["child_policy" if "child_policy" in replay else "child_visits"].cpu().numpy()
    worst = 0.0
    for i in range(n):
        share = normalised(weights[i])
        live = share > 0
        assert live.any(), i
        kids = dict(zip(flat[i, :cnt[i]].tolist(), prior[i, :cnt[i]].astype(np.float64).tolist()))
        assert set(kids) == set(legal_flats(R, recs[i]).tolist()), i
        got = np.array([kids[int(f)] for f in cflat[i][live]])
        np.testing.assert_allclose(got, share[live], rtol=PRIOR_RTOL, atol=0, err_msg=f"entry {i}, k {recs[i][g.off_turn]}")
        assert got.sum() >= 1 - 1e-5, i
        worst = max(worst, float(np.max(np.abs(got - share[live]) / share[live])))
    return worst


def distinct(replay):
    """The replay's entries at distinct positions (a position can recur across games with other visits)."""
    _, first = np.unique(replay["boards"].cpu().numpy(), axis=0, return_index=True)
    idx = torch.from_numpy(np.sort(first)).to(replay["boards"].device)
    return {f: replay[f][idx] for f in FIELDS if f in replay}


@pytest.mark.parametrize("mode", ["plain", "gumbel"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_search_reads_selfplay_targets_as_the_moves_they_weigh(runs, name, mode):
    sp, replay = runs(name, mode)
    sub = distinct(replay)
    assert set(sub["boards"][:, sp.geom.off_turn].tolist()) == {0, 1, 2, 3}
    worst = check_frame(sp, sub)
    print(f"{name} {mode}: {len(sub['boards'])} positions, max relative prior error {worst:.2e}")


@pytest.mark.parametrize("source", ["visits", "gumbel"])
@pytest.mark.parametrize("R", [10, 13])
def test_search_reads_synthetic_targets_as_the_moves_they_weigh(R, source):
    """Random positions (every colour to move, all piece types), the oracle's legal flats in random order as the
    children, random visits with zeros or an f32 soft-max row as the weights."""
    g = GEOMETRIES[R]
    o = oracle_for(R)
    recs = random_positions(R, 160, seed=100 + R)
    recs = recs[[o.game_result(r)[0] == 0 and len(legal_flats(R, r)) > 0 for r in recs]]
    flat, w = synthetic_children(R, recs, np.random.default_rng(R), source)
    keep = w.astype(np.float64).sum(axis=1) > 0
    recs, flat, w = recs[keep], flat[keep], w[keep]
    assert set(recs[:, g.off_turn]) == {0, 1, 2, 3}
    replay = {"boards": torch.from_numpy(recs).cuda(), "child_flat": torch.from_numpy(flat).cuda(),
              "child_visits" if source == "visits" else "child_policy": torch.from_numpy(w).cuda()}
    sp = SelfPlay(R, 1, None, dict(ARGS, max_game_length=1), start_record(START[R]))
    worst = check_frame(sp, replay)
    print(f"R={R} {source}: {len(recs)} positions, max relative prior error {worst:.2e}")


@pytest.mark.parametrize("R", [8, 10, 13, 14])
def test_heuristic_kernel_matches_the_oracle_on_random_positions(R):
    g = GEOMETRIES[R]
    o = oracle_for(R)
    recs = random_positions(R, 512, seed=200 + R)
    pieces = recs[:, :g.nsq]
    present = pieces[(pieces & 0x80) != 0]
    for team in (0, 1):
        types = {int(p >> 2) & 7 for p in present if (p >> 5) & 1 == team}
        assert types == set(range(PAWN, KING + 1)), team
    assert (recs[:, g.off_king:g.off_king + 4] == g.nsq).any(), "no position with a king missing"
    env = BatchedEnv(R, len(recs))
    env.load(recs)
    got = env.heuristic().cpu().numpy()
    want = np.array([o.heuristic(r, int(r[g.off_turn]) & 1) for r in recs])
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:8]
