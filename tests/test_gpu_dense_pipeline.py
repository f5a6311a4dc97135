"""-m gpu: the dense-output pipeline across kinds of call.

Tracked calls (each BatchedEnv has its own fpc_dense_track handle, one of them updates incrementally) and handle-less
fpc_observe / fpc_playout_step calls into tensors of their own, interleaved on one host thread and one stream, with
FPC_FLAG_ASYNC_DENSE on and off, planes-only, mask-only and both.  The handle-less batches grow mid-sequence, so the
library's records workspace is reallocated while an asynchronous expansion may still be running, and fpc_shutdown
drops the per-thread state midway.  After fpc_join every tensor must equal the same sequence run synchronously, bit
for bit, and a sample must equal the oracle."""
import functools

import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200 import _lib
from alphazero_4_player_chess_b200.env import BatchedEnv
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.geometry import GEOMETRIES
from tests.util import SEED, oracle_for

pytestmark = pytest.mark.gpu

R = 14
MAX_PLIES = 40          # short games, so finished slots are re-seeded along the way
STEPS = 12
SHUTDOWN_AT = 6
SIZES = (100, 300, 1000, 300)  # handle-less batch of steps 0-2, 3-5, 6-8, 9-11
VARIANTS = ((True, True), (True, False), (False, True))  # (planes, mask)


def _ptr(t):
    return None if t is None else t.data_ptr()


class Rig:
    """What one device holds: tracked envs `a` (full rewrites) and `b` (incremental), and one handle-less batch per
    size, whose tensors only the handle-less entry points write."""

    def __init__(self, device):
        self.device = torch.device(device)
        self.a = BatchedEnv(R, 512, self.device)
        self.b = BatchedEnv(R, 384, self.device)
        self.h = {n: BatchedEnv(R, n, self.device) for n in sorted(set(SIZES))}
        start = start_record("STANDARD", castling=True)
        for i, e in enumerate(self.envs()):
            e.reset_playout(start, first_game=10000 * i)
            e.planes_buffer().zero_()
            e.mask_buffer().zero_()

    def envs(self):
        return [self.a, self.b, *self.h.values()]

    def playout(self, e, planes=True, mask=True, async_dense=False):
        with torch.cuda.device(self.device):
            _lib.check(e.L.fpc_playout_step(
                R, e.boards.data_ptr(), e.n, SEED, e.game.data_ptr(), e.ply.data_ptr(), e.start.data_ptr(), MAX_PLIES,
                e.n, None, e.counts.data_ptr(), e.status.data_ptr(), _ptr(e.planes_buffer() if planes else None),
                None, -1, _ptr(e.mask_buffer() if mask else None), e.counters.data_ptr(), int(async_dense),
                e._stream()))

    def observe(self, e, planes=True, mask=True, async_dense=False):
        with torch.cuda.device(self.device):
            _lib.check(e.L.fpc_observe(
                R, e.boards.data_ptr(), e.n, None, None, e.counts.data_ptr(), e.status.data_ptr(),
                _ptr(e.planes_buffer() if planes else None), None, -1, _ptr(e.mask_buffer() if mask else None),
                int(async_dense), e._stream()))

    def shutdown(self):
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().fpc_shutdown())

    def join(self):
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().fpc_join(torch.cuda.current_stream(self.device).cuda_stream))
        torch.cuda.synchronize(self.device)


def calls(rig, asyn):
    """The calls of the whole sequence on one rig, in order.  With asyn, two of every three dense calls set
    FPC_FLAG_ASYNC_DENSE; without, none does."""
    a, b = rig.a, rig.b
    out = []

    def add(fn, **kw):
        out.append(functools.partial(fn, async_dense=asyn and len(out) % 3 != 2, **kw))

    for step in range(STEPS):
        if step == SHUTDOWN_AT:
            out.append(rig.shutdown)
        h = rig.h[SIZES[step // 3]]
        ph, mh = VARIANTS[step % 3]
        pa, ma = VARIANTS[(step + 1) % 3]
        pb, mb = VARIANTS[(step + 2) % 3]
        add(a.playout_step, seed=SEED, max_plies=MAX_PLIES)
        add(rig.playout, e=h)
        add(b.playout_step, seed=SEED, max_plies=MAX_PLIES, incremental=True)
        add(rig.observe, e=h, planes=ph, mask=mh)
        add(a.observe, planes=pa, mask=ma)
        add(b.observe, planes=pb, mask=mb, incremental=True)
    # last: both tensors of every env from its current boards, for the oracle
    add(a.observe)
    add(b.observe, incremental=True)
    for e in rig.h.values():
        add(rig.observe, e=e)
    return out


def run(devices, asyn):
    rigs = [Rig(f"cuda:{d}") for d in devices]
    sequences = [calls(r, asyn) for r in rigs]
    for k in range(len(sequences[0])):  # one call per device in turn
        for seq in sequences:
            seq[k]()
    for r in rigs:
        r.join()
    return rigs


def check_against_sync(devices):
    got, want = run(devices, asyn=True), run(devices, asyn=False)
    o, g = oracle_for(R), GEOMETRIES[R]
    for rg, rw in zip(got, want):
        for eg, ew in zip(rg.envs(), rw.envs()):
            for name in ("boards", "counts", "status", "game", "ply"):
                assert torch.equal(getattr(eg, name), getattr(ew, name)), (eg.n, name)
            assert torch.equal(eg.planes_buffer(), ew.planes_buffer()), eg.n
            assert torch.equal(eg.mask_buffer(), ew.mask_buffer()), eg.n
            rows = torch.arange(0, eg.n, 13)
            recs = eg.boards[rows].cpu().numpy()
            assert np.array_equal(eg.planes_buffer()[rows].cpu().numpy(),
                                  o.encode(recs, recs[:, g.off_turn].astype(np.int32))), eg.n
            assert np.array_equal(eg.mask_buffer()[rows].cpu().numpy(), o.mask(recs)), eg.n


def test_tracked_and_handle_less_calls_interleave():
    check_against_sync([0])


def test_tracked_and_handle_less_calls_interleave_on_two_devices():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible CUDA devices")
    check_against_sync([0, 1])
