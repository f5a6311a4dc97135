"""-m gpu: the rules kernel on crowded positions (tests/util.crowded_bands), up to and past the 300-move buffer, against
the oracle's full legal list (Oracle.legal_moves_wide), bit-exact as in test_gpu_parity.py.

At most 300 legal moves: counts, moves, flats, result and status flags, planes, mask, the boards after every legal move,
heuristic, attack maps and one playout step.  More than 300 legal moves: the overflow contract of include/fpc.h
(FPC_STATUS_OVERFLOW)."""
import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200 import _lib
from alphazero_4_player_chess_b200.env import BatchedEnv
from alphazero_4_player_chess_b200.geometry import GEOMETRIES
from tests.util import CROWDED_BANDS, SEED, crowded_bands, crowded_positions, mixed_positions, oracle_for

pytestmark = pytest.mark.gpu
R_SIZES = [14, 13]


def crowded(R, over: bool):
    """The band records with more (over) or at most 300 legal moves, concatenated."""
    bands = crowded_bands(R)
    print(f"R={R} band counts:", {b: len(bands[b]) for b in CROWDED_BANDS})
    o = oracle_for(R)
    recs = np.concatenate([bands[b] for b in CROWDED_BANDS])
    keep = [(len(o.legal_moves_wide(r)[0]) > 300) == over for r in recs]
    return np.ascontiguousarray(recs[keep])


def oracle_mask(o, recs, lists):
    out = np.zeros((len(recs), o.A * o.nsq), dtype=np.float32)
    for i, moves in enumerate(lists):
        out[i, [o.move_flat_index(m) for m in moves]] = 1.0
    return out.reshape(len(recs), o.A, o.R, o.R)


def observe(R, recs):
    env = BatchedEnv(R, len(recs))
    env.load(recs)
    env.observe(planes=True, mask=True, moves=True, flat=True)
    torch.cuda.synchronize()
    return env


@pytest.mark.parametrize("R", R_SIZES)
def test_crowded_lists_flags_and_dense_outputs(R):
    g = GEOMETRIES[R]
    o = oracle_for(R)
    recs = crowded(R, over=False)
    n = len(recs)
    env = observe(R, recs)
    counts, status = env.counts.cpu().numpy(), env.status.cpu().numpy()
    moves = env.moves_buffer().cpu().numpy().view(np.uint64)
    flat = env.flat_buffer().cpu().numpy()
    lists = []
    for i in range(n):
        want, _ = o.legal_moves_wide(recs[i])
        lists.append(want)
        assert counts[i] == len(want) and (moves[i, : len(want)] == want).all(), i
        assert flat[i, : len(want)].tolist() == [o.move_flat_index(m) for m in want], i
        turn = int(recs[i][g.off_turn]) & 3
        kc = any((int(m) >> 16) & 0x80 and ((int(m) >> 18) & 7) == 5 for m in want)
        chk = o.king_in_check(recs[i], turn)
        want_status = (3 if not chk else (2 if turn & 1 == 0 else 1)) if len(want) == 0 else 0
        want_status |= (_lib.STATUS_CAN_TAKE_KING if kc else 0) | (0x1000 if chk else 0)
        want_status |= 0x100 if chk and len(want) == 0 else 0
        assert status[i] == want_status, (i, hex(status[i]), hex(want_status))
    assert max(counts) == 300
    turns = recs[:, g.off_turn].astype(np.int32)
    assert np.array_equal(env.planes_buffer().cpu().numpy(), o.encode(recs, turns))
    assert np.array_equal(env.mask_buffer().cpu().numpy(), oracle_mask(o, recs, lists))
    for k in range(4):
        assert np.array_equal(env.encode(k=k).cpu().numpy(), o.encode(recs, k))
    kt = torch.arange(n, dtype=torch.int32, device="cuda") % 4
    assert np.array_equal(env.encode(k=kt).cpu().numpy(), o.encode(recs, kt.cpu().numpy()))
    # heuristic of the team to move, attack maps
    assert env.heuristic().cpu().numpy().tolist() == [o.heuristic(r, int(r[g.off_turn]) & 1) for r in recs]
    d = torch.as_tensor(recs).cuda()
    amap = torch.empty((n, g.nsq), dtype=torch.uint8, device="cuda")
    _lib.check(_lib.lib().fpc_attack_maps(R, d.data_ptr(), n, amap.data_ptr(), torch.cuda.current_stream().cuda_stream))
    got = amap.cpu().numpy()
    for i in range(n):
        assert np.array_equal(got[i], o.attack_map(recs[i])), i


@pytest.mark.parametrize("R", R_SIZES)
def test_crowded_boards_after_every_legal_move(R):
    """fpc_make_moves (full move) and fpc_make_index (index-built) on every legal move of every position."""
    o = oracle_for(R)
    L = _lib.lib()
    recs = crowded(R, over=False)
    parents, full, idx = [], [], []
    for r in recs:
        for m in o.legal_moves_wide(r)[0]:
            parents.append(r)
            full.append(m)
            idx.append(o.move_flat_index(m))
    parents = np.stack(parents)
    n = len(full)
    d_par = torch.as_tensor(parents).cuda()
    d_mv = torch.as_tensor(np.array(full, dtype=np.uint64).view(np.int64)).cuda()
    d_ix = torch.as_tensor(np.array(idx, dtype=np.int32)).cuda()
    out, err = torch.empty_like(d_par), torch.zeros(n, dtype=torch.int32, device="cuda")
    _lib.check(L.fpc_make_moves(R, d_par.data_ptr(), d_mv.data_ptr(), n, out.data_ptr(), err.data_ptr(), None))
    got = out.cpu().numpy()
    assert not err.any()
    for i in range(n):
        assert np.array_equal(got[i], o.make_move(parents[i], full[i])), i
    _lib.check(L.fpc_make_index(R, d_par.data_ptr(), d_ix.data_ptr(), n, out.data_ptr(), err.data_ptr(), None))
    got = out.cpu().numpy()
    assert not err.any()
    for i in range(n):
        assert np.array_equal(got[i], o.make_index(parents[i], idx[i])), i
    print(f"R={R}: {n} moves from {len(recs)} positions")


@pytest.mark.parametrize("R", R_SIZES)
def test_crowded_playout_step(R):
    """One fpc_playout_step: the move played is the oracle's mix-picked index into the full canonical list."""
    o = oracle_for(R)
    recs = crowded(R, over=False)
    n = len(recs)
    env = BatchedEnv(R, n)
    env.reset_playout(recs[0])
    env.load(recs)
    env.playout_step(seed=SEED, max_plies=1000, planes=False, mask=False, chosen=True)
    torch.cuda.synchronize()
    chosen = env.chosen.cpu().numpy().view(np.uint64)
    boards, counts = env.boards.cpu().numpy(), env.counts.cpu().numpy()
    for i in range(n):
        want, _ = o.legal_moves_wide(recs[i])
        assert counts[i] == len(want), i
        if len(want) == 0:
            continue
        pick = ((o.mix(SEED, i, 0) >> 32) * len(want)) >> 32
        assert chosen[i] == want[pick], i
        assert np.array_equal(boards[i], o.make_move(recs[i], want[pick])), i


@pytest.mark.parametrize("R", R_SIZES)
def test_overflow_contract(R):
    """More than 300 legal moves: STATUS_OVERFLOW set exactly there, counts <= 300, the listed moves and flats a strictly
    ascending subset of the canonical list, the mask at exactly the listed flats, CAN_TAKE_KING and CHECK those of the
    full list.  Below 300 (mixed in) no overflow.  At 14x14 at least one position must have its only king captures in a
    dropped generation round, so that the flag is seen to come from the full list."""
    g = GEOMETRIES[R]
    o = oracle_for(R)
    over = crowded(R, over=True)
    recs = np.concatenate([over, crowded_positions(R, 256, seed=5)])
    env = observe(R, recs)
    counts, status = env.counts.cpu().numpy(), env.status.cpu().numpy()
    moves = env.moves_buffer().cpu().numpy().view(np.uint64)
    flat = env.flat_buffer().cpu().numpy()
    mask = env.mask_buffer().cpu().numpy().reshape(len(recs), -1)
    dropped_capture = 0
    for i, rec in enumerate(recs):
        want, _ = o.legal_moves_wide(rec)
        assert bool(status[i] & _lib.STATUS_OVERFLOW) == (len(want) > 300), i
        assert counts[i] <= 300
        got = moves[i, : counts[i]]
        keys = [o.move_flat_index(m) * 8 + ((int(m) >> 24) & 0xff) for m in got]
        assert all(a < b for a, b in zip(keys, keys[1:])), i
        assert set(got.tolist()) <= set(want.tolist()), i
        assert flat[i, : counts[i]].tolist() == [o.move_flat_index(m) for m in got], i
        assert np.flatnonzero(mask[i]).tolist() == sorted(set(flat[i, : counts[i]].tolist())), i
        turn = int(rec[g.off_turn]) & 3
        takers = [m for m in want if (int(m) >> 16) & 0x80 and ((int(m) >> 18) & 7) == 5]
        assert bool(status[i] & _lib.STATUS_CAN_TAKE_KING) == bool(takers), i
        assert bool(status[i] & 0x1000) == o.king_in_check(rec, turn), i
        assert (status[i] & 3) == 0 or len(want) <= 300
        if len(want) > 300:
            assert counts[i] < len(want)
            dropped_capture += bool(takers) and not set(int(m) for m in takers) & set(got.tolist())
    assert len(over) > 0
    # the hand-built late king captures (none at 13x13) put a king capture in a dropped round
    assert dropped_capture > 0 or len(crowded_bands(R)["late king capture"]) == 0
    print(f"R={R}: {len(over)} positions past 300 legal moves, {dropped_capture} with every king capture dropped")


@pytest.mark.parametrize("R", R_SIZES)
def test_incremental_update_crowded_and_sparse(R):
    """FPC_FLAG_INCREMENTAL through fpc_observe_tracked: every slot alternates between a crowded position (up to 300 mask
    entries, or a partial list past 300) and a sparse one, call after call; each call equals a full rewrite."""
    name = {14: "STANDARD", 13: "THIRTEEN"}[R]
    dense = np.concatenate([crowded(R, over=False), crowded(R, over=True)])
    n = len(dense)
    sparse = mixed_positions(name, n)[:n]
    a, b = BatchedEnv(R, n), BatchedEnv(R, n)
    a.planes_buffer().fill_(7.0)
    a.mask_buffer().fill_(7.0)
    for call in range(6):
        recs = np.where((np.arange(n)[:, None] + call) % 2 == 0, dense, sparse) if call % 3 else \
            (dense if call % 2 == 0 else sparse)
        recs = np.ascontiguousarray(recs)
        a.load(recs)
        b.load(recs)
        a.observe(planes=True, mask=True, incremental=True)
        b.observe(planes=True, mask=True)
        torch.cuda.synchronize()
        assert torch.equal(a.planes_buffer(), b.planes_buffer()), call
        assert torch.equal(a.mask_buffer(), b.mask_buffer()), call
        assert torch.equal(a.counts, b.counts) and torch.equal(a.status, b.status), call
