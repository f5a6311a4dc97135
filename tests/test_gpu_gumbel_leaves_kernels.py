"""-m gpu: the leaf-parallel Gumbel kernels (fpc_tree_select_gumbel_leaves, fpc_tree_gumbel_result_leaves) on the
hand-built, sentinel-filled slabs of tests/test_gpu_gumbel_kernels.py, one launch at a time.

- At L = 1 the select, root-only and interior, must write what fpc_tree_select_gumbel / _interior write in every tree
  array, word for word, on root child counts 1, 2, 20, 38 and 300 at and around the schedule's phase boundaries, beside
  an unexpanded root, a dropped game and a root whose visits left the schedule; issued must gain exactly the chosen
  child's visit, in_flight carry the path's marks, and the slot the leaf.
- The result must equal fpc_tree_gumbel_result when I == N, and when a child lost a visit to a collision (I_i = N_i + 1)
  it must take its survivors from I: the restatement's choice over {I_i == max I}, with the policy from N.
- Refusals before any launch."""
import ctypes as C

import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200._lib import (FPC_ERR_ARG, FPC_MAX_MOVES, FPC_OK, SLOT_EMPTY, SLOT_LEAF,
                                                LeafBatchDesc)
from tests.gumbel_oracle import argmax_among, gumbels, logits_sigma, scores, warp_sum
from tests.test_gpu_gumbel_kernels import CASES, SEED, boundaries, build, desc, gumbel_result
from tests.test_gpu_puct_kernels import SENT_I32, STATE, bits, put, snapshot

pytestmark = pytest.mark.gpu

# what the sequential select writes for its leaf and the leaf batch writes per slot instead
LEAF_ROWS = ("leaf_boards", "leaf_flat", "leaf_counts", "leaf_status", "k")


class Batch:
    """A struct fpc_leaf_batch for tree t, sentinel-filled, plus issued."""

    def __init__(self, t, L, vl=1):
        n, dev = t.n, "cuda"
        i32 = dict(dtype=torch.int32, device=dev)
        self.in_flight = torch.zeros((n, t.node_cap), **i32)
        self.slot_node = torch.full((n * L,), SENT_I32, **i32)
        self.slot_kind = torch.full((n * L,), SENT_I32, **i32)
        self.boards = torch.zeros((n * L, t.geom.record_bytes), dtype=torch.uint8, device=dev)
        self.flat = torch.zeros((n * L, FPC_MAX_MOVES), **i32)
        self.counts = torch.zeros(n * L, **i32)
        self.status = torch.zeros(n * L, **i32)
        self.k = torch.zeros(n * L, **i32)
        self.priors = torch.zeros((n * L, FPC_MAX_MOVES), dtype=torch.float32, device=dev)
        self.collisions = torch.zeros(n, **i32)
        self.issued = torch.full((n, FPC_MAX_MOVES), SENT_I32, **i32)
        self.planes = torch.empty((n * L, 24, t.R, t.R), dtype=torch.float32, device=dev)
        d = LeafBatchDesc()
        d.L, d.virtual_loss = L, vl
        for field, name in (("in_flight", "in_flight"), ("slot_node", "slot_node"), ("slot_kind", "slot_kind"),
                            ("leaf_boards", "boards"), ("leaf_flat", "flat"), ("leaf_counts", "counts"),
                            ("leaf_status", "status"), ("k", "k"), ("priors", "priors"),
                            ("collisions", "collisions")):
            setattr(d, field, getattr(self, name).data_ptr())
        self.desc = d

    def select(self, t, gd, node_value=None, issued=True):
        rc = t.L.fpc_tree_select_gumbel_leaves(C.byref(t.desc), C.byref(gd) if gd is not None else None,
                                               C.byref(self.desc), self.issued.data_ptr() if issued else None,
                                               node_value.data_ptr() if node_value is not None else None, 0,
                                               self.planes.data_ptr(), 0, None, t._stream())
        torch.cuda.synchronize()
        return rc


def issued_from_visits(st, info):
    """I = N on every expanded root, the sentinel elsewhere."""
    out = np.full((len(info), FPC_MAX_MOVES), SENT_I32, np.int32)
    for g, d in enumerate(info):
        if d["k"]:
            out[g, :d["k"]] = st["visits"][g, d["fc"]: d["fc"] + d["k"]] - 1
    return out


@pytest.mark.parametrize("R", [8, 14])
@pytest.mark.parametrize("m,n_sims", [(1, 47), (4, 47), (16, 63), (300, 299)])
@pytest.mark.parametrize("interior", [False, True])
def test_one_slot_is_the_sequential_select_word_for_word(R, m, n_sims, interior):
    rng = np.random.default_rng(R * 1000 + m + n_sims + interior)
    n = len(CASES) * len(boundaries(m, n_sims))
    a, before, info, rv_a = build(R, n, rng, m, n_sims)
    b, _, _, _ = build(R, n, np.random.default_rng(0), m, n_sims)
    for name in STATE:
        put(b, name, before[name])
    rv_b = rv_a.clone()
    keys = torch.from_numpy(rng.integers(-2**63, 2**63 - 1, n, dtype=np.int64)).cuda()
    gd_a, gd_b = desc(keys, rv_a, m, n_sims), desc(keys, rv_b, m, n_sims)
    nv_a = nv_b = None
    if interior:  # planted values: the select must read and write the same entries on both sides
        nv = rng.normal(0.0, 1.0, (n, a.node_cap))
        nv_a, nv_b = torch.from_numpy(nv).cuda(), torch.from_numpy(nv).cuda()
        rc = a.L.fpc_tree_select_gumbel_interior(C.byref(a.desc), C.byref(gd_a), nv_a.data_ptr(), 0,
                                                 a.planes.data_ptr(), 0, None, a._stream())
    else:
        rc = a.L.fpc_tree_select_gumbel(C.byref(a.desc), C.byref(gd_a), 0, a.planes.data_ptr(), 0, None, a._stream())
    assert rc == FPC_OK
    batch = Batch(b, 1)
    issued0 = issued_from_visits(before, info)
    batch.issued.copy_(torch.from_numpy(issued0))
    assert batch.select(b, gd_b, nv_b) == FPC_OK
    got, want = snapshot(b), snapshot(a)
    for name in STATE:
        if name not in LEAF_ROWS:
            assert np.array_equal(got[name], want[name]), name
    assert np.array_equal(bits(rv_a), bits(rv_b))
    if interior:
        assert np.array_equal(bits(nv_a), bits(nv_b))
    leaf = want["leaf"]
    kind, node = batch.slot_kind.cpu().numpy(), batch.slot_node.cpu().numpy()
    issued, in_flight = batch.issued.cpu().numpy(), batch.in_flight.cpu().numpy()
    parent = want["parent"]
    for g, d in enumerate(info):
        if leaf[g] < 0:
            assert kind[g] == SLOT_EMPTY and node[g] == -1, g
            assert not in_flight[g].any()
            assert np.array_equal(issued[g], issued0[g]), g
            continue
        assert kind[g] == SLOT_LEAF and node[g] == leaf[g], g
        assert np.array_equal(bits(batch.boards[g]), want["leaf_boards"][g])
        assert batch.k[g] == want["k"][g]
        path, x = [], int(leaf[g])
        while x > 0:
            path.append(x)
            x = int(parent[g, x])
        path.append(0)
        marks = np.zeros(b.node_cap, np.int32)
        marks[path] = 1
        assert np.array_equal(in_flight[g], marks), g
        inc = issued0[g].copy()
        if len(path) > 1:  # the root child on the leaf's path gained its visit
            inc[path[-2] - d["fc"]] += 1
        assert np.array_equal(issued[g], inc), g
    assert not batch.collisions.any()
    print(f"R={R} m={m} n_sims={n_sims} interior={interior}: {n} games, {int((leaf >= 0).sum())} leaves")


def oracle_result(st, d, g, I, rv, key, scale=1.0):
    fc, k = d["fc"], d["k"]
    N = st["visits"][g, fc: fc + k] - 1
    vs = st["value_sum"][g, fc: fc + k].view(np.float64)
    prior = st["prior"][g, fc: fc + k].view(np.float32)
    root = st["value_sum"][g, 0:1].view(np.float64)[0] if int(N.sum()) == 0 else rv
    z, _ = logits_sigma(N, vs, prior, root)
    best = argmax_among(scores(z, gumbels(SEED, key, k, scale)), I == I.max())
    e = np.exp(z - z.max())
    return int(st["move_flat"][g, fc + best]), (e / warp_sum(e)).astype(np.float32)


@pytest.mark.parametrize("m,n_sims", [(4, 47), (16, 63)])
def test_result_takes_its_survivors_from_issued(m, n_sims):
    R = 14
    rng = np.random.default_rng(m + n_sims)
    n = len(CASES) * len(boundaries(m, n_sims))
    t, st, info, rv = build(R, n, rng, m, n_sims)
    keys = torch.from_numpy(rng.integers(-2**63, 2**63 - 1, n, dtype=np.int64)).cuda()
    gd = desc(keys, rv, m, n_sims)
    batch = Batch(t, 2)
    issued0 = issued_from_visits(st, info)

    def result_leaves():
        a = torch.full((n,), -7, dtype=torch.int32, device="cuda")
        p = torch.full((n, FPC_MAX_MOVES), -7.0, dtype=torch.float32, device="cuda")
        rc = t.L.fpc_tree_gumbel_result_leaves(C.byref(t.desc), C.byref(gd), batch.issued.data_ptr(), a.data_ptr(),
                                               p.data_ptr(), t._stream())
        torch.cuda.synchronize()
        return rc, a.cpu().numpy(), p.cpu().numpy()

    batch.issued.copy_(torch.from_numpy(issued0))
    rc, a0, p0 = gumbel_result(t, gd)
    assert rc == FPC_OK
    rc, a1, p1 = result_leaves()
    assert rc == FPC_OK and np.array_equal(a0, a1) and np.array_equal(bits(torch.from_numpy(p0)),
                                                                      bits(torch.from_numpy(p1)))
    # a child one visit short of the most visited lost a visit to a collision: under I it is a survivor too
    lost = issued0.copy()
    changed = 0
    for g, d in enumerate(info):
        k = d["k"]
        if k < 2:
            continue
        N = lost[g, :k].astype(np.int64)
        short = np.flatnonzero(N == N.max() - 1) if N.max() > 0 else []
        if len(short):
            lost[g, short[0]] += 1
            changed += 1
    batch.issued.copy_(torch.from_numpy(lost))
    rc, a2, p2 = result_leaves()
    assert rc == FPC_OK
    rvh = rv.cpu().numpy()
    for g, d in enumerate(info):
        if not d["k"]:
            assert a2[g] == -1 and not p2[g].any()
            continue
        flat, pol = oracle_result(st, d, g, lost[g, :d["k"]].astype(np.int64), rvh[g], int(keys[g]))
        assert a2[g] == flat, g
        np.testing.assert_allclose(p2[g, :d["k"]], pol, rtol=1e-6, atol=0)
        assert np.array_equal(p2[g], p1[g]), g  # the improved policy comes from N, not from I
    assert changed >= n // 4
    assert np.array_equal(snapshot(t)["visits"], st["visits"])


def test_refusals_before_any_launch():
    R, m, n_sims = 8, 4, 15
    rng = np.random.default_rng(5)
    t, st, info, rv = build(R, len(CASES), rng, m, n_sims)
    keys = torch.zeros(t.n, dtype=torch.int64, device="cuda")
    gd = desc(keys, rv, m, n_sims)
    batch = Batch(t, 2)
    assert batch.select(t, gd, issued=False) == FPC_ERR_ARG
    assert batch.select(t, None) == FPC_ERR_ARG
    for L, vl in ((0, 1), (257, 1), (2, 0)):
        batch.desc.L, batch.desc.virtual_loss = L, vl
        assert batch.select(t, gd) == FPC_ERR_ARG
    batch.desc.L, batch.desc.virtual_loss = 2, 1
    assert batch.select(t, desc(keys, rv, 0, n_sims)) == FPC_ERR_ARG
    a = torch.zeros(t.n, dtype=torch.int32, device="cuda")
    p = torch.zeros((t.n, FPC_MAX_MOVES), dtype=torch.float32, device="cuda")
    L_ = t.L
    assert L_.fpc_tree_gumbel_result_leaves(C.byref(t.desc), C.byref(gd), None, a.data_ptr(), p.data_ptr(), None) \
        == FPC_ERR_ARG
    assert L_.fpc_tree_gumbel_result_leaves(C.byref(t.desc), C.byref(gd), batch.issued.data_ptr(), None, p.data_ptr(),
                                            None) == FPC_ERR_ARG
    torch.cuda.synchronize()
    got = snapshot(t)
    for name in STATE:
        assert np.array_equal(got[name], st[name]), name
    assert (batch.slot_kind == SENT_I32).all() and (batch.issued == SENT_I32).all()
