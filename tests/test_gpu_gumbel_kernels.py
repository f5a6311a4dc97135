"""-m gpu: the Gumbel root search's kernels (fpc_tree_select_gumbel, fpc_tree_gumbel_result) on hand-built,
sentinel-filled slabs, one launch at a time, against the numpy restatement of include/fpc.h (tests/gumbel_oracle.py).

Root child counts 1, 2, 20, 38 and 300 (children not starting at node 1, some with expanded subtrees below them), with
visits laid out along the halving schedule at and around its phase boundaries, beside an unexpanded root, a dropped game
and a root whose visits left the schedule.  The select must take the restatement's root child and then descend exactly
as fpc_tree_select does from that child: a twin tree whose root keeps only the chosen child, run through
fpc_tree_select, must end with the same words everywhere.  root_value must be written exactly where s == 0, and the
result's actions must equal the restatement's and its policy match within rtol 1e-6."""
import ctypes as C

import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200._lib import FPC_ERR_ARG, FPC_MAX_MOVES, FPC_OK, GumbelDesc, TreeDesc
from alphazero_4_player_chess_b200.mcts import ERR_NO_CHILD
from tests.gumbel_oracle import C_SCALE, C_VISIT, considered_visits, result, root_choice
from tests.test_gpu_puct_kernels import NODE_I32, SENT_F64, STATE, new_tree, put, snapshot

pytestmark = pytest.mark.gpu

NODE_CAP = 420
CASES = [("k1", 1), ("k2", 2), ("k20", 20), ("k38", 38), ("k300", 300), ("unexpanded", 0), ("dropped", 20),
         ("off", 2)]
SEED = 0x5EEDF00D


def boundaries(m, n_sims):
    """Simulation indices at and around the schedule's phase boundaries, and past n_sims."""
    if m <= 1:
        return [0, 1, n_sims - 1, n_sims, n_sims + 2]
    out, s, c, l2 = [0, 1], 0, m, (m - 1).bit_length()
    while s <= n_sims:
        s += max(1, n_sims // (l2 * c)) * c
        out += [s - 1, s, s + 1]
        c = max(2, c // 2)
    return sorted({x for x in out + [n_sims - 1, n_sims] if x >= 0})


def on_schedule(rng, k, m, n_sims, s):
    """Root visits N after s simulations that followed the schedule (candidates ranked by a random order)."""
    rank, N = rng.permutation(k), np.zeros(k, np.int64)
    for t in range(s):
        cand = np.flatnonzero(N == considered_visits(t, min(m, k), n_sims))
        N[cand[np.argmin(rank[cand])]] += 1
    return N


def build(R, n, rng, m, n_sims, cases=CASES, s_list=None, fc_list=None):
    """n games, game g of case cases[g % len(cases)] at s = s_list[g // len(cases) % len(s_list)].  Every node is
    materialised on board slot 0 (the start position); a few root children carry a subtree of three children.  Returns
    (tree, state, per-game info dicts, root_value [n] f64 on the device)."""
    t = new_tree(R, n, NODE_CAP)
    st = snapshot(t)
    s_list = s_list or boundaries(m, n_sims)
    root_value = np.full(n, SENT_F64, np.int64).view(np.float64)
    info = []
    for g in range(n):
        case, k = cases[g % len(cases)]
        s = s_list[(g // len(cases)) % len(s_list)]
        fc = fc_list[g] if fc_list is not None else 1 + int(rng.integers(0, 20))
        if case == "off":
            N = np.array([3, 0])
        elif k:
            N = on_schedule(rng, k, m, n_sims, min(s, 3 * k + n_sims))
        else:
            N = np.zeros(0, np.int64)
        used = fc + k
        for name in NODE_I32:
            st[name][g, :used + 12] = rng.integers(-1, used, used + 12)
        st["board_idx"][g, :used + 12] = 0
        st["n_children"][g, :used + 12] = 0
        st["first_child"][g, :used + 12] = 0
        st["parent"][g, 1:fc] = 0
        st["value_sum"][g, :used + 12] = rng.normal(0.0, 3.0, used + 12).view(np.int64)
        st["prior"][g, :used + 12] = rng.uniform(1e-4, 1.0, used + 12).astype(np.float32).view(np.int32)
        st["visits"][g, 0] = 1 + int(N.sum())
        if k:
            st["first_child"][g, 0], st["n_children"][g, 0] = fc, k
            st["parent"][g, fc:used] = 0
            st["visits"][g, fc:used] = N + 1
            q = rng.uniform(-1.0, 1.0, k)
            st["value_sum"][g, fc:used] = np.where(N > 0, q * N, 0.0).view(np.int64)
            visited = np.flatnonzero(N > 0)
            for j, c in enumerate(rng.permutation(visited)[:3]):  # subtrees below some visited children
                gc = used + 3 * j
                st["first_child"][g, fc + c], st["n_children"][g, fc + c] = gc, 3
                st["parent"][g, gc: gc + 3] = fc + c
                st["visits"][g, gc: gc + 3] = rng.integers(1, 4, 3)
        st["n_nodes"][g] = used + 12
        st["dropped"][g] = case == "dropped"
        if k and int(N.sum()) > 0:
            root_value[g] = rng.normal(0.0, 1.0)
        info.append(dict(case=case, k=k, fc=fc, s=int(N.sum())))
    st["leaf"][:] = rng.integers(-1, 50, n)
    st["error"][:] = 0
    for name in STATE:
        put(t, name, st[name])
    return t, snapshot(t), info, torch.from_numpy(root_value).cuda()


def desc(keys, root_value, m, n_sims, scale=1.0, seed=SEED):
    """A struct fpc_gumbel over the caller's tensors, which must outlive it."""
    d = GumbelDesc()
    d.seed, d.keys, d.root_value = seed, keys.data_ptr() if keys is not None else None, \
        root_value.data_ptr() if root_value is not None else None
    d.max_considered, d.n_sims, d.scale, d.c_visit, d.c_scale = m, n_sims, scale, C_VISIT, C_SCALE
    return d


def select(t, gd, tree_desc=None):
    rc = t.L.fpc_tree_select_gumbel(C.byref(tree_desc if tree_desc is not None else t.desc),
                                    C.byref(gd) if gd is not None else None, 0, t.planes.data_ptr(), 0, None,
                                    t._stream())
    torch.cuda.synchronize()
    return rc


def gumbel_result(t, gd, tree_desc=None, action=True, policy=True):
    a = torch.full((t.n,), -7, dtype=torch.int32, device="cuda")
    p = torch.full((t.n, FPC_MAX_MOVES), -7.0, dtype=torch.float32, device="cuda")
    rc = t.L.fpc_tree_gumbel_result(C.byref(tree_desc if tree_desc is not None else t.desc), C.byref(gd),
                                    a.data_ptr() if action else None, p.data_ptr() if policy else None, t._stream())
    torch.cuda.synchronize()
    return rc, a.cpu().numpy(), p.cpu().numpy()


def expected(st, info, g, rv, key, m, n_sims, scale=1.0):
    """(root choice index or -1, N) of game g by the restatement; rv = root_value as the select reads it."""
    fc, k = info[g]["fc"], info[g]["k"]
    N = st["visits"][g, fc: fc + k] - 1
    vs = st["value_sum"][g, fc: fc + k].view(np.float64)
    prior = st["prior"][g, fc: fc + k].view(np.float32)
    root = st["value_sum"][g, 0:1].view(np.float64)[0] if int(N.sum()) == 0 else rv
    return root_choice(N, vs, prior, root, SEED, key, m, n_sims, scale)[0], (N, vs, prior, root)


@pytest.mark.parametrize("R", [8, 14])
@pytest.mark.parametrize("m,n_sims", [(1, 47), (4, 47), (16, 63), (300, 299)])
def test_select_and_result_against_the_restatement(R, m, n_sims):
    rng = np.random.default_rng(R * 1000 + m + n_sims)
    n = len(CASES) * len(boundaries(m, n_sims))
    t, before, info, rv = build(R, n, rng, m, n_sims)
    keys = torch.from_numpy(rng.integers(-2**63, 2**63 - 1, n, dtype=np.int64)).cuda()
    rv_before = rv.cpu().numpy().copy()
    gd = desc(keys, rv, m, n_sims)
    # the twin: fpc_tree_select on the same slabs, each root cut down to the child the restatement chooses
    twin, _, _, _ = build(R, n, np.random.default_rng(0), m, n_sims)
    twin_st = {name: before[name].copy() for name in STATE}
    want_error = before["error"].copy()
    chosen = 0
    for g, d in enumerate(info):
        if d["case"] in ("dropped", "unexpanded"):
            continue
        i, _ = expected(before, info, g, rv_before[g], int(keys[g]), m, n_sims)
        if i < 0:
            assert d["case"] == "off" and m > 1
            twin_st["dropped"][g] = 1
            want_error[g] |= ERR_NO_CHILD
        else:
            twin_st["first_child"][g, 0], twin_st["n_children"][g, 0] = d["fc"] + i, 1
            chosen += 1
    for name in STATE:
        put(twin, name, twin_st[name])
    assert select(t, gd) == FPC_OK
    twin.select()
    got, want = snapshot(t), snapshot(twin)
    for name in STATE:
        if name in ("first_child", "n_children"):
            assert np.array_equal(got[name], before[name]), name
        elif name == "error":
            assert np.array_equal(got[name], want_error)
        else:
            assert np.array_equal(got[name], want[name]), name
    assert torch.equal(t.planes, twin.planes)
    # root_value: written exactly on the live games whose root is expanded with s == 0
    rv_got = rv.cpu().numpy()
    for g, d in enumerate(info):
        if d["case"] not in ("dropped", "unexpanded") and d["s"] == 0:
            assert rv_got[g].view(np.int64) == before["value_sum"][g, 0]
        else:
            assert rv_got[g].view(np.int64) == rv_before[g].view(np.int64), g
    # the result, on the slabs as the select left them
    st = snapshot(t)
    rc, action, policy = gumbel_result(t, gd)
    assert rc == FPC_OK
    after = snapshot(t)
    for name in STATE:
        assert np.array_equal(after[name], st[name]), name
    for g, d in enumerate(info):
        if d["k"] == 0:
            assert action[g] == -1 and not policy[g].any()
            continue
        N, vs, prior, root = expected(st, info, g, rv_got[g], int(keys[g]), m, n_sims)[1]
        i, pol = result(N, vs, prior, root, SEED, int(keys[g]), 1.0)
        assert action[g] == st["move_flat"][g, d["fc"] + i], (g, d)
        np.testing.assert_allclose(policy[g, :d["k"]], pol, rtol=1e-6, atol=0, err_msg=str(g))
        assert not policy[g, d["k"]:].any()
    print(f"R={R} m={m} n_sims={n_sims}: {n} games, {chosen} root choices, s in {boundaries(m, n_sims)}")


def test_scale_zero_and_a_key_gives_the_same_choice_at_any_place_in_the_batch():
    R, rng = 14, np.random.default_rng(5)
    case, s = [("k38", 38)], [9]
    t8, st8, info8, rv8 = build(R, 8, rng, 16, 63, case, s, fc_list=[7] * 8)
    t1, _, info1, rv1 = build(R, 1, rng, 16, 63, case, s, fc_list=[7])
    for name in STATE:
        if name not in ("leaf", "leaf_boards", "leaf_flat", "leaf_counts", "leaf_status", "k"):
            put(t1, name, st8[name][5:6])
    rv1.copy_(rv8[5:6])
    keys = torch.from_numpy(rng.integers(0, 2**40, 8, dtype=np.int64)).cuda()
    key1 = keys[5:6].clone()  # held here: the descriptor keeps only its address
    for scale in (1.0, 0.0):
        g8, g1 = desc(keys, rv8, 16, 63, scale), desc(key1, rv1, 16, 63, scale)
        _, a8, p8 = gumbel_result(t8, g8)
        _, a1, p1 = gumbel_result(t1, g1)
        assert a8[5] == a1[0] and np.array_equal(p8[5], p1[0])
        assert select(t8, g8) == FPC_OK and select(t1, g1) == FPC_OK
        assert int(t8.leaf[5]) == int(t1.leaf[0])
    # scale 0: the same slabs under eight keys choose alike
    for name in NODE_I32 + ("value_sum", "prior"):
        put(t8, name, np.repeat(st8[name][5:6], 8, axis=0))
    rv8.fill_(float(rv8[5]))
    _, a, _ = gumbel_result(t8, desc(keys, rv8, 16, 63, 0.0))
    assert len(set(a.tolist())) == 1


def test_bad_arguments_are_refused_before_any_launch():
    R, rng = 8, np.random.default_rng(6)
    t, before, _, rv = build(R, 16, rng, 16, 47)
    keys = torch.arange(16, dtype=torch.int64, device="cuda")
    rv_before = rv.cpu().numpy().copy()
    bad_r = TreeDesc()
    C.memmove(C.byref(bad_r), C.byref(t.desc), C.sizeof(TreeDesc))
    bad_r.R = 12
    bad = []
    for field, value in [("max_considered", 0), ("max_considered", FPC_MAX_MOVES + 1), ("n_sims", -1),
                         ("scale", -1.0), ("scale", float("nan")), ("scale", float("inf")), ("c_visit", -50.0),
                         ("c_visit", float("inf")), ("c_scale", float("nan")), ("c_scale", -0.1), ("keys", None),
                         ("root_value", None)]:
        d = desc(keys, rv, 16, 47)
        setattr(d, field, value)
        bad.append(d)
    for d in bad:
        assert select(t, d) == FPC_ERR_ARG and t.L.fpc_last_error()
        assert gumbel_result(t, d)[0] == FPC_ERR_ARG
    good = desc(keys, rv, 16, 47)
    assert select(t, good, bad_r) == FPC_ERR_ARG and gumbel_result(t, good, bad_r)[0] == FPC_ERR_ARG
    assert select(t, None) == FPC_ERR_ARG
    for kw in ({"action": False}, {"policy": False}):
        rc, action, policy = gumbel_result(t, good, **kw)
        assert rc == FPC_ERR_ARG and (action == -7).all() and (policy == -7.0).all()
    after = snapshot(t)
    for name in STATE:
        assert np.array_equal(after[name], before[name]), name
    assert np.array_equal(rv.cpu().numpy().view(np.int64), rv_before.view(np.int64))
