"""-m gpu: fpc_tree_select_gumbel_interior on hand-built, sentinel-filled trees three levels deep, one launch at a time,
against the numpy restatement of include/fpc.h (tests/gumbel_interior_oracle.py).

The root's single child x1 has 1, 2, 20, 38 or 300 children; its visited children carry three children each.  Nodes
sit at s == 0 (node_value must be written) and at s > 0 with node_value planted away from value_sum (which proves the
cache is read), beside zero priors, exact ties, a NaN value sum, paths ending on an unmaterialised child, on an existing
board and with board_cap met exactly and one over, and the root cases of the Gumbel select (unexpanded, dropped, off the
schedule).  The leaf must be the restatement's.  A twin tree whose path nodes keep only the restatement's child, run
through fpc_tree_select, must end with the same words everywhere (so the materialisation, leaf_boards and k match and
nothing else is written), and node_value must change exactly at the nodes passed at s == 0."""
import ctypes as C

import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200._lib import FPC_ERR_ARG, FPC_OK, TreeDesc
from alphazero_4_player_chess_b200.fen import start_record
from tests.gumbel_interior_oracle import TIE, interior_choice
from tests.gumbel_oracle import root_choice
from tests.test_gpu_gumbel_kernels import SEED, desc
from tests.test_gpu_gumbel_kernels import build as build_root
from tests.test_gpu_gumbel_kernels import select as select_root
from tests.test_gpu_puct_kernels import NODE_I32, SENT_F64, START, STATE, new_tree, put, snapshot
from tests.util import oracle_for

pytestmark = pytest.mark.gpu

NODE_CAP = 1300
FANOUTS = (1, 2, 20, 38, 300)
# (name, x1 at s == 0, tie, zero prior, NaN value sum, n_boards)
KINDS = [("s0", True, False, False, False, "free"), ("s>0", False, False, False, False, "free"),
         ("zero_prior", False, False, True, False, "free"), ("tie", True, True, False, False, "free"),
         ("tie_visited", False, True, False, False, "free"), ("cap_exact", False, False, False, False, "exact"),
         ("cap_over", False, False, False, False, "over"), ("nan", False, False, False, True, "free")]
ROOT_CASES = [("unexpanded", 0), ("dropped", 20), ("off", 2)]


def select(t, gd, node_value, tree_desc=None):
    rc = t.L.fpc_tree_select_gumbel_interior(C.byref(tree_desc if tree_desc is not None else t.desc),
                                             C.byref(gd) if gd is not None else None,
                                             node_value.data_ptr() if node_value is not None else None, 0,
                                             t.planes.data_ptr(), 0, None, t._stream())
    torch.cuda.synchronize()
    return rc


def nan_slab(n):
    return torch.from_numpy(np.full((n, NODE_CAP), SENT_F64, np.int64)).cuda()


def build(R, rng):
    """Games: every (fan-out, kind) of the interior, then the root cases.  Returns (tree, state, info, root_value,
    node_value [n, NODE_CAP] f64 as i64 bits on the device)."""
    cases = [("interior", F, kind) for F in FANOUTS for kind in KINDS] + [("root", k, name) for name, k in ROOT_CASES]
    n = len(cases)
    t = new_tree(R, n, NODE_CAP)
    st = snapshot(t)
    o = oracle_for(R)
    legal = [o.move_flat_index(m) for m in o.legal_moves(start_record(START[R]))]
    root_value = np.full(n, SENT_F64, np.int64).view(np.float64)
    node_value = np.full((n, NODE_CAP), SENT_F64, np.int64)
    info = []
    for g, (what, F, kind) in enumerate(cases):
        if what == "root":
            info.append(dict(case=kind))
            continue
        name, s0, tie, zero, nan, boards = kind
        fc1 = 2 + int(rng.integers(0, 5))
        N1 = np.zeros(F, np.int64) if s0 else np.where(rng.random(F) < 0.5, rng.integers(1, 6, F), 0)
        if not s0 and not N1.any():
            N1[int(rng.integers(0, F))] = 1
        if tie and not s0:
            N1[:] = 2
        used = fc1 + F
        kids = {}  # level-2 node -> (first child, N of its three children)
        for c in np.flatnonzero(N1 > 0):
            N2 = np.zeros(3, np.int64) if rng.random() < 0.5 else rng.integers(0, 3, 3)
            kids[fc1 + int(c)] = (used, N2)
            used += 3
        nn = used
        for nm in NODE_I32:
            st[nm][g, :nn + 4] = rng.integers(0, nn, nn + 4)
        st["n_children"][g, :nn + 4] = 0
        st["first_child"][g, :nn + 4] = 0
        st["board_idx"][g, :nn + 4] = np.where(rng.random(nn + 4) < 0.5, 0, -1)
        st["board_idx"][g, :fc1] = 0
        st["move_flat"][g, :nn + 4] = rng.choice(legal, nn + 4)
        vs = rng.normal(0.0, 1.0, nn + 4)
        prior = rng.uniform(1e-3, 1.0, nn + 4).astype(np.float32)
        # root -> x1 (node 1), on the schedule of a one-child root: cv(s) = s
        s_root = int(N1.sum()) + 1
        st["first_child"][g, 0], st["n_children"][g, 0], st["visits"][g, 0] = 1, 1, 1 + s_root
        st["parent"][g, 1] = 0
        st["visits"][g, 1] = 1 + s_root
        root_value[g] = rng.normal()
        st["first_child"][g, 1], st["n_children"][g, 1], st["board_idx"][g, 1] = fc1, F, 0
        st["parent"][g, fc1:fc1 + F] = 1
        st["visits"][g, fc1:fc1 + F] = N1 + 1
        vs[fc1:fc1 + F] = np.where(N1 > 0, rng.uniform(-1.0, 1.0, F) * N1, 0.0)
        if tie:
            prior[fc1:fc1 + F] = np.float32(0.25)
            vs[fc1:fc1 + F] = 0.5 * N1
        if zero and F > 1:  # a zero prior among others (all-zero priors are NaN logits)
            z = fc1 + int(rng.integers(0, F))
            prior[z], st["visits"][g, z] = 0.0, 1
        if nan:
            vs[fc1 + int(np.flatnonzero(N1 > 0)[0])] = np.nan
        for x, (fc2, N2) in kids.items():
            st["first_child"][g, x], st["n_children"][g, x], st["board_idx"][g, x] = fc2, 3, 0
            st["parent"][g, fc2:fc2 + 3] = x
            st["visits"][g, fc2:fc2 + 3] = N2 + 1
            vs[fc2:fc2 + 3] = np.where(N2 > 0, rng.uniform(-1.0, 1.0, 3) * N2, 0.0)
            if N2.any():
                node_value[g, x] = np.float64(rng.normal()).view(np.int64)  # planted away from value_sum
        if not s0:
            node_value[g, 1] = np.float64(vs[1] + 1.0 + rng.random()).view(np.int64)
        if boards != "free":  # every path ends on a board to materialise
            leafy = np.flatnonzero(st["n_children"][g, :nn] == 0)
            st["board_idx"][g, leafy[leafy >= fc1]] = -1
        st["value_sum"][g, :nn + 4] = vs.view(np.int64)
        st["prior"][g, :nn + 4] = prior.view(np.int32)
        st["n_nodes"][g] = nn + 4
        st["n_boards"][g] = {"free": 1, "exact": t.board_cap - 1, "over": t.board_cap}[boards]
        info.append(dict(case=name, F=F, fc1=fc1))
    # the root cases, laid out as the Gumbel kernel test lays them out
    _, sub_st, sub_info, sub_rv = build_root(R, len(ROOT_CASES), rng, 4, 47, cases=ROOT_CASES, s_list=[5])
    for j in range(len(ROOT_CASES)):
        g = len(cases) - len(ROOT_CASES) + j
        for nm in STATE:
            if sub_st[nm].ndim == 1:
                st[nm][g] = sub_st[nm][j]
            else:
                st[nm][g, :sub_st[nm].shape[1]] = sub_st[nm][j]
        root_value[g] = sub_rv[j].item()
        info[g].update(sub_info[j])
    st["leaf"][:] = rng.integers(-1, 50, n)
    st["error"][:] = 0
    for nm in STATE:
        put(t, nm, st[nm])
    return t, snapshot(t), info, torch.from_numpy(root_value).cuda(), torch.from_numpy(node_value).cuda()


def stats(st, g, x, fc, k):
    N = st["visits"][g, fc:fc + k] - 1
    vs = st["value_sum"][g, fc:fc + k].view(np.float64)
    prior = st["prior"][g, fc:fc + k].view(np.float32)
    return N, vs, prior


def expected_path(st, g, rv, nv, dev_leaf, m, n_sims, key):
    """The restatement's descent of game g: (path [nodes], nodes written at s == 0, failed, adopted).  At an interior
    choice where the device's path differs, the device's child is adopted on an absolute near-tie only."""
    parent = st["parent"][g]
    dev_path = []
    x = int(dev_leaf)
    while x > 0:
        dev_path.append(x)
        x = int(parent[x])
    dev_path = [0] + dev_path[::-1]  # aligned with path: node 0 first
    k, fc = int(st["n_children"][g, 0]), int(st["first_child"][g, 0])
    if k == 0:
        return [0], [], False, 0
    N, vs, prior = stats(st, g, 0, fc, k)
    u = st["value_sum"][g, 0:1].view(np.float64)[0] if int(N.sum()) == 0 else rv
    i, _ = root_choice(N, vs, prior, u, SEED, key, m, n_sims, 1.0)
    if i < 0:
        return [0], [], True, 0
    path, written, adopted = [0, fc + i], [], 0
    x = fc + i
    while st["n_children"][g, x] > 0:
        k, fc = int(st["n_children"][g, x]), int(st["first_child"][g, x])
        N, vs, prior = stats(st, g, x, fc, k)
        if int(N.sum()) == 0:
            u = st["value_sum"][g, x:x + 1].view(np.float64)[0]
            written.append(x)
        else:
            u = nv[g, x:x + 1].view(np.float64)[0]
        i, sc = interior_choice(N, vs, prior, u)
        if i < 0:
            return path, written, True, adopted
        d = len(path)
        if d < len(dev_path) and dev_path[d] != fc + i:
            j = dev_path[d] - fc
            assert 0 <= j < k and abs(sc[j] - sc[i]) <= TIE, (g, x, i, j)
            i, adopted = j, adopted + 1
        x = fc + i
        path.append(x)
    return path, written, False, adopted


@pytest.mark.parametrize("R", [8, 14])
def test_interior_select_against_the_restatement(R):
    rng = np.random.default_rng(100 + R)
    m, n_sims = 4, 47
    t, before, info, rv, nv = build(R, rng)
    n = t.n
    keys = torch.from_numpy(rng.integers(-2**63, 2**63 - 1, n, dtype=np.int64)).cuda()
    rv_before, nv_before = rv.cpu().numpy().copy(), nv.cpu().numpy().copy()
    gd = desc(keys, rv, m, n_sims)
    assert select(t, gd, nv.view(torch.float64)) == FPC_OK
    got = snapshot(t)
    twin, _, _, _, _ = build(R, np.random.default_rng(0))
    twin_st = {name: before[name].copy() for name in STATE}
    nv_want = nv_before.copy()
    adopted = counted = 0
    for g, d in enumerate(info):
        if d["case"] in ("dropped", "unexpanded"):
            continue
        path, written, failed, a = expected_path(before, g, rv_before[g], nv_before, got["leaf"][g], m, n_sims,
                                                 int(keys[g]))
        adopted += a
        for x in written:
            nv_want[g, x] = before["value_sum"][g, x]
        for x, c in zip(path, path[1:]):  # the twin keeps only the path's children
            twin_st["first_child"][g, x], twin_st["n_children"][g, x] = c, 1
        if failed:  # SelectChild fails on the same node when it keeps only a NaN child or nothing
            x = path[-1]
            if d["case"] == "nan":
                bad = [c for c in range(int(before["first_child"][g, x]),
                                        int(before["first_child"][g, x] + before["n_children"][g, x]))
                       if np.isnan(before["value_sum"][g, c:c + 1].view(np.float64)[0])]
                twin_st["first_child"][g, x], twin_st["n_children"][g, x] = bad[0], 1
            else:
                assert d["case"] == "off"
                twin_st["dropped"][g] = 1
                twin_st["error"][g] |= 4
        else:
            assert got["leaf"][g] == path[-1] or got["dropped"][g], (g, d, path, got["leaf"][g])
            counted += 1
    for name in STATE:
        put(twin, name, twin_st[name])
    twin.select()
    want = snapshot(twin)
    for name in STATE:
        if name in ("first_child", "n_children"):
            assert np.array_equal(got[name], before[name]), name
        else:
            assert np.array_equal(got[name], want[name]), name
    assert torch.equal(t.planes, twin.planes)
    assert np.array_equal(nv.cpu().numpy(), nv_want)
    assert adopted <= 1, adopted
    # every root here has s > 0: root_value is read, never written
    assert np.array_equal(rv.cpu().numpy().view(np.int64), rv_before.view(np.int64))
    by_case = {}
    for g, d in enumerate(info):
        by_case.setdefault(d["case"], []).append(g)
    assert all(got["error"][g] == 4 and got["leaf"][g] == -1 for g in by_case["nan"] + by_case["off"])
    assert all(got["error"][g] == 2 and got["leaf"][g] == -1 for g in by_case["cap_over"])
    assert all(got["error"][g] == 0 and got["n_boards"][g] == t.board_cap for g in by_case["cap_exact"])
    assert all(got["leaf"][g] >= 0 and got["error"][g] == 0 for c in ("s0", "s>0", "zero_prior", "tie", "tie_visited")
               for g in by_case[c])
    # exact ties: the first child wins at x1
    assert all(got["leaf"][g] == d["fc1"] or before["parent"][g, got["leaf"][g]] == d["fc1"]
               for g, d in enumerate(info) if d["case"] in ("tie", "tie_visited"))
    print(f"R={R}: {n} games, {counted} leaves, {adopted} near-tie choices adopted")


@pytest.mark.parametrize("R", [8, 14])
def test_depth_one_is_the_gumbel_select(R):
    """Every root child unexpanded: the interior select is fpc_tree_select_gumbel word for word, node_value untouched."""
    m, n_sims = 16, 63
    out = []
    for interior in (False, True):
        t, before, info, rv = build_root(R, 40, np.random.default_rng(7 + R), m, n_sims)
        nc = before["n_children"].copy()
        nc[:, 1:] = 0
        put(t, "n_children", nc)
        keys = torch.arange(40, dtype=torch.int64, device="cuda") * 977
        gd = desc(keys, rv, m, n_sims)
        nv = nan_slab(40)
        assert (select(t, gd, nv.view(torch.float64)) if interior else select_root(t, gd)) == FPC_OK
        out.append((snapshot(t), rv.cpu().numpy().view(np.int64), nv.cpu().numpy(), t.planes.clone()))
    (a, ra, _, pa), (b, rb, nvb, pb) = out
    for name in STATE:
        assert np.array_equal(a[name], b[name]), name
    assert np.array_equal(ra, rb) and torch.equal(pa, pb)
    assert (nvb == SENT_F64).all()


def test_bad_arguments_are_refused_and_write_nothing():
    R, rng = 8, np.random.default_rng(6)
    t, before, _, rv = build_root(R, 16, rng, 16, 47)
    keys = torch.arange(16, dtype=torch.int64, device="cuda")
    nv = nan_slab(16)
    rv_before = rv.cpu().numpy().copy()
    bad_r = TreeDesc()
    C.memmove(C.byref(bad_r), C.byref(t.desc), C.sizeof(TreeDesc))
    bad_r.R = 12
    for field, value in [("max_considered", 0), ("n_sims", -1), ("scale", float("nan")), ("c_visit", -50.0),
                         ("c_scale", float("inf")), ("keys", None), ("root_value", None)]:
        d = desc(keys, rv, 16, 47)
        setattr(d, field, value)
        assert select(t, d, nv.view(torch.float64)) == FPC_ERR_ARG and t.L.fpc_last_error()
    good = desc(keys, rv, 16, 47)
    assert select(t, good, nv.view(torch.float64), bad_r) == FPC_ERR_ARG
    assert select(t, None, nv.view(torch.float64)) == FPC_ERR_ARG
    assert select(t, good, None) == FPC_ERR_ARG
    after = snapshot(t)
    for name in STATE:
        assert np.array_equal(after[name], before[name]), name
    assert np.array_equal(rv.cpu().numpy().view(np.int64), rv_before.view(np.int64))
    assert (nv.cpu().numpy() == SENT_F64).all()
