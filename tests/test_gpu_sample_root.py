"""-m gpu: fpc_tree_sample_root (keyed move sampling from the root's visit counts) on hand-built, sentinel-filled
slabs, against the numpy restatement of include/fpc.h's recipe (tests/sample_oracle.py).

Root child counts 1, 2, 20 and 300 with uneven visits (zeros among them), children not starting at node 1, beside a
root whose visits are all zero, an unexpanded root and a dropped game, each of which must give -1.  At temperature 1
the choice must equal the restatement's exactly; at other temperatures too, except where U*W lies within 1e-12 of a
prefix boundary (the device's pow may differ from numpy's in the last bit), and these inputs have no such case."""
import ctypes as C

import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200._lib import FPC_ERR_ARG, FPC_OK, TreeDesc
from tests.sample_oracle import near_boundary, sample_index
from tests.test_gpu_puct_kernels import NODE_I32, STATE, new_tree, put, snapshot

pytestmark = pytest.mark.gpu

NODE_CAP = 400
CASES = [("k1", 1), ("k2", 2), ("k20", 20), ("k300", 300), ("zero", 20), ("unexpanded", 0), ("dropped", 20)]
SEED = 0x0123456789ABCDEF
SENT_ACTION = -31337


def build(R, n, rng, cases=CASES, layouts=None):
    """n games, game g of case cases[g % len(cases)]: random words in the used nodes, the root's k children at
    first_child = 1 + pad with distinct move_flat and uneven visits.  Returns (m, per-game (case, first_child, k))."""
    m = new_tree(R, n, NODE_CAP)
    st = snapshot(m)
    info = []
    for g in range(n):
        case, k = cases[g % len(cases)]
        fc, used = layouts[g] if layouts is not None else (1 + int(rng.integers(0, 21)), None)
        used = used or fc + k + int(rng.integers(0, 40))
        for name in NODE_I32:
            st[name][g, :used] = rng.integers(-1, used, used)
        st["value_sum"][g, :used] = rng.normal(0.0, 10.0, used).view(np.int64)
        st["prior"][g, :used] = rng.uniform(0.0, 1.0, used).astype(np.float32).view(np.int32)
        if k:
            st["move_flat"][g, fc: fc + k] = rng.permutation(5000)[:k]
            v = (rng.integers(1, 12, k) ** 3).astype(np.int32)  # uneven: 1 .. 1331
            v[rng.random(k) < 0.15] = 0
            if case == "zero":
                v[:] = 0
            elif not v.any():
                v[0] = 1
            st["visits"][g, fc: fc + k] = v
        st["first_child"][g, 0], st["n_children"][g, 0] = (fc, k) if k else (0, 0)
        st["n_nodes"][g] = used
        st["dropped"][g] = case == "dropped"
        info.append((case, fc, k))
    st["leaf"][:] = rng.integers(-1, 50, n)
    st["error"][:] = 0
    for name in STATE:
        put(m, name, st[name])
    return m, info


def call(m, keys, temperature, seed=SEED, desc=None, action=None, keys_ptr=True):
    keys_t = torch.as_tensor(np.asarray(keys, np.int64)).cuda()
    rc = m.L.fpc_tree_sample_root(C.byref(desc if desc is not None else m.desc), seed,
                                  keys_t.data_ptr() if keys_ptr else None, temperature,
                                  action.data_ptr() if action is not None else None, m._stream())
    torch.cuda.synchronize()
    return rc


def expected(before, info, keys, temperature):
    """(want action [n], near-boundary count) from the restatement."""
    want, near = [], 0
    for g, (case, fc, k) in enumerate(info):
        if case in ("dropped", "unexpanded"):
            want.append(-1)
            continue
        visits = before["visits"][g, fc: fc + k]
        i, t, P = sample_index(visits, temperature, SEED, int(keys[g]))
        near += temperature != 1.0 and i >= 0 and near_boundary(t, P)
        want.append(-1 if i < 0 else int(before["move_flat"][g, fc + i]))
    return np.array(want), near


@pytest.mark.parametrize("R,temperature", [(14, 1.0), (8, 1.0), (14, 0.5), (8, 1.7), (14, 0.25), (8, 3.0)])
def test_sampling_against_the_restatement(R, temperature):
    rng = np.random.default_rng(R * 100 + int(temperature * 10))
    n = 40 * len(CASES)
    m, info = build(R, n, rng)
    before = snapshot(m)
    for rep in range(3):
        keys = rng.integers(-2**63, 2**63 - 1, n, dtype=np.int64)
        action = torch.full((n + 8,), SENT_ACTION, dtype=torch.int32, device="cuda")
        assert call(m, keys, temperature, action=action) == FPC_OK
        got = action.cpu().numpy()
        want, near = expected(before, info, keys, temperature)
        assert near == 0
        assert np.array_equal(got[:n], want), np.flatnonzero(got[:n] != want)[:10]
        assert (got[n:] == SENT_ACTION).all()  # nothing past d_action[n_games - 1]
        for g, (case, _, _) in enumerate(info):
            if case in ("zero", "unexpanded", "dropped"):
                assert got[g] == -1, (g, case)
        after = snapshot(m)
        for name in STATE:
            assert np.array_equal(after[name], before[name]), name  # the slabs are only read
    # through BatchedMCTS.sample_root: the same call
    keys = rng.integers(0, 2**40, n, dtype=np.int64)
    got = m.sample_root(SEED, torch.as_tensor(keys), temperature).cpu().numpy()
    assert np.array_equal(got, expected(before, info, keys, temperature)[0])


def test_a_key_draws_the_same_move_in_any_slot():
    R, rng = 14, np.random.default_rng(3)
    layout = (7, 7 + 300 + 5)
    cases = [("k300", 300)]
    m8, _ = build(R, 8, rng, cases, layouts=[layout] * 8)
    m1, _ = build(R, 1, rng, cases, layouts=[layout])
    st = snapshot(m8)
    for name in ("visits", "move_flat"):
        put(m8, name, np.repeat(st[name][5:6], 8, axis=0))  # every game the same root
        put(m1, name, st[name][5:6])
    keys = rng.integers(0, 2**40, 8, dtype=np.int64)
    for temperature in (1.0, 0.7):
        a8 = m8.sample_root(SEED, torch.as_tensor(keys), temperature).cpu().numpy()
        a1 = m1.sample_root(SEED, torch.as_tensor(keys[5:6]), temperature).cpu().numpy()
        assert a8[5] == a1[0]
        assert len(set(a8.tolist())) > 1  # other keys, other draws


def test_bad_arguments_are_refused_before_any_launch():
    R, rng = 8, np.random.default_rng(4)
    n = 16
    m, _ = build(R, n, rng)
    keys = np.arange(n, dtype=np.int64)
    before = snapshot(m)
    action = torch.full((n,), SENT_ACTION, dtype=torch.int32, device="cuda")
    bad_r, bad_visits = TreeDesc(), TreeDesc()
    for d in (bad_r, bad_visits):
        C.memmove(C.byref(d), C.byref(m.desc), C.sizeof(TreeDesc))
    bad_r.R, bad_visits.visits = 12, None
    for temperature, kw in [(0.0, {}), (-1.0, {}), (float("nan"), {}), (float("inf"), {}), (-float("inf"), {}),
                            (1.0, {"keys_ptr": False}), (1.0, {"action": None}), (1.0, {"desc": bad_r}),
                            (1.0, {"desc": bad_visits})]:
        kw = {"action": action, **kw}
        assert call(m, keys, temperature, **kw) == FPC_ERR_ARG, (temperature, kw.keys())
        assert m.L.fpc_last_error()
    keys_t = torch.as_tensor(keys).cuda()
    assert m.L.fpc_tree_sample_root(None, SEED, keys_t.data_ptr(), 1.0, action.data_ptr(), m._stream()) == FPC_ERR_ARG
    torch.cuda.synchronize()
    after = snapshot(m)
    for name in STATE:
        assert np.array_equal(after[name], before[name]), name
    assert (action.cpu().numpy() == SENT_ACTION).all()
