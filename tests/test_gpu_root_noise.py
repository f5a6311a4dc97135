"""-m gpu: fpc_tree_root_noise (Dirichlet noise on the root's children priors) on hand-built, sentinel-filled slabs,
one launch at a time, against the numpy restatement of include/fpc.h's recipe (tests/noise_oracle.py).

Root child counts 1, 2, 19, 38 and 300 (children not starting at node 1), beside an unexpanded root, a dropped game and
a game already marked done.  The noised priors must equal the restatement within rtol 1e-6, every other word of every
slab must be unchanged, `done` must be set exactly on the noised games, and a second call must change nothing."""
import ctypes as C

import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200._lib import FPC_ERR_ARG, FPC_OK, TreeDesc
from tests.noise_oracle import noised
from tests.test_gpu_puct_kernels import NODE_I32, STATE, new_tree, put, snapshot

pytestmark = pytest.mark.gpu

NODE_CAP = 400
CASES = [("k1", 1), ("k2", 2), ("k19", 19), ("k38", 38), ("k300", 300), ("unexpanded", 0), ("dropped", 19),
         ("done", 19)]
SEED = 0x0123456789ABCDEF


def build(R, n, rng, cases=CASES, layouts=None):
    """n games, game g of case cases[g % len(cases)]: random words in the used nodes, the root's k children at
    first_child = 1 + pad.  Returns (m, done [n] i32 on the device, per-game (case, first_child, k))."""
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
        st["first_child"][g, 0], st["n_children"][g, 0] = (fc, k) if k else (0, 0)
        st["n_nodes"][g] = used
        st["dropped"][g] = case == "dropped"
        info.append((case, fc, k))
    st["leaf"][:] = rng.integers(-1, 50, n)
    st["error"][:] = 0
    for name in STATE:
        put(m, name, st[name])
    done = torch.tensor([case == "done" for case, _, _ in info], dtype=torch.int32, device="cuda")
    return m, done, info


def call(m, keys, alpha, eps, done, seed=SEED, desc=None):
    keys_t = torch.as_tensor(np.asarray(keys, np.int64)).cuda()
    rc = m.L.fpc_tree_root_noise(C.byref(desc if desc is not None else m.desc), seed, keys_t.data_ptr(), alpha, eps,
                                 done.data_ptr() if done is not None else None, m._stream())
    torch.cuda.synchronize()
    return rc


@pytest.mark.parametrize("R,alpha,eps", [(14, 0.03, 0.25), (14, 0.3, 0.25), (8, 1.0, 0.25), (8, 2.5, 0.25),
                                         (14, 0.3, 1.0), (8, 0.3, 0.0)])
def test_noise_against_the_restatement(R, alpha, eps):
    rng = np.random.default_rng(int(alpha * 1000) + R + int(eps * 10))
    n = 5 * len(CASES)
    m, done, info = build(R, n, rng)
    keys = rng.integers(-2**63, 2**63 - 1, n, dtype=np.int64)
    before = snapshot(m)
    assert call(m, keys, alpha, eps, done) == FPC_OK
    got = snapshot(m)
    for name in STATE:
        if name != "prior":
            assert np.array_equal(got[name], before[name]), name
    want_prior = before["prior"].copy()
    noised_games = []
    for g, (case, fc, k) in enumerate(info):
        if case in ("dropped", "done", "unexpanded"):
            continue
        noised_games.append(g)
        p0 = before["prior"][g, fc: fc + k].view(np.float32)
        want = noised(p0, SEED, keys[g], alpha, eps)
        p1 = got["prior"][g, fc: fc + k].view(np.float32)
        np.testing.assert_allclose(p1, want, rtol=1e-6, atol=0, err_msg=f"game {g} ({case})")
        if eps == 0.0:
            assert np.array_equal(p1, p0)
        elif eps == 1.0:
            assert abs(float(p1.astype(np.float64).sum()) - 1.0) < 1e-5
        want_prior[g, fc: fc + k] = got["prior"][g, fc: fc + k]
    assert np.array_equal(got["prior"], want_prior)  # nothing outside the noised children moved
    want_done = np.zeros(n, np.int32)
    want_done[noised_games] = 1
    want_done[[g for g, (case, _, _) in enumerate(info) if case == "done"]] = 1
    assert done.cpu().numpy().tolist() == want_done.tolist()
    # a second call: every game is done, dropped or unexpanded
    assert call(m, keys, alpha, eps, done) == FPC_OK
    again = snapshot(m)
    for name in STATE:
        assert np.array_equal(again[name], got[name]), name
    assert done.cpu().numpy().tolist() == want_done.tolist()


def test_draws_depend_on_the_key_not_on_the_place_in_the_batch():
    R, rng = 14, np.random.default_rng(3)
    layout = (7, 7 + 38 + 5)
    cases = [("k38", 38)]
    m8, done8, _ = build(R, 8, rng, cases, layouts=[layout] * 8)
    m1, done1, _ = build(R, 1, rng, cases, layouts=[layout])
    prior = snapshot(m8)["prior"][5:6]
    put(m8, "prior", np.repeat(prior, 8, axis=0))  # every game the same children priors
    put(m1, "prior", prior)
    keys = rng.integers(0, 2**40, 8, dtype=np.int64)
    assert call(m8, keys, 0.3, 0.25, done8) == FPC_OK
    assert call(m1, keys[5:6], 0.3, 0.25, done1) == FPC_OK
    a, b = snapshot(m8)["prior"], snapshot(m1)["prior"]
    assert np.array_equal(a[5], b[0])
    assert not np.array_equal(a[4], a[5])  # another key, other draws


def test_bad_arguments_are_refused_before_any_launch():
    R, rng = 8, np.random.default_rng(4)
    m, done, _ = build(R, 16, rng)
    keys = np.arange(16, dtype=np.int64)
    before, done_before = snapshot(m), done.cpu().numpy().copy()
    bad_r, bad_prior = TreeDesc(), TreeDesc()
    for d in (bad_r, bad_prior):
        C.memmove(C.byref(d), C.byref(m.desc), C.sizeof(TreeDesc))
    bad_r.R, bad_prior.prior = 12, None
    for alpha, eps, kw in [(0.0, 0.25, {}), (-0.3, 0.25, {}), (float("nan"), 0.25, {}), (float("inf"), 0.25, {}),
                           (0.3, -0.01, {}), (0.3, 1.01, {}), (0.3, float("nan"), {}), (0.3, 0.25, {"done": None}),
                           (0.3, 0.25, {"desc": bad_r}), (0.3, 0.25, {"desc": bad_prior})]:
        kw = {"done": done, **kw}
        assert call(m, keys, alpha, eps, **kw) == FPC_ERR_ARG, (alpha, eps, kw.keys())
        assert m.L.fpc_last_error()
    keys_t = torch.as_tensor(keys).cuda()
    assert m.L.fpc_tree_root_noise(C.byref(m.desc), SEED, None, 0.3, 0.25, done.data_ptr(), m._stream()) == FPC_ERR_ARG
    assert m.L.fpc_tree_root_noise(None, SEED, keys_t.data_ptr(), 0.3, 0.25, done.data_ptr(), m._stream()) == FPC_ERR_ARG
    torch.cuda.synchronize()
    after = snapshot(m)
    for name in STATE:
        assert np.array_equal(after[name], before[name]), name
    assert np.array_equal(done.cpu().numpy(), done_before)
