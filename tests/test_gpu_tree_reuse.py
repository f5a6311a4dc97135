"""-m gpu: fpc_tree_advance (tree reuse between moves) on hand-built trees, one launch at a time, against a numpy
restatement of the re-rooting: keep the played child's subtree, renumbered in ascending order of the old index, with its
boards compacted in ascending slot order -- or a fresh root exactly as fpc_tree_reset writes it.

Trees are grown the way the kernels grow them (children appended at n_nodes when their parent is expanded, a node
materialised before it is expanded), with the played child's subtree interleaved with the rest of the tree.  Every slab
is filled with sentinels first, so a word written outside the region the contract names shows as a difference."""
import ctypes as C

import numpy as np
import pytest
import torch

from alphazero_4_player_chess_b200._lib import TREE_ADVANCE_MAX_NODE_CAP, FpcError, check
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.geometry import GEOMETRIES
from alphazero_4_player_chess_b200.mcts import BatchedMCTS
from tests.test_gpu_puct_kernels import NODE_I32, SENT_F32, SENT_F64, SENT_I32, STATE, assert_state, put, snapshot
from tests.util import oracle_for

pytestmark = pytest.mark.gpu

NODE_CAP, SIMS = 2048, 250  # board_cap = 2 * SIMS + 2 with reuse_tree=True
LIM_N, LIM_B = 600, 80      # the limits of the launch that probes them


def new_tree(R, n, node_cap, sims, seed):
    m = BatchedMCTS(R, n, None, {"C": 3.0, "num_searches": sims}, node_cap=node_cap, reuse_tree=True)
    for name in NODE_I32:
        getattr(m, name).fill_(SENT_I32)
    m.value_sum.view(torch.int64).fill_(SENT_F64)
    m.prior.view(torch.int32).fill_(SENT_F32)
    g = torch.Generator(device="cuda").manual_seed(seed)
    m.boards.copy_(torch.randint(0, 256, m.boards.shape, generator=g, device="cuda", dtype=torch.uint8))
    return m


def advance(m, actions, roots, max_nodes, max_boards):
    acts = torch.from_numpy(np.ascontiguousarray(actions, np.int32)).cuda()
    rb = torch.from_numpy(np.ascontiguousarray(roots)).cuda()
    kept = torch.full((m.n,), -5, dtype=torch.int32, device="cuda")
    check(m.L.fpc_tree_advance(C.byref(m.desc), acts.data_ptr(), rb.data_ptr(), max_nodes, max_boards, kept.data_ptr(),
                               m._stream()))
    torch.cuda.synchronize()
    return kept.cpu().numpy()


class Grow:
    """One game's tree, grown as the kernels grow it.  `sub` marks the subtree of the root child that will be played."""

    def __init__(self, rng, asz):
        self.rng, self.asz = rng, asz
        self.parent, self.fc, self.nc, self.flat, self.bidx, self.sub = [-1], [0], [0], [-1], [0], [False]
        self.nb = 1
        self.open = {True: [], False: []}  # unexpanded, unmaterialised nodes in / outside the subtree
        self.n_sub = self.b_sub = 0

    def __len__(self):
        return len(self.parent)

    def materialise(self, v):
        if self.bidx[v] < 0:
            self.bidx[v] = self.nb
            self.nb += 1
            self.b_sub += self.sub[v]

    def expand(self, v, k=None, flats=None):
        self.materialise(v)
        if flats is None:
            flats = np.unique(self.rng.integers(0, self.asz, k))
        n0, k, s = len(self.parent), len(flats), self.sub[v]
        self.fc[v], self.nc[v] = n0, k
        self.parent += [v] * k
        self.fc += [0] * k
        self.nc += [0] * k
        self.flat += [int(f) for f in flats]
        self.bidx += [-1] * k
        self.sub += [s] * k
        self.open[s] += range(n0, n0 + k)
        self.n_sub += k * s
        return n0, k

    def pick(self, s):
        lst = self.open[s]
        i = int(self.rng.integers(len(lst)))
        lst[i], lst[-1] = lst[-1], lst[i]
        return lst.pop()

    def take(self, v):
        self.open[self.sub[v]].remove(v)

    def choose(self, c):
        self.take(c)
        self.sub[c] = True
        self.open[True].append(c)
        self.n_sub = 1

    def step(self, s, kmax, cap, touch=0.15):
        """Select an open node in (s) or outside the subtree: materialise it only (a terminal leaf) or expand it."""
        if not self.open[s]:
            s = not s
            if not self.open[s]:
                return
        k = int(self.rng.integers(1, kmax + 1))
        if len(self) + k > cap:
            return
        v = self.pick(s)
        if self.rng.random() < touch:
            self.materialise(v)
        else:
            self.expand(v, k)


def grow_case(rng, R, case, cap):
    """(Grow, action, c or -1, root board kind) for one game of the given case."""
    asz = GEOMETRIES[R].action_space_size
    t = Grow(rng, asz)
    if case == "unexpanded_root":
        return t, int(rng.integers(0, asz)), -1, "random"
    n0, k = t.expand(0, int(rng.integers(1, 300)) if case != "only_child" else 1)
    ci = {"first": 0, "last": k - 1}.get(case, int(rng.integers(0, k)))
    c = n0 + ci
    t.choose(c)
    action, kind = t.flat[c], "match"
    if case == "chain":  # an ancestor chain of 300 below c, interleaved with other expansions
        v = c
        t.take(c)
        for _ in range(300):
            a, kk = t.expand(v, int(rng.integers(1, 3)))
            v = a + int(rng.integers(kk))
            t.take(v)
            if rng.random() < 0.3 and t.open[False]:
                t.step(False, 6, cap)
        t.open[True].append(v)
    elif case == "unexpanded_child":
        for _ in range(int(rng.integers(0, 30))):
            if t.open[False]:
                t.step(False, 40, cap)
        kind = "random"
    elif case == "terminal_child":
        t.take(c)
        t.materialise(c)
        for _ in range(int(rng.integers(0, 30))):
            if t.open[False]:
                t.step(False, 40, cap)
    elif case in ("nodes_at", "nodes_over"):
        target = LIM_N + (case == "nodes_over")
        while t.n_sub < target:
            if rng.random() < 0.5 and t.open[False]:
                t.step(False, 10, cap - (target - t.n_sub))
            else:
                v = t.pick(True)
                t.expand(v, min(int(rng.integers(5, 41)), target - t.n_sub))
    elif case in ("boards_at", "boards_over"):
        target = LIM_B + (case == "boards_over")
        while t.b_sub < target:
            if rng.random() < 0.3 and t.open[False]:
                t.step(False, 10, cap - 4 * (target - t.b_sub))
            v = t.pick(True)
            if len(t.open[True]) == 0 or rng.random() < 0.6:
                t.expand(v, int(rng.integers(1, 4)))
            else:
                t.materialise(v)
    else:
        for _ in range(int(rng.integers(0, 80))):
            t.step(bool(rng.random() < 0.5), 40, cap)
    if case == "absent":
        action = int(np.setdiff1d(np.arange(asz), t.flat[n0: n0 + k])[int(rng.integers(0, asz - k))])
    elif case == "none":
        action = -1
    elif case == "mismatch":
        if c in t.open[True]:
            t.take(c)
        t.materialise(c)
        kind = "mismatch"
    assert len(t) <= cap
    return t, action, c, kind


CASES_A = ["first", "middle", "last", "none", "absent", "unexpanded_root", "unexpanded_child", "terminal_child", "chain",
           "mismatch", "stale_state", "only_child"]
CASES_B = ["nodes_at", "nodes_over", "boards_at", "boards_over", "middle"]


def build_launch(R, n, cases, seed, cap=NODE_CAP, sims=SIMS):
    """A tree object filled with one hand-built game per slot; returns (m, actions, roots, per-game case)."""
    g = GEOMETRIES[R]
    rng = np.random.default_rng(seed)
    m = new_tree(R, n, cap, sims, seed)
    st = snapshot(m)
    actions = np.zeros(n, np.int32)
    roots = rng.integers(0, 256, (n, g.record_bytes)).astype(np.uint8)
    names = []
    promo = promotion_boards() if R == 14 else None
    for gi in range(n):
        case = cases[gi % len(cases)]
        t, action, c, kind = grow_case(rng, R, case, cap)
        nn = len(t)
        assert t.nb <= m.board_cap, (case, t.nb)
        st["parent"][gi, :nn], st["first_child"][gi, :nn], st["n_children"][gi, :nn] = t.parent, t.fc, t.nc
        st["move_flat"][gi, :nn], st["board_idx"][gi, :nn] = t.flat, t.bidx
        st["visits"][gi, :nn] = rng.integers(1, 1000, nn)
        st["value_sum"][gi, :nn] = rng.normal(0.0, 30.0, nn).view(np.int64)
        st["prior"][gi, :nn] = rng.uniform(0.0, 1.0, nn).astype(np.float32).view(np.int32)
        st["n_nodes"][gi], st["n_boards"][gi] = nn, t.nb
        if kind == "match":
            roots[gi] = st["boards"][gi, t.bidx[c]] if t.bidx[c] >= 0 else roots[gi]
        elif kind == "mismatch":
            if promo is not None and gi % 2:  # a promotion made with the full move, where the tree holds the index-built one
                parent_rec, index_built, full = promo
                st["boards"][gi, 0], st["boards"][gi, t.bidx[c]], roots[gi] = parent_rec, index_built, full
            else:
                roots[gi] = st["boards"][gi, t.bidx[c]]
                roots[gi, int(rng.integers(0, R * R))] ^= 0x20
        actions[gi] = action
        names.append(case)
    st["leaf"][:] = rng.integers(-1, 50, n)
    st["dropped"][:] = rng.integers(0, 2, n)
    st["error"][:] = rng.integers(0, 16, n)
    for name in STATE:
        put(m, name, st[name])
    return m, actions, roots, names


def promotion_boards():
    """(position, child made with the index-built move, child made with the full move) for a red pawn promoting on the
    14x14 board: the index-built make leaves the pawn a pawn, so the two children differ."""
    R = 14
    g = GEOMETRIES[R]
    o = oracle_for(R)
    rec = g.empty_record()

    def place(r, c, color, ptype):
        rec[r * R + c] = 0x80 | (color << 5) | (ptype << 2)
        if ptype == 5:
            rec[g.off_king + color] = r * R + c
    place(13, 7, 0, 5), place(7, 0, 1, 5), place(0, 6, 2, 5), place(6, 13, 3, 5)
    place(R // 4 + 1, 5, 0, 0)
    promo = next(mv for mv in o.legal_moves(rec) if ((int(mv) >> 24) & 0xFF) != 6)
    index_built = o.make_index(rec, o.move_flat_index(promo))
    full = o.make_move(rec, promo)
    assert not np.array_equal(index_built, full)
    return rec, index_built, full


def reference(before, actions, roots, max_nodes, max_boards):
    """The state fpc_tree_advance must leave, and kept[]."""
    want = {k: v.copy() for k, v in before.items()}
    n = len(actions)
    kept = np.zeros(n, np.int32)
    for g in range(n):
        nn = int(before["n_nodes"][g])
        nc0, fc0 = int(before["n_children"][g, 0]), int(before["first_child"][g, 0])
        c = -1
        if actions[g] >= 0 and nc0 > 0:
            hit = np.flatnonzero(before["move_flat"][g, fc0: fc0 + nc0] == actions[g])
            c = fc0 + int(hit[0]) if len(hit) else -1
        ok = c > 0
        if ok:
            par = before["parent"][g, :nn]
            member = np.zeros(nn, bool)
            member[c] = True
            idx = np.arange(c + 1, nn)
            while True:  # parent[i] < i: a fixed point after (depth) rounds
                nxt = member.copy()
                nxt[idx] = member[par[idx]]
                if np.array_equal(nxt, member):
                    break
                member = nxt
            keep = np.flatnonzero(member)
            bix = before["board_idx"][g, keep]
            cs = int(bix[0])
            ok = (len(keep) <= max_nodes and int((bix >= 0).sum()) <= max_boards and
                  (cs < 0 or np.array_equal(before["boards"][g, cs], roots[g])))
        if not ok:
            fresh_root(want, g, roots[g])
            continue
        k = len(keep)
        new = np.full(nn, -1, np.int64)
        new[keep] = np.arange(k)
        nch = before["n_children"][g, keep]
        want["parent"][g, :k] = new[before["parent"][g, keep]]
        want["first_child"][g, :k] = np.where(nch > 0, new[np.clip(before["first_child"][g, keep], 0, nn - 1)], 0)
        for name in ("n_children", "visits", "move_flat", "value_sum", "prior"):
            want[name][g, :k] = before[name][g, keep]
        want["parent"][g, 0] = want["move_flat"][g, 0] = -1
        want["prior"][g, 0] = 0
        off = int(cs < 0)
        slots = np.sort(bix[bix >= 0])
        slot_new = {int(s): i + off for i, s in enumerate(slots)}
        want["board_idx"][g, :k] = [slot_new[int(b)] if b >= 0 else -1 for b in bix]
        want["board_idx"][g, 0] = 0
        for s in slots:
            want["boards"][g, slot_new[int(s)]] = before["boards"][g, s]
        if off:
            want["boards"][g, 0] = roots[g]
        want["n_nodes"][g], want["n_boards"][g] = k, len(slots) + off
        want["leaf"][g], want["dropped"][g], want["error"][g] = -1, 0, 0
        kept[g] = k
    return want, kept


def fresh_root(want, g, root):
    for name, v in (("parent", -1), ("first_child", 0), ("n_children", 0), ("visits", 1), ("move_flat", -1),
                    ("board_idx", 0), ("value_sum", 0), ("prior", 0)):
        want[name][g, 0] = v  # 0.0 in f32 and f64 is the all-zero bit pattern
    want["boards"][g, 0] = root
    want["n_nodes"][g], want["n_boards"][g], want["leaf"][g], want["dropped"][g], want["error"][g] = 1, 1, -1, 0, 0


def run_launch(R, cases, seed, max_nodes, max_boards, n=1024):
    m, actions, roots, names = build_launch(R, n, cases, seed)
    before = snapshot(m)
    kept = advance(m, actions, roots, max_nodes, max_boards)
    got = snapshot(m)
    want, want_kept = reference(before, actions, roots, max_nodes, max_boards)
    assert_state(got, want)
    assert np.array_equal(kept, want_kept), np.flatnonzero(kept != want_kept)[:8]
    # a fresh root is fpc_tree_reset's root, word for word
    ref = new_tree(R, n, NODE_CAP, SIMS, seed)
    for name in STATE:
        put(ref, name, before[name])
    ref.reset(torch.from_numpy(roots))
    reset = snapshot(ref)
    fresh = np.flatnonzero(kept == 0)
    for name in STATE:
        assert np.array_equal(got[name][fresh], reset[name][fresh]), name
    return names, kept, before


@pytest.mark.parametrize("R", [8, 10, 13, 14])
def test_advance_against_the_numpy_reference(R):
    names, kept, before = run_launch(R, CASES_A, 500 + R, NODE_CAP, 2 * SIMS + 2)
    by = {case: kept[[i for i, c in enumerate(names) if c == case]] for case in CASES_A}
    for case in ("none", "absent", "unexpanded_root", "mismatch"):
        assert (by[case] == 0).all(), case
    for case in ("first", "middle", "last", "chain", "stale_state", "only_child"):
        assert (by[case] > 0).all(), case
    assert (by["unexpanded_child"] == 1).all() and (by["terminal_child"] >= 1).all()
    assert (by["chain"] > 300).all()
    # the subtrees were interleaved with the rest of the tree: kept nodes are not one contiguous old range
    print(f"R={R}: kept nodes per case: " + ", ".join(f"{c} {int(v.mean())}" for c, v in by.items()) +
          f"; {int(before['n_nodes'].sum())} nodes before")


@pytest.mark.parametrize("R", [8, 14])
def test_limits_are_inclusive(R):
    names, kept, _ = run_launch(R, CASES_B, 700 + R, LIM_N, LIM_B)
    by = {case: kept[[i for i, c in enumerate(names) if c == case]] for case in CASES_B}
    assert (by["nodes_at"] == LIM_N).all() and (by["nodes_over"] == 0).all()
    assert (by["boards_at"] > 0).all() and (by["boards_over"] == 0).all()


def test_largest_node_cap_and_one_above():
    R, cap = 8, TREE_ADVANCE_MAX_NODE_CAP
    rng = np.random.default_rng(9)
    asz = GEOMETRIES[R].action_space_size
    m = new_tree(R, 2, cap, 1100, 9)  # board_cap 2,202
    st = snapshot(m)
    actions = np.zeros(2, np.int32)
    roots = np.zeros((2, GEOMETRIES[R].record_bytes), np.uint8)
    for gi in range(2):  # a full slab: c's subtree and the rest interleaved up to the last node
        t = Grow(rng, asz)
        n0, k = t.expand(0, 40)
        c = n0 + 7 + gi
        t.choose(c)
        while len(t) < cap:
            s = bool(rng.random() < 0.5) or not t.open[False]
            v = t.pick(s)
            t.expand(v, min(300, cap - len(t)))
        nn = len(t)
        assert nn == cap and t.nb <= m.board_cap
        st["parent"][gi], st["first_child"][gi], st["n_children"][gi] = t.parent, t.fc, t.nc
        st["move_flat"][gi], st["board_idx"][gi] = t.flat, t.bidx
        st["visits"][gi] = rng.integers(1, 1000, nn)
        st["value_sum"][gi] = rng.normal(0.0, 30.0, nn).view(np.int64)
        st["prior"][gi] = rng.uniform(0.0, 1.0, nn).astype(np.float32).view(np.int32)
        st["n_nodes"][gi], st["n_boards"][gi] = nn, t.nb
        actions[gi] = t.flat[c]
        roots[gi] = st["boards"][gi, t.bidx[c]]
    for name in STATE:
        put(m, name, st[name])
    before = snapshot(m)
    kept = advance(m, actions, roots, cap, m.board_cap)
    want, want_kept = reference(before, actions, roots, cap, m.board_cap)
    assert_state(snapshot(m), want)
    assert np.array_equal(kept, want_kept) and (kept > cap // 4).all(), kept
    # one above the largest supported node_cap: refused before any launch, nothing written
    big = new_tree(R, 1, cap + 1, 4, 10)
    before = snapshot(big)
    with pytest.raises(FpcError, match="node_cap"):
        advance(big, np.zeros(1, np.int32), np.zeros((1, GEOMETRIES[R].record_bytes), np.uint8), 1, 1)
    assert_state(snapshot(big), before)


def test_advance_needs_a_tree_and_checks_its_arguments():
    R = 8
    m = BatchedMCTS(R, 2, None, {"C": 3.0, "num_searches": 4}, reuse_tree=True)
    roots = torch.from_numpy(np.stack([start_record("EIGHT_SIMPLE")] * 2))
    with pytest.raises(FpcError, match="needs a tree"):
        m.advance(torch.zeros(2, dtype=torch.int32), roots)
    with pytest.raises(FpcError, match="there are none"):
        m.search(None)
    m.reset(roots)
    with pytest.raises(FpcError, match="negative limit"):
        advance(m, np.zeros(2, np.int32), roots.numpy(), -1, 0)
    assert m.node_cap == 1 + 2 * 96 * 4 and m.board_cap == 2 * 4 + 2
    plain = BatchedMCTS(R, 2, None, {"C": 3.0, "num_searches": 4})
    assert plain.node_cap == 1 + 96 * 4 and plain.board_cap == 4 + 2
