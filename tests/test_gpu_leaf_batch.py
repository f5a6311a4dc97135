"""-m gpu: the leaf-parallel kernels (fpc_tree_select_leaves / fpc_tree_expand_backup_leaves) on hand-loaded trees, one
batch at a time, against the restatement in tests/leaves_oracle.py.

The trees are those of a restatement search (mcts_port.search with FakeNet), copied into sentinel-filled slabs (a NaN
bit pattern in the float arrays, -7777 in the int arrays), so that a write outside what the semantics allow shows as a
changed word.  Integer state and f64 value sums must be bit-exact; priors within the rtol of tests/test_gpu_mcts.py.
Games take roles within one launch: plain; a root child whose children all have NaN priors (a descent error in
mid-batch); node_cap met exactly and one over at a middle slot; board_cap likewise; a 300-deep chain."""
import copy
import ctypes as C
import functools

import numpy as np
import pytest
import torch

import tests.leaves_oracle as lo
from alphazero_4_player_chess_b200 import _lib
from alphazero_4_player_chess_b200._lib import FPC_MAX_MOVES, MAX_LEAVES_PER_GAME
from alphazero_4_player_chess_b200.fen import start_record
from alphazero_4_player_chess_b200.mcts import BatchedMCTS
from oracle.mcts_port import Tree, search
from tests.golden.fake_net import FakeNet
from tests.test_gpu_mcts import search_roots
from tests.util import oracle_for

pytestmark = pytest.mark.gpu

START = {8: "EIGHT_SIMPLE", 10: "TEN", 13: "THIRTEEN", 14: "STANDARD"}
SENT_I32, SENT_F32, SENT_F64 = -7777, 0x7FC0DEAD, 0x7FF8DEADBEEF0001
NODE_I32 = ("parent", "first_child", "n_children", "visits", "move_flat", "board_idx")
PRIOR_RTOL = 2e-6
C_PUCT = 3.0
SORTED_BACKUP_ENTRIES = 4096  # LB_ENTRIES of leaves_commit_kernel: more (node, slot) backup entries take its serial walk


@functools.lru_cache(maxsize=None)
def searched_trees(R, n, sims):
    o = oracle_for(R)
    roots = search_roots(START[R], R, n)
    return search(o, FakeNet(R), roots, C_PUCT, sims, batch_rotation=False)


def clone(t):
    return copy.deepcopy(t, {id(t.o): t.o})  # the oracle's rules library is shared, not copied


def new_mcts(R, n, L, vl, node_cap, board_room):
    alloc = max(L, 2)  # L = 1 runs the leaf calls on a batch allocated for two slots per game
    sims = alloc * (1 + board_room // alloc)  # board_cap = sims + 2
    m = BatchedMCTS(R, n, FakeNet(R, device="cuda"), {"C": C_PUCT, "num_searches": sims}, node_cap=node_cap,
                    leaves_per_game=alloc, virtual_loss=vl)
    m.batch.L = L
    return m


def pad_nodes(t, k):
    """k unreachable nodes appended (parent 0, never a child): they only move n_nodes."""
    for _ in range(k):
        t.parent.append(0)
        t.children.append([])
        t.visits.append(1)
        t.value_sum.append(0.0)
        t.prior.append(0.0)
        t.move_flat.append(-1)
        t.rec.append(t.rec[0])


def load(m, trees, n_boards):
    """The trees into m's slabs (sentinels elsewhere); boards: the materialised nodes in ascending order."""
    n, nc = m.n, m.node_cap
    a = {name: np.full((n, nc), SENT_I32, np.int32) for name in NODE_I32}
    vs = np.full((n, nc), SENT_F64, np.int64)
    pr = np.full((n, nc), SENT_F32, np.int32)
    boards = np.zeros(tuple(m.boards.shape), np.uint8)
    for gi, t in enumerate(trees):
        nn = len(t.parent)
        a["parent"][gi, :nn] = t.parent
        a["first_child"][gi, :nn] = [ch[0] if ch else 0 for ch in t.children]
        a["n_children"][gi, :nn] = [len(ch) for ch in t.children]
        a["visits"][gi, :nn] = t.visits
        a["move_flat"][gi, :nn] = t.move_flat
        mat = sorted(t.materialised)
        slot = {node: i for i, node in enumerate(mat)}
        a["board_idx"][gi, :nn] = [slot.get(i, -1) for i in range(nn)]
        for node, i in slot.items():
            boards[gi, i] = t.rec[node]
        vs[gi, :nn] = np.asarray(t.value_sum, np.float64).view(np.int64)
        pr[gi, :nn] = np.asarray(t.prior, np.float32).view(np.int32)
    for name in NODE_I32:
        getattr(m, name).copy_(torch.from_numpy(a[name]))
    m.value_sum.view(torch.int64).copy_(torch.from_numpy(vs))
    m.prior.view(torch.int32).copy_(torch.from_numpy(pr))
    m.boards.copy_(torch.from_numpy(boards))
    m.n_nodes.copy_(torch.tensor([len(t.parent) for t in trees], dtype=torch.int32))
    m.n_boards.copy_(torch.as_tensor(n_boards, dtype=torch.int32))
    m.dropped.zero_()
    m.error.zero_()
    m.in_flight.zero_()
    m.slot_boards.copy_(torch.from_numpy(np.stack([trees[0].rec[0]] * m.slot_boards.shape[0])))


def host(t):
    if t.dtype == torch.float64:
        t = t.view(torch.int64)
    elif t.dtype == torch.float32:
        t = t.view(torch.int32)
    return t.cpu().numpy().copy()


def unique_legal(o, rec):
    return len({o.move_flat_index(mv) for mv in o.legal_moves(rec)})


def plan(o, trees, L, vl, roles):
    """Adapt the games to their roles on copies run through the restatement; returns (trees, n_boards, node_cap,
    board_cap, applied): applied = the games whose role could be set up (a cap role needs two qualifying slots)."""
    trees = [lo.prepare(clone(t)) for t in trees]
    pre, applied = [], set()
    for t in trees:
        slots, _ = lo.select_batch(clone(t), L, vl)
        pre.append(slots)
    for gi, (t, role) in enumerate(zip(trees, roles)):
        if role == "nan_child":  # every child of an expanded root child off slot 0's first step gets a NaN prior
            first = pre[gi][0][1]
            while first > 0 and t.parent[first] != 0:
                first = t.parent[first]
            xs = [c for c in t.children[0] if t.children[c] and c != first]
            if xs:
                applied.add(gi)
                for ch in t.children[xs[0]]:
                    t.prior[ch] = float("nan")
            pre[gi] = lo.select_batch(clone(t), L, vl)[0]
    # node_cap: a middle slot of the in-progress leaves fits exactly (node_exact) or is one over (node_over)
    need = []
    for gi, t in enumerate(trees):
        cnt = {j: unique_legal(o, t.rec[node]) for j, (k, node) in enumerate(pre[gi])
               if k == lo.LEAF and o.game_result(t.rec[node])[0] == 0}
        need.append(cnt)
    node_cap = max(len(t.parent) + sum(c.values()) for t, c in zip(trees, need)) + 8
    n_boards = [len(t.materialised) for t in trees]
    board_room = max(len(t.materialised) for t in trees) + L + 8
    board_cap = L * (1 + board_room // L) + 2
    for gi, (t, role) in enumerate(zip(trees, roles)):
        js = sorted(need[gi])
        if role in ("node_exact", "node_over") and len(js) >= 2:
            mid = js[len(js) // 2]
            upto = sum(need[gi][j] for j in js if j <= mid)
            applied.add(gi)
            pad_nodes(t, node_cap - len(t.parent) - upto + (role == "node_over"))
        new = [j for j, (k, node) in enumerate(pre[gi]) if k == lo.LEAF and node not in t.materialised]
        if role in ("board_exact", "board_over") and len(new) >= 2:
            mid = new[len(new) // 2]
            room = sum(j <= mid for j in new) - (role == "board_over")
            n_boards[gi] = board_cap - room
            applied.add(gi)
    return trees, n_boards, node_cap, board_cap, applied


ROLES = ["plain", "nan_child", "node_exact", "node_over", "board_exact", "board_over", "plain", "nan_child"]


def run_batch(R, L, vl, trees, roles, n_boards, node_cap, board_cap):
    """One select + FakeNet + expand/backup on the device and on the restatement; every check.  Returns counts over the
    batch and, per game, what happened: select / expand error bits, final node and board counts against the caps, and
    the backup entries (nodes on the leaf slots' paths)."""
    o = oracle_for(R)
    n = len(trees)
    m = new_mcts(R, n, L, vl, node_cap, board_cap - 2)
    assert m.board_cap >= board_cap
    n_boards = [nb + (m.board_cap - board_cap) for nb in n_boards]  # the same room with the device's board_cap
    load(m, trees, n_boards)
    slabs_before = {name: host(getattr(m, name)) for name in NODE_I32 + ("value_sum", "prior")}
    planes = m.select()
    torch.cuda.synchronize()
    kind, snode = host(m.slot_kind).reshape(n, -1)[:, :L], host(m.slot_node).reshape(n, -1)[:, :L]
    sboards, sstatus = host(m.slot_boards), host(m.slot_status)
    inf, err, drop = host(m.in_flight), host(m.error), host(m.dropped)
    board_idx, nb_dev, pool = host(m.board_idx), host(m.n_boards), host(m.boards)
    stats = dict(leaf=0, coll=0, empty=0, terminal_mid=0, err=0)
    games = [dict() for _ in trees]
    slots_all, results_all = [], []
    for gi, t in enumerate(trees):
        before_mat = set(t.materialised)
        room = m.board_cap - n_boards[gi]
        slots, e = lo.select_batch(t, L, vl, board_room=room)
        slots_all.append(slots)
        assert [k for k, _ in slots] == kind[gi].tolist(), (gi, roles[gi])
        assert [nd for _, nd in slots] == snode[gi].tolist(), (gi, roles[gi])
        assert err[gi] == e and drop[gi] == (1 if e else 0), (gi, roles[gi], err[gi], e)
        want_inf = np.zeros(m.node_cap, np.int32)
        for x, c in t.in_flight.items():
            want_inf[x] = c
        assert np.array_equal(inf[gi], want_inf), (gi, roles[gi])
        nb = n_boards[gi]
        res = []
        for j, (k, node) in enumerate(slots):
            s = gi * m.leaves + j
            if k == lo.EMPTY:
                res.append(0)
                continue
            assert np.array_equal(sboards[s], t.rec[node]), (gi, j)
            r = o.game_result(t.rec[node])[0]
            assert (sstatus[s] & 3) == r, (gi, j)
            res.append(r)
            if k == lo.LEAF and node not in before_mat:
                assert board_idx[gi, node] == nb and np.array_equal(pool[gi, nb], t.rec[node]), (gi, j)
                nb += 1
            stats["terminal_mid"] += k == lo.LEAF and r != 0 and j > 0
        assert nb_dev[gi] == nb, gi
        results_all.append(res)
        stats["leaf"] += sum(k == lo.LEAF for k, _ in slots)
        stats["coll"] += sum(k == lo.COLLISION for k, _ in slots)
        stats["empty"] += sum(k == lo.EMPTY for k, _ in slots)
        stats["err"] += bool(e)
        entries = 0
        for k, node in slots:
            while k == lo.LEAF and node >= 0:
                entries += 1
                node = t.parent[node]
        games[gi].update(select_err=int(err[gi]), entries=entries)
    assert host(m.collisions).tolist() == [t.collisions for t in trees]

    logits, value = m.net(planes)
    m.expand_backup(logits, value)
    torch.cuda.synchronize()
    lg, val = logits.cpu(), value.reshape(-1).cpu().numpy()
    ks = host(m.slot_k)
    got = {name: host(getattr(m, name)) for name in NODE_I32 + ("value_sum", "prior")}
    assert not host(m.in_flight).any()
    errs, drops, nn_dev = host(m.error), host(m.dropped), host(m.n_nodes)
    for gi, t in enumerate(trees):
        base = gi * m.leaves

        def children(j, gi=gi, t=t):
            s = base + j
            rec = t.rec[slots_all[gi][j][1]]
            ((flats, probs),) = lo.leaf_priors(o, lg[s: s + 1], [int(ks[s])], rec[None], False)
            return flats, probs

        n0 = len(t.parent)
        e2, d2 = lo.expand_backup_batch(t, slots_all[gi], results_all[gi], val[base: base + L], children,
                                        node_cap=m.node_cap)
        assert errs[gi] == err[gi] | e2, (gi, roles[gi], errs[gi], e2)
        assert drops[gi] == int(bool(drop[gi] or d2)), gi
        nn = len(t.parent)
        assert nn_dev[gi] == nn, (gi, roles[gi])
        games[gi].update(expand_err=int(e2), nodes_full=nn == m.node_cap, boards_full=int(nb_dev[gi]) == m.board_cap)
        assert got["parent"][gi, :nn].tolist() == t.parent
        assert got["visits"][gi, :nn].tolist() == t.visits
        assert got["move_flat"][gi, :nn].tolist() == t.move_flat
        assert got["value_sum"][gi, :nn].view(np.float64).tolist() == t.value_sum  # f64, bit-exact
        np.testing.assert_allclose(got["prior"][gi, n0:nn].view(np.float32), np.array(t.prior[n0:], np.float32),
                                   rtol=PRIOR_RTOL, atol=0)
        for node in range(nn):
            ch = t.children[node]
            assert got["n_children"][gi, node] == len(ch)
            if ch:
                assert got["first_child"][gi, node] == ch[0], (gi, node)
        for name in NODE_I32 + ("value_sum", "prior"):  # nothing past the node count was touched
            assert np.array_equal(got[name][gi, nn:], slabs_before[name][gi, nn:]), (gi, name)
    return stats, games


@pytest.mark.parametrize("R", [8, 10, 13, 14])
@pytest.mark.parametrize("L", [2, 8, 64, MAX_LEAVES_PER_GAME])
def test_leaf_batch_matches_the_restatement(R, L):
    o = oracle_for(R)
    base = searched_trees(R, 8, 40)
    roles = ROLES[: len(base)]
    trees, n_boards, node_cap, board_cap, applied = plan(o, base, L, 1, roles)
    stats, games = run_batch(R, L, 1, trees, roles, n_boards, node_cap, board_cap)
    # every role that could be set up did what it is there for
    for gi in applied:
        g, role = games[gi], roles[gi]
        if role == "node_exact":
            assert g["nodes_full"], (gi, g)  # the middle slot's children end exactly at node_cap
        elif role == "node_over":
            assert g["expand_err"] & lo.ERR_NODE_CAP, (gi, g)
        elif role == "board_exact":
            assert g["boards_full"], (gi, g)  # the middle slot's board takes the arena's last slot
        elif role == "board_over":
            assert g["select_err"] & lo.ERR_BOARD_CAP, (gi, g)
    if L >= 8:
        assert {roles[gi] for gi in applied} == set(ROLES) - {"plain"}, applied
    if L >= 64:  # a later slot reached the child whose children all have NaN priors
        assert any(games[gi]["select_err"] & lo.ERR_NO_CHILD for gi in applied if roles[gi] == "nan_child")
    # a second batch with a larger virtual loss on the same trees (marks cleared, arenas as left by the first)
    trees2 = [lo.prepare(clone(t)) for t in searched_trees(R, 8, 40)]
    stats2, _ = run_batch(R, L, 3, trees2, ["plain"] * len(trees2), [len(t.materialised) for t in trees2],
                       max(len(t.parent) for t in trees2) + L * FPC_MAX_MOVES,
                       max(len(t.materialised) for t in trees2) + L + 10)
    print(f"R={R} L={L}: VL 1 {stats}; VL 3 {stats2}")
    assert stats["err"] >= 1  # the NaN-prior child or a cap ended some game's batch in the middle
    if R == 8 and L >= 64:
        assert stats["terminal_mid"] >= 1  # a terminal leaf in mid-batch (late 8x8 positions)


def chain_tree(o, R, depth):
    """root -> a chain of `depth` single children (every node on the root's board) -> a node expanded with one child per
    legal move of that board."""
    rec = start_record(START[R])
    t = Tree(o, C_PUCT, rec)
    rng = np.random.default_rng(depth + R)
    node = 0
    for _ in range(depth):
        t.parent.append(node)
        t.children.append([])
        t.visits.append(int(rng.integers(20, 60)))
        t.value_sum.append(float(rng.normal(0.0, 5.0)))
        t.prior.append(float(np.float32(rng.uniform(0.1, 1.0))))
        t.move_flat.append(-1)
        t.rec.append(rec)
        t.children[node].append(len(t.parent) - 1)
        node = len(t.parent) - 1
    flats = sorted({o.move_flat_index(mv) for mv in o.legal_moves(rec)})
    probs = [float(np.float32(p)) for p in rng.dirichlet(np.ones(len(flats)))]
    t.expand(node, flats, probs)
    t.visits[0] = 100
    lo.prepare(t)
    t.materialised = set(range(depth + 1))
    return t


@pytest.mark.parametrize("R", [8, 14])
@pytest.mark.parametrize("L", [8, 64])
def test_300_deep_chain(R, L):
    """Paths of 302 nodes: past the descent's shared-memory path (walk up for the marks) and, at L = 64, more backup
    entries than the commit kernel sorts in shared memory (its serial fallback)."""
    o = oracle_for(R)
    trees = [chain_tree(o, R, 300) for _ in range(2)]
    stats, games = run_batch(R, L, 1, trees, ["chain"] * 2, [301, 301], 301 + 400 + L * FPC_MAX_MOVES, 301 + L + 10)
    entries = [g["entries"] for g in games]
    print(f"R={R} L={L} chain: {stats}; backup entries per game {entries}")
    assert stats["leaf"] >= 2 * min(L, 2)
    if L == 8:
        assert all(SORTED_BACKUP_ENTRIES >= e > 300 for e in entries)  # the sorted backup
    else:
        assert all(e > SORTED_BACKUP_ENTRIES for e in entries)  # the serial fallback


@pytest.mark.parametrize("R", [8, 10, 13, 14])
@pytest.mark.parametrize("batch_rotation", [0, 1])
def test_one_slot_equals_fpc_tree_select(R, batch_rotation):
    """At L = 1 the leaf calls give the slabs of fpc_tree_select + fpc_tree_expand_backup bit for bit, and, for every
    game with a leaf, the same k and planes (batch_rotation: leaves_batch_k_kernel against tree_batch_k_kernel)."""
    trees = [lo.prepare(clone(t)) for t in searched_trees(R, 8, 40)]
    n = len(trees)
    node_cap = max(len(t.parent) for t in trees) + 400
    out, seen = [], []
    L_ = _lib.lib()
    for leafy in (False, True):
        m = new_mcts(R, n, 1, 1, node_cap, 60)
        load(m, trees, [len(t.materialised) for t in trees])
        net = FakeNet(R, device="cuda")
        seen.append([])
        for _ in range(3):  # three batches: the later ones descend through the children the earlier ones made
            planes = torch.zeros((n, 24, R, R), device="cuda")
            st = torch.cuda.current_stream().cuda_stream
            if leafy:
                _lib.check(L_.fpc_tree_select_leaves(C.byref(m.desc), C.byref(m.batch), batch_rotation,
                                                     planes.data_ptr(), 0, None, st))
                k = m.slot_k[:n]
            else:
                _lib.check(L_.fpc_tree_select(C.byref(m.desc), batch_rotation, planes.data_ptr(), 0, None, st))
                k = m.k
            live = m.leaf >= 0  # a dropped game's row is evaluated from a stale board and ignored
            seen[-1].append((host(live), host(k)[host(live)], host(planes)[host(live)]))
            logits, value = net(planes)
            logits, value = logits.contiguous(), value.reshape(-1).contiguous()
            if leafy:
                _lib.check(L_.fpc_tree_expand_backup_leaves(C.byref(m.desc), C.byref(m.batch), logits.data_ptr(),
                                                            value.data_ptr(), st))
            else:
                _lib.check(L_.fpc_tree_expand_backup(C.byref(m.desc), logits.data_ptr(), value.data_ptr(), st))
        torch.cuda.synchronize()
        out.append({name: host(getattr(m, name)) for name in NODE_I32 + ("value_sum", "prior", "n_nodes", "n_boards",
                                                                           "boards", "dropped", "error", "leaf")})
        if leafy:
            assert not host(m.in_flight).any() and not host(m.collisions).any()
    for name in out[0]:
        assert np.array_equal(out[0][name], out[1][name]), name
    for (la, ka, pa), (lb, kb, pb) in zip(*seen):
        assert np.array_equal(la, lb) and la.any()
        assert np.array_equal(ka, kb) and np.array_equal(pa, pb)


def test_bad_arguments_are_rejected_before_any_launch():
    R, n = 8, 4
    m = new_mcts(R, n, 2, 1, 64, 8)
    L_ = _lib.lib()
    planes = torch.zeros((2 * n, 24, R, R), device="cuda")
    logits = torch.zeros((2 * n, m.geom.action_space_size + 1), device="cuda")
    values = torch.zeros(2 * n, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    before = {name: host(getattr(m, name)) for name in NODE_I32 + ("in_flight", "slot_kind", "n_nodes")}
    for L, vl in ((0, 1), (MAX_LEAVES_PER_GAME + 1, 1), (2, 0), (-1, 1)):
        m.batch.L, m.batch.virtual_loss = L, vl
        assert L_.fpc_tree_select_leaves(C.byref(m.desc), C.byref(m.batch), 0, planes.data_ptr(), 0, None,
                                         st) == _lib.FPC_ERR_ARG
        assert L_.fpc_tree_expand_backup_leaves(C.byref(m.desc), C.byref(m.batch), logits.data_ptr(),
                                                values.data_ptr(), st) == _lib.FPC_ERR_ARG
    m.batch.L, m.batch.virtual_loss = 2, 1
    assert L_.fpc_tree_expand_backup_leaves(C.byref(m.desc), C.byref(m.batch), logits.data_ptr() + 4,
                                            values.data_ptr(), st) == _lib.FPC_ERR_ARG
    assert b"aligned" in L_.fpc_last_error()
    m.batch.in_flight = None
    assert L_.fpc_tree_select_leaves(C.byref(m.desc), C.byref(m.batch), 0, planes.data_ptr(), 0, None,
                                     st) == _lib.FPC_ERR_ARG
    assert L_.fpc_tree_select_leaves(C.byref(m.desc), None, 0, planes.data_ptr(), 0, None, st) == _lib.FPC_ERR_ARG
    torch.cuda.synchronize()
    after = {name: host(getattr(m, name)) for name in before}
    for name in before:
        assert np.array_equal(before[name], after[name]), name
    with pytest.raises(ValueError):
        BatchedMCTS(R, n, None, {"C": 3, "num_searches": 10}, leaves_per_game=4)
    with pytest.raises(ValueError):
        BatchedMCTS(R, n, None, {"C": 3, "num_searches": 10}, leaves_per_game=2, virtual_loss=0)
