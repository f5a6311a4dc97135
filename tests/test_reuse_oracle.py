"""CPU: tree reuse on top of the MCTS restatement (tests/reuse_oracle.py: reroot and search_on), the reference that
fpc_tree_advance and BatchedMCTS.search(None) are checked against in tests/test_gpu_mcts_reuse.py."""
import numpy as np

from alphazero_4_player_chess_b200.fen import start_record
from oracle.mcts_port import Tree, search
from tests.reuse_oracle import reroot, search_on
from tests.golden.fake_net import FakeNet
from tests.util import oracle_for

R, C_PUCT = 8, 3.0


def searched_tree(sims=60):
    o = oracle_for(R)
    (t,) = search(o, FakeNet(R), [start_record("EIGHT_SIMPLE")], C_PUCT, sims, batch_rotation=False)
    return o, t


def subtree(t, c):
    out, stack = [], [c]
    while stack:
        node = stack.pop()
        out.append(node)
        stack += t.children[node]
    return sorted(out)


def fields(t):
    return dict(parent=t.parent, children=t.children, visits=t.visits, value_sum=t.value_sum, prior=t.prior,
                move_flat=t.move_flat, rec=[r.tolist() for r in t.rec])


def test_reroot_on_an_unexpanded_child_equals_a_fresh_tree():
    o, t = searched_tree()
    leaf = next(ch for ch in t.children[0] if not t.children[ch])
    flat = t.move_flat[leaf]
    got = reroot(t, flat)
    assert fields(got) == fields(Tree(o, C_PUCT, o.make_index(t.rec[0], flat)))
    assert got.visits == [t.visits[leaf]] == [1]


def test_reroot_keeps_every_node_of_the_subtree_in_index_order():
    o, t = searched_tree()
    expanded = [ch for ch in t.children[0] if t.children[ch]]
    assert len(expanded) >= 2
    for c in expanded:
        got = reroot(t, t.move_flat[c])
        keep = subtree(t, c)
        assert len(got.parent) == len(keep) > 1
        new = {old: k for k, old in enumerate(keep)}
        assert got.parent[0] == -1 and got.move_flat[0] == -1 and got.prior[0] == 0.0
        assert got.visits[0] == t.visits[c] and got.value_sum[0] == t.value_sum[c]
        assert np.array_equal(got.rec[0], o.make_index(t.rec[0], t.move_flat[c]))
        for old, k in new.items():
            assert got.visits[k] == t.visits[old] and got.value_sum[k] == t.value_sum[old]
            assert got.children[k] == [new[ch] for ch in t.children[old]]
            assert np.array_equal(got.rec[k], t.rec[old])
            if k:
                assert got.parent[k] == new[t.parent[old]] < k
                assert got.prior[k] == t.prior[old] and got.move_flat[k] == t.move_flat[old]
            kids = got.children[k]  # contiguous, ascending flat order
            if kids:
                assert kids == list(range(kids[0], kids[0] + len(kids)))
            assert [got.move_flat[ch] for ch in kids] == sorted(got.move_flat[ch] for ch in kids)


def test_search_continues_given_trees():
    o, t = searched_tree()
    c = max(t.children[0], key=lambda ch: t.visits[ch])
    kept = reroot(t, t.move_flat[c])
    before = fields(kept)
    n0, v0 = len(kept.parent), kept.visits[0]
    sims = 25
    (got,) = search_on(o, FakeNet(R), [kept], C_PUCT, sims, batch_rotation=False)
    assert got is kept
    assert got.visits[0] == v0 + sims  # no terminal leaf within reach of this opening: every simulation backs up
    assert len(got.parent) > n0
    for name in ("parent", "move_flat", "prior"):  # the carried nodes keep their places
        assert getattr(got, name)[:n0] == before[name][:n0]
    # a fresh search from the same position is a different tree: the carried statistics steer the descent
    (fresh,) = search(o, FakeNet(R), [kept.rec[0]], C_PUCT, sims, batch_rotation=False)
    assert fresh.visits[0] == 1 + sims and fields(fresh) != fields(got)

