"""CPU: the leaf-parallel restatement (tests/leaves_oracle.py), the reference that the leaf-batch kernels and
BatchedMCTS(leaves_per_game=L) are checked against in tests/test_gpu_leaf_batch.py and tests/test_gpu_mcts_leaves.py."""
import numpy as np
import pytest

import tests.leaves_oracle as lo
from alphazero_4_player_chess_b200.fen import start_record
from oracle.mcts_port import search
from tests.golden.fake_net import FakeNet
from tests.util import mixed_positions, oracle_for

R, C_PUCT = 8, 3.0


def roots(n):
    o = oracle_for(R)
    pool = mixed_positions("EIGHT_SIMPLE", 300)
    return np.stack([r for r in pool[100::7] if o.game_result(r)[0] == 0][:n])


def fields(t):
    return dict(parent=t.parent, children=t.children, visits=t.visits, value_sum=t.value_sum, prior=t.prior,
                move_flat=t.move_flat)


@pytest.mark.parametrize("batch_rotation", [True, False])
def test_one_leaf_per_game_is_the_restatement(batch_rotation):
    o = oracle_for(R)
    rs = roots(6)
    want = search(o, FakeNet(R), rs, C_PUCT, 30, batch_rotation=batch_rotation)
    got = lo.search_leaves(o, FakeNet(R), rs, C_PUCT, 30, 1, 1, batch_rotation=batch_rotation)
    assert [fields(t) for t in got] == [fields(t) for t in want]
    assert all(t.collisions == 0 for t in got)


@pytest.mark.parametrize("L", [2, 8, 32])
def test_first_batch_from_a_fresh_root_has_L_minus_1_collisions(L):
    o = oracle_for(R)
    (t,) = lo.search_leaves(o, FakeNet(R), [start_record("EIGHT_SIMPLE")], C_PUCT, L, L, 1)
    assert t.collisions == L - 1
    assert t.visits[0] == 2 and len(t.children[0]) > 0


@pytest.mark.parametrize("L,vl", [(4, 1), (8, 3), (16, 1)])
def test_marks_clear_and_root_visits_count_the_leaf_slots(monkeypatch, L, vl):
    o = oracle_for(R)
    kinds = []
    select, expand = lo.select_batch, lo.expand_backup_batch

    def logged_select(t, *a, **k):
        slots, err = select(t, *a, **k)
        kinds.append((id(t), [kd for kd, _ in slots]))
        return slots, err

    def checked_expand(t, *a, **k):
        out = expand(t, *a, **k)
        assert t.in_flight == {}
        return out

    monkeypatch.setattr(lo, "select_batch", logged_select)
    monkeypatch.setattr(lo, "expand_backup_batch", checked_expand)
    rs = roots(5)
    trees = lo.search_leaves(o, FakeNet(R), rs, C_PUCT, 64, L, vl, batch_rotation=False)
    for t in trees:
        ks = [k for tid, ks in kinds if tid == id(t) for k in ks]
        assert t.visits[0] == 1 + ks.count(lo.LEAF)
        assert t.collisions == ks.count(lo.COLLISION) >= L - 1
        assert t.in_flight == {}
    n_coll = sum(t.collisions for t in trees)
    print(f"L={L} VL={vl}: {n_coll} collisions over {len(trees) * 64} slots")


def test_virtual_loss_spreads_one_batch_over_distinct_leaves():
    o = oracle_for(R)
    (t,) = search(o, FakeNet(R), [start_record("EIGHT_SIMPLE")], C_PUCT, 40, batch_rotation=False)
    lo.prepare(t)
    slots, err = lo.select_batch(t, 8, 1)
    leaves = [n for k, n in slots if k == lo.LEAF]
    assert err == 0 and len(set(leaves)) == len(leaves) > 1
    assert t.in_flight[0] == 8
    assert all(not t.children[n] for _, n in slots)
    # slot 0 is the one-leaf selection
    node = 0
    while t.children[node]:
        node = t.select_child(node)
    assert slots[0] == (lo.LEAF, node)


def test_L_must_divide_the_simulations():
    with pytest.raises(ValueError):
        lo.search_leaves(oracle_for(R), FakeNet(R), roots(1), C_PUCT, 30, 4, 1)
