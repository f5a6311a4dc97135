"""CPU: the leaf-parallel Gumbel restatement (tests/gumbel_leaves_oracle.py) -- at L = 1 it is the sequential Gumbel
search of tests/gumbel_oracle.py and tests/gumbel_interior_oracle.py, tree for tree; its schedule on `issued` follows
the halving schedule step by step whatever the scores do between batches; and a search whose batches collide only at
the unexpanded root gives the root the schedule's visit counts, whatever L is."""
import numpy as np
import pytest

from alphazero_4_player_chess_b200.fen import start_record
from tests.golden.fake_net import FakeNet
from tests.gumbel_interior_oracle import GumbelInteriorTree
from tests.gumbel_leaves_oracle import make_trees, root_slot, search
from tests.gumbel_oracle import GumbelTree, considered_visits
from tests.reuse_oracle import search_on
from tests.util import oracle_for, playout_positions

SEED, C_PUCT = 0xB0A7, 3


def roots8(n):
    p = playout_positions("EIGHT_SIMPLE", False, n, 8)
    return [np.ascontiguousarray(r) for r in p["recs"][p["ply"] == 3]]


def same_tree(a, b):
    for name in ("parent", "children", "visits", "value_sum", "prior", "move_flat"):
        assert getattr(a, name) == getattr(b, name), name


@pytest.mark.parametrize("interior", [False, True])
def test_one_leaf_per_batch_is_the_sequential_gumbel_search(interior):
    o, sims, m = oracle_for(8), 16, 4
    roots = roots8(6)
    net = FakeNet(8)
    base = GumbelInteriorTree if interior else GumbelTree
    seq = [base(o, C_PUCT, r).setup_gumbel(SEED, g, m, sims - 1, 1.0) for g, r in enumerate(roots)]
    if interior:
        seq = [t.setup_interior() for t in seq]
    seq = search_on(o, net, seq, C_PUCT, sims, batch_rotation=False)
    par = search(o, net, make_trees(o, C_PUCT, roots, SEED, range(len(roots)), m, sims - 1, 1.0, 1, 1, interior),
                 sims, batch_rotation=False)
    for a, b in zip(seq, par):
        same_tree(a, b)
        assert b.collisions == 0
        if a.children[0]:
            assert list(b.issued) == [a.visits[c] - 1 for c in a.children[0]]
            assert a.root_value == b.root_value
            fa, pa = a.result()
            fb, pb = b.result_leaves()
            assert fa == fb and np.array_equal(pa, pb)
        if interior:
            assert a.node_value == b.node_value


@pytest.mark.parametrize("seed", range(6))
def test_issued_follows_the_schedule_step_by_step(seed):
    """Scores are redrawn every batch (collisions and backups move the committed statistics arbitrarily); the slots of
    a batch take candidates in turn.  Whatever the scores, every step's candidate set is non-empty and the issued
    counts, sorted, are those of the plain schedule after the same number of steps."""
    rng = np.random.default_rng(seed)
    for _ in range(40):
        k = int(rng.integers(1, 40))
        m = int(rng.integers(1, 20))
        L = int(rng.choice([1, 2, 3, 4, 8, 16]))
        n_sims = int(rng.integers(1, 80))
        mp = min(m, k)
        issued = np.zeros(k, np.int64)
        ref = np.zeros(k, np.int64)
        for step in range(n_sims + 2 * L):  # past n_sims too: the extended schedule
            if step % L == 0:
                sc = rng.normal(size=k)
                sc[rng.random(k) < 0.2] = -1e9  # floored scores tie
            i, cand = root_slot(issued, sc, mp, n_sims)
            assert i >= 0 and cand.any(), (k, m, L, n_sims, step)
            assert issued[i] == considered_visits(step, mp, n_sims)
            issued[i] += 1
            r, _ = root_slot(ref, np.zeros(k), mp, n_sims)
            ref[r] += 1
            assert np.array_equal(np.sort(issued), np.sort(ref)), step


@pytest.mark.parametrize("L", [2, 4, 8])
@pytest.mark.parametrize("interior", [False, True])
def test_collision_free_searches_give_the_schedules_visits(L, interior):
    """14x14 positions (20 and more moves): with m = 16 every batch can take L distinct root children.  In every
    search N_i <= I_i, and the visits lost are the collisions after the first batch; where there are none, N is
    the schedule's."""
    o, sims, m = oracle_for(14), 32, 16
    p = playout_positions("STANDARD", False, 6, 4)
    roots = [start_record("STANDARD")] + [np.ascontiguousarray(r) for r in p["recs"][p["ply"] == 2]]
    n_sims = sims - L
    trees = search(o, FakeNet(14), make_trees(o, C_PUCT, roots, SEED, range(len(roots)), m, n_sims, 1.0, L, 1,
                                              interior), sims, batch_rotation=False)
    clean = 0
    for t in trees:
        k = len(t.children[0])
        N = np.array([t.visits[c] - 1 for c in t.children[0]])
        assert (N <= t.issued).all()
        assert int((t.issued - N).sum()) == t.collisions - (L - 1) or int(t.issued.sum()) < n_sims
        if t.collisions != L - 1 or int(t.issued.sum()) != n_sims:
            continue  # collisions after the first batch, or a terminal leaf ended the search
        clean += 1
        assert np.array_equal(N, t.issued)
        ref = np.zeros(k, np.int64)
        for _ in range(n_sims):
            r, _ = root_slot(ref, np.zeros(k), min(m, k), n_sims)
            ref[r] += 1
        assert np.array_equal(np.sort(N), np.sort(ref))
        assert t.visits[0] == 1 + 1 + n_sims  # created with 1, its own expansion, then one visit per issue
    print(f"L={L} interior={interior}: {clean} of {len(trees)} searches collision-free below the root")
    assert clean >= 1
