"""TEST INFRASTRUCTURE.  Tree reuse on top of the MCTS restatement (oracle/mcts_port.py), the reference that the
device's fpc_tree_advance and BatchedMCTS.search(None) are checked against.  Reuse is outside the reference, which builds
a fresh Node per move (`mcts.py:28-31`), so the restatement itself has no notion of it; this module adds the two pieces
without changing the restatement: re-rooting a Tree, and running its search on top of given trees."""
from __future__ import annotations

from oracle import mcts_port
from oracle.mcts_port import Tree


def reroot(t: Tree, flat: int) -> Tree:
    """The subtree of t's root child that played `flat`, as a new Tree.  Nodes keep their statistics and are renumbered
    in ascending order of their old index, so the numbering matches the device's in-place compaction (and a recorded
    prior_source stays aligned); the new root gets parent -1, move -1 and prior 0.  A move that is not a root child gives
    a fresh Tree at the position after it."""
    c = next((ch for ch in t.children[0] if t.move_flat[ch] == flat), None)
    if c is None:
        return Tree(t.o, t.C, t.o.make_index(t.rec[0], int(flat)))
    member = [False] * len(t.parent)
    member[c] = True
    for i in range(c + 1, len(t.parent)):
        member[i] = member[t.parent[i]]  # parent[i] < i
    keep = [i for i in range(c, len(t.parent)) if member[i]]
    new = {old: k for k, old in enumerate(keep)}
    out = Tree(t.o, t.C, t.rec[c])
    out.parent = [-1] + [new[t.parent[i]] for i in keep[1:]]
    out.children = [[new[ch] for ch in t.children[i]] for i in keep]
    out.visits = [t.visits[i] for i in keep]
    out.value_sum = [t.value_sum[i] for i in keep]
    out.prior = [0.0] + [t.prior[i] for i in keep[1:]]
    out.move_flat = [-1] + [t.move_flat[i] for i in keep[1:]]
    out.rec = [t.rec[i] for i in keep]
    return out


def search_on(o, net, trees, C: float, num_searches: int, **kwargs):
    """mcts_port.search for num_searches more simulations on top of `trees` (updated in place and returned) instead of
    fresh roots.  The restatement's own loop runs unchanged: only the trees it starts from are swapped in, by handing
    its Tree constructor the given trees one by one for the duration of the call.  kwargs: those of mcts_port.search."""
    given = iter(trees)
    fresh = mcts_port.Tree
    mcts_port.Tree = lambda _o, _C, _rec: next(given)
    try:
        return mcts_port.search(o, net, [t.rec[0] for t in trees], C, num_searches, **kwargs)
    finally:
        mcts_port.Tree = fresh
