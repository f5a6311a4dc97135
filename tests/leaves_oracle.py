"""TEST INFRASTRUCTURE.  Leaf-parallel PUCT (several leaf slots per game in one network batch, with a virtual loss) on top
of the MCTS restatement (oracle/mcts_port.py), the reference that fpc_tree_select_leaves / fpc_tree_expand_backup_leaves
and BatchedMCTS(leaves_per_game=L) are checked against.  Leaf parallelism is outside the reference (one leaf per game
and simulation, `mcts.py:17-43`); this module restates the batch semantics of include/fpc.h without changing the
restatement's Tree:

- selection, slots j = 0 .. L-1 in order: descend with SelectChild over N_eff = visits + VL*in_flight and
  W_eff = value_sum - VL*in_flight; an endpoint with in_flight > 0 is a collision, else a leaf; +1 in_flight on the
  whole root -> endpoint path; a descent error drops the game and leaves this and the later slots empty;
- expand / backup in slot order: terminal leaf -> backup 0 / -1 and the game drops after the batch; leaf in progress
  -> backup, then its children (node_cap checked per slot against the running node count); in_flight back to zero.

A Tree gets three attributes here: in_flight (dict node -> count, empty between batches), collisions (running count)
and materialised (the set of nodes whose board the device would hold: the root and every node selected as a leaf)."""
from __future__ import annotations

import math

import numpy as np
import torch

from oracle.mcts_port import Tree

EMPTY, LEAF, COLLISION = 0, 1, 2
ERR_NODE_CAP, ERR_BOARD_CAP, ERR_NO_CHILD = 1, 2, 4


def prepare(t: Tree) -> Tree:
    if not hasattr(t, "in_flight"):
        t.in_flight = {}
        t.collisions = 0
        t.materialised = {0} | {i for i, v in enumerate(t.visits) if v > 1}
    return t


def select_child_vl(t: Tree, node: int, vl: int) -> int:
    """node.cpp:49-78 over the effective statistics; -1 when no child is selectable."""
    f = t.in_flight
    best, best_ucb = -1, -math.inf
    lg = math.log(math.sqrt(float(t.visits[node] + vl * f.get(node, 0))))
    for ch in t.children[node]:
        loss = vl * f.get(ch, 0)
        n = t.visits[ch] + loss
        q = (t.value_sum[ch] - float(loss)) / n if n > 0 else 0.0
        ucb = q + t.C * math.sqrt(lg / (1 + n)) * t.prior[ch]
        if ucb > best_ucb:
            best, best_ucb = ch, ucb
    return best


def select_batch(t: Tree, L: int, vl: int, board_room: int | None = None):
    """The L slots of one game: ([(kind, node)] * L, error bits).  board_room = boards the arena can still take (None:
    unlimited)."""
    prepare(t)
    slots, err = [], 0
    for _ in range(L):
        path = [0]
        while t.children[path[-1]]:
            ch = select_child_vl(t, path[-1], vl)
            if ch < 0:
                err = ERR_NO_CHILD
                break
            path.append(ch)
        if err:
            break
        e = path[-1]
        coll = t.in_flight.get(e, 0) > 0
        if not coll and e not in t.materialised:
            if board_room is not None and board_room <= 0:
                err = ERR_BOARD_CAP
                break
            t.materialised.add(e)
            board_room = None if board_room is None else board_room - 1
        for x in path:
            t.in_flight[x] = t.in_flight.get(x, 0) + 1
        t.collisions += coll
        slots.append((COLLISION if coll else LEAF, e))
    return slots + [(EMPTY, -1)] * (L - len(slots)), err


def expand_backup_batch(t: Tree, slots, results, values, children, node_cap: int | None = None):
    """Slots in order; results[j] = GameResult of slot j's board, values[j] its value, children(j) -> (flats, priors)
    of a leaf in progress.  Returns (error bits, whether the game drops)."""
    err, drop = 0, False
    for j, (kind, node) in enumerate(slots):
        if kind != LEAF:
            continue
        if results[j]:
            t.backpropagate(node, 0.0 if results[j] == 3 else -1.0)
            drop = True
            continue
        t.backpropagate(node, float(values[j]))
        flats, probs = children(j)
        if node_cap is not None and len(t.parent) + len(flats) > node_cap:
            err |= ERR_NODE_CAP
            continue
        t.expand(node, flats, probs)
    t.in_flight.clear()
    return err, drop


def leaf_priors(o, logits: torch.Tensor, ks, recs, batch_rotation: bool):
    """mcts.py:67-76 on a batch of leaves: soft-max, rot90 by -k, legal mask, renormalise, op for op as mcts_port.search
    does it (the whole batch rotated at once under batch_rotation: the layout decides the order of the f32 sum).
    Returns [(flats, probs)] in row order, nonzero() order = ascending flat index."""
    R, A = o.R, o.A
    pol = torch.softmax(logits, dim=1).view(-1, A, R, R)
    if batch_rotation:
        pol = torch.rot90(pol, -int(ks[0]), (-2, -1))
    else:
        pol = torch.stack([torch.rot90(pol[i], -int(ks[i]), (-2, -1)) for i in range(len(recs))])
    pol = pol * torch.from_numpy(o.mask(recs))
    pol = pol / torch.sum(pol, dim=(1, 2, 3), keepdim=True)
    flat = pol.reshape(len(recs), -1)
    out = []
    for i in range(len(recs)):
        nz = torch.nonzero(flat[i]).view(-1)
        out.append((nz.tolist(), flat[i][nz].tolist()))
    return out


def search_leaves(o, net, root_recs, C: float, num_searches: int, L: int, vl: int, batch_rotation: bool = True,
                  replay=None, prior_source=None, prior_rtol: float = 2e-6, trees=None):
    """num_searches / L batches of L leaf slots per game, from fresh roots at root_recs (or on top of `trees`, updated
    in place).  replay(batch, slots) -> (logits [k, A*R*R], value [k, 1]) stands in for the network, slots = the
    [(game, j)] leaf slots in progress of the batch in g-major / j-minor order; prior_source [n_games][node_cap] f32
    pins the stored priors to recorded bits after checking them against the ones computed here within prior_rtol (as
    in mcts_port.search)."""
    if num_searches % L:
        raise ValueError(f"L={L} does not divide num_searches={num_searches}")
    off_turn = o.R * o.R
    trees = [Tree(o, C, r) for r in root_recs] if trees is None else list(trees)
    for t in trees:
        prepare(t)
    live = [True] * len(trees)
    for batch in range(num_searches // L):
        slots = [select_batch(t, L, vl)[0] if live[gi] else [(EMPTY, -1)] * L for gi, t in enumerate(trees)]
        results = [[o.game_result(trees[gi].rec[node])[0] if kind == LEAF else 0 for kind, node in s]
                   for gi, s in enumerate(slots)]
        evals = [(gi, j) for gi, s in enumerate(slots) for j, (kind, _) in enumerate(s)
                 if kind == LEAF and results[gi][j] == 0]
        out = {}
        if evals:
            recs = np.stack([trees[gi].rec[slots[gi][j][1]] for gi, j in evals])
            turns = recs[:, off_turn].astype(np.int32)
            ks = np.full(len(evals), turns[0], np.int32) if batch_rotation else turns
            if replay is not None:
                logits, value = replay(batch, evals)
            else:
                logits, value = net(torch.from_numpy(o.encode(recs, ks)))
            pri = leaf_priors(o, logits, ks, recs, batch_rotation)
            vals = value.reshape(-1)
            for i, key in enumerate(evals):
                out[key] = (float(vals[i]), pri[i])
        for gi, t in enumerate(trees):
            if not live[gi]:
                continue

            def children(j, gi=gi, t=t):
                flats, probs = out[(gi, j)][1]
                if prior_source is not None:
                    first = len(t.parent)
                    rec = prior_source[gi][first: first + len(probs)]
                    np.testing.assert_allclose(rec, np.array(probs, dtype=np.float32), rtol=prior_rtol, atol=0)
                    probs = [float(x) for x in rec]
                return flats, probs

            values = [out[(gi, j)][0] if (gi, j) in out else 0.0 for j in range(L)]
            err, drop = expand_backup_batch(t, slots[gi], results[gi], values, children)
            if drop or any(k == EMPTY for k, _ in slots[gi]):
                live[gi] = False  # a terminal leaf, or a descent error (the restatement raises on the latter)
    return trees
