"""TEST INFRASTRUCTURE.  The leaf-parallel Gumbel search restated in numpy from include/fpc.h
(fpc_tree_select_gumbel_leaves / fpc_tree_gumbel_result_leaves), the reference that the kernels and
BatchedMCTS(gumbel=True, gumbel_leaves=L) are checked against.  It joins the two restatements it is built from without
changing either: tests/leaves_oracle.py's leaf batch (effective statistics, collisions, in_flight marks, the slot-order
commit) and tests/gumbel_oracle.py / tests/gumbel_interior_oracle.py's root and interior rules.

A `GumbelLeavesTree` is a GumbelInteriorTree (the Gumbel root recipe, the interior rule and its node_value cache) that
also carries the leaf batch's state (leaves_oracle.prepare) and `issued`, the schedule's visit count I_i per root child.
Its select_batch() is one batch's selection of one game:
- root not expanded: every slot ends at the root, one LEAF and L - 1 COLLISIONs; issued untouched;
- root expanded: the scores once per batch from the committed statistics (root_value cached at s == 0), then per slot
  the first maximum over {I_i == cv(sum I)} with the schedule planned for n_sims, I_i += 1, and the descent below with
  SelectChild over the effective statistics (or, interior, the interior rule over them, its node value following the
  committed s);
- a failed descent sets its error bit, leaves this and every later slot EMPTY and gives the slot's issue back.
Near-ties: where a device choice (device_slots: the endpoint the device recorded per batch and slot) differs from the
restatement's, it is adopted only within the tolerances of the Gumbel restatements, and counted."""
from __future__ import annotations

import numpy as np
import torch

from tests.gumbel_interior_oracle import TIE, GumbelInteriorTree, interior_choice
from tests.gumbel_oracle import argmax_among, considered_visits, gumbels, logits_sigma, scores, warp_sum
from tests.leaves_oracle import (COLLISION, EMPTY, ERR_BOARD_CAP, ERR_NO_CHILD, LEAF, expand_backup_batch, leaf_priors,
                                 prepare, select_child_vl)


def root_slot(issued, sc, mp: int, n_sims: int):
    """(child index a slot takes, the candidate mask): the first maximum of sc over {I_i == cv(sum I)}, -1 when empty."""
    cand = np.asarray(issued) == considered_visits(int(np.sum(issued)), mp, n_sims)
    return argmax_among(sc, cand), cand


class GumbelLeavesTree(GumbelInteriorTree):
    def setup_leaves(self, L: int, vl: int = 1, interior: bool = False, device_slots=None):
        """device_slots (optional): [batch][j] the endpoint node of slot j as the device recorded it (-1 for EMPTY)."""
        prepare(self)
        self.setup_interior()
        self.L, self.vl, self.interior = int(L), int(vl), bool(interior)
        self.issued = None  # np.int64 [k] once the root is expanded
        self.device_slots, self.batches = device_slots, 0
        return self

    # ---- the device's choice at a node, read off the endpoint it recorded ----------------------------------------------
    def _device_child(self, x: int, j: int):
        if self.device_slots is None:
            return None
        node = int(self.device_slots[self.batches][j])
        while node >= 0 and self.parent[node] != x:
            node = self.parent[node]
        return node if node >= 0 else None

    def _interior_step(self, x: int, j: int) -> int:
        """the interior rule at x over the effective statistics; x's value follows the committed s."""
        f, vl = self.in_flight, self.vl
        ch = self.children[x]
        committed = np.array([self.visits[c] - 1 for c in ch], np.int64)
        loss = np.array([vl * f.get(c, 0) for c in ch], np.int64)
        N = committed + loss
        W = np.array([self.value_sum[c] - float(vl * f.get(c, 0)) for c in ch])
        prior = np.array([self.prior[c] for c in ch], np.float32)
        if int(committed.sum()) == 0:
            assert self.node_value.get(x, self.value_sum[x]) == self.value_sum[x], ("node_value changed", x)
            if x not in self.node_value:
                self.log.append(("w", x, self.batches))
            self.node_value[x] = self.value_sum[x]
        else:
            assert x in self.node_value, ("node_value read before it was written", x, self.batches)
            self.log.append(("r", x, self.batches))
        i, sc = interior_choice(N, W, prior, self.node_value[x])
        d = self._device_child(x, j)
        if d is not None and i >= 0 and d != ch[i]:
            k = ch.index(d)
            assert abs(sc[k] - sc[i]) <= TIE, (self.batches, j, x, i, k, sc[i], sc[k])
            i, self.adopted_interior = k, self.adopted_interior + 1
        return ch[i] if i >= 0 else -1

    def select_batch(self, board_room: int | None = None):
        """The L slots of this game's next batch: ([(kind, node)] * L, error bits)."""
        L, vl, gb = self.L, self.vl, self.gb
        root_ch = self.children[0]
        k = len(root_ch)
        if k:
            N, vs, prior = self.root_stats()
            if int(N.sum()) == 0:
                self.root_value = self.value_sum[0]
            if self.issued is None:
                self.issued = np.zeros(k, np.int64)
            z, _ = logits_sigma(N, vs, prior, self.root_value)
            sc = scores(z, gumbels(gb["seed"], gb["key"], k, gb["scale"]))
            mp = min(gb["m"], k)
        slots, err = [], 0
        for j in range(L):
            path, took = [0], -1
            if k:
                i, cand = root_slot(self.issued, sc, mp, gb["n_sims"])
                d = self._device_child(0, j)
                if d is not None and i >= 0 and d != root_ch[i]:
                    jd = root_ch.index(d)
                    assert cand[jd] and abs(sc[jd] - sc[i]) <= 1e-12 * abs(sc[i]), (self.batches, j, i, jd)
                    i, self.adopted = jd, self.adopted + 1
                if i < 0:
                    err = ERR_NO_CHILD
                    break
                self.issued[i] += 1
                took = i
                path.append(root_ch[i])
            while self.children[path[-1]]:
                x = path[-1]
                ch = self._interior_step(x, j) if self.interior else select_child_vl(self, x, vl)
                if ch < 0:
                    err = ERR_NO_CHILD
                    break
                path.append(ch)
            e = path[-1]
            coll = not err and self.in_flight.get(e, 0) > 0
            if not err and not coll and e not in self.materialised:
                if board_room is not None and board_room <= 0:
                    err = ERR_BOARD_CAP
                else:
                    self.materialised.add(e)
                    board_room = None if board_room is None else board_room - 1
            if err:
                if took >= 0:
                    self.issued[took] -= 1  # an EMPTY slot issues no visit
                break
            for x in path:
                self.in_flight[x] = self.in_flight.get(x, 0) + 1
            self.collisions += coll
            slots.append((COLLISION if coll else LEAF, e))
        self.batches += 1
        return slots + [(EMPTY, -1)] * (L - len(slots)), err

    def result_leaves(self):
        """(action flat, improved policy [k] f32): gumbel_oracle.result with the survivors {I_i == max I}."""
        if not self.children[0]:
            return -1, np.zeros(0, np.float32)
        N, vs, prior = self.root_stats()
        root = self.value_sum[0] if int(N.sum()) == 0 else self.root_value
        issued = self.issued if self.issued is not None else np.zeros(len(N), np.int64)
        z, _ = logits_sigma(N, vs, prior, root)
        best = argmax_among(scores(z, gumbels(self.gb["seed"], self.gb["key"], len(N), self.gb["scale"])),
                            issued == issued.max())
        e = np.exp(z - z.max())
        return self.move_flat[self.children[0][best]], (e / warp_sum(e)).astype(np.float32)


def make_trees(o, C, root_recs, seed, keys, m, n_sims, scale, L, vl=1, interior=False, device_slots=None):
    return [GumbelLeavesTree(o, C, r).setup_gumbel(seed, keys[g], m, n_sims, scale)
            .setup_leaves(L, vl, interior, None if device_slots is None else device_slots[g])
            for g, r in enumerate(root_recs)]


def search(o, net, trees, num_searches: int, batch_rotation: bool = True, replay=None, prior_source=None,
           prior_rtol: float = 2e-6):
    """num_searches / L batches over `trees` (GumbelLeavesTree, updated in place and returned): tests/leaves_oracle.py's
    search_leaves loop with the trees' own select_batch.  replay(batch, slots) -> (logits, value) stands in for the
    network, slots = the [(game, j)] LEAF slots in progress in g-major / j-minor order; prior_source pins the stored
    priors to the device's bits after an rtol check."""
    L = trees[0].L
    if num_searches % L:
        raise ValueError(f"L={L} does not divide num_searches={num_searches}")
    off_turn = o.R * o.R
    live = [True] * len(trees)
    for batch in range(num_searches // L):
        slots = []
        for gi, t in enumerate(trees):
            if live[gi]:
                slots.append(t.select_batch()[0])
            else:
                slots.append([(EMPTY, -1)] * L)
                t.batches += 1
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
            _, drop = expand_backup_batch(t, slots[gi], results[gi], values, children)
            if drop or any(kind == EMPTY for kind, _ in slots[gi]):
                live[gi] = False
    return trees
