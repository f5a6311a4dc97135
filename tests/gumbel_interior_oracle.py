"""TEST INFRASTRUCTURE.  Gumbel MuZero's interior selection restated in numpy from include/fpc.h
(fpc_tree_select_gumbel_interior), the reference that the kernel and BatchedMCTS(gumbel_interior=True) are checked
against.  `GumbelInteriorTree` is tests/gumbel_oracle.GumbelTree (the Gumbel root step, unchanged) whose steps below the
root take the interior rule instead of the restatement's SelectChild, with its own node_value cache.

The scores are built from tests/gumbel_oracle.py's pieces, in the kernel's sum order, so they are the kernel's up to the
last bits of log / exp.  Scores are differences in [-1, 1] near 0, so a near-tie is an absolute difference."""
from __future__ import annotations

import numpy as np

from tests.gumbel_oracle import C_SCALE, C_VISIT, GumbelTree, logits_sigma, warp_sum

TIE = 1e-12  # absolute: two interior scores this close may be ordered either way by CUDA's and numpy's log / exp


def improved_policy(N, vs, prior, u, c_visit=C_VISIT, c_scale=C_SCALE):
    """(pi' [k] f64, s) at a node whose children have N (visits - 1), value sums and f32 priors; u = the node's network
    value (v = -u)."""
    z, s = logits_sigma(N, vs, prior, u, c_visit, c_scale)
    e = np.exp(z - np.fmax.reduce(z))
    return e / warp_sum(e), s


def interior_scores(N, vs, prior, u, c_visit=C_VISIT, c_scale=C_SCALE):
    """score_i = pi'_i - N_i / (1 + s) [k] f64."""
    N = np.asarray(N, np.int64)
    pi, s = improved_policy(N, vs, prior, u, c_visit, c_scale)
    return pi - N.astype(np.float64) / (1.0 + float(s))


def first_max(score) -> int:
    """the first maximum of score in ascending i, -1 when no score compares greater than -inf (NaN)."""
    ok = score > -np.inf
    if not ok.any():
        return -1
    return int(np.argmax(np.where(ok, score, -np.inf)))


def interior_choice(N, vs, prior, u, c_visit=C_VISIT, c_scale=C_SCALE):
    """(child index the interior step takes or -1, the score vector)."""
    sc = interior_scores(N, vs, prior, u, c_visit, c_scale)
    return first_max(sc), sc


class GumbelInteriorTree(GumbelTree):
    """A GumbelTree whose descent below the root applies the interior rule.  node_value: the cache, {node: value},
    written at a node's first pass (s == 0) and read at every later one; `log` lists ("w" | "r", node, select) in
    order.  device_leaves (optional): the leaf the device took at each of this tree's selects; where the device's
    interior choice (the child of x above that leaf) differs from the restatement's, it is adopted only when the two
    scores are within an absolute TIE, counted in `adopted_interior`."""

    def setup_interior(self, device_leaves=None):
        self.node_value, self.log, self.device_leaves, self.adopted_interior = {}, [], device_leaves, 0
        return self

    def node_stats(self, x):
        ch = self.children[x]
        return (np.array([self.visits[c] - 1 for c in ch]), np.array([self.value_sum[c] for c in ch]),
                np.array([self.prior[c] for c in ch], np.float32))

    def device_child(self, x):
        """the child of x on the path to the device's leaf of the current select, None when unknown."""
        if self.device_leaves is None:
            return None
        node = int(self.device_leaves[self.selects - 1])
        while node >= 0 and self.parent[node] != x:
            node = self.parent[node]
        return node if node >= 0 else None

    def select_child(self, node: int) -> int:
        """the interior step at node > 0 (GumbelTree takes the root's step itself)"""
        N, vs, prior = self.node_stats(node)
        sel = self.selects - 1
        if int(N.sum()) == 0:
            assert node not in self.node_value, ("node_value written twice", node, sel)
            self.node_value[node] = self.value_sum[node]
            self.log.append(("w", node, sel))
        else:
            assert node in self.node_value, ("node_value read before it was written", node, sel)
            self.log.append(("r", node, sel))
        i, sc = interior_choice(N, vs, prior, self.node_value[node])
        ch = self.children[node]
        d = self.device_child(node)
        if d is not None and i >= 0 and d != ch[i]:
            j = ch.index(d)
            assert abs(sc[j] - sc[i]) <= TIE, (sel, node, i, j, sc[i], sc[j])
            i, self.adopted_interior = j, self.adopted_interior + 1
        if i < 0:
            raise RuntimeError("Failed to select a child.")
        return ch[i]
