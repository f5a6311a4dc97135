"""TEST INFRASTRUCTURE.  The Gumbel root search restated in numpy from include/fpc.h (fpc_tree_select_gumbel /
fpc_tree_gumbel_result), the reference that the kernels and BatchedMCTS(gumbel=True) are checked against.  Gumbel root
search is outside the reference, so the MCTS restatement has no notion of it; `GumbelTree` adds it without changing the
restatement: a Tree whose choose_leaf takes the Gumbel root step and then descends with the restatement's SelectChild.

Sums run in the kernel's order (child i on lane i % 32, lanes ascending, then the xor butterfly 16 .. 1), so the f64
scores are the kernel's up to the last bits of log / exp.  The uniforms are tests/noise_oracle.py's at j = 2^31."""
from __future__ import annotations

import numpy as np

from oracle.mcts_port import Tree
from tests.noise_oracle import uniform

C_VISIT, C_SCALE = 50.0, 0.1
J = 1 << 31
FLOOR = -1e9


def considered_visits(s: int, m: int, n_sims: int) -> int:
    """cv(s) as the kernel computes it: mctx's schedule in closed form, the c = 2 tail summed at once."""
    if m <= 1:
        return s
    l2 = (m - 1).bit_length()  # ceil(log2 m)
    c, v = m, 0
    while c > 2:
        e = max(1, n_sims // (l2 * c))
        if s < e * c:
            return v + s // c
        s, v, c = s - e * c, v + e, max(2, c // 2)
    return v + s // 2


def warp_sum(x, mask=None) -> float:
    """sum of x[i] (over mask) in the kernel's order."""
    part = [0.0] * 32
    for i, v in enumerate(np.asarray(x, np.float64)):
        if mask is None or mask[i]:
            part[i % 32] += float(v)
    p = np.array(part)
    for o in (16, 8, 4, 2, 1):
        p = p + p[np.arange(32) ^ o]
    return float(p[0])


def gumbels(seed, key, k: int, scale: float):
    """g_i = scale * (-log(-log U_i)) for i < k; key may be an array (rows)."""
    key = np.asarray(key)
    u = uniform(seed, key[..., None], np.arange(k), J)
    return scale * -np.log(-np.log(u))


def logits_sigma(N, vs, prior, root: float, c_visit=C_VISIT, c_scale=C_SCALE):
    """z = l + sigma [k] f64 and s for the root children's N (visits - 1), value sums and f32 priors; root = the root's
    value_sum as the select found it at s == 0 (v = -root)."""
    N = np.asarray(N, np.int64)
    vs = np.asarray(vs, np.float64)
    p = np.asarray(prior, np.float32).astype(np.float64)
    s, nmax = int(N.sum()), int(N.max())
    with np.errstate(divide="ignore"):
        lp = np.log(p)
    vis = N > 0
    q = np.zeros(len(N))
    q[vis] = vs[vis] / N[vis]
    w = np.maximum(p, 2.0 ** -126)
    ws, wq = warp_sum(w, vis), warp_sum(w * q, vis)
    w_mean = wq / ws if ws > 0.0 else 0.0
    v_mix = (-root + float(s) * w_mean) / (1.0 + float(s))
    cq = np.where(vis, q, v_mix)
    lo, hi = cq.min(), cq.max()
    a = (c_visit + float(nmax)) * c_scale
    return (lp - lp.max()) + a * ((cq - lo) / max(hi - lo, 1e-8)), s


def scores(z, g):
    x = g + z
    return np.where(x > FLOOR, x, FLOOR)


def argmax_among(score, cand) -> int:
    """first maximum of score over cand, -1 when cand is empty."""
    if not np.any(cand):
        return -1
    return int(np.argmax(np.where(cand, score, -np.inf)))


def root_choice(N, vs, prior, root, seed, key, m, n_sims, scale, c_visit=C_VISIT, c_scale=C_SCALE):
    """(child index the select takes, its score vector) -- index -1 when no child is on the schedule."""
    N = np.asarray(N, np.int64)
    z, s = logits_sigma(N, vs, prior, root, c_visit, c_scale)
    sc = scores(z, gumbels(seed, key, len(N), scale))
    return argmax_among(sc, N == considered_visits(s, min(m, len(N)), n_sims)), sc


def result(N, vs, prior, root, seed, key, scale, c_visit=C_VISIT, c_scale=C_SCALE):
    """(child index of the action, improved policy [k] f32)."""
    N = np.asarray(N, np.int64)
    z, _ = logits_sigma(N, vs, prior, root, c_visit, c_scale)
    best = argmax_among(scores(z, gumbels(seed, key, len(N), scale)), N == N.max())
    e = np.exp(z - z.max())
    return best, (e / warp_sum(e)).astype(np.float32)


class GumbelTree(Tree):
    """A restatement Tree whose choose_leaf takes the Gumbel root step.  device_roots (optional): the root child (node)
    the device took at each of this tree's selects; where it differs from the restatement's choice, the device's is
    adopted only when the two scores are within a relative 1e-12 (a last-ulp difference of log between CUDA and numpy),
    counted in `adopted`."""

    def setup_gumbel(self, seed, key, m, n_sims, scale, device_roots=None):
        self.gb = dict(seed=seed, key=int(key), m=int(m), n_sims=int(n_sims), scale=float(scale))
        self.root_value, self.device_roots, self.selects, self.adopted = None, device_roots, 0, 0
        return self

    def root_stats(self):
        ch = self.children[0]
        return (np.array([self.visits[c] - 1 for c in ch]), np.array([self.value_sum[c] for c in ch]),
                np.array([self.prior[c] for c in ch], np.float32))

    def choose_leaf(self):
        sel, self.selects = self.selects, self.selects + 1
        ch = self.children[0]
        if not ch:
            return super().choose_leaf()
        N, vs, prior = self.root_stats()
        if int(N.sum()) == 0:
            self.root_value = self.value_sum[0]
        gb = self.gb
        i, sc = root_choice(N, vs, prior, self.root_value, gb["seed"], gb["key"], gb["m"], gb["n_sims"], gb["scale"])
        if self.device_roots is not None and self.device_roots[sel] >= 0 and ch[i] != self.device_roots[sel]:
            j = ch.index(self.device_roots[sel])
            assert abs(sc[j] - sc[i]) <= 1e-12 * abs(sc[i]), (sel, i, j, sc[i], sc[j])
            i, self.adopted = j, self.adopted + 1
        if i < 0:
            raise RuntimeError("Failed to select a child.")
        node = ch[i]
        while self.children[node]:
            node = self.select_child(node)
        res, _, _ = self.o.game_result(self.rec[node])
        if res != 0:
            self.backpropagate(node, 0.0 if res == 3 else -1.0)
            return None
        return node

    def result(self):
        """(action flat, improved policy [k] f32) after the search; (-1, []) for a root without children."""
        if not self.children[0]:
            return -1, np.zeros(0, np.float32)
        N, vs, prior = self.root_stats()
        root = self.value_sum[0] if int(N.sum()) == 0 else self.root_value
        i, pol = result(N, vs, prior, root, self.gb["seed"], self.gb["key"], self.gb["scale"])
        return self.move_flat[self.children[0][i]], pol
