"""TEST INFRASTRUCTURE.  Dirichlet noise at the search root, restated in numpy from the recipe in include/fpc.h
(fpc_tree_root_noise), the reference that the kernel and BatchedMCTS(root_noise=True) are checked against.  Root noise
is outside the reference (alphazero.py:291-306 carries dirichlet_alpha / dirichlet_epsilon, mcts.py:45 defines
add_dirichlet_noise and nothing calls it), so the MCTS restatement has no notion of it; `NoisedTree` adds the hook
without changing the restatement: a Tree that noises its root's children once, when they exist.

Counter-based draws: child i of the game with key `key` reads U(i, j) = ((mix64(seed, key, i << 32 | j) >> 11) + 0.5)
* 2^-53; Gamma by Marsaglia-Tsang over at most 64 attempts of three uniforms each (3t, 3t+1, 3t+2), the alpha < 1
boost from U(i, 192)."""
from __future__ import annotations

import numpy as np

from oracle.mcts_port import Tree

ATTEMPTS = 64
TWO_PI = 6.283185307179586
M64 = (1 << 64) - 1


def mix64(seed, key, ctr):
    """csrc/fpc_device.cuh mix64 on uint64 arrays (wrapping arithmetic)."""
    seed, key, ctr = (np.asarray(x, dtype=np.uint64) for x in (seed, key, ctr))
    with np.errstate(over="ignore"):
        z = seed ^ (key * np.uint64(0x9E3779B97F4A7C15)) ^ (ctr * np.uint64(0xBF58476D1CE4E5B9))
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def as_u64(x):
    """Python / numpy integers (an i64 key may be negative) as their uint64 bit patterns."""
    return np.asarray(np.asarray(x, dtype=np.int64) if np.asarray(x).dtype.kind == "i" else x).astype(np.uint64)


def uniform(seed, key, i, j):
    ctr = (as_u64(i) << np.uint64(32)) | as_u64(j)
    return ((mix64(np.uint64(int(seed) & M64), as_u64(key), ctr) >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53


def gamma(seed, key, i, alpha: float):
    """Gamma(alpha, 1) draws for the (key, i) pairs (broadcast arrays), f64."""
    key, i = np.broadcast_arrays(as_u64(key), as_u64(i))
    a = alpha + 1.0 if alpha < 1.0 else float(alpha)
    d = a - 1.0 / 3.0
    c = 1.0 / np.sqrt(9.0 * d)
    g = np.full(key.shape, d)  # the fallback after ATTEMPTS rejections
    todo = np.ones(key.shape, bool)
    for t in range(ATTEMPTS):
        if not todo.any():
            break
        k, ii = key[todo], i[todo]
        x = np.sqrt(-2.0 * np.log(uniform(seed, k, ii, 3 * t))) * np.cos(TWO_PI * uniform(seed, k, ii, 3 * t + 1))
        v = 1.0 + c * x
        with np.errstate(invalid="ignore"):
            v3 = v * v * v
            ok = (v > 0.0) & (np.log(uniform(seed, k, ii, 3 * t + 2)) < 0.5 * x * x + d - d * v3 + d * np.log(v3))
        idx = np.flatnonzero(todo)[ok]
        g[idx] = d * v3[ok]
        todo[idx] = False
    if alpha < 1.0:
        g = g * uniform(seed, key, i, 3 * ATTEMPTS) ** (1.0 / alpha)
    return g


def dirichlet(seed, key, k: int, alpha: float):
    """eta [k] f64 for one game."""
    gam = gamma(seed, key, np.arange(k), alpha)
    s = gam.sum()
    return gam / s if s > 0.0 else np.full(k, 1.0 / k)


def noised(prior, seed, key, alpha: float, eps: float):
    """The root children's f32 priors after fpc_tree_root_noise (alpha and eps as the f32 values the call receives)."""
    prior = np.asarray(prior, np.float32)
    alpha, eps = float(np.float32(alpha)), float(np.float32(eps))
    eta = dirichlet(seed, key, len(prior), alpha)
    return ((1.0 - eps) * prior.astype(np.float64) + eps * eta).astype(np.float32)


class NoisedTree(Tree):
    """A restatement Tree whose root children get the noise once: at once when the root is already expanded (call
    `noise_root`), else when the search expands the root.  adopt [k] f32 (optional): the device's noised priors, checked
    against the restatement within rtol and then stored as they are, so that everything downstream compares exactly
    (as mcts_port.search's prior_source does for the network's priors)."""

    def setup_noise(self, seed, key, alpha, eps, adopt=None, rtol=1e-6):
        self.noise = dict(seed=seed, key=int(key), alpha=alpha, eps=eps)
        self.adopt, self.rtol, self.noised_root = adopt, rtol, False
        return self

    def noise_root(self):
        ch = self.children[0]
        if self.noised_root or not ch:
            return
        want = noised([self.prior[c] for c in ch], **self.noise)
        got = want
        if self.adopt is not None:
            got = np.asarray(self.adopt, np.float32)
            np.testing.assert_allclose(got, want, rtol=self.rtol, atol=0)
        for c, p in zip(ch, got):
            self.prior[c] = float(p)
        self.noised_root = True

    def expand(self, node, flats, probs):
        super().expand(node, flats, probs)
        if node == 0:
            self.noise_root()


def noised_tree(t: Tree, seed, key, alpha, eps, adopt=None) -> NoisedTree:
    """t (a Tree, e.g. re-rooted) as a NoisedTree sharing its state, with its root noised now if it has children."""
    out = NoisedTree.__new__(NoisedTree)
    out.__dict__.update(t.__dict__)
    out.setup_noise(seed, key, alpha, eps, adopt)
    out.noise_root()
    return out
