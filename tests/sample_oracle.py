"""TEST INFRASTRUCTURE.  Keyed move sampling from the root's visit counts, restated in numpy from the recipe in
include/fpc.h (fpc_tree_sample_root): the reference that the kernel, BatchedMCTS.sample_root and SelfPlay.play_games are
checked against.  The uniform is tests/noise_oracle.py's U(i, j) at i = 0, j = SAMPLE_J."""
from __future__ import annotations

import numpy as np

from tests.noise_oracle import uniform

SAMPLE_J = 2**31 + 1


def weights(visits, temperature: float) -> np.ndarray:
    """w [k] f64 of one root: the counts at temperature 1, else (v / V) ** (1 / temperature); counts below 0 count 0."""
    v = np.maximum(np.asarray(visits, np.int64), 0)
    if float(temperature) == 1.0:
        return v.astype(np.float64)
    V = float(v.sum())
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.power(v.astype(np.float64) / V, 1.0 / float(temperature))


def sample_index(visits, temperature: float, seed: int, key: int):
    """(index i into the root's children or -1, t = U * W, prefix sums P [k]) for one root."""
    w = weights(visits, temperature)
    P = np.cumsum(w)  # one rounded addition per child in ascending i, as the kernel adds
    W = P[-1] if len(P) else 0.0
    if not W > 0.0:
        return -1, 0.0, P
    t = float(uniform(seed, key, 0, SAMPLE_J)) * W
    above = np.flatnonzero(P > t)
    if len(above):
        return int(above[0]), t, P
    return int(np.flatnonzero(w > 0.0)[-1]), t, P


def sample_many(visits, temperature: float, seed: int, keys) -> np.ndarray:
    """The index sample_index picks for one root under each of many keys, [len(keys)] i64."""
    w = weights(visits, temperature)
    P = np.cumsum(w)
    if not len(P) or not P[-1] > 0.0:
        return np.full(len(keys), -1, np.int64)
    t = uniform(seed, np.asarray(keys, np.int64), 0, SAMPLE_J) * P[-1]
    idx = np.searchsorted(P, t, side="right")  # the smallest i with P_i > t
    return np.where(idx < len(P), idx, np.flatnonzero(w > 0.0)[-1]).astype(np.int64)


def near_boundary(t: float, P: np.ndarray, rel: float = 1e-12) -> bool:
    """Whether t lies within rel (relative to W) of a prefix boundary: where a last-bit difference in the weights
    (the device's pow against numpy's) could move the choice."""
    return len(P) > 0 and bool(np.any(np.abs(P - t) <= rel * P[-1]))
