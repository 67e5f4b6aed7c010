"""Synthetic benchmark workloads (SURVEY.md section 8d): the C3 pair (BASELINE.json configs[2])
and the C5 batch of small pairs (configs[4]).  Pure NumPy input generators — kept inside the
package so that the product arm of bench.py needs no test infrastructure; a CPU test checks they
produce the very arrays the CPU arm's generator does."""
from __future__ import annotations

import numpy as np

from . import mathutils


def surface(n: int, seed: int, extent: float = 100.0, x0: float = 0.0) -> np.ndarray:
    """Tilted, gently undulating plane with 1 cm noise (all six rigid-body parameters are
    observable on it; a perfect plane would leave three of them free), sampled over
    [x0, x0 + extent] x [0, extent]: patches with different x0 overlap partly."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(x0, x0 + extent, n)
    y = rng.uniform(0, extent, n)
    z = 0.05 * x + 0.03 * y + 2 * np.sin(2 * np.pi * x / 25) * np.cos(2 * np.pi * y / 40)
    z = z + rng.normal(0, 0.01, n)
    return np.column_stack((x, y, z))


def H_from_rbp(x) -> np.ndarray:
    return mathutils.create_homogeneous_transformation_matrix(
        mathutils.euler_angles_to_rotation_matrix(x[0], x[1], x[2]), np.asarray(x[3:6], dtype=float))


def apply_H(X: np.ndarray, H: np.ndarray) -> np.ndarray:
    Xh = np.column_stack((X, np.ones(X.shape[0])))
    Xh = np.transpose(H @ Xh.T)
    return np.column_stack((Xh[:, 0] / Xh[:, 3], Xh[:, 1] / Xh[:, 3], Xh[:, 2] / Xh[:, 3]))


H_TRUE_C3 = (np.deg2rad(0.3), np.deg2rad(-0.2), np.deg2rad(0.5), 0.15, -0.10, 0.05)


def c3_pair(n: int = 1_000_000, shift: int = 0):
    """X_fix = surface(n, 1234 + shift); X_mov = H_true^-1 * surface(n, 5678 + shift).  `shift`
    gives the independent pairs of the weak-scaling runs (10 x rank)."""
    H_true = H_from_rbp(H_TRUE_C3)
    X_fix = surface(n, 1234 + shift)
    X_mov = apply_H(surface(n, 5678 + shift), np.linalg.inv(H_true))
    return np.ascontiguousarray(X_fix), np.ascontiguousarray(X_mov), H_true


def c5_transforms(n_pairs: int) -> np.ndarray:
    """The rigid-body parameters of all pairs of a C5 batch: angles U(-1 deg, 1 deg),
    translations U(-0.2, 0.2), one generator (seed 99) for the whole batch."""
    rng = np.random.default_rng(99)
    return np.column_stack((np.deg2rad(rng.uniform(-1.0, 1.0, (n_pairs, 3))), rng.uniform(-0.2, 0.2, (n_pairs, 3))))


def c5_pair(i: int, n: int = 100_000, n_pairs_total: int = 512):
    """Pair i of the C5 batch: a 30 x 30 patch of the surface sampled twice (seeds 10000 + 2 i and
    10001 + 2 i), the second sample moved by the inverse of H_i."""
    H = H_from_rbp(c5_transforms(n_pairs_total)[i])
    X_fix = surface(n, 10_000 + 2 * i, extent=30.0)
    X_mov = apply_H(surface(n, 10_001 + 2 * i, extent=30.0), np.linalg.inv(H))
    return np.ascontiguousarray(X_fix), np.ascontiguousarray(X_mov), H
