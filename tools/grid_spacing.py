"""Largest nearest-neighbour angle of the HEALPix SO(3) grids, levels 0..5, measured on the CPU (DESIGN 4.7).

The default `neighbour_radius` of `evalpath.estimate_rotation_modes` is 1.5x this angle per level: a ball of that radius around
any grid point holds at least its nearest neighbour, so the local-maximum test of `rotation_modes` always looks at a neighbour.
Grids from `oracle.rnf_oracle.healpix_grid` (fp64 math -> fp32, as the device grid); neighbours by `scipy.spatial.cKDTree` on the
unit quaternions and their negatives (q and -q are the same rotation).  The chord d between unit quaternions is a rotation angle
of 4 asin(d / 2).

    python tools/grid_spacing.py          # prints one line per level and the table as JSON
"""
import json
import os
import sys

import numpy as np
from scipy.spatial import cKDTree

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import rnf_oracle as orc  # noqa: E402


def quaternions(R: np.ndarray) -> np.ndarray:
    """[N,3,3] -> unit quaternions [N,4] (real first), best-conditioned of the four candidate rows, fp64."""
    m = R.reshape(-1, 9).astype(np.float64)
    m00, m01, m02, m10, m11, m12, m20, m21, m22 = m.T
    q_abs = np.sqrt(np.maximum(np.stack([1 + m00 + m11 + m22, 1 + m00 - m11 - m22, 1 - m00 + m11 - m22, 1 - m00 - m11 + m22], -1), 0))
    cand = np.stack([np.stack([q_abs[:, 0] ** 2, m21 - m12, m02 - m20, m10 - m01], -1),
                     np.stack([m21 - m12, q_abs[:, 1] ** 2, m10 + m01, m02 + m20], -1),
                     np.stack([m02 - m20, m10 + m01, q_abs[:, 2] ** 2, m12 + m21], -1),
                     np.stack([m10 - m01, m20 + m02, m21 + m12, q_abs[:, 3] ** 2], -1)], -2)
    best = q_abs.argmax(-1)
    q = cand[np.arange(m.shape[0]), best] / (2.0 * q_abs[np.arange(m.shape[0]), best])[:, None]
    return q / np.linalg.norm(q, axis=-1, keepdims=True)


def largest_nn_angle(level: int) -> float:
    q = quaternions(orc.healpix_grid(level).numpy())
    tree = cKDTree(np.concatenate([q, -q]))
    d, _ = tree.query(q, k=2)
    return float(4.0 * np.arcsin(np.minimum(d[:, 1].max() / 2.0, 1.0)))


if __name__ == "__main__":
    table = {}
    for level in range(6):
        a = largest_nn_angle(level)
        table[level] = a
        print(f"level {level}: {72 * 8 ** level} rotations, largest nearest-neighbour angle {a:.6f} rad "
              f"({np.degrees(a):.3f} deg), 1.5x = {1.5 * a:.6f} rad", flush=True)
    print(json.dumps(table))
