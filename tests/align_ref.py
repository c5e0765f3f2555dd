"""numpy restatement of moleculekit's superposition (align.py `_pp_measure_fit` / `_pp_align`, `Molecule.align`,
`util.molRMSD`), the yardstick of K14 (csrc/align.cu).

``dtype=np.float32`` reproduces the reference's own arithmetic: float32 coordinates give float32 means, dot products and
LAPACK ``sgesdd``.  ``dtype=np.float64`` is the accuracy target the GPU results are held to.
"""
from __future__ import annotations

import numpy as np


def measure_fit(P, Q):
    """P, Q centred (n, 3): (R, rmsd) with R the proper rotation that best maps P onto Q."""
    cov = P.T @ Q
    V, S, W = np.linalg.svd(cov)
    W = W.T
    rmsd = np.sqrt(np.abs((np.sum(P * P) + np.sum(Q * Q) - 2 * np.sum(S)) / P.shape[0]))
    if np.linalg.det(W) * np.linalg.det(V) < 0:
        W[:, 2] = -W[:, 2]  # proper rotation only
    return W @ V.T, rmsd


def pp_align(coords, refcoords, sel, refsel, frames, refframe, matchingframes, inplace=False, dtype=np.float64):
    """Every atom of every listed frame moved by the fit of ``sel`` onto ``refsel``: (x - cP) R^T + cQ.  The result has
    ``coords``' dtype (float32 in), computed in ``dtype``."""
    out = coords if inplace else coords.copy()
    for f in frames:
        P = coords[sel, :, f].astype(dtype)
        Q = refcoords[refsel, :, f if matchingframes else refframe].astype(dtype)
        cP, cQ = P.mean(axis=0), Q.mean(axis=0)
        R, _ = measure_fit(P - cP, Q - cQ)
        out[:, :, f] = (coords[:, :, f].astype(dtype) - cP) @ R.T + cQ
    return out


def transforms(coords, refcoords, sel, refsel, frames, refframe, matchingframes, dtype=np.float64):
    """(n_frames, 15) [R row-major | cP | cQ] per listed frame, the layout of mkb_align_fit."""
    out = np.zeros((len(frames), 15), dtype=np.float64)
    for i, f in enumerate(frames):
        P = coords[sel, :, f].astype(dtype)
        Q = refcoords[refsel, :, f if matchingframes else refframe].astype(dtype)
        cP, cQ = P.mean(axis=0), Q.mean(axis=0)
        R, _ = measure_fit(P - cP, Q - cQ)
        out[i] = np.concatenate([R.ravel(), cP, cQ])
    return out


def molRMSD(coords, refcoords, rmsdsel1, rmsdsel2, dtype=np.float64):
    """util.molRMSD on coordinate arrays: the reference broadcasts when it has one frame."""
    d = coords[rmsdsel1, :, :].astype(dtype) - refcoords[rmsdsel2, :, :].astype(dtype)
    return np.squeeze(np.sqrt(np.mean(np.sum(d * d, axis=1), axis=0)))


def random_rotation(rng):
    """A uniformly distributed proper rotation (QR of a Gaussian matrix with the sign fix)."""
    q, r = np.linalg.qr(rng.normal(size=(3, 3)))
    q = q * np.sign(np.diag(r))
    if np.linalg.det(q) < 0:
        q[:, 0] = -q[:, 0]
    return q


def rigid_trajectory(rng, base, F, noise=0.5, spread=20.0):
    """(N, 3, F) float32: frame f is a random rigid motion of ``base`` (N, 3) plus Gaussian noise, and the motions."""
    N = base.shape[0]
    out = np.empty((N, 3, F), dtype=np.float32)
    Rs, ts = [], []
    for f in range(F):
        R = random_rotation(rng)
        t = rng.uniform(-spread, spread, size=3)
        out[:, :, f] = (base @ R.T + t + rng.normal(0, noise, size=(N, 3))).astype(np.float32)
        Rs.append(R)
        ts.append(t)
    return out, np.array(Rs), np.array(ts)
