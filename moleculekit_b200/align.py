"""Superposition of trajectory frames on the GPU (K14): mirror of moleculekit's ``Molecule.align`` and ``util.molRMSD``.

  _pp_align(coords, refcoords, sel, refsel, frames, refframe, matchingframes, inplace)   moleculekit/align.py
  align(mol, sel, refmol, refsel, frames, matchingframes, mode)                          Molecule.align
  molRMSD(mol, refmol, rmsdsel1, rmsdsel2)                                               moleculekit/util.py

The fit (float64 centroids and covariance, Horn's quaternion for the optimal proper rotation), the rigid transform of
every atom and the RMSD reduction run in ``mkb_align_fit`` / ``mkb_align_apply`` / ``mkb_rmsd`` (csrc/align.cu).  The
``*_device`` functions take CUDA tensors in the (N, 3, F) float32 frame-minor layout and leave results on the device.
Arithmetic contract: the transform is computed and applied in float64 and rounded once to float32, so aligned coordinates
lie within one float32 ulp of a float64 evaluation of the reference's formulas (the reference itself works in float32).
No CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .distance_utils import _ptr, _traj
from .occupancy_utils import _dev, _stream_ptr

_SIZE_MISMATCH = ("Cannot align molecules. The two selections produced different number of atoms. Either fix the "
                  "selections or use mode='structure'")


# ---------------------------------------------------------------------------------------------- device level
def _frames(frames, dev) -> torch.Tensor:
    if isinstance(frames, torch.Tensor):
        return frames.to(device=dev, dtype=torch.int64).contiguous()
    return torch.from_numpy(np.ascontiguousarray(frames, dtype=np.int64)).to(dev)


def _ref_view(ref: torch.Tensor) -> tuple[torch.Tensor, int]:
    """(tensor, row stride) of a (n, 3, Fr) float32 frame-minor reference (contiguous or a frame slice of one)."""
    assert ref.is_cuda and ref.dtype == torch.float32 and ref.ndim == 3 and ref.shape[1] == 3
    if ref.shape[2] <= 1 or ref.shape[0] == 0:
        ref = ref.contiguous()
        return ref, max(int(ref.shape[2]), 1)
    assert ref.stride(2) == 1 and ref.stride(0) == 3 * ref.stride(1), "ref must be (n, 3, Fr) frame-minor"
    return ref, int(ref.stride(1))


def _no_box(coords: torch.Tensor) -> torch.Tensor:
    F = coords.shape[2]
    return torch.zeros((3, max(F, 1)), dtype=torch.float32, device=coords.device)[:, :F]


def align_fit_device(coords: torch.Tensor, frames, sel: torch.Tensor, ref: torch.Tensor,
                     matchingframes: bool = False) -> torch.Tensor:
    """K14 fit on CUDA tensors: (n_frames, 15) float64 transforms [R row-major | cP | cQ], one per listed frame, that
    superpose the ``sel`` atoms of ``coords`` (N, 3, F) onto ``ref`` (n_sel, 3, Fr), the reference rows in selection
    order.  ``ref`` column 0 is the target of every frame, or with ``matchingframes`` column ``frames[i]``."""
    dev = coords.device
    fr = _frames(frames, dev)
    ref, rs = _ref_view(ref)
    out = torch.empty((fr.numel(), 15), dtype=torch.float64, device=dev)
    h = _lib.handle(dev.index)
    tr = _traj(coords, _no_box(coords))
    with torch.cuda.device(dev):
        rc = _lib.load().mkb_align_fit(h, _stream_ptr(dev), C.byref(tr), _ptr(fr), int(fr.numel()), _ptr(sel),
                                       int(sel.numel()), _ptr(ref), rs, int(bool(matchingframes)), _ptr(out))
    _lib.check(rc, h)
    return out


def align_apply_device(coords: torch.Tensor, frames, transforms: torch.Tensor) -> torch.Tensor:
    """K14 apply: moves every atom of the listed frames of ``coords`` (N, 3, F) IN PLACE, x' = (x - cP) R^T + cQ in
    float64 rounded once to float32, and returns ``coords``.  Frames must not repeat."""
    dev = coords.device
    fr = _frames(frames, dev)
    assert transforms.is_cuda and transforms.dtype == torch.float64 and tuple(transforms.shape) == (fr.numel(), 15)
    if coords.shape[2] <= 1 and not coords.is_contiguous():
        raise ValueError("coords must be contiguous for in-place alignment")
    transforms = transforms.contiguous()
    h = _lib.handle(dev.index)
    tr = _traj(coords, _no_box(coords))
    with torch.cuda.device(dev):
        rc = _lib.load().mkb_align_apply(h, _stream_ptr(dev), C.byref(tr), _ptr(fr), int(fr.numel()), _ptr(transforms))
    _lib.check(rc, h)
    return coords


def rmsd_device(coords: torch.Tensor, frames, sel: torch.Tensor, ref: torch.Tensor,
                transforms: torch.Tensor | None = None) -> torch.Tensor:
    """K14 RMSD: (n_frames,) float32, per listed frame the RMSD between the ``sel`` atoms of ``coords`` and ``ref``
    (n_sel, 3, Fr), summed in float64.  Fr == 1 broadcasts, else column ``frames[i]`` is used.  With ``transforms``
    (from align_fit_device) the coordinates are the float32 values align_apply_device would store, without storing them."""
    dev = coords.device
    fr = _frames(frames, dev)
    ref, rs = _ref_view(ref)
    if transforms is not None:
        assert transforms.is_cuda and transforms.dtype == torch.float64 and tuple(transforms.shape) == (fr.numel(), 15)
        transforms = transforms.contiguous()
    out = torch.empty(fr.numel(), dtype=torch.float32, device=dev)
    h = _lib.handle(dev.index)
    tr = _traj(coords, _no_box(coords))
    with torch.cuda.device(dev):
        rc = _lib.load().mkb_rmsd(h, _stream_ptr(dev), C.byref(tr), _ptr(fr), int(fr.numel()), _ptr(sel),
                                  int(sel.numel()), _ptr(ref), rs, int(ref.shape[2]), _ptr(transforms), _ptr(out))
    _lib.check(rc, h)
    return out


def sel_tensor(idx, dev) -> torch.Tensor:
    """int32 CUDA tensor of atom indexes (the uint32 selections of the C-ABI)."""
    return torch.from_numpy(np.ascontiguousarray(idx, dtype=np.int64).astype(np.int32)).to(dev)


# ------------------------------------------------------------------------------------------------ host mirrors
def _as_index(sel, n_atoms: int, what: str) -> np.ndarray:
    sel = np.asarray(sel)
    if sel.dtype == bool:
        if sel.shape != (n_atoms,):
            raise IndexError(f"{what}: boolean mask of length {sel.shape} for {n_atoms} atoms")
        return np.where(sel)[0]
    idx = sel.astype(np.int64).reshape(-1)
    if idx.size and (idx.min() < 0 or idx.max() >= n_atoms):
        raise IndexError(f"{what}: atom index out of range for {n_atoms} atoms")
    return idx


def _check_coords(name, coords):
    if not isinstance(coords, np.ndarray) or coords.dtype != np.float32 or coords.ndim != 3 or coords.shape[1] != 3:
        raise ValueError(f"{name} must be a float32 (natoms, 3, nframes) array")


def _pp_align(coords, refcoords, sel, refsel, frames, refframe, matchingframes, inplace=False, device=None):
    """Drop-in for moleculekit's align._pp_align: every atom of every listed frame is moved by the fit of ``sel`` onto
    ``refsel`` of ``refcoords`` (frame ``refframe``, or the same frame with ``matchingframes``).  Returns the result
    (``coords`` itself when ``inplace``).

    One deviation: when ``refcoords`` is ``coords`` and ``inplace`` is set, the reference aligns frame by frame in place,
    so a later frame is fitted against the already aligned (float32-perturbed) reference frame.  Here every frame is fitted
    against the reference rows as they were when the call started.  The difference is within the float32 rounding of the
    reference frame."""
    _check_coords("coords", coords)
    _check_coords("refcoords", refcoords)
    N, _, F = coords.shape
    sel = _as_index(sel, N, "sel")
    refsel = _as_index(refsel, refcoords.shape[0], "refsel")
    if sel.size != refsel.size:
        raise RuntimeError(_SIZE_MISMATCH)
    if sel.size == 0:
        raise RuntimeError("Alignment selection resulted in 0 atoms.")
    frames = np.asarray(frames, dtype=np.int64).reshape(-1)
    if frames.size and (frames.min() < 0 or frames.max() >= F):
        raise IndexError(f"frames out of range for a trajectory of {F} frames")
    if np.unique(frames).size != frames.size:
        raise ValueError("frames must not repeat")
    Fr = refcoords.shape[2]
    if matchingframes:
        if frames.size and frames.max() >= Fr:
            raise ValueError(f"matchingframes: the reference has {Fr} frames, frame {int(frames.max())} was asked for")
    elif not 0 <= int(refframe) < Fr:
        raise IndexError(f"refframe {refframe} out of range for a reference of {Fr} frames")
    out = coords if inplace else coords.copy()
    if frames.size == 0 or N == 0:
        return out
    dev = _dev(device)
    ref_rows = refcoords[refsel] if matchingframes else refcoords[refsel, :, int(refframe)][:, :, None]
    d_ref = torch.from_numpy(np.ascontiguousarray(ref_rows)).to(dev)
    d_coords = torch.from_numpy(np.ascontiguousarray(coords)).to(dev)
    d_frames = _frames(frames, dev)
    xf = align_fit_device(d_coords, d_frames, sel_tensor(sel, dev), d_ref, matchingframes)
    align_apply_device(d_coords, d_frames, xf)
    out[...] = d_coords.cpu().numpy()
    return out


def align(mol, sel, refmol=None, refsel=None, frames=None, matchingframes=False, mode="index", device=None):
    """Mirror of Molecule.align: superposes ``sel`` of every listed frame (default all) onto ``refsel`` (default ``sel``)
    of ``refmol`` (default ``mol``) at ``refmol.frame`` (or the same frame with ``matchingframes``) and moves every atom
    of those frames; ``mol.coords`` is updated in place.  ``mol`` is duck-typed (coords, numFrames, frame, atomselect).
    With ``refmol`` omitted, every frame is fitted against the reference frame as it was before the call (see
    ``_pp_align``)."""
    if mode == "structure":
        raise NotImplementedError(
            "mode='structure' (TM-align sequence-independent superposition) is not accelerated here: use "
            "moleculekit's Molecule.align for it")
    if mode != "index":
        raise ValueError(f"Unknown alignment mode {mode!r}: expected 'index' or 'structure'")
    if refmol is None:
        refmol = mol
    if refsel is None:
        refsel = sel
    if frames is None:
        frames = range(mol.coords.shape[2])
    frames = np.array(frames)
    sel = mol.atomselect(sel, indexes=True)
    refsel = refmol.atomselect(refsel, indexes=True)
    if np.size(sel) != np.size(refsel):
        raise RuntimeError(_SIZE_MISMATCH)
    mol.coords = _pp_align(mol.coords, refmol.coords, np.asarray(sel, dtype=np.int64),
                           np.asarray(refsel, dtype=np.int64), frames, refmol.frame, matchingframes, inplace=True,
                           device=device)


def molRMSD(mol, refmol, rmsdsel1, rmsdsel2, device=None):
    """Drop-in for moleculekit.util.molRMSD: per frame, the RMSD between ``rmsdsel1`` of ``mol`` and ``rmsdsel2`` of
    ``refmol`` (masks or indexes) without any fit; a one-frame reference broadcasts.  Squeezed float32, summed in float64.
    Only the selected rows travel to the device."""
    _check_coords("mol.coords", mol.coords)
    _check_coords("refmol.coords", refmol.coords)
    i1 = _as_index(rmsdsel1, mol.coords.shape[0], "rmsdsel1")
    i2 = _as_index(rmsdsel2, refmol.coords.shape[0], "rmsdsel2")
    if i1.size != i2.size:
        raise ValueError(f"the two RMSD selections have {i1.size} and {i2.size} atoms")
    if i1.size == 0:
        raise RuntimeError("RMSD atom selection resulted in 0 atoms.")
    F, Fr = mol.coords.shape[2], refmol.coords.shape[2]
    if Fr not in (1, F):
        raise ValueError(f"the reference has {Fr} frames: expected 1 or {F}")
    if F == 0:
        return np.squeeze(np.zeros(0, dtype=np.float32))
    dev = _dev(device)
    d_c = torch.from_numpy(np.ascontiguousarray(mol.coords[i1])).to(dev)
    d_r = torch.from_numpy(np.ascontiguousarray(refmol.coords[i2])).to(dev)
    out = rmsd_device(d_c, torch.arange(F, device=dev), sel_tensor(np.arange(i1.size), dev), d_r)
    return np.squeeze(out.cpu().numpy())
