"""Periodic wrapping of bonded groups on the GPU (K9, SURVEY 8f row 4).

Mirrors the reference's ``moleculekit.wrapping``:

  wrap_box(groups, coords, box, centersel, center)   moleculekit/wrapping/wrapping.pyx:91-144  (in place, K9)
  wrap_triclinic_unitcell(groups, coords, boxvectors, centersel, center)        wrapping.pyx:147-250  (in place, K9b)
  wrap_compact_unitcell(groups, coords, boxvectors, centersel, center, mode)    wrapping.pyx:255-344  (in place, K9b)
  get_bonded_groups / getBondedGroups                 wrapping.pyx:24-86, moleculekit/molecule.py:3807-3856
  wrap(mol, ...)                                      Molecule.wrap, moleculekit/molecule.py:1987-2090

The per-frame/per-group arithmetic runs in ``mkb_wrap_box`` / ``mkb_wrap_triclinic`` (csrc/wrapping.cu) and is bit-identical
to the reference;
the connected-components bookkeeping is host logic (one pass over the bond list).  No CPU fallback for the kernel.
"""
from __future__ import annotations

import ctypes as C
import logging

import numpy as np
import torch

from . import _lib
from .distance_utils import _check, _ptr, _traj
from .occupancy_utils import _dev, _stream_ptr

logger = logging.getLogger(__name__)


# ---------------------------------------------------------------------------------------------- device level
def wrap_box_device(coords: torch.Tensor, box: torch.Tensor, groups: torch.Tensor, centersel: torch.Tensor | None,
                    center=None) -> torch.Tensor:
    """K9 on CUDA tensors: wraps ``coords`` (N, 3, F) float32 frame-minor IN PLACE and returns it.  ``groups`` /
    ``centersel`` are int32/uint32-valued CUDA tensors; ``center`` (3 floats) is used when centersel is empty."""
    dev = coords.device
    ncs = 0 if centersel is None else int(centersel.numel())
    cen = (C.c_float * 3)(*([0.0, 0.0, 0.0] if center is None else [float(np.float32(c)) for c in center]))
    if coords.shape[2] <= 1 and not coords.is_contiguous():
        raise ValueError("coords must be contiguous for in-place wrapping")
    h = _lib.handle(dev.index)
    tr = _traj(coords, box)
    with torch.cuda.device(dev):
        rc = _lib.load().mkb_wrap_box(h, _stream_ptr(dev), C.byref(tr), _ptr(groups), int(groups.numel()),
                                      _ptr(centersel) if ncs else C.c_void_p(0), ncs, cen)
    _lib.check(rc, h)
    return coords


UNITCELL_MODES = {"rectangular": 0, "compact": 1, "triclinic": 2}


def wrap_triclinic_device(coords: torch.Tensor, boxvectors: torch.Tensor, groups: torch.Tensor,
                          centersel: torch.Tensor | None, center=None, unitcell: str | int = "triclinic") -> torch.Tensor:
    """K9b on CUDA tensors: wraps ``coords`` (N, 3, F) float32 frame-minor IN PLACE for a triclinic cell and returns it.
    ``boxvectors`` (3, 3, F) float64 (row i = box vector i, as Molecule.boxvectors; a frame slice of a contiguous array is
    fine); ``unitcell``: "rectangular" / "compact" (wrap_compact_unitcell modes 0 / 1) or "triclinic"."""
    dev = coords.device
    mode = UNITCELL_MODES[unitcell] if isinstance(unitcell, str) else int(unitcell)
    ncs = 0 if centersel is None else int(centersel.numel())
    cen = (C.c_float * 3)(*([0.0, 0.0, 0.0] if center is None else [float(np.float32(c)) for c in center]))
    N, _, F = coords.shape
    assert boxvectors.is_cuda and boxvectors.dtype == torch.float64 and tuple(boxvectors.shape) == (3, 3, F)
    if F <= 1:
        boxvectors = boxvectors.contiguous()
        bvs = max(F, 1)
    else:
        assert boxvectors.stride(2) == 1 and boxvectors.stride(0) == 3 * boxvectors.stride(1)
        bvs = boxvectors.stride(1)
    h = _lib.handle(dev.index)
    tr = _traj(coords, torch.zeros((3, max(F, 1)), dtype=torch.float32, device=dev)[:, :F])
    with torch.cuda.device(dev):
        rc = _lib.load().mkb_wrap_triclinic(h, _stream_ptr(dev), C.byref(tr), _ptr(boxvectors), int(bvs), _ptr(groups),
                                            int(groups.numel()), _ptr(centersel) if ncs else C.c_void_p(0), ncs, cen, mode)
    if rc != 0 and b"Too many triclinic vectors" in (_lib.load().mkb_last_error(h) or b""):
        raise ValueError("Too many triclinic vectors!!")  # wrapping.pyx:439-441
    _lib.check(rc, h)
    return coords


# ------------------------------------------------------------------------------------------------ host mirrors
def _check_index_ranges(groups, centersel, n_atoms):
    if groups.size and int(groups.max()) > n_atoms:
        raise IndexError("group offset out of range")
    if centersel.size and int(centersel.max()) >= n_atoms:
        raise IndexError("centersel index out of range")
    # K9 wraps all groups in parallel: the offsets must be ascending (disjoint [groups[i], groups[i+1]) ranges), as
    # getBondedGroups + the reference's contiguous-molecule assumption produce.  The reference walks them sequentially and
    # tolerates anything; overlapping ranges here would race, so they are rejected instead of wrapped nondeterministically.
    if groups.size > 1 and np.any(np.diff(groups.astype(np.int64)) < 0):
        raise ValueError("wrap_box: group offsets must be ascending (bonded groups have to be contiguous in atom order); "
                         "reorder the atoms or wrap the offending groups separately")


def wrap_box(groups, coords, box, centersel, center, device=None):
    """Drop-in for wrapping.pyx:91-97: ``coords`` (N, 3, F) float32 is wrapped in place (numpy), nothing is returned."""
    _check("groups", groups, np.uint32, 1); _check("coords", coords, np.float32, 3)
    _check("box", box, np.float32, 2); _check("centersel", centersel, np.uint32, 1)
    _check("center", center, np.float32, 1)
    if coords.shape[0] == 0 or coords.shape[2] == 0 or groups.shape[0] < 2:
        return
    _check_index_ranges(groups, centersel, coords.shape[0])
    dev = _dev(device)
    d_coords = torch.from_numpy(np.ascontiguousarray(coords)).to(dev)
    d_box = torch.from_numpy(np.ascontiguousarray(box)).to(dev)
    d_groups = torch.from_numpy(np.ascontiguousarray(groups).view(np.int32)).to(dev)
    d_cs = torch.from_numpy(np.ascontiguousarray(centersel).view(np.int32)).to(dev) if centersel.size else None
    wrap_box_device(d_coords, d_box, d_groups, d_cs, center)
    coords[...] = d_coords.cpu().numpy()


def _wrap_tric_host(groups, coords, boxvectors, centersel, center, unitcell, device):
    _check("groups", groups, np.uint32, 1); _check("coords", coords, np.float32, 3)
    _check("boxvectors", boxvectors, np.float64, 3); _check("centersel", centersel, np.uint32, 1)
    _check("center", center, np.float32, 1)
    if coords.shape[0] == 0 or coords.shape[2] == 0:
        return
    _check_index_ranges(groups, centersel, coords.shape[0])
    dev = _dev(device)
    d_coords = torch.from_numpy(np.ascontiguousarray(coords)).to(dev)
    d_bv = torch.from_numpy(np.ascontiguousarray(boxvectors)).to(dev)
    d_groups = torch.from_numpy(np.ascontiguousarray(groups).view(np.int32)).to(dev)
    d_cs = torch.from_numpy(np.ascontiguousarray(centersel).view(np.int32)).to(dev) if centersel.size else None
    wrap_triclinic_device(d_coords, d_bv, d_groups, d_cs, center, unitcell)
    coords[...] = d_coords.cpu().numpy()


def wrap_triclinic_unitcell(groups, coords, boxvectors, centersel, center, device=None):
    """Drop-in for wrapping.pyx:147-155: ``coords`` (N, 3, F) float32 wrapped in place into the triclinic unit cell."""
    _wrap_tric_host(groups, coords, boxvectors, centersel, center, 2, device)


def wrap_compact_unitcell(groups, coords, boxvectors, centersel, center, mode, device=None):
    """Drop-in for wrapping.pyx:255-264: mode 0 = rectangular image of the triclinic cell, 1 = compact (minimum distance
    to the cell centre); in place."""
    if mode not in (0, 1):
        return  # the reference's pbc_dx leaves dx untouched for other modes; nobody calls it that way (molecule.py:2083-2090)
    _wrap_tric_host(groups, coords, boxvectors, centersel, center, int(mode), device)


def box_vectors(box, boxangles):
    """Molecule.boxvectors (moleculekit/molecule.py:428-454) / unitcell.lengths_and_angles_to_box_vectors
    (moleculekit/unitcell.py:33-125): (3, 3, F) float64 from lengths (3, F) and angles (3, F) in degrees."""
    box, boxangles = np.asarray(box), np.asarray(boxangles)
    F = box.shape[1]
    if np.all(boxangles == 0) and np.all(box == 0):
        return np.zeros((3, 3, F), dtype=np.float64)
    assert np.all(boxangles != 0), "Box angles should not be 0"
    a_len, b_len, c_len = (box[i].astype(np.float64) for i in range(3))
    alpha, beta, gamma = (boxangles[i].astype(np.float64) * np.pi / 180 for i in range(3))
    a = np.array([a_len, np.zeros_like(a_len), np.zeros_like(a_len)])
    b = np.array([b_len * np.cos(gamma), b_len * np.sin(gamma), np.zeros_like(b_len)])
    cx = c_len * np.cos(beta)
    cy = c_len * (np.cos(alpha) - np.cos(beta) * np.cos(gamma)) / np.sin(gamma)
    cz = np.sqrt(c_len * c_len - cx * cx - cy * cy)
    c = np.array([cx, cy, cz])
    tol = 1e-6
    for v in (a, b, c):
        v[np.logical_and(v > -tol, v < tol)] = 0.0
    return np.transpose(np.stack((a.T, b.T, c.T), axis=1), (1, 2, 0)).copy()


def get_bonded_groups(bonds, n_atoms: int, parent, size) -> None:
    """Host mirror of wrapping.pyx:65-86: union-by-size disjoint sets over the bond list, then every atom's parent is
    its root.  ``parent`` / ``size`` (uint32, length n_atoms) are updated in place like the reference's buffers; the
    identity of each root (first argument wins a size tie, pyx:57-62) is what orders the groups downstream."""
    par = parent.tolist()
    siz = size.tolist()

    def root(x):
        r = x
        while par[r] != r:
            r = par[r]
        while par[x] != r:  # full path compression, as the reference's recursive find
            par[x], x = r, par[x]
        return r

    for a, b in np.asarray(bonds).reshape(-1, 2).tolist():
        ra, rb = root(a), root(b)
        if ra == rb:
            continue
        if siz[ra] < siz[rb]:
            par[ra] = rb
            siz[rb] += siz[ra]
        else:
            par[rb] = ra
            siz[ra] += siz[rb]
    for i in range(n_atoms):
        root(i)
    parent[:] = np.asarray(par, dtype=np.uint32)
    size[:] = np.asarray(siz, dtype=np.uint32)


def getBondedGroups(mol, bonds=None):
    """molecule.py:3807-3856: (groups, group) -- the first atom of every bonded group plus a closing numAtoms entry,
    ordered by root id exactly like the reference's np.unique(parent), and the group index of every atom."""
    if bonds is None:
        bonds = mol.bonds
    n = int(mol.numAtoms)
    parent = np.arange(n).astype(np.uint32)
    size = np.ones(n, dtype=np.uint32)
    get_bonded_groups(np.asarray(bonds, dtype=np.uint32), n, parent, size)
    _, grouplist, grouparray = np.unique(parent, return_index=True, return_inverse=True)
    return np.hstack((grouplist, [n])).astype(np.uint32), grouparray


def wrap_plan(mol, wrapsel="all", fileBonds=True, guessBonds=False, wrapcenter=None, unitcell="rectangular"):
    """Host bookkeeping of Molecule.wrap (molecule.py:1987-2090) without touching the coordinates: bonded groups, centre
    selection or fixed centre, and the kernel choice.  Returns None when the reference skips the wrap (zero box), else a
    dict with ``groups``, ``centersel``, ``center`` and ``unitcell`` (None = orthorhombic box, K9; else the triclinic
    ``unitcell`` name, K9b, with ``boxvectors`` (3, 3, F) float64).  ``wrap`` and ``wrap_device`` both run on it."""
    unitcell = unitcell.lower()
    if unitcell not in ["rectangular", "triclinic", "compact"]:
        raise ValueError(f"Invalid unit cell type: {unitcell}. Must be one of: rectangular, triclinic, compact")
    nbonds = np.asarray(mol.bonds).reshape(-1, 2).shape[0]
    guess_sel = guessBonds
    if nbonds < (mol.numAtoms / 2):
        logger.warning(
            f"Wrapping detected {nbonds} bonds and {mol.numAtoms} atoms. "
            "Ignore this message if you believe this is correct, otherwise make sure you "
            "have loaded a topology containing all the bonds of the system before wrapping. "
            "The results may be inaccurate. If you want to use guessed bonds use the guessBonds argument.")
        guess_sel = True
    centersel = np.array([], dtype=np.uint32)
    if wrapcenter is None:
        if isinstance(wrapsel, str):
            try:
                sel = mol.atomselect(wrapsel, indexes=True, guessBonds=guess_sel)
            except TypeError:  # containers without the guessBonds keyword
                sel = mol.atomselect(wrapsel, indexes=True)
        else:
            sel = np.asarray(wrapsel)
            sel = np.where(sel)[0] if sel.dtype == bool else sel
        centersel = np.asarray(sel).astype(np.uint32)
        wrapcenter = np.array([0, 0, 0], dtype=np.float32)
    else:
        wrapcenter = np.array(wrapcenter, dtype=np.float32)
    if np.all(mol.box == 0):
        logger.warning(
            "Zero box size detected in `Molecule.box`; skipping wrap. "
            "Read a topology / trajectory containing box information, "
            "or set `mol.box` and `mol.boxangles` manually before calling `wrap`.")
        return None
    if mol.box.shape[1] != mol.coords.shape[2]:
        raise RuntimeError(
            "Detected different number of simulation frames in `Molecule.box` and `Molecule.coords`. "
            "This could mean that you have not read correctly the box information from the simulation.")
    if hasattr(mol, "_getBonds"):
        bonds = mol._getBonds(fileBonds, guessBonds)
    else:
        bonds = np.asarray(mol.bonds, dtype=np.uint32).reshape(-1, 2) if fileBonds else np.zeros((0, 2), np.uint32)
        if guessBonds:
            from .bondguesser import guess_bonds
            bonds = np.vstack((bonds, guess_bonds(mol))).astype(np.uint32)
    groups, _ = getBondedGroups(mol, bonds)
    plan = {"groups": groups, "centersel": centersel, "center": wrapcenter, "unitcell": None, "boxvectors": None}
    boxangles = getattr(mol, "boxangles", None)
    if boxangles is None or not np.any(np.asarray(boxangles) != 90):  # molecule.py:2075-2077
        return plan
    boxvectors = getattr(mol, "boxvectors", None)
    if boxvectors is None:
        boxvectors = box_vectors(mol.box, boxangles)
    plan["unitcell"] = unitcell
    plan["boxvectors"] = np.ascontiguousarray(boxvectors, dtype=np.float64)
    return plan


def wrap(mol, wrapsel="all", fileBonds=True, guessBonds=False, wrapcenter=None, unitcell="rectangular", device=None):
    """Mirror of Molecule.wrap (molecule.py:1987-2090); ``mol.coords`` is wrapped in place.  ``mol`` is duck-typed: coords,
    box, numAtoms, bonds, atomselect (for a string ``wrapsel``), optionally boxangles / boxvectors and ``_getBonds``.
    Cells with a box angle != 90 take the triclinic kernels with the reference's ``unitcell`` choice."""
    plan = wrap_plan(mol, wrapsel, fileBonds, guessBonds, wrapcenter, unitcell)
    if plan is None:
        return
    groups, centersel, wrapcenter = plan["groups"], plan["centersel"], plan["center"]
    if plan["unitcell"] is None:
        wrap_box(groups, mol.coords, mol.box, centersel, wrapcenter, device=device)
    elif plan["unitcell"] == "triclinic":
        wrap_triclinic_unitcell(groups, mol.coords, plan["boxvectors"], centersel, wrapcenter, device=device)
    else:
        wrap_compact_unitcell(groups, mol.coords, plan["boxvectors"], centersel, wrapcenter,
                              1 if plan["unitcell"] == "compact" else 0, device=device)


def wrap_device(coords: torch.Tensor, box, plan) -> torch.Tensor:
    """Runs a ``wrap_plan`` on a resident (N, 3, F) float32 trajectory in place (K9 / K9b) and returns it; ``box`` is the
    host (3, F) box of the plan's molecule.  The same index checks as the host entry points run before the device call."""
    if plan is None or coords.shape[0] == 0 or coords.shape[2] == 0:
        return coords
    groups, centersel = plan["groups"], plan["centersel"]
    _check_index_ranges(groups, centersel, coords.shape[0])
    dev = coords.device
    d_groups = torch.from_numpy(np.ascontiguousarray(groups).view(np.int32)).to(dev)
    d_cs = torch.from_numpy(np.ascontiguousarray(centersel).view(np.int32)).to(dev) if centersel.size else None
    if plan["unitcell"] is None:
        if groups.shape[0] < 2:
            return coords
        d_box = torch.from_numpy(np.ascontiguousarray(box, dtype=np.float32)).to(dev)
        return wrap_box_device(coords, d_box, d_groups, d_cs, plan["center"])
    d_bv = torch.from_numpy(plan["boxvectors"]).to(dev)
    return wrap_triclinic_device(coords, d_bv, d_groups, d_cs, plan["center"], plan["unitcell"])
