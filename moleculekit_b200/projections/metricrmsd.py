"""Drop-in for ``moleculekit.projections.metricrmsd.MetricRmsd``: RMSD of every frame to a reference structure after
superposition.

The reference copies the molecule, wraps it, aligns every frame with Molecule.align and reduces with util.molRMSD, all in
numpy.  Here the trajectory goes to the device once: with ``pbc`` it is wrapped there (K9 / K9b on the plan of
``wrapping.wrap_plan``), then fitted and reduced by K14's fused RMSD kernel, so the aligned trajectory is never written and
only one float per frame comes back.  Without ``pbc`` only the rows of the fit and RMSD selections travel.  ``mol`` is
duck-typed like the other projections (coords, box, numAtoms, numFrames, atomselect, and bonds for ``pbc``).
"""
from __future__ import annotations

import numpy as np

from .projection import Projection


class MetricRmsd(Projection):
    """Same constructor as the reference: ``refmol`` (copied), ``trajrmsdstr`` (RMSD atoms of the trajectory),
    ``trajalnstr`` (fit atoms, default ``trajrmsdstr``), ``refrmsdstr`` (default ``trajrmsdstr``), ``refalnstr`` (default
    ``trajalnstr``), ``centerstr`` (wrap centre selection) and ``pbc``.  Every frame is fitted onto ``refmol`` at
    ``refmol.frame``; the RMSD is taken against every frame of ``refmol`` when it has as many frames as the trajectory,
    else against its single frame."""

    def __init__(self, refmol, trajrmsdstr, trajalnstr=None, refrmsdstr=None, refalnstr=None, centerstr="protein",
                 pbc=True):
        super().__init__()
        if trajalnstr is None:
            trajalnstr = trajrmsdstr
        if refalnstr is None:
            refalnstr = trajalnstr
        if refrmsdstr is None:
            refrmsdstr = trajrmsdstr
        self._refmol = refmol.copy()
        self._refalnsel = self._refmol.atomselect(refalnstr)
        self._refrmsdsel = self._refmol.atomselect(refrmsdstr)
        self._trajalnsel = trajalnstr
        self._trajrmsdsel = trajrmsdstr
        self._centersel = centerstr
        self._pbc = pbc
        self.device = None  # CUDA device for project(); None = current device

    def _calculateMolProp(self, mol, props="all"):
        props = ("trajalnsel", "trajrmsdsel", "centersel") if props == "all" else props
        res = {}
        if "trajalnsel" in props:
            res["trajalnsel"] = mol.atomselect(self._trajalnsel)
            if np.sum(res["trajalnsel"]) == 0:
                raise RuntimeError("Alignment selection resulted in 0 atoms.")
        if "trajrmsdsel" in props:
            res["trajrmsdsel"] = mol.atomselect(self._trajrmsdsel)
            if np.sum(res["trajrmsdsel"]) == 0:
                raise RuntimeError("RMSD atom selection resulted in 0 atoms.")
        if "centersel" in props and self._pbc:
            res["centersel"] = mol.atomselect(self._centersel)
            if np.sum(res["centersel"]) == 0:
                raise RuntimeError("Centering selection resulted in 0 atoms.")
        return res

    def project(self, mol):
        """(numFrames,) float32 RMSD, squeezed like the reference (a 0-d array for one frame)."""
        import torch

        from .. import align as al
        from ..occupancy_utils import _dev
        from ..wrapping import wrap_device, wrap_plan

        props = self._getMolProp(mol, "all")
        aln = np.where(props["trajalnsel"])[0]
        rms = np.where(props["trajrmsdsel"])[0]
        refaln = np.where(self._refalnsel)[0]
        refrms = np.where(self._refrmsdsel)[0]
        if aln.size != refaln.size:
            raise RuntimeError(al._SIZE_MISMATCH)
        if rms.size != refrms.size:
            raise ValueError(f"the RMSD selections have {rms.size} (trajectory) and {refrms.size} (reference) atoms")
        ref = self._refmol
        F, Fr = mol.coords.shape[2], ref.coords.shape[2]
        if Fr not in (1, F):
            raise ValueError(f"the reference has {Fr} frames: expected 1 or {F}")
        if not 0 <= int(ref.frame) < Fr:
            raise IndexError(f"refmol.frame {ref.frame} out of range for a reference of {Fr} frames")
        coords = np.asarray(mol.coords)
        if coords.dtype != np.float32:
            raise ValueError("mol.coords must be float32")
        plan = wrap_plan(mol, props["centersel"]) if self._pbc else None
        if F == 0:
            return np.array(np.squeeze(np.zeros(0)), dtype=np.float32)
        dev = _dev(self.device)
        if self._pbc:
            d = torch.from_numpy(np.ascontiguousarray(coords)).to(dev)
            wrap_device(d, mol.box, plan)
        else:  # only the rows the fit and the RMSD read
            rows = np.union1d(aln, rms)
            d = torch.from_numpy(np.ascontiguousarray(coords[rows])).to(dev)
            aln, rms = np.searchsorted(rows, aln), np.searchsorted(rows, rms)
        frames = torch.arange(F, device=dev)
        f0 = int(ref.frame)
        d_refaln = torch.from_numpy(np.ascontiguousarray(ref.coords[refaln, :, f0:f0 + 1], dtype=np.float32)).to(dev)
        d_refrms = torch.from_numpy(np.ascontiguousarray(ref.coords[refrms], dtype=np.float32)).to(dev)
        xf = al.align_fit_device(d, frames, al.sel_tensor(aln, dev), d_refaln)
        out = al.rmsd_device(d, frames, al.sel_tensor(rms, dev), d_refrms, xf)
        return np.array(np.squeeze(out.cpu().numpy()), dtype=np.float32)

    def getMapping(self, mol):
        from pandas import DataFrame

        types = ["rmsd"]
        indexes = [np.where(self._getMolProp(mol, "trajrmsdsel"))[0]]
        description = ["RMSD to reference structure."]
        return DataFrame({"type": types, "atomIndexes": indexes, "description": description})
