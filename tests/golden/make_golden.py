"""Generate the committed golden fixtures in tests/golden/ from the REFERENCE itself.

Runs only in the build container (needs /root/reference).  Two sources are used:

 1. the reference's own stored goldens under /root/reference/tests (3PTB_voxres_old.npy,
    metricdistance/{distances,mindistances,selfmindistance}.npy, inline constants of
    tests/test_metricdistance.py / tests/test_interactions.py), sliced/sparsified so they are small;
 2. outputs of the reference's compiled Cython kernels (oracle/_ref, built from the .pyx files in
    place by oracle/build_ref.py) on seeded inputs, for cases the reference has no stored golden for
    (arbitrary centres, multi-sigma atoms, ordered contact pairs, COM reductions, cdist/pdist).

Reading PDB/XTC files needs the full reference Python package with its extensions built; as
/root/reference is read-only that build lives in a scratch copy (SURVEY.md appendix A):

    mkdir /tmp/refcopy && cd /tmp/refcopy && cp -r /root/reference/moleculekit /root/reference/setup.py . \
      && chmod -R u+w . && python setup.py build_ext --inplace
    cd /root/repo && PYTHONPATH=/tmp/refcopy LOCAL_PDB_REPO=/root/reference/tests/pdb python tests/golden/make_golden.py

The fixtures carry only numbers (coordinates, masks, outputs) -- no reference source.
"""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REFT = "/root/reference/tests"


def scratch_copy(path: str) -> str:
    """The reference's XTC reader drops index-cache files (.name, .name.numframes) next to the trajectory it reads;
    /root/reference must not be written to, so trajectories are read from a scratch copy."""
    import shutil
    import tempfile

    d = tempfile.mkdtemp(prefix="mkb_golden_")
    dst = os.path.join(d, os.path.basename(path))
    shutil.copyfile(path, dst)
    return dst


def strarr(a):
    """object string array -> fixed-width unicode (npz without pickle)"""
    return np.array([str(x) for x in a])


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def wrapping_fixture():
    """wrap.npz (K9, wrap_box): the reference's own orthorhombic test system (tests/test_wrapping.py:9-16), cut to the
    protein + the first solvent groups and 3 frames, with (a) the output of the reference's compiled wrap_box on that cut
    (bit-exact target), (b) the same atoms/frames of the reference's STORED golden output_wrapped.xtc (atol 1e-2, the
    reference test's own tolerance) and (c) the bond list / bonded groups of the cut; plus seeded random cases."""
    from oracle import build_ref

    wref = build_ref.load()[3]
    from moleculekit.molecule import Molecule, getBondedGroups

    d = os.path.join(REFT, "test_wrapping")
    mol = Molecule(os.path.join(d, "structure.prmtop"))
    mol.read(scratch_copy(os.path.join(d, "output.xtc")))
    refmol = Molecule(os.path.join(d, "structure.prmtop"))
    refmol.read(scratch_copy(os.path.join(d, "output_wrapped.xtc")))
    groups, _ = getBondedGroups(mol)
    centersel = mol.atomselect("protein or resname ACE NME", indexes=True, guessBonds=False).astype(np.uint32)
    ncut_groups = 900
    K = int(groups[ncut_groups])
    assert centersel.max() < K
    frames = [0, 11, 29]
    w = {}
    w["coords"] = np.ascontiguousarray(mol.coords[:K][:, :, frames])
    w["box"] = np.ascontiguousarray(mol.box[:, frames])
    w["groups"] = groups[: ncut_groups + 1].copy()
    w["centersel"] = centersel
    w["bonds"] = mol.bonds[(mol.bonds < K).all(axis=1)].astype(np.uint32)
    out = w["coords"].copy()
    wref.wrap_box(w["groups"], out, w["box"], centersel, np.zeros(3, np.float32))
    w["ref_wrapped"] = out
    w["gold_wrapped_xtc"] = np.ascontiguousarray(refmol.coords[:K][:, :, frames])
    assert np.allclose(out, w["gold_wrapped_xtc"], atol=1e-2)  # the reference reproduces its stored golden on the cut
    assert not np.array_equal(out, w["coords"])
    # fixed-centre variant (tests/test_wrapping.py:18-24 wraps 6X18 around a given point)
    cen = np.array([94.64, 3.69, 1.11], dtype=np.float32)
    out2 = w["coords"].copy()
    wref.wrap_box(w["groups"], out2, w["box"], np.zeros(0, np.uint32), cen)
    w["center_fixed"] = cen
    w["ref_wrapped_fixed"] = out2
    # seeded random cases incl. empty groups, single-atom groups, a zero box component (NaN translation)
    rng = np.random.default_rng(99)
    ncase = 6
    for c in range(ncase):
        N = int(rng.integers(5, 300)); F = int(rng.integers(1, 7))
        cuts = np.unique(np.concatenate([[0], rng.integers(0, N, size=int(rng.integers(0, 40))), [N]])).astype(np.uint32)
        if c == 1:
            cuts = np.sort(np.concatenate([cuts, cuts[1:3]])).astype(np.uint32)  # repeated offsets = empty groups
        box = rng.uniform(6, 25, size=(3, F)).astype(np.float32)
        if c == 2:
            box[1, 0] = 0.0
        xyz = rng.normal(0, 35, size=(N, 3, F)).astype(np.float32)
        cs = np.zeros(0, np.uint32) if c % 2 else np.sort(rng.choice(N, size=min(N, 17), replace=False)).astype(np.uint32)
        cen = rng.normal(0, 4, 3).astype(np.float32)
        o = xyz.copy()
        with np.errstate(all="ignore"):
            wref.wrap_box(cuts, o, box, cs, cen)
        for k, v in (("groups", cuts), ("coords", xyz), ("box", box), ("centersel", cs), ("center", cen), ("ref", o)):
            w[f"r{c}_{k}"] = v
    w["ncase"] = np.array(ncase)
    np.savez_compressed(os.path.join(HERE, "wrap.npz"), **w)


def triclinic_fixture():
    """tric.npz (K9b): the reference's triclinic test system tests/test_readers/dodecahedral_box (tests/test_wrapping.py:26-44),
    cut to the protein + the first solvent groups and 3 frames, with (a) the output of the reference's compiled
    wrap_triclinic_unitcell / wrap_compact_unitcell (modes 0, 1) on that cut (bit-exact targets) and (b) the same atoms /
    frames of the reference's STORED goldens output_{triclinic,compact,rectangular}_wrapped.xtc (atol 1e-2, the reference
    test's tolerance); plus a fixed-centre variant and seeded random cases (rhombic dodecahedron, truncated octahedron,
    general reduced cells; empty groups, atoms outside all groups)."""
    from oracle import build_ref

    wref = build_ref.load()[3]
    from moleculekit.molecule import Molecule, getBondedGroups

    d = os.path.join(REFT, "test_readers", "dodecahedral_box")
    mol = Molecule(os.path.join(d, "3ptb_dodecahedron.psf"))
    mol.read(scratch_copy(os.path.join(d, "output.xtc")))
    groups, _ = getBondedGroups(mol)
    centersel = mol.atomselect("protein", indexes=True, guessBonds=False).astype(np.uint32)
    ncut_groups = int(np.searchsorted(groups, centersel.max() + 1)) + 800
    K = int(groups[ncut_groups])
    assert centersel.max() < K
    frames = [0, mol.numFrames // 2, mol.numFrames - 1]
    w = {}
    w["coords"] = np.ascontiguousarray(mol.coords[:K][:, :, frames])
    w["box"] = np.ascontiguousarray(mol.box[:, frames])
    w["boxangles"] = np.ascontiguousarray(mol.boxangles[:, frames])
    w["boxvectors"] = np.ascontiguousarray(mol.boxvectors[:, :, frames])
    w["groups"] = groups[: ncut_groups + 1].copy()
    w["centersel"] = centersel
    zero = np.zeros(3, np.float32)
    for name, fn in (("triclinic", lambda c: wref.wrap_triclinic_unitcell(w["groups"], c, w["boxvectors"], centersel, zero)),
                     ("compact", lambda c: wref.wrap_compact_unitcell(w["groups"], c, w["boxvectors"], centersel, zero, 1)),
                     ("rectangular", lambda c: wref.wrap_compact_unitcell(w["groups"], c, w["boxvectors"], centersel, zero, 0))):
        out = w["coords"].copy()
        fn(out)
        w[f"ref_{name}"] = out
        gold = Molecule(scratch_copy(os.path.join(d, f"output_{name}_wrapped.xtc")))
        w[f"gold_{name}_xtc"] = np.ascontiguousarray(gold.coords[:K][:, :, frames])
        # the cut reproduces the stored golden: a group's translation depends only on its own atoms and the protein centre
        assert np.max(np.abs(out - w[f"gold_{name}_xtc"])) < 1e-2, name
        assert not np.array_equal(out, w["coords"])
    cen = np.array([12.5, -3.0, 40.25], dtype=np.float32)
    w["center_fixed"] = cen
    for name, mode in (("triclinic", None), ("compact", 1), ("rectangular", 0)):
        out = w["coords"].copy()
        if mode is None:
            wref.wrap_triclinic_unitcell(w["groups"], out, w["boxvectors"], np.zeros(0, np.uint32), cen)
        else:
            wref.wrap_compact_unitcell(w["groups"], out, w["boxvectors"], np.zeros(0, np.uint32), cen, mode)
        w[f"ref_{name}_fixed"] = out
    rng = np.random.default_rng(2024)
    ncase = 9
    for c in range(ncase):
        N = int(rng.integers(5, 300)); F = int(rng.integers(1, 7))
        cuts = np.unique(np.concatenate([[0], rng.integers(0, N, size=int(rng.integers(0, 40))), [N]])).astype(np.uint32)
        if c == 1:
            cuts = np.sort(np.concatenate([cuts, cuts[1:3]])).astype(np.uint32)  # repeated offsets = empty groups
        if c == 2 and len(cuts) > 3:
            cuts = cuts[1:-1].copy()  # atoms before the first / after the last group are only centred
        bv = np.zeros((3, 3, F))
        for f in range(F):
            L = rng.uniform(20, 40)
            if c % 3 == 0:    # rhombic dodecahedron (GROMACS xy-square form)
                vec = [[L, 0, 0], [0, L, 0], [L / 2, L / 2, L * np.sqrt(2) / 2]]
            elif c % 3 == 1:  # truncated octahedron
                vec = [[L, 0, 0], [L / 3, 2 * np.sqrt(2) * L / 3, 0], [-L / 3, np.sqrt(2) * L / 3, np.sqrt(6) * L / 3]]
            else:             # a mildly skewed reduced cell
                vec = [[L, 0, 0], [rng.uniform(-.3, .3) * L, L * rng.uniform(.9, 1.1), 0],
                       [rng.uniform(-.3, .3) * L, rng.uniform(-.3, .3) * L, L * rng.uniform(.9, 1.1)]]
            bv[:, :, f] = np.array(vec) * (1 + 0.001 * rng.normal())
        xyz = rng.normal(0, 45, size=(N, 3, F)).astype(np.float32)
        cs = np.zeros(0, np.uint32) if c % 2 else np.sort(rng.choice(N, size=min(N, 17), replace=False)).astype(np.uint32)
        cen = rng.normal(0, 4, 3).astype(np.float32)
        for k, v in (("groups", cuts), ("coords", xyz), ("boxvectors", bv), ("centersel", cs), ("center", cen)):
            w[f"r{c}_{k}"] = v
        for name, mode in (("triclinic", None), ("compact", 1), ("rectangular", 0)):
            o = xyz.copy()
            if mode is None:
                wref.wrap_triclinic_unitcell(cuts, o, bv, cs, cen)
            else:
                wref.wrap_compact_unitcell(cuts, o, bv, cs, cen, mode)
            w[f"r{c}_ref_{name}"] = o
    w["ncase"] = np.array(ncase)
    np.savez_compressed(os.path.join(HERE, "tric.npz"), **w)
    print("tric.npz", K, "atoms", len(frames), "frames")


def hbonds_fixture():
    """hbonds.npz (K12): the reference's hydrogen-bond test (tests/test_interactions.py:7-55) rebuilt without rdkit: the
    protein's donors / acceptors come from the reference's get_donors_acceptors, the benzamidine ligand is read from the SDF
    by hand (its donors are the four N-H pairs the test's expected rows name, it has no acceptors).  Stored: coordinates
    (two identical frames as in the test), donors, acceptors, selection masks, the reference's hbonds_calculate outputs --
    whose 'protein' vs 'resname BEN' rows equal the constants in the reference test and whose 'all' result has its 178
    rows -- plus ignore_hs / threshold variants and seeded random periodic cases from the compiled hbonds.calculate."""
    from oracle import build_ref

    href = build_ref.load()[6]
    from moleculekit.interactions.interactions import get_donors_acceptors, hbonds_calculate
    from moleculekit.molecule import Molecule

    d = os.path.join(REFT, "test_interactions")
    mol = Molecule(os.path.join(d, "3PTB_prepared.pdb"))
    mol.guessBonds()
    donors, acceptors = get_donors_acceptors(mol, exclude_water=True, exclude_backbone=False)
    lines = open(os.path.join(d, "3PTB_BEN.sdf")).read().splitlines()
    na, nb = int(lines[3][:3]), int(lines[3][3:6])
    xyz = np.array([[float(l[0:10]), float(l[10:20]), float(l[20:30])] for l in lines[4:4 + na]], dtype=np.float32)
    elem = [l[31:34].strip() for l in lines[4:4 + na]]
    lbonds = np.array([[int(l[0:3]) - 1, int(l[3:6]) - 1] for l in lines[4 + na:4 + na + nb]])
    lig = Molecule().empty(na)
    lig.coords = xyz[:, :, None].copy()
    lig.element[:] = elem
    lig.name[:] = [f"{e}{i}" for i, e in enumerate(elem)]
    lig.resname[:] = "BEN"
    lig.record[:] = "HETATM"
    lig.resid[:] = 1
    lig.bonds = lbonds.astype(np.uint32)
    lig.bondtype = np.array(["1"] * nb, dtype=object)
    mol.append(lig)
    lig_idx = np.where(mol.resname == "BEN")[0][0]
    lig_don = np.array([[a, b] if elem[a] == "N" else [b, a] for a, b in lbonds
                        if {elem[a], elem[b]} == {"N", "H"}], dtype=np.uint32)
    mol.bonds = mol._guessBonds()
    mol.coords = np.tile(mol.coords, (1, 1, 2)).copy()
    mol.box = np.tile(mol.box, (1, 2)).copy()
    donors = np.vstack((donors, lig_don + lig_idx)).astype(np.uint32)
    acceptors = np.asarray(acceptors, dtype=np.uint32)
    w = {"coords": mol.coords.astype(np.float32), "box": mol.box.astype(np.float32), "donors": donors,
         "acceptors": acceptors, "protein": mol.atomselect("protein"), "ben": mol.atomselect("resname BEN")}
    hb = hbonds_calculate(mol, donors, acceptors, "protein", "resname BEN")
    expected = np.array([[3414, 3421, 2471], [3414, 3422, 2789], [3415, 3423, 2472], [3415, 3424, 2482]])
    assert len(hb) == 2 and np.array_equal(hb[0], expected) and np.array_equal(hb[1], expected), hb  # test_interactions.py:41-51
    w["hb_prot_ben"] = hb[0]
    hb = hbonds_calculate(mol, donors, acceptors, "all")
    assert np.array(hb[0]).shape == (178, 3)  # test_interactions.py:53-55
    w["hb_all"] = hb[0]
    w["hb_all_nohs"] = hbonds_calculate(mol, donors, acceptors, "all", ignore_hs=True)[0]
    w["hb_all_wide"] = hbonds_calculate(mol, donors, acceptors, "all", dist_threshold=3.2, angle_threshold=100)[1]
    w["hb_prot_ben_nohs"] = hbonds_calculate(mol, donors, acceptors, "protein", "resname BEN", ignore_hs=True,
                                             dist_threshold=3.5)[0]
    rng = np.random.default_rng(77)
    ncase = 8
    for c in range(ncase):
        N = int(rng.integers(30, 250)); F = int(rng.integers(1, 6))
        L = rng.uniform(8, 15, size=(3, F)).astype(np.float32)
        if c == 1:
            L[1, 0] = 0
        if c == 2:
            L[:] = 0
        xyz = (rng.uniform(0, 1, size=(N, 3, F)) * 12).astype(np.float32) if c % 2 else rng.normal(0, 6, size=(N, 3, F)).astype(np.float32)
        nd = int(rng.integers(1, 60)); nacc = int(rng.integers(1, 60))
        heavy = rng.integers(0, N, nd); hyd = rng.integers(0, N, nd)
        for k in range(nd):
            if hyd[k] != heavy[k]:
                v = rng.normal(size=(3, F)); v /= np.linalg.norm(v, axis=0)
                xyz[hyd[k]] = xyz[heavy[k]] + v.astype(np.float32)
        if c == 3:
            xyz[hyd[0]] = xyz[heavy[0]]  # overlapping donor pair (dist2_b == 0)
        if c == 4:
            xyz[5, 1, 0] = np.nan
        dn = np.stack([heavy, hyd], 1).astype(np.uint32)
        acc = rng.integers(0, N, nacc).astype(np.uint32)
        s1 = (rng.random(N) < .6).astype(np.uint32); s2 = (rng.random(N) < .6).astype(np.uint32)
        dth = float(rng.uniform(2, 6)); ath = float(rng.uniform(60, 150))
        for k, v in (("coords", xyz), ("box", L), ("donors", dn), ("acceptors", acc), ("sel1", s1), ("sel2", s2),
                     ("thr", np.array([dth, ath]))):
            w[f"r{c}_{k}"] = v
        for intra in (0, 1):
            for ign in (0, 1):
                dd = dn if not ign else np.unique(dn[:, 0])[:, None].astype(np.uint32)
                with np.errstate(all="ignore"):
                    r = href.calculate(dd, acc, xyz, L, s1, s2, dist_threshold=dth, angle_threshold=ath, intra=bool(intra),
                                       ignore_hs=bool(ign))
                w[f"r{c}_out_{intra}{ign}_counts"] = np.array([len(x) // 3 for x in r])
                w[f"r{c}_out_{intra}{ign}"] = np.array([v for x in r for v in x], dtype=np.int32).reshape(-1, 3)
    w["ncase"] = np.array(ncase)
    np.savez_compressed(os.path.join(HERE, "hbonds.npz"), **w)
    print("hbonds.npz", mol.numAtoms, "atoms,", len(donors), "donors,", len(acceptors), "acceptors")


def _sdf_molecule(path, resname):
    """A Molecule from a V2000 SDF read by hand (no rdkit): coordinates, elements, bonds."""
    from moleculekit.molecule import Molecule

    lines = open(path).read().splitlines()
    na, nb = int(lines[3][:3]), int(lines[3][3:6])
    xyz = np.array([[float(l[0:10]), float(l[10:20]), float(l[20:30])] for l in lines[4:4 + na]], dtype=np.float32)
    elem = [l[31:34].strip() for l in lines[4:4 + na]]
    lbonds = np.array([[int(l[0:3]) - 1, int(l[3:6]) - 1] for l in lines[4 + na:4 + na + nb]])
    lig = Molecule().empty(na)
    lig.coords = xyz[:, :, None].copy()
    lig.element[:] = elem
    lig.name[:] = [f"{e}{i}" for i, e in enumerate(elem)]
    lig.resname[:] = resname
    lig.record[:] = "HETATM"
    lig.resid[:] = 1
    lig.bonds = lbonds.astype(np.uint32)
    lig.bondtype = np.array(["1"] * nb, dtype=object)
    return lig, elem, lbonds


def waterbridge_fixture():
    """waterbridge.npz: the reference's water-bridge test (tests/test_interactions.py:255-326) rebuilt without rdkit (the
    glycerol ligand read from the SDF by hand).  Stored: coordinates, donors / acceptors of the reference's
    get_donors_acceptors(exclude_water=False), the selection masks the test uses, and the reference's outputs -- asserted
    equal to the constants written in the test before they are stored."""
    from moleculekit.interactions.interactions import get_donors_acceptors, waterbridge_calculate
    from moleculekit.molecule import Molecule

    d = os.path.join(REFT, "test_interactions")
    mol = Molecule(os.path.join(d, "5gw6_receptor_H_wet.pdb"))
    mol.bonds = mol._guessBonds()
    lig, _, _ = _sdf_molecule(os.path.join(d, "5gw6_ligand-RDK.sdf"), "GOL")
    mol.append(lig)
    donors, acceptors = get_donors_acceptors(mol, exclude_water=False, exclude_backbone=False)
    asn = "protein and resname ASN and resid 155"
    w = {"coords": mol.coords.astype(np.float32), "box": mol.box.astype(np.float32), "donors": donors, "acceptors": acceptors,
         "gol": mol.atomselect("resname GOL"), "asn155": mol.atomselect(asn), "protein": mol.atomselect("protein"),
         "water": mol.atomselect("water")}
    kw = dict(dist_threshold=3.8, ignore_hs=True)
    wb1 = waterbridge_calculate(mol, donors, acceptors, "resname GOL", asn, order=1, **kw)
    assert np.array_equal(wb1, [[[3140, 2899, 2024]]]), wb1
    wb2 = waterbridge_calculate(mol, donors, acceptors, "resname GOL", asn, order=2, **kw)
    assert [list(map(int, p)) for p in wb2[0]] == [[3140, 2899, 2944, 2023], [3140, 2899, 2024]], wb2
    wb3 = waterbridge_calculate(mol, donors, acceptors, "resname GOL", "protein", order=1, **kw)
    assert np.array_equal(wb3, [[[3140, 2899, 2024], [3142, 2857, 1317], [3142, 2857, 2720], [3142, 2857, 2737],
                                 [3142, 2857, 2789]]]), wb3
    wb4 = waterbridge_calculate(mol, donors, acceptors, "resname GOL", "protein", order=1, dist_threshold=2.6)  # with hydrogens

    def flat(wb):  # ragged paths of frame 0 -> (lengths, concatenated indices)
        return np.array([len(p) for p in wb[0]], dtype=np.int64), np.array([i for p in wb[0] for i in p], dtype=np.int64)

    for name, wb in (("wb1", wb1), ("wb2", wb2), ("wb3", wb3), ("wb4", wb4)):
        w[f"{name}_len"], w[f"{name}_idx"] = flat(wb)
    np.savez_compressed(os.path.join(HERE, "waterbridge.npz"), **w)
    print("waterbridge.npz", mol.numAtoms, "atoms", len(donors), "donors", len(acceptors), "acceptors; with-H bridges:", len(wb4[0]))


def rings_fixture():
    """rings.npz (K13): (a) the reference's pipi_calculate / cationpi_calculate on a real structure -- the protein of its
    interaction tests (tests/test_interactions/3PTB_prepared.pdb, two frames: the second one jittered), rings from the
    reference's get_protein_rings, cations from get_protein_charged, wide thresholds so that the lists are not empty --
    and (b) seeded synthetic systems (planar 5/6-rings, cations above ring centres, halogen bonds; periodic boxes incl. zero
    components) through the compiled pipi / cationpi / sigmahole kernels.  The reference's own tests for these detectors
    need rdkit for the ligand rings (tests/test_interactions.py:57-253), so their constants cannot be rebuilt here."""
    from oracle import build_ref

    mods = build_ref.load()
    pipi, cat, sig = mods[7], mods[8], mods[9]
    from moleculekit.interactions.interactions import (cationpi_calculate, get_protein_charged, get_protein_rings,
                                                       pipi_calculate)
    from moleculekit.molecule import Molecule

    mol = Molecule(os.path.join(REFT, "test_interactions", "3PTB_prepared.pdb"))
    rng = np.random.default_rng(4)
    mol.coords = np.concatenate([mol.coords, mol.coords + rng.normal(0, 0.15, size=mol.coords.shape).astype(np.float32)], axis=2)
    mol.box = np.zeros((3, 2), np.float32)
    rings = get_protein_rings(mol)
    pos, _ = get_protein_charged(mol)
    w = {"p_coords": mol.coords.astype(np.float32), "p_box": mol.box, "p_ring_atoms": np.hstack(rings).astype(np.uint32),
         "p_ring_starts": np.insert(np.cumsum([len(r) for r in rings]), 0, 0).astype(np.uint32), "p_cations": pos}
    pp, da = pipi_calculate(mol, rings, rings, dist_threshold1=6.0, angle_threshold1_max=40, dist_threshold2=7.0,
                            angle_threshold2_min=50)
    cp, cda = cationpi_calculate(mol, rings, pos, dist_threshold=7.0, angle_threshold_min=30)
    for f in range(2):
        w[f"p_pipi_{f}"] = np.array(pp[f], dtype=np.int32).reshape(-1, 2); w[f"p_pipi_da_{f}"] = np.array(da[f], dtype=np.float32).reshape(-1, 2)
        w[f"p_cat_{f}"] = np.array(cp[f], dtype=np.int32).reshape(-1, 2); w[f"p_cat_da_{f}"] = np.array(cda[f], dtype=np.float32).reshape(-1, 2)
    assert len(pp[0]) > 3 and len(cp[0]) > 3, (len(pp[0]), len(cp[0]))
    rng = np.random.default_rng(11)
    ncase = 10
    for c in range(ncase):
        N = int(rng.integers(80, 300)); F = int(rng.integers(1, 5))
        L = rng.uniform(14, 25, size=(3, F)).astype(np.float32)
        if c == 0:
            L[:] = 0
        if c == 3:
            L[2, 0] = 0
        xyz = (rng.uniform(0, 1, size=(N, 3, F)) * 16 + rng.integers(-2, 3, size=(N, 3, 1)) * L[None]).astype(np.float32)
        rings_c, used = [], 0
        for r in range(int(rng.integers(4, 14))):
            k = int(rng.choice([5, 6])); idx = np.arange(used, used + k)
            if used + k > N - 12:
                break
            used += k
            ctr = rng.uniform(0, 16, size=(3, 1)); u = rng.normal(size=3); u /= np.linalg.norm(u)
            v = np.cross(u, rng.normal(size=3)); v /= np.linalg.norm(v)
            for j, a in enumerate(idx):
                ang = 2 * np.pi * j / k
                xyz[a] = (ctr + 1.39 * (np.cos(ang) * u[:, None] + np.sin(ang) * v[:, None]) + rng.normal(0, .05, size=(3, F))).astype(np.float32)
            rings_c.append(idx)
        k = len(rings_c) // 2
        if c % 3 == 0:   # a set against itself: identical rings are skipped
            ra = np.hstack(rings_c).astype(np.uint32)
            s1 = np.insert(np.cumsum([len(r) for r in rings_c]), 0, 0).astype(np.uint32); s2 = s1.copy()
        else:
            ra = np.hstack(rings_c).astype(np.uint32)
            s1 = np.insert(np.cumsum([len(r) for r in rings_c[:k]]), 0, 0).astype(np.uint32)
            s2 = (np.insert(np.cumsum([len(r) for r in rings_c[k:]]), 0, 0) + s1.max()).astype(np.uint32)
        sa = np.insert(np.cumsum([len(r) for r in rings_c]), 0, 0).astype(np.uint32)
        cations = rng.integers(used, N, size=int(rng.integers(2, 14))).astype(np.uint32)
        for q in cations[:4]:
            rr = rings_c[int(rng.integers(len(rings_c)))]
            ctr = xyz[rr].mean(axis=0); n = np.cross(xyz[rr[0]] - xyz[rr[2]], xyz[rr[1]] - xyz[rr[2]], axis=0); n /= np.linalg.norm(n, axis=0)
            xyz[q] = (ctr + 3.5 * n + rng.normal(0, .4, size=ctr.shape)).astype(np.float32)
        hal = np.stack([cations, rng.integers(used, N, size=len(cations))], 1).astype(np.uint32)
        th = np.array([rng.uniform(3.5, 8), rng.uniform(10, 50), rng.uniform(5, 10), rng.uniform(40, 80),
                       rng.uniform(4, 7), rng.uniform(20, 70)], dtype=np.float64)
        for kname, v in (("coords", xyz), ("box", L), ("ring_atoms", ra), ("s1", s1), ("s2", s2), ("sa", sa), ("cations", cations),
                         ("hal", hal), ("th", th)):
            w[f"r{c}_{kname}"] = v
        with np.errstate(all="ignore"):
            outs = (pipi.calculate(ra, s1, s2, xyz, L, *[float(x) for x in th[:4]]),
                    cat.calculate(ra, sa, cations, xyz, L, float(th[4]), float(th[5])),
                    sig.calculate(ra, sa, hal, xyz, L, float(th[4]), float(th[5]) / 4))
        for name, (res, da_) in zip(("pipi", "cat", "sig"), outs):
            w[f"r{c}_{name}_counts"] = np.array([len(x) // 2 for x in res])
            w[f"r{c}_{name}"] = np.array([v for x in res for v in x], dtype=np.int32).reshape(-1, 2)
            w[f"r{c}_{name}_da"] = np.array([v for x in da_ for v in x], dtype=np.float32).reshape(-1, 2)
    w["ncase"] = np.array(ncase)
    np.savez_compressed(os.path.join(HERE, "rings.npz"), **w)
    print("rings.npz", len(rings), "protein rings,", len(pos), "cations; pipi", len(pp[0]), "cation-pi", len(cp[0]),
          "synthetic hits", sum(int(w[f"r{c}_{n}_counts"].sum()) for c in range(ncase) for n in ("pipi", "cat", "sig")))


def rotation_fixture():
    """rotate.npz: outputs of the reference's rotateCoordinates (tools/voxeldescriptors.py:78-114) and rotationMatrix
    (util.py:70-117) on seeded inputs -- the float64 targets of mkb_rotate_coords."""
    from moleculekit.tools.voxeldescriptors import rotateCoordinates
    from moleculekit.util import rotationMatrix

    rng = np.random.default_rng(314)
    r = {}
    n = 5
    for c in range(n):
        coords = (rng.normal(0, 20, size=(int(rng.integers(1, 400)), 3)) + rng.normal(0, 50, size=3)).astype(np.float32)
        rot = rng.uniform(-2 * np.pi, 2 * np.pi, size=3)
        cen = coords.mean(axis=0).astype(np.float64) if c % 2 else rng.normal(0, 30, size=3)
        out = rotateCoordinates(coords, list(rot), list(cen))
        assert out.dtype == np.float64
        r[f"c{c}_coords"], r[f"c{c}_rot"], r[f"c{c}_center"], r[f"c{c}_out"] = coords, rot, cen, out
        r[f"c{c}_mats"] = np.stack([rotationMatrix([1, 0, 0], rot[0]), rotationMatrix([0, 1, 0], rot[1]),
                                    rotationMatrix([0, 0, 1], rot[2])])
    r["ncase"] = np.array(n)
    np.savez_compressed(os.path.join(HERE, "rotate.npz"), **r)


def within_fixture():
    """within.npz (K10): `within` / `exwithin` selections of the reference on its own test structures.  Expected masks come
    from the reference's STORED goldens tests/test_atomselect/selections.pickle where the selection string is stored
    ('within 5 of nucleic', 'exwithin 5 of nucleic'), else from the live reference atomselect; the live result is
    asserted equal to the stored golden wherever both exist (incl. the composite 'protein and within 8.3 of ...')."""
    import pickle

    from moleculekit.molecule import Molecule

    with open(os.path.join(REFT, "test_atomselect", "selections.pickle"), "rb") as f:
        stored = pickle.load(f)
    w = {}
    cases = []
    for pid in ("3ptb", "1bna", "3wbm", "6a5j"):
        mol = Molecule(pid)
        mol.serial[10] = -88  # tests/test_atomselect.py:139-141 mutate the molecule before selecting
        mol.beta[:] = 0
        mol.beta[1000:] = -1
        n = mol.numAtoms
        w[f"{pid}_coords"] = np.ascontiguousarray(mol.coords[:, :, mol.frame])
        for op, cutoff, src in (("within", 5, "nucleic"), ("exwithin", 5, "nucleic"), ("within", 8.3, "resname ALA"),
                                ("exwithin", 4, "index 2"), ("within", 8, "resid 100"), ("exwithin", 3.05, "name CA")):
            sel = f"{op} {cutoff} of {src}"
            live = mol.atomselect(sel)
            if (pid, sel) in stored:
                ref = np.zeros(n, dtype=bool)
                ref[np.asarray(stored[(pid, sel)], dtype=np.int64)] = True
                assert np.array_equal(ref, live), (pid, sel)
                origin = "stored"
            else:
                origin = "live"
            key = f"{pid}_{len(cases)}"
            w[key + "_source"] = mol.atomselect(src)
            w[key + "_expected"] = live
            cases.append((pid, op, str(cutoff), src, origin, key))
        comp = "protein and within 8.3 of resname ALA"
        ref = np.zeros(n, dtype=bool)
        ref[np.asarray(stored[(pid, comp)], dtype=np.int64)] = True
        assert np.array_equal(ref, mol.atomselect("protein") & mol.atomselect("within 8.3 of resname ALA")), pid
    w["cases"] = np.array(cases)
    np.savez_compressed(os.path.join(HERE, "within.npz"), **w)
    print("within cases:", len(cases), "stored-golden backed:", sum(c[4] == "stored" for c in cases))


def interactions_fixture():
    """interactions.npz: the reference's contact-type detectors on its own test structures (tests/test_interactions.py:
    117-161 salt bridges on 5ME6_prepared with its inline expected pairs; :329-351 metal coordination on 5vl5 / 3ptb) plus
    hydrophobic contacts and a two-frame periodic salt-bridge case from the live reference."""
    from moleculekit.interactions.interactions import (get_protein_charged, hydrophobic_calculate,
                                                       metal_coordination_calculate, saltbridge_calculate)
    from moleculekit.molecule import Molecule

    w = {}
    mol = Molecule(os.path.join(REFT, "test_interactions", "5ME6_prepared.pdb"))
    pos, neg = get_protein_charged(mol)
    br = saltbridge_calculate(mol, pos, neg, "protein", "protein")
    expected = np.array([[694, 725], [2146, 2183], [2158, 2346]])  # tests/test_interactions.py:158
    assert np.array_equal(expected, br[0])
    for k, v in (("coords", mol.coords), ("box", mol.box), ("resname", strarr(mol.resname)), ("name", strarr(mol.name)),
                 ("element", strarr(mol.element)), ("protein", mol.atomselect("protein")), ("pos", pos), ("neg", neg),
                 ("bridges", br[0])):
        w["me6_" + k] = v
    s1 = mol.atomselect("protein and resid 100 to 125")
    hy = hydrophobic_calculate(mol, s1, "protein", 4.0)
    w["me6_hyd_sel1"] = s1
    w["me6_hyd"] = hy[0]
    # two frames in a periodic box: the second frame is shifted by one box length along x for half of the atoms
    m2 = mol.copy()
    m2.coords = np.tile(m2.coords, (1, 1, 2)).copy()
    L = np.float32(150.0)
    m2.box = np.full((3, 2), L, dtype=np.float32)
    m2.coords[::2, 0, 1] += L
    half = np.zeros(m2.numAtoms, dtype=bool)
    half[::2] = True
    br2 = saltbridge_calculate(m2, pos, neg, half & m2.atomselect("protein"), ~half & m2.atomselect("protein"))
    assert len(br2) == 2 and len(br2[0]) > 0 and np.array_equal(br2[0], br2[1])  # images are found across the box
    w["me6_coords2"], w["me6_box2"], w["me6_half"], w["me6_bridges2"] = m2.coords, m2.box, half, br2[1]
    for pid, a, b, ref in (("5vl5", "all", "resname S31 and not element Cu",
                            [[933, 922], [933, 932], [933, 934], [933, 935], [933, 937], [933, 944]]),
                           ("3ptb", "not protein", "protein", [[1629, 383], [1629, 396], [1629, 420], [1629, 460]])):
        m = Molecule(pid)
        res = metal_coordination_calculate(m, a, b)
        assert np.array_equal(res[0], np.array(ref, dtype=np.uint32))  # tests/test_interactions.py:338-351
        w[pid + "_coords"], w[pid + "_box"], w[pid + "_element"] = m.coords, m.box, strarr(m.element)
        w[pid + "_sel1"], w[pid + "_sel2"], w[pid + "_metal"] = m.atomselect(a), m.atomselect(b), res[0]
    np.savez_compressed(os.path.join(HERE, "interactions.npz"), **w)
    print("interactions: hydrophobic pairs", len(hy[0]))


def xtc_fixture():
    """tests/golden/xtc/*.xtc + xtc.npz (K11): XTC files written by the reference's own writer (xtc.pyx:91-104 write_xtc)
    from seeded coordinates -- water-like triples (runs + the first-atom swap), a globular cloud, tightly clustered atoms
    (small-range adaptation), ranges above 2^24 (the plain bit-field branch), 3 / 9 / 10 atoms (the uncompressed branch
    and its boundary) and three re-encoded frames of the reference's real test trajectory -- with the arrays the
    reference's read_xtc returns for them.  The reference reader is also run on its full real trajectories (scratch
    copies) and must agree with the oracle frame for frame."""
    from oracle import build_ref, cpu_oracle

    xr = build_ref.load()[5]
    out_dir = os.path.join(HERE, "xtc")
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(2024)

    def water(nw, F, L):
        o = rng.uniform(0, L, size=(nw, 1, 3, 1))
        h = o + rng.normal(0, 0.06, size=(nw, 2, 3, 1))
        return (np.concatenate([o, h], axis=1).reshape(nw * 3, 3, 1) +
                np.cumsum(rng.normal(0, 0.05, size=(nw * 3, 3, F)), axis=2)).astype(np.float32)

    real_src = scratch_copy(os.path.join(REFT, "test_projections", "trajectory", "traj.xtc"))
    real = xr.read_xtc(real_src.encode())
    cases = {
        "water": water(120, 6, 3.0),
        "globule": rng.normal(0, 1.5, size=(257, 3, 5)).astype(np.float32),
        "clustered": (rng.normal(0, 0.02, size=(500, 3, 3)) + 5).astype(np.float32),
        "wide_x": np.stack([np.linspace(-8500, 8500, 60), rng.normal(0, 1, 60), rng.normal(0, 1, 60)], 1)[:, :, None]
        .repeat(2, 2).astype(np.float32),
        "wide_xyz": (np.linspace(-9000, 9000, 50)[:, None, None] * np.ones((1, 3, 2))).astype(np.float32),
        "atoms3": rng.normal(0, 1, size=(3, 3, 4)).astype(np.float32),
        "atoms9": rng.normal(0, 1, size=(9, 3, 2)).astype(np.float32),
        "atoms10": rng.normal(0, 1, size=(10, 3, 2)).astype(np.float32),
        "real3": np.ascontiguousarray(real[0][:, :, [0, 100, 199]]),
    }
    w = {"names": np.array(list(cases))}
    for name, xyz in cases.items():
        F = xyz.shape[2]
        box = np.zeros((3, 3, F), np.float32)
        box[0, 0] = 3.1; box[1, 1] = 3.2; box[2, 2] = 3.3; box[1, 0] = 0.25
        time = (np.arange(F) * 0.5 + 1).astype(np.float32)
        step = (np.arange(F) * 10 + 5).astype(np.uint32)
        fn = os.path.join(out_dir, name + ".xtc")
        xr.write_xtc(fn.encode(), np.ascontiguousarray(xyz), box, time, step)
        ref = xr.read_xtc(fn.encode())
        got = cpu_oracle.read_xtc(open(fn, "rb").read())
        for a, b in zip(ref, got):
            assert np.array_equal(np.asarray(a), np.asarray(b)), name
        assert np.abs(ref[0] - xyz).max() < 2e-3, name  # the reference round-trips within its precision
        for k, v in zip(("coords", "box", "time", "step"), ref):
            w[f"{name}_{k}"] = np.asarray(v)
    # full real trajectories: the oracle agrees with the reference on every frame (not committed: megabytes)
    for rel in (("test_projections", "trajectory", "traj.xtc"), ("test_wrapping", "6X18.xtc")):
        src = scratch_copy(os.path.join(REFT, *rel))
        ref = xr.read_xtc(src.encode())
        got = cpu_oracle.read_xtc(open(src, "rb").read())
        assert all(np.array_equal(np.asarray(a), np.asarray(b)) for a, b in zip(ref, got)), rel
        print("real trajectory", rel[-1], ref[0].shape, "oracle == reference")
    np.savez_compressed(os.path.join(HERE, "xtc.npz"), **w)
    for fcache in os.listdir(out_dir):  # index caches the reference reader leaves next to every file it opens
        if fcache.startswith("."):
            os.remove(os.path.join(out_dir, fcache))


def live_pins():
    """live_reference.json: sha256 of the oracle's outputs on the seeded cases of the *_vs_live_reference tests of
    tests/test_oracle_golden.py, so those comparisons also run where oracle/_ref is absent.  The tests record them
    themselves (MKB_RECORD_LIVE=1); with oracle/_ref built they first assert that every output equals the reference
    binary's, and the file notes per test whether that was the case."""
    import subprocess

    if os.path.isfile(os.path.join(HERE, "live_reference.json")):
        os.remove(os.path.join(HERE, "live_reference.json"))
    subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider",
                    os.path.join(ROOT, "tests", "test_oracle_golden.py"), "-k", "live_reference or float_overloads"],
                   check=True, cwd=ROOT, env=dict(os.environ, MKB_RECORD_LIVE="1"))


def main():
    from oracle import build_ref

    if "--only-live" in sys.argv:
        live_pins()
        return
    if "--only-xtc" in sys.argv:
        assert build_ref.build()
        xtc_fixture()
        return
    if "--only-interactions" in sys.argv:
        interactions_fixture()
        return
    if "--only-within" in sys.argv:
        within_fixture()
        return
    if "--only-rotation" in sys.argv:
        rotation_fixture()
        return
    if "--only-triclinic" in sys.argv:
        assert build_ref.build()
        triclinic_fixture()
        return
    if "--only-rings" in sys.argv:
        assert build_ref.build()
        rings_fixture()
        return
    if "--only-waterbridge" in sys.argv:
        waterbridge_fixture()
        return
    if "--only-hbonds" in sys.argv:
        assert build_ref.build()
        hbonds_fixture()
        return
    if "--only-wrapping" in sys.argv:
        assert build_ref.build()
        wrapping_fixture()
        return

    assert build_ref.build(), "oracle/_ref could not be built (is /root/reference present?)"
    occ_ref, dist_ref = build_ref.load()[:2]

    from moleculekit.molecule import Molecule  # the reference (scratch build on PYTHONPATH)
    from moleculekit.tools.voxeldescriptors import getCenters
    from moleculekit.periodictable import periodictable

    # ------------------------------------------------------------------ voxel: 3PTB (reference golden)
    vd = os.path.join(REFT, "test_voxeldescriptors")
    coords = np.load(os.path.join(vd, "3PTB_coords_inp.npy"))
    sigmas = np.load(os.path.join(vd, "3PTB_channels_inp.npy"))
    centers_inp = np.load(os.path.join(vd, "3PTB_centers_inp.npy"))
    gold_feat, gold_centers, gold_nvox = np.load(os.path.join(vd, "3PTB_voxres_old.npy"), allow_pickle=True)
    assert coords.dtype == np.float32 and sigmas.dtype == np.float64
    # The orphan *_inp.npy inputs predate the current vdW table: their single metal atom (the Ca2+ ion,
    # channels 6 and 7) carries sigma 1.37, whereas the stored golden was produced with today's
    # periodictable["Ca"].vdw_radius = 2.31 (reference test: mol.element "CA" -> "Ca",
    # tests/test_voxeldescriptors.py:71-86).  Patch that one row so inputs and golden agree.
    metal = sigmas[:, 6] != 0
    assert metal.sum() == 1
    sigmas = sigmas.copy()
    sigmas[metal] = np.where(sigmas[metal] != 0, periodictable["Ca"].vdw_radius, 0.0)

    class _M:  # minimal duck for reference getCenters/boundingBox
        def __init__(self, c):
            self.c = c

        def get(self, what, sel=None):
            return self.c

    centers, nvox = getCenters(_M(coords.copy()), buffer=8, voxelsize=1)
    assert np.array_equal(centers, centers_inp) and np.array_equal(centers, gold_centers)
    assert np.array_equal(nvox, gold_nvox) and list(nvox) == [60, 55, 65]
    out = np.zeros((centers.shape[0], 8))
    occ_ref.calculate_occupancy(centers, coords, sigmas, out)
    assert np.allclose(out, gold_feat), "today's reference kernel no longer matches its stored golden"
    assert np.array_equal(out != 0, gold_feat != 0)
    nz = np.flatnonzero(gold_feat.reshape(-1))
    np.savez_compressed(
        os.path.join(HERE, "voxel_3ptb.npz"),
        coords=coords, sigmas=sigmas, buffer=np.float64(8), voxelsize=np.float64(1),
        nvoxels=np.asarray(nvox, dtype=np.int64), bb_min=centers[0].copy(),
        centers_sha256=np.array(sha(centers)), centers_head=centers[:4], centers_tail=centers[-4:],
        # the reference's stored golden (tests/test_voxeldescriptors/3PTB_voxres_old.npy), sparse, f32 values
        gold_nz_idx=nz.astype(np.uint32), gold_nz_val=gold_feat.reshape(-1)[nz].astype(np.float32),
        # today's reference kernel on the same inputs, bit pattern pinned by hash + f64 checksum
        refkernel_sha256=np.array(sha(out)), refkernel_sum=np.float64(out.sum()),
        refkernel_nnz=np.int64(np.count_nonzero(out)),
    )

    # ------------------------------------------------------------------ voxel: small seeded cases (_ref outputs)
    rng = np.random.default_rng(1234)
    cases = {}
    # (a) arbitrary user centres, per-channel distinct sigmas, zero sigmas, negative sigma, coincident point
    N, M, C = 48, 700, 8
    xyz = (rng.normal(size=(N, 3)) * 4.0 + 20.0).astype(np.float32)
    ctr = rng.uniform(8.0, 32.0, size=(M, 3))
    ctr[0] = xyz[3].astype(np.float64)                      # d2 == 0 -> value 1
    ctr[1] = xyz[5].astype(np.float64) + [3.0, 4.0, 0.0]    # d2 == 25 exactly?  (only if exact in fp) gate check
    sg = rng.choice([0.0, 1.1, 1.52, 1.55, 1.7, 1.8, 2.0], size=(N, C), p=[.5, .1, .1, .1, .1, .05, .05])
    sg[7, 2] = -1.7
    o = np.zeros((M, C))
    occ_ref.calculate_occupancy(ctr, xyz, sg, o)
    cases["a"] = (xyz, ctr, sg, o)
    # (b) lattice points and lattice atoms: many exact d2 == 25 ties (3-4-0 triangles), C = 3
    g = np.arange(0, 9, dtype=np.float64)
    ctr = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    xyz = rng.integers(0, 9, size=(20, 3)).astype(np.float32)
    sg = rng.choice([0.0, 1.7, 3.4], size=(20, 3))
    o = np.zeros((ctr.shape[0], 3))
    occ_ref.calculate_occupancy(ctr, xyz, sg, o)
    cases["b"] = (xyz, ctr, sg, o)
    # (c) big coordinates (fp32 ulp ~ 1.5e-5) on a 0.5 A grid with f64 origin, C = 8 bool-like sigmas
    xyz = (rng.normal(size=(60, 3)) * 3.0 + np.array([210.0, -180.0, 95.0])).astype(np.float32)
    origin = np.array([210.0, -180.0, 95.0]) - 6.0 + 0.123456789
    ii = np.arange(24) * 0.5
    ctr = np.stack(np.meshgrid(ii, ii, ii, indexing="ij"), -1).reshape(-1, 3) + origin
    rad = rng.choice([1.52, 1.55, 1.7, 1.8], size=60)
    sg = rad[:, None] * (rng.random((60, 8)) < 0.4)
    o = np.zeros((ctr.shape[0], 8))
    occ_ref.calculate_occupancy(ctr, xyz, sg, o)
    cases["c"] = (xyz, ctr, sg, o)
    np.savez_compressed(os.path.join(HERE, "voxel_small.npz"),
                        **{f"{k}_{n}": v for k, tup in cases.items()
                           for n, v in zip(("coords", "centers", "sigmas", "out"), tup)})

    # ------------------------------------------------------------------ trajectory (every 10th frame)
    tr = os.path.join(REFT, "test_projections", "trajectory")
    md = os.path.join(REFT, "test_projections", "metricdistance")
    mol = Molecule(os.path.join(tr, "filtered.pdb"))
    mol.read(scratch_copy(os.path.join(tr, "traj.xtc")))
    molskip = Molecule(os.path.join(tr, "filtered.pdb"))
    molskip.read(scratch_copy(os.path.join(tr, "traj.xtc")), skip=10)
    assert np.array_equal(molskip.coords, mol.coords[:, :, ::10])
    sels = ["protein and name CA", "resname MOL and noh", "protein and noh",
            "protein and resid 1 to 50 and noh", "protein and resid 1 to 20 and noh", "protein"]
    masks = np.stack([mol.atomselect(s) for s in sels])
    from moleculekit.projections.metricdistance import MetricDistance, MetricSelfDistance

    def strarr(a):
        return np.array([str(x) for x in a])

    fx = dict(
        coords=molskip.coords, box=molskip.box, name=strarr(mol.name), resname=strarr(mol.resname),
        resid=mol.resid.astype(np.int64), chain=strarr(mol.chain), segid=strarr(mol.segid),
        element=strarr(mol.element), sel_strings=np.array(sels), sel_masks=masks,
        # reference stored goldens, frames ::10 (tests/test_metricdistance.py:182-278)
        gold_distances=np.load(os.path.join(md, "distances.npy"))[::10],
        gold_mindistances=np.load(os.path.join(md, "mindistances.npy"))[::10],
        gold_selfmindistance=np.load(os.path.join(md, "selfmindistance.npy"))[::10],
    )
    # sanity: the reference on the 20 skipped frames reproduces its goldens
    d = MetricDistance("protein and name CA", "resname MOL and noh", metric="distances", periodic="selections").project(molskip)
    assert np.allclose(d, fx["gold_distances"], atol=1e-3)
    fx["ref_distances"] = d  # exact float32 output of today's kernel on these frames
    fx["ref_mindistances"] = MetricDistance("protein and noh", "resname MOL and noh", periodic="selections",
                                            groupsel1="residue", groupsel2="all").project(molskip)
    fx["ref_selfmindistance"] = MetricSelfDistance("protein and resid 1 to 50 and noh", groupsel="residue").project(molskip)
    fx["ref_chains_distances"] = MetricDistance("protein and resid 1 to 20 and noh", "resname MOL and noh",
                                                periodic="chains").project(molskip)
    fx["ref_com_com"] = MetricDistance("protein and resid 1 to 50 and noh", "resname MOL and noh", "selections",
                                       groupsel1="residue", groupsel2="all", groupreduce1="com",
                                       groupreduce2="com").project(molskip)
    fx["ref_com_closest"] = MetricDistance("protein and resid 1 to 50 and noh", "resname MOL and noh", "selections",
                                           groupsel1="residue", groupsel2="all", groupreduce1="com",
                                           groupreduce2="closest").project(molskip)
    # MetricShell (tests/test_metricshell.py:8-26): stored golden refdata.npy, frames ::10, + today's output
    from moleculekit.projections.metricshell import MetricShell
    fx["gold_shell"] = np.load(os.path.join(REFT, "test_projections", "metricshell", "refdata.npy"))[::10]
    fx["ref_shell"] = MetricShell("protein and name CA", "resname MOL and noh", periodic="selections").project(molskip)
    assert np.allclose(fx["ref_shell"], fx["gold_shell"])
    fx["ref_shell_self"] = MetricShell("resname MOL and noh", "resname MOL and noh", periodic=None, numshells=6,
                                       shellwidth=1.5, truncate=7.0).project(molskip)
    # ordered contact pairs from the reference's contacts_trajectory (bit-exact target)
    from moleculekit.distance import calculate_contacts

    def pack(lst):
        cnt = np.array([len(x) for x in lst], dtype=np.int64)
        return cnt, (np.vstack(lst) if cnt.sum() else np.zeros((0, 2), np.uint32)).astype(np.uint32)

    ca, lig, noh = masks[0], masks[1], masks[2]
    fx["ct_ca_lig_sel8_cnt"], fx["ct_ca_lig_sel8_pairs"] = pack(calculate_contacts(molskip, ca, lig, "selections", 8))
    fx["ct_ca_ca_none6_cnt"], fx["ct_ca_ca_none6_pairs"] = pack(calculate_contacts(molskip, ca, ca, None, 6))
    fx["ct_noh_lig_chains5_cnt"], fx["ct_noh_lig_chains5_pairs"] = pack(calculate_contacts(molskip, noh, lig, "chains", 5))
    np.savez_compressed(os.path.join(HERE, "traj20.npz"), **fx)

    # ------------------------------------------------------------------ single-structure cases (3ptb, 5vl5)
    def molfix(pdbid):
        m = Molecule(pdbid)
        return m, dict(coords=m.coords.copy(), box=m.box.copy(), element=strarr(m.element), resname=strarr(m.resname),
                       resid=m.resid.astype(np.int64), name=strarr(m.name), chain=strarr(m.chain),
                       segid=strarr(m.segid),
                       masses=np.array([periodictable[e].mass for e in m.element], dtype=np.float32))

    m3, f3 = molfix("3ptb")
    f3["sel_protein"] = m3.atomselect("protein")
    f3["sel_ben"] = m3.atomselect("resname BEN")
    f3["sel_residue_1_2"] = m3.atomselect("residue 1 2")
    f3["sel_residue_3_4"] = m3.atomselect("residue 3 4")
    f3["sel_residue_1"] = m3.atomselect("residue 1"); f3["sel_residue_2"] = m3.atomselect("residue 2")
    f3["sel_residue_3"] = m3.atomselect("residue 3"); f3["sel_residue_4"] = m3.atomselect("residue 4")
    kw = dict(groupsel1="all", groupsel2="all")
    f3["ref_com_com"] = MetricDistance("protein", "resname BEN", None, groupreduce1="com", groupreduce2="com", **kw).project(m3)
    f3["ref_com_closest"] = MetricDistance("protein", "resname BEN", None, groupreduce1="com", groupreduce2="closest", **kw).project(m3)
    f3["ref_closest_com"] = MetricDistance("protein", "resname BEN", None, groupreduce1="closest", groupreduce2="com", **kw).project(m3)
    f3["ref_closest_closest"] = MetricDistance("protein", "resname BEN", None, groupreduce1="closest", groupreduce2="closest", **kw).project(m3)
    f3["ref_pairs_residue"] = MetricDistance("residue 1 2", "residue 3 4", None, pairs=True, groupsel1="residue",
                                             groupsel2="residue").project(m3)
    from moleculekit.periodictable import METAL_ELEMENTS
    metals = sorted(METAL_ELEMENTS)
    lig_el = ["N", "O", "Cl", "F", "Br", "I", "CL", "BR", "S"]
    s1, s2 = m3.atomselect("not protein"), m3.atomselect("protein")
    f3["mc_sel1"] = s1 & np.isin(m3.element, metals)
    f3["mc_sel2"] = s2 & np.isin(m3.element, lig_el)
    f3["mc_expected"] = np.array([[1629, 383], [1629, 396], [1629, 420], [1629, 460]], dtype=np.uint32)  # tests/test_interactions.py:346-349
    np.savez_compressed(os.path.join(HERE, "pdb_3ptb.npz"), **f3)

    m5, f5 = molfix("5vl5")
    s1, s2 = m5.atomselect("all"), m5.atomselect("resname S31 and not element Cu")
    f5 = dict(coords=f5["coords"], box=f5["box"], element=f5["element"])
    f5["mc_a_sel1"] = s1 & np.isin(m5.element, metals); f5["mc_a_sel2"] = s2 & np.isin(m5.element, lig_el)
    f5["mc_b_sel1"] = s1 & np.isin(m5.element, lig_el); f5["mc_b_sel2"] = s2 & np.isin(m5.element, metals)
    f5["mc_expected"] = np.array([[933, 922], [933, 932], [933, 934], [933, 935], [933, 937], [933, 944]],
                                 dtype=np.uint32)  # tests/test_interactions.py:338-341
    np.savez_compressed(os.path.join(HERE, "pdb_5vl5.npz"), **f5)

    # ------------------------------------------------------------------ seeded raw-kernel cases (_ref outputs, bit-exact targets)
    rng = np.random.default_rng(77)
    N, F = 120, 7
    L = np.array([18.0, 21.0, 16.5], dtype=np.float32)
    c = np.empty((N, 3, F), dtype=np.float32)
    c[:, :, 0] = rng.uniform(0, 1, size=(N, 3)) * L
    for f in range(1, F):
        c[:, :, f] = c[:, :, f - 1] + rng.normal(0, 1.5, size=(N, 3)).astype(np.float32)   # unwrapped walk, |n| up to ~3
    bx = (L[:, None] * (1 + 0.01 * rng.normal(size=(3, F)))).astype(np.float32)
    chains = rng.integers(0, 3, size=N).astype(np.uint32)
    s1 = np.sort(rng.choice(N, 37, replace=False)).astype(np.uint32)
    s2 = np.sort(rng.choice(N, 53, replace=False)).astype(np.uint32)
    rk = dict(coords=c, box=bx, chains=chains, sel1=s1, sel2=s2)
    r = np.zeros((F, 37 * 53), np.float32); dist_ref.dist_trajectory(c, bx, s1, s2, chains, False, True, r); rk["dist_pbc"] = r
    r = np.zeros((F, 37 * 53), np.float32); dist_ref.dist_trajectory(c, bx, s1, s2, chains, False, False, r); rk["dist_nopbc"] = r
    r = np.zeros((F, 37 * 36 // 2), np.float32); dist_ref.dist_trajectory(c, bx, s1, s1, chains, True, True, r); rk["dist_self_pbc"] = r
    ct = dist_ref.contacts_trajectory(c, bx, s1, s2, chains, False, True, 6.5)
    rk["ct_cnt"] = np.array([len(x) // 2 for x in ct], dtype=np.int64)
    rk["ct_pairs"] = np.concatenate([np.array(x, dtype=np.uint32) for x in ct]).reshape(-1, 2)
    ct = dist_ref.contacts_trajectory(c, bx, s1, s1, chains, True, True, 7.25)
    rk["ct_self_cnt"] = np.array([len(x) // 2 for x in ct], dtype=np.int64)
    rk["ct_self_pairs"] = np.concatenate([np.array(x, dtype=np.uint32) for x in ct]).reshape(-1, 2)
    groups1 = [sorted(rng.choice(N, rng.integers(1, 9), replace=False).tolist()) for _ in range(11)]
    groups2 = [sorted(rng.choice(N, rng.integers(1, 9), replace=False).tolist()) for _ in range(6)]
    masses = rng.choice([1.00794, 12.0107, 14.0067, 15.9994, 32.065], size=N).astype(np.float32)
    gc1 = np.array([chains[g[0]] for g in groups1], dtype=np.uint32)
    gc2 = np.array([chains[g[0]] for g in groups2], dtype=np.uint32)
    rk["g1_off"] = np.cumsum([0] + [len(g) for g in groups1]).astype(np.int64); rk["g1_atoms"] = np.concatenate(groups1).astype(np.int32)
    rk["g2_off"] = np.cumsum([0] + [len(g) for g in groups2]).astype(np.int64); rk["g2_atoms"] = np.concatenate(groups2).astype(np.int32)
    rk["masses"] = masses
    for r1 in (0, 1):
        for r2 in (0, 1):
            r = np.zeros((F, 11 * 6), np.float32)
            dist_ref.dist_trajectory_reduction(c, bx, groups1, groups2, gc1, gc2, False, True, masses, r1, r2, r)
            rk[f"red_{r1}{r2}"] = r
    r = np.zeros((F, 11 * 10 // 2), np.float32)
    dist_ref.dist_trajectory_reduction(c, bx, groups1, groups1, gc1, gc1, True, True, masses, 0, 0, r); rk["red_self"] = r
    r = np.zeros((F, 6), np.float32)
    dist_ref.dist_trajectory_reduction_pairs(c, bx, groups1[:6], groups2, gc1[:6], gc2, True, masses, 0, 1, r); rk["red_pairs_01"] = r
    for D in (1, 2, 3, 5):
        a = rng.normal(size=(13, D)).astype(np.float32) * 5; b = rng.normal(size=(9, D)).astype(np.float32) * 5
        r = np.zeros((13, 9), np.float32); dist_ref.cdist(a, b, r)
        p = np.zeros(13 * 12 // 2, np.float32); dist_ref.pdist(a, p)
        rk[f"cd{D}_a"], rk[f"cd{D}_b"], rk[f"cd{D}_out"], rk[f"pd{D}_out"] = a, b, r, p
    rk["sq_out"] = np.array(dist_ref.squareform(rk["pd3_out"]))
    rk["coll_out"] = np.array(dist_ref.get_collisions(rk["cd3_a"], rk["cd3_b"], 6.0), dtype=np.uint32).reshape(-1, 2)
    np.savez_compressed(os.path.join(HERE, "rawkernels.npz"), **rk)

    # ------------------------------------------------------------------ bond guessing (row a13): reference csv goldens
    from moleculekit.bondguesser import guess_bonds, vdw_radii as ref_vdw
    from moleculekit.molecule import calculateUniqueBonds

    bg = {}
    pdbids = ["3ptb", "3hyd", "6a5j", "5vbl", "7q5b", "1unc", "3zhi", "1a25", "1u5u", "1gzm", "6va1", "1bna", "3wbm",
              "1awf", "5vav"]  # tests/test_bondguesser.py:10-26
    for pid in pdbids:
        m = Molecule(pid)
        ref = np.loadtxt(os.path.join(REFT, "test_bondguesser", f"{pid}.csv"), delimiter=",").astype(np.uint32)
        got, _ = calculateUniqueBonds(guess_bonds(m).astype(np.uint32), [])
        assert np.array_equal(got, ref), pid  # the reference reproduces its own golden here
        bg[f"{pid}_coords"] = m.coords[:, :, m.frame].copy()
        bg[f"{pid}_element"] = strarr(m.element)
        bg[f"{pid}_name"] = strarr(m.name)
        bg[f"{pid}_bonds"] = ref
    bg["pdbids"] = np.array(pdbids)
    bg["vdw_keys"] = np.array(list(ref_vdw.keys()))
    bg["vdw_vals"] = np.array([float(v) for v in ref_vdw.values()])
    np.savez_compressed(os.path.join(HERE, "bonds.npz"), **bg)

    wrapping_fixture()
    rotation_fixture()
    within_fixture()
    interactions_fixture()
    xtc_fixture()

    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
