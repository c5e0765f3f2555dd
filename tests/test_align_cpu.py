"""Superposition (K14) without a GPU: the numpy restatement of the reference (tests/align_ref.py) and its identities, the
argument checks of the host entry points (all raise before any device call), MetricRmsd's mapping, and the split of
Molecule.wrap's bookkeeping (wrapping.wrap_plan) that MetricRmsd shares with wrapping.wrap."""
import numpy as np
import pytest

import align_ref as ar


@pytest.fixture
def no_device(monkeypatch):
    """Any attempt to reach a device fails the test."""
    from moleculekit_b200 import _lib, align

    def boom(*a, **k):
        raise AssertionError("the device was touched before the arguments were checked")

    monkeypatch.setattr(align, "_dev", boom)
    monkeypatch.setattr(_lib, "handle", boom)


def _cloud(seed=5, N=5000, F=50, nsel=715):
    rng = np.random.default_rng(seed)
    base = rng.normal(0, 12, size=(N, 3)) + 30.0
    coords, _, _ = ar.rigid_trajectory(rng, base, F, noise=0.5, spread=20.0)
    sel = np.sort(rng.choice(N, nsel, replace=False))
    return coords, sel


def test_oracle_proper_rotation_and_mirror():
    rng = np.random.default_rng(1)
    for trial in range(50):
        n = int(rng.integers(3, 200))
        P = rng.normal(size=(n, 3)) * 10
        Q = -P + rng.normal(size=(n, 3)) * 0.1 if trial % 2 else P @ ar.random_rotation(rng).T
        P, Q = P - P.mean(0), Q - Q.mean(0)
        R, rmsd = ar.measure_fit(P, Q)
        assert np.allclose(R @ R.T, np.eye(3), atol=1e-12) and np.linalg.det(R) == pytest.approx(1.0, abs=1e-12)
        # the returned rmsd (a difference of sums, so good to ~1e-6 here) is that of the optimal proper rotation unless
        # the target is a mirror image
        direct = np.sqrt(np.mean(np.sum((P @ R.T - Q) ** 2, axis=1)))
        if trial % 2 == 0:
            assert direct == pytest.approx(rmsd, abs=1e-5)
        else:
            assert direct >= rmsd - 1e-9


def test_oracle_identity_at_zero_covariance():
    """A one-atom selection has a zero covariance: the reference's SVD gives the identity, the alignment is a pure
    translation of every atom."""
    coords, _ = _cloud(F=4)
    ref = coords[:, :, 2:3].copy()
    xf = ar.transforms(coords, ref, np.array([17]), np.array([17]), range(4), 0, False)
    assert np.array_equal(xf[:, :9], np.tile(np.eye(3).ravel(), (4, 1)))
    out = ar.pp_align(coords, ref, np.array([17]), np.array([17]), range(4), 0, False)
    shift = ref[17, :, 0].astype(np.float64) - coords[17].astype(np.float64).T
    assert np.allclose(out.astype(np.float64) - coords.astype(np.float64), shift.T[None, :, :], atol=1e-4)
    assert np.allclose(out[17], ref[17], atol=1e-5)


def test_oracle_float32_within_bound_of_float64():
    """The reference's own float32 arithmetic against the float64 target on the seeded 5000-atom cloud."""
    coords, sel = _cloud()
    a32 = ar.pp_align(coords, coords, sel, sel, range(coords.shape[2]), 0, False, dtype=np.float32)
    a64 = ar.pp_align(coords, coords, sel, sel, range(coords.shape[2]), 0, False, dtype=np.float64)
    assert a32.dtype == a64.dtype == np.float32
    assert np.max(np.abs(a32.astype(np.float64) - a64)) < 5e-4
    r32 = ar.molRMSD(a32, coords[:, :, :1], sel, sel, dtype=np.float32)
    r64 = ar.molRMSD(a64, coords[:, :, :1], sel, sel)
    assert np.max(np.abs(r32 - r64) / r64[1:].min()) < 1e-5
    # the rigid motions are recovered: what is left is the noise of two frames, sqrt(6) * 0.5 A
    assert np.all(np.abs(r64[1:] - np.sqrt(6) * 0.5) < 0.1) and r64[0] < 1e-4


def test_pp_align_argument_checks(no_device):
    from moleculekit_b200.align import _pp_align

    c = np.zeros((10, 3, 4), np.float32)
    r = np.zeros((10, 3, 2), np.float32)
    s = np.arange(5)
    with pytest.raises(RuntimeError, match="0 atoms"):
        _pp_align(c, r, np.zeros(0, int), np.zeros(0, int), range(4), 0, False)
    with pytest.raises(RuntimeError, match="different number of atoms"):
        _pp_align(c, r, s, np.arange(4), range(4), 0, False)
    with pytest.raises(IndexError):
        _pp_align(c, r, s, s, [0, 4], 0, False)
    with pytest.raises(IndexError):
        _pp_align(c, r, s, s, [-1], 0, False)
    with pytest.raises(IndexError):
        _pp_align(c, r, np.array([0, 10]), np.array([0, 1]), range(4), 0, False)
    with pytest.raises(IndexError):
        _pp_align(c, r, s, s, range(4), 2, False)
    with pytest.raises(ValueError, match="matchingframes"):
        _pp_align(c, r, s, s, range(4), 0, True)
    with pytest.raises(ValueError, match="repeat"):
        _pp_align(c, r, s, s, [1, 1], 0, False)
    with pytest.raises(ValueError, match="float32"):
        _pp_align(c.astype(np.float64), r, s, s, range(4), 0, False)
    # nothing to do: no frames listed
    out = _pp_align(c, r, s, s, [], 0, False)
    assert out is not c and np.array_equal(out, c)


def test_align_and_molrmsd_argument_checks(no_device):
    from moleculekit_b200.align import align, molRMSD
    from moleculekit_b200.molecule_lite import MolLite

    rng = np.random.default_rng(0)
    mol = MolLite(rng.normal(size=(8, 3, 5)).astype(np.float32))
    with pytest.raises(NotImplementedError, match="moleculekit"):
        align(mol, np.arange(4), mode="structure")
    with pytest.raises(ValueError, match="mode"):
        align(mol, np.arange(4), mode="sequence")
    with pytest.raises(RuntimeError, match="different number of atoms"):
        align(mol, np.arange(4), refsel=np.arange(3))
    with pytest.raises(RuntimeError, match="0 atoms"):
        align(mol, np.zeros(8, bool))
    with pytest.raises(IndexError):
        align(mol, np.arange(4), frames=[5])
    ref3 = MolLite(rng.normal(size=(8, 3, 3)).astype(np.float32))
    with pytest.raises(ValueError, match="matchingframes"):
        align(mol, np.arange(4), refmol=ref3, matchingframes=True)
    with pytest.raises(ValueError, match="expected 1 or 5"):
        molRMSD(mol, ref3, np.arange(4), np.arange(4))
    with pytest.raises(ValueError):
        molRMSD(mol, mol, np.arange(4), np.arange(3))
    with pytest.raises(RuntimeError, match="0 atoms"):
        molRMSD(mol, mol, np.zeros(8, bool), np.zeros(8, bool))
    with pytest.raises(IndexError):
        molRMSD(mol, mol, np.array([8]), np.array([0]))


def test_metricrmsd_checks_and_mapping(no_device):
    from moleculekit_b200.molecule_lite import MolLite
    from moleculekit_b200.projections.metricrmsd import MetricRmsd

    rng = np.random.default_rng(2)
    ca = np.zeros(30, bool)
    ca[::3] = True
    sels = {"name CA": ca, "none": np.zeros(30, bool), "protein": np.ones(30, bool)}
    mol = MolLite(rng.normal(size=(30, 3, 4)).astype(np.float32), named_selections=sels,
                  resname=["ALA"] * 30, resid=np.arange(30) // 3, name=["N", "CA", "C"] * 10)
    ref = MolLite(mol.coords[:, :, :1], named_selections=sels)
    m = MetricRmsd(ref, "name CA", pbc=False)
    assert m._refmol is not ref
    mp = m.getMapping(mol)
    assert list(mp.columns) == ["type", "atomIndexes", "description"] and len(mp) == 1
    assert mp["type"][0] == "rmsd" and mp["description"][0] == "RMSD to reference structure."
    assert np.array_equal(mp["atomIndexes"][0], np.where(ca)[0])
    with pytest.raises(RuntimeError, match="RMSD atom selection resulted in 0 atoms"):
        MetricRmsd(ref, "none", trajalnstr="name CA", refrmsdstr="name CA", pbc=False).project(mol)
    with pytest.raises(RuntimeError, match="Alignment selection resulted in 0 atoms"):
        MetricRmsd(ref, "name CA", trajalnstr="none", refalnstr="name CA", pbc=False).project(mol)
    with pytest.raises(RuntimeError, match="Centering selection resulted in 0 atoms"):
        MetricRmsd(ref, "name CA", centerstr="none", pbc=True).project(mol)
    with pytest.raises(RuntimeError, match="different number of atoms"):
        MetricRmsd(ref, "name CA", refalnstr="protein", pbc=False).project(mol)
    ref3 = MolLite(mol.coords[:, :, :3], named_selections=sels)
    with pytest.raises(ValueError, match="expected 1 or 4"):
        MetricRmsd(ref3, "name CA", pbc=False).project(mol)


# ------------------------------------------------------------------------------------------- wrap_plan split
def _record_wraps(monkeypatch):
    from moleculekit_b200 import wrapping as wr

    calls = []
    monkeypatch.setattr(wr, "wrap_box", lambda g, c, b, cs, cen, device=None: calls.append(("box", g, cs, cen, None)))
    monkeypatch.setattr(wr, "wrap_triclinic_unitcell",
                        lambda g, c, bv, cs, cen, device=None: calls.append(("triclinic", g, cs, cen, bv)))
    monkeypatch.setattr(wr, "wrap_compact_unitcell",
                        lambda g, c, bv, cs, cen, mode, device=None: calls.append((mode, g, cs, cen, bv)))
    return calls


def test_wrap_decisions_unchanged(g_wrap, g_tric, monkeypatch):
    """wrap() still hands the same groups, centre selection / fixed centre and box vectors to the same kernel entry as
    before the split, and wrap_plan returns exactly what wrap() dispatches on."""
    from moleculekit_b200 import wrapping as wr
    from moleculekit_b200.molecule_lite import MolLite

    calls = _record_wraps(monkeypatch)
    g = g_wrap
    mask = np.zeros(g["coords"].shape[0], dtype=bool)
    mask[g["centersel"]] = True
    mol = MolLite(g["coords"].copy(), box=g["box"], bonds=g["bonds"], named_selections={"protein": mask})
    wr.wrap(mol, "protein")
    kind, groups, cs, cen, _ = calls.pop()
    assert kind == "box" and np.array_equal(groups, g["groups"]) and np.array_equal(cs, g["centersel"])
    assert np.array_equal(cen, np.zeros(3, np.float32))
    plan = wr.wrap_plan(mol, "protein")
    assert plan["unitcell"] is None and np.array_equal(plan["groups"], groups) and np.array_equal(plan["centersel"], cs)
    wr.wrap(mol, wrapcenter=g["center_fixed"])
    kind, groups, cs, cen, _ = calls.pop()
    assert kind == "box" and cs.size == 0 and np.array_equal(cen, g["center_fixed"].astype(np.float32))
    # zero box: no kernel, no plan
    mol0 = MolLite(g["coords"].copy(), box=np.zeros_like(g["box"]), bonds=g["bonds"])
    wr.wrap(mol0, wrapsel=mask)
    assert not calls and wr.wrap_plan(mol0, wrapsel=mask) is None
    with pytest.raises(RuntimeError, match="different number of simulation frames"):
        wr.wrap_plan(MolLite(g["coords"].copy(), box=g["box"][:, :2], bonds=g["bonds"]), wrapsel=mask)
    with pytest.raises(ValueError, match="Invalid unit cell type"):
        wr.wrap_plan(mol, unitcell="cubic")
    # triclinic cells: box vectors from lengths and angles, the reference's unitcell choice
    t = g_tric
    gr = t["groups"].astype(np.int64)
    bonds = np.concatenate([np.stack([np.arange(a, b - 1), np.arange(a + 1, b)], 1) for a, b in zip(gr[:-1], gr[1:])
                            if b - a > 1]).astype(np.uint32)
    sel = np.zeros(t["coords"].shape[0], bool)
    sel[t["centersel"]] = True
    for unitcell, want in (("triclinic", "triclinic"), ("compact", 1), ("rectangular", 0)):
        m = MolLite(t["coords"].copy(), box=t["box"], bonds=bonds, boxangles=t["boxangles"])
        with np.errstate(all="ignore"):
            wr.wrap(m, wrapsel=sel, unitcell=unitcell)
        kind, groups, cs, cen, bv = calls.pop()
        assert kind == want and np.array_equal(groups, t["groups"]) and np.array_equal(cs, t["centersel"])
        assert np.array_equal(bv, wr.box_vectors(t["box"], t["boxangles"]))
        plan = wr.wrap_plan(m, wrapsel=sel, unitcell=unitcell)
        assert plan["unitcell"] == unitcell and np.array_equal(plan["boxvectors"], bv)
