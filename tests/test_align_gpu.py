"""GPU parity of K14 (superposition: Molecule.align, molRMSD, MetricRmsd) against the numpy restatement of the reference
(tests/align_ref.py): the float64 restatement is the accuracy target, the float32 one the reference's own arithmetic."""
import numpy as np
import pytest

import align_ref as ar

pytestmark = pytest.mark.gpu


def _within_ulp(got, want64, ulps=1):
    """every float32 of ``got`` within ``ulps`` float32 ulp of the float64 ``want64``.  A coordinate that lands next to
    zero is a difference of terms of tens of Angstrom, which float64 carries to ~1e-13 A: there the ulp is floored at
    1e-10 A."""
    spacing = np.maximum(np.spacing(np.abs(want64).astype(np.float32)).astype(np.float64), 1e-10)
    return np.all(np.abs(got.astype(np.float64) - want64) <= ulps * spacing)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _rmsd_ok(got, want64):
    got = np.asarray(got, dtype=np.float64)
    return np.all(np.abs(got - want64) <= 1e-6 * np.abs(want64) + 1e-6)


def _exact(coords, xfs, frames):
    """float64 (x - cP) R^T + cQ of the listed frames with the oracle's transforms; other frames as given"""
    out = coords.astype(np.float64)
    for i, f in enumerate(frames):
        xf = xfs[i]
        out[:, :, f] = (coords[:, :, f].astype(np.float64) - xf[9:12]) @ xf[:9].reshape(3, 3).T + xf[12:]
    return out


def _dev_fit(coords, frames, sel, ref_rows, matching=False):
    import torch

    from moleculekit_b200 import align as al

    dev = torch.device("cuda:0")
    d = torch.from_numpy(np.ascontiguousarray(coords)).to(dev)
    xf = al.align_fit_device(d, np.asarray(frames), al.sel_tensor(sel, dev),
                             torch.from_numpy(np.ascontiguousarray(ref_rows)).to(dev), matching)
    return d, xf


# ---------------------------------------------------------------------------------------------- real trajectory
@pytest.fixture(scope="module")
def traj20(g_traj):
    g = dict(g_traj)
    names = list(g["sel_strings"])
    g["ca"] = np.where(g["sel_masks"][names.index("protein and name CA")])[0]
    g["protein"] = g["sel_masks"][names.index("protein")]
    return g


def test_traj20_align_to_frame0(traj20):
    from moleculekit_b200.align import align, molRMSD
    from moleculekit_b200.molecule_lite import MolLite

    g = traj20
    c0 = g["coords"]
    ca = g["ca"]
    assert ca.size == 277
    mol = MolLite(c0.copy())
    align(mol, ca)
    # float64 target with the GPU path's semantics: every frame fitted against frame 0 as it was before the call
    exact = _exact(c0, ar.transforms(c0, c0, ca, ca, range(20), 0, False), range(20))
    # the reference's own arithmetic: in place, frame 0 is aligned to itself first and later frames see that copy
    want32 = c0.copy()
    ar.pp_align(want32, want32, ca, ca, range(20), 0, False, inplace=True, dtype=np.float32)
    assert _within_ulp(mol.coords, exact)
    assert np.max(np.abs(mol.coords.astype(np.float64) - want32)) < 5e-4
    assert _within_ulp(mol.coords[:, :, 0], c0[:, :, 0].astype(np.float64))
    assert _rmsd_ok(molRMSD(mol, MolLite(c0[:, :, :1].copy()), ca, ca), ar.molRMSD(exact, c0[:, :, :1], ca, ca))


def test_traj20_align_to_separate_refmol(traj20):
    """a single-frame refmol: frame 7 moved by a known rigid motion; RMSD of the aligned CA against it"""
    from moleculekit_b200.align import align, molRMSD
    from moleculekit_b200.molecule_lite import MolLite

    g = traj20
    c0, ca = g["coords"], g["ca"]
    rng = np.random.default_rng(3)
    R = ar.random_rotation(rng)
    refc = ((c0[:, :, 7].astype(np.float64) @ R.T) + [5.0, -12.0, 40.0]).astype(np.float32)[:, :, None]
    refmol = MolLite(refc)
    mol = MolLite(c0.copy())
    align(mol, ca, refmol=refmol)
    exact = _exact(c0, ar.transforms(c0, refc, ca, ca, range(20), 0, False), range(20))
    assert _within_ulp(mol.coords, exact)
    want32 = ar.pp_align(c0, refc, ca, ca, range(20), 0, False, dtype=np.float32)
    assert np.max(np.abs(mol.coords.astype(np.float64) - want32)) < 5e-4
    assert _rmsd_ok(molRMSD(mol, refmol, ca, ca), ar.molRMSD(exact, refc, ca, ca))
    # frame 7 is the reference up to rounding
    assert np.max(np.abs(mol.coords[:, :, 7] - refc[:, :, 0])) < 1e-3


# -------------------------------------------------------------------------------------------- seeded synthetic
@pytest.fixture(scope="module")
def synth():
    rng = np.random.default_rng(11)
    N, F = 20000, 300
    base = rng.normal(0, 15, size=(N, 3))
    coords, _, _ = ar.rigid_trajectory(rng, base, F, noise=0.5, spread=25.0)
    sel = np.sort(rng.choice(2000, 300, replace=False))
    return coords, sel


def test_frames_subset_and_pp_align(synth):
    from moleculekit_b200.align import _pp_align

    coords, sel = synth
    frames = np.array([0, 3, 4, 5, 17, 100, 101, 299, 150])
    ref = coords[:, :, 40:41].copy()
    got = _pp_align(coords, ref, sel, sel, frames, 0, False)
    want = _exact(coords, ar.transforms(coords, ref, sel, sel, frames, 0, False), frames)
    assert _within_ulp(got[:, :, frames], want[:, :, frames])
    rest = np.setdiff1d(np.arange(300), frames)
    assert np.array_equal(_bits(got[:, :, rest]), _bits(coords[:, :, rest]))
    # inplace returns the caller's array
    c = coords.copy()
    assert _pp_align(c, ref, sel, sel, frames, 0, False, inplace=True) is c
    assert np.array_equal(_bits(c), _bits(got))


def test_matchingframes_and_different_refsel(synth):
    from moleculekit_b200.align import align
    from moleculekit_b200.molecule_lite import MolLite

    coords, sel = synth
    rng = np.random.default_rng(4)
    # the reference trajectory holds the same atoms 5 rows further down, each frame moved differently
    refc = np.zeros((coords.shape[0] + 5, 3, 300), np.float32)
    for f in range(300):
        refc[5:, :, f] = (coords[:, :, f].astype(np.float64) @ ar.random_rotation(rng).T + rng.normal(0, 9, 3)
                          + rng.normal(0, 0.2, size=(coords.shape[0], 3))).astype(np.float32)
    refmol = MolLite(refc, frame=3)
    mol = MolLite(coords.copy())
    align(mol, sel, refmol=refmol, refsel=sel + 5, matchingframes=True)
    want = _exact(coords, ar.transforms(coords, refc, sel, sel + 5, range(300), 3, True), range(300))
    assert _within_ulp(mol.coords, want)
    mol = MolLite(coords.copy())
    align(mol, sel, refmol=refmol, refsel=sel + 5)  # refmol.frame = 3 for every frame
    want = _exact(coords, ar.transforms(coords, refc, sel, sel + 5, range(300), 3, False), range(300))
    assert _within_ulp(mol.coords, want)


def test_mirror_image_target(synth):
    """a mirror image cannot be reached by a rotation: det +1, and the RMSD equals the oracle's reflection-corrected one"""
    import torch

    from moleculekit_b200 import align as al

    coords, sel = synth
    ref = -coords[sel][:, :, 10:11]
    d, xf = _dev_fit(coords, range(300), sel, ref)
    R = xf[:, :9].cpu().numpy().reshape(-1, 3, 3)
    assert np.allclose(np.linalg.det(R), 1.0, atol=1e-12)
    assert np.allclose(R @ R.transpose(0, 2, 1), np.eye(3), atol=1e-12)
    want_xf = ar.transforms(coords, ref, sel, np.arange(sel.size), range(300), 0, False)
    rmsd = al.rmsd_device(d, range(300), al.sel_tensor(sel, d.device), torch.from_numpy(ref).to(d.device), xf)
    want = ar.molRMSD(_exact(coords[sel], want_xf, range(300)), ref, slice(None), slice(None))
    assert _rmsd_ok(rmsd.cpu().numpy(), want)


def test_frame_shard_equals_whole(synth):
    import torch

    from moleculekit_b200 import align as al

    coords, sel = synth
    dev = torch.device("cuda:0")
    ref = torch.from_numpy(np.ascontiguousarray(coords[sel][:, :, :1])).to(dev)
    dsel = al.sel_tensor(sel, dev)
    whole = torch.from_numpy(coords).to(dev)
    xw = al.align_fit_device(whole, range(300), dsel, ref)
    rw = al.rmsd_device(whole, range(300), dsel, ref, xw)
    al.align_apply_device(whole, range(300), xw)
    d = torch.from_numpy(coords).to(dev)
    shard = d[:, :, 64:192]
    xs = al.align_fit_device(shard, range(128), dsel, ref)
    rs = al.rmsd_device(shard, range(128), dsel, ref, xs)
    assert al.align_apply_device(shard, range(128), xs).data_ptr() == shard.data_ptr()
    assert torch.equal(xs, xw[64:192]) and torch.equal(rs, rw[64:192])
    got, want = d.cpu().numpy(), whole.cpu().numpy()
    assert np.array_equal(_bits(got[:, :, 64:192]), _bits(want[:, :, 64:192]))
    assert np.array_equal(_bits(got[:, :, :64]), _bits(coords[:, :, :64]))
    assert np.array_equal(_bits(got[:, :, 192:]), _bits(coords[:, :, 192:]))


def test_fused_rmsd_and_determinism(synth):
    import torch

    from moleculekit_b200 import align as al

    coords, sel = synth
    dev = torch.device("cuda:0")
    rsel = np.arange(500, 4500, 7)  # an RMSD selection other than the fit selection
    ref_fit = torch.from_numpy(np.ascontiguousarray(coords[sel][:, :, 0:1])).to(dev)
    ref_rms = torch.from_numpy(np.ascontiguousarray(coords[rsel][:, :, 0:1])).to(dev)
    d = torch.from_numpy(coords).to(dev)
    dsel, drsel = al.sel_tensor(sel, dev), al.sel_tensor(rsel, dev)
    xf = al.align_fit_device(d, range(300), dsel, ref_fit)
    fused = al.rmsd_device(d, range(300), drsel, ref_rms, xf)
    xf2 = al.align_fit_device(d, range(300), dsel, ref_fit)
    fused2 = al.rmsd_device(d, range(300), drsel, ref_rms, xf2)
    assert np.array_equal(xf.cpu().numpy().view(np.uint64), xf2.cpu().numpy().view(np.uint64))
    assert np.array_equal(_bits(fused.cpu().numpy()), _bits(fused2.cpu().numpy()))
    al.align_apply_device(d, range(300), xf)
    plain = al.rmsd_device(d, range(300), drsel, ref_rms)
    f, p = fused.cpu().numpy().astype(np.float64), plain.cpu().numpy().astype(np.float64)
    assert np.all(np.abs(f - p) <= 1e-6 * p)
    want = ar.molRMSD(_exact(coords, ar.transforms(coords, coords[:, :, :1], sel, sel, range(300), 0, False),
                             range(300)), coords[:, :, :1], rsel, rsel)
    assert _rmsd_ok(f, want)


# --------------------------------------------------------------------------------------------- degenerate inputs
def test_one_atom_and_coincident_points(synth):
    coords, _ = synth
    c = coords[:3000, :, :40].copy()
    ref = c[[123]][:, :, 5:6]
    d, xf = _dev_fit(c, range(40), np.array([123]), ref)
    x = xf.cpu().numpy()
    assert np.array_equal(x[:, :9], np.tile(np.eye(3).ravel(), (40, 1)))  # exactly the identity: a pure translation
    assert np.array_equal(x[:, 12:], np.tile(ref[0, :, 0].astype(np.float64), (40, 1)))
    # coincident points: every fit atom at the same place in every frame
    c2 = c.copy()
    c2[100:110] = c2[100:101]
    d, xf = _dev_fit(c2, range(40), np.arange(100, 110), c[200:210, :, :1])
    assert np.array_equal(xf.cpu().numpy()[:, :9], np.tile(np.eye(3).ravel(), (40, 1)))


def test_collinear_selection(synth):
    """a rank-one covariance: the rotation is not unique; check the invariants instead"""
    import torch

    from moleculekit_b200 import align as al

    rng = np.random.default_rng(8)
    F, n = 64, 40
    t = rng.normal(size=n) * 10
    coords = np.zeros((n + 10, 3, F), np.float32)
    for f in range(F):
        u = rng.normal(size=3)
        coords[:n, :, f] = (np.outer(t, u / np.linalg.norm(u)) + rng.normal(0, 30, 3)).astype(np.float32)
        coords[n:, :, f] = rng.normal(0, 10, size=(10, 3)).astype(np.float32)
    ref = coords[:n, :, 0:1].copy()
    d, xf = _dev_fit(coords, range(F), np.arange(n), ref)
    R = xf[:, :9].cpu().numpy().reshape(-1, 3, 3)
    assert np.allclose(R @ R.transpose(0, 2, 1), np.eye(3), atol=1e-12) and np.allclose(np.linalg.det(R), 1, atol=1e-12)
    got = al.rmsd_device(d, range(F), al.sel_tensor(np.arange(n), d.device), torch.from_numpy(ref).to(d.device), xf)
    want = ar.molRMSD(_exact(coords, ar.transforms(coords, coords, np.arange(n), np.arange(n), range(F), 0, False),
                             range(F)), coords[:, :, :1], np.arange(n), np.arange(n))
    assert _rmsd_ok(got.cpu().numpy(), want)


def test_single_frame_million_atoms():
    from moleculekit_b200.align import _pp_align

    rng = np.random.default_rng(21)
    N = 1_000_000
    base = rng.uniform(-150, 150, size=(N, 3))
    coords = (base + rng.normal(0, 0.3, size=(N, 3))).astype(np.float32)[:, :, None]
    R = ar.random_rotation(rng)
    ref = (base @ R.T + [3.0, 4.0, -5.0]).astype(np.float32)[:, :, None]
    sel = np.sort(rng.choice(N, 200_000, replace=False))  # a fit selection of many chunks
    got = _pp_align(coords, ref, sel, sel, [0], 0, False)
    want = _exact(coords, ar.transforms(coords, ref, sel, sel, [0], 0, False), [0])
    assert _within_ulp(got, want)


def test_many_frames_three_atoms():
    from moleculekit_b200.align import _pp_align

    rng = np.random.default_rng(22)
    F = 20000
    base = rng.normal(0, 5, size=(50, 3))
    coords, _, _ = ar.rigid_trajectory(rng, base, F, noise=0.1, spread=30.0)
    sel = np.array([3, 17, 40])
    got = _pp_align(coords, coords, sel, sel, range(F), 0, False)
    want = _exact(coords, ar.transforms(coords, coords, sel, sel, range(F), 0, False), range(F))
    assert _within_ulp(got, want)


# ------------------------------------------------------------------------------------------------- MetricRmsd
@pytest.mark.parametrize("pbc", [True, False])
def test_metricrmsd_traj20(traj20, oracle, pbc):
    from moleculekit_b200.bondguesser import guess_bonds
    from moleculekit_b200.molecule_lite import MolLite
    from moleculekit_b200.projections.metricrmsd import MetricRmsd
    from moleculekit_b200.wrapping import getBondedGroups

    g = traj20
    c0, ca, prot = g["coords"], g["ca"], g["protein"]
    camask = np.zeros(c0.shape[0], bool)
    camask[ca] = True
    sels = {"protein and name CA": camask, "protein": prot}
    kw = dict(element=g["element"], name=g["name"], resname=g["resname"], resid=g["resid"], chain=g["chain"],
              named_selections=sels)
    mol = MolLite(c0.copy(), box=g["box"], **kw)
    mol.bonds = guess_bonds(mol)
    refmol = MolLite(c0[:, :, 0:1].copy(), **kw)
    m = MetricRmsd(refmol, "protein and name CA", pbc=pbc)
    got = m.project(mol)
    assert got.dtype == np.float32 and got.shape == (20,)
    assert np.array_equal(mol.coords, c0)  # the caller's molecule is untouched
    # oracle pipeline: wrap_box, float64 align, molRMSD
    w = c0.copy()
    if pbc:
        groups, _ = getBondedGroups(mol, mol.bonds)
        oracle.wrap_box(groups, w, g["box"], np.where(prot)[0].astype(np.uint32), np.zeros(3, np.float32))
    aligned = _exact(w, ar.transforms(w, refmol.coords, ca, ca, range(20), 0, False), range(20))
    want = ar.molRMSD(aligned, refmol.coords, ca, ca)
    assert _rmsd_ok(got, want)
    mp = m.getMapping(mol)
    assert len(mp) == 1 and mp["type"][0] == "rmsd" and np.array_equal(mp["atomIndexes"][0], ca)
    # a one-frame trajectory squeezes to a 0-d array like the reference
    one = MolLite(c0[:, :, 3:4].copy(), box=g["box"][:, 3:4], bonds=mol.bonds, **kw)
    r1 = m.project(one)
    assert r1.shape == () and abs(float(r1) - float(got[3])) <= 1e-6 * float(got[3]) + 1e-6
