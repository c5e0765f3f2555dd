"""Pin the CPU oracle (oracle/mkb_oracle.c) against the reference.

Sources of truth, strongest first:
  * outputs of the reference's own compiled Cython kernels (oracle/_ref) -- live when present,
    and frozen in tests/golden/*.npz (tests/golden/make_golden.py) otherwise;
  * the reference's stored goldens (3PTB_voxres_old.npy, distances/mindistances/selfmindistance.npy).
Integer / float32 outputs must be bit-identical; the float64 occupancy must be bit-identical to the
reference kernel on the same libm (hash) and within allclose of the stored golden.
"""
import hashlib
import json
import os

import numpy as np
import pytest

LIVE_PINS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "live_reference.json")


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _lists(x):
    """a list of index lists (contacts / bonds per frame) as one int64 array: the lengths, then the entries"""
    return np.concatenate([np.array([len(v) for v in x], np.int64), np.array([w for v in x for w in v], np.int64)])


def _pin(name, outputs, live):
    """The oracle's outputs on the seeded cases of a *_vs_live_reference test, pinned by sha256 in
    tests/golden/live_reference.json, so the comparison runs without oracle/_ref.  With oracle/_ref present (``live``)
    the test has just compared the same outputs with the reference's binaries, so the pins are checked against the
    reference as well.  ``tests/golden/make_golden.py --only-live`` records them (MKB_RECORD_LIVE=1)."""
    digests = [_sha(o) for o in outputs]
    if os.environ.get("MKB_RECORD_LIVE"):
        pins = json.load(open(LIVE_PINS)) if os.path.isfile(LIVE_PINS) else {}
        pins[name] = digests
        pins.setdefault("_recorded_against", {})[name] = "reference binaries (oracle/_ref)" if live else "oracle only"
        with open(LIVE_PINS, "w") as f:
            json.dump(pins, f, indent=1, sort_keys=True)
        return
    with open(LIVE_PINS) as f:
        assert digests == json.load(f)[name], name


def _grid_centers(bb_min, nvox, vs):
    ix, iy, iz = [np.arange(n) * vs for n in nvox]
    g = np.stack(np.meshgrid(ix, iy, iz, indexing="ij"), -1).reshape(-1, 3).astype(np.float64)
    return g + bb_min


def test_occupancy_3ptb_golden(oracle, g_voxel3ptb):
    g = g_voxel3ptb
    centers = _grid_centers(g["bb_min"], g["nvoxels"], float(g["voxelsize"]))
    assert _sha(centers) == str(g["centers_sha256"])
    out = np.zeros((centers.shape[0], 8))
    oracle.calculate_occupancy(centers, g["coords"], g["sigmas"], out)
    # reference's stored golden (f32-rounded sparse copy): allclose like tests/test_voxeldescriptors.py:84
    gold = np.zeros(out.size, dtype=np.float64)
    gold[g["gold_nz_idx"]] = g["gold_nz_val"]
    assert np.array_equal(np.flatnonzero(out.reshape(-1)), g["gold_nz_idx"])
    assert np.allclose(out.reshape(-1), gold, rtol=1e-5, atol=1e-8)
    # today's reference kernel: identical bit pattern (same glibc exp) or, failing that, 1e-12 checksum
    assert int(g["refkernel_nnz"]) == np.count_nonzero(out)
    if _sha(out) != str(g["refkernel_sha256"]):
        assert abs(out.sum() - float(g["refkernel_sum"])) < 1e-9 * float(g["refkernel_sum"])


@pytest.mark.parametrize("case", ["a", "b", "c"])
def test_occupancy_small_golden(oracle, g_voxelsmall, case):
    g = g_voxelsmall
    out = np.zeros_like(g[f"{case}_out"])
    oracle.calculate_occupancy(g[f"{case}_centers"], g[f"{case}_coords"], g[f"{case}_sigmas"], out)
    assert np.array_equal(out != 0, g[f"{case}_out"] != 0)
    assert np.allclose(out, g[f"{case}_out"], rtol=1e-14, atol=0)


def test_occupancy_accumulates_and_ignores_nan(oracle):
    rng = np.random.default_rng(0)
    xyz = rng.normal(size=(10, 3)).astype(np.float32) * 3
    ctr = rng.normal(size=(50, 3)) * 3
    sg = np.full((10, 2), 1.7)
    sg[0, 0] = np.nan
    a = np.zeros((50, 2)); oracle.calculate_occupancy(ctr, xyz, sg, a)
    assert not np.isnan(a).any()
    b = np.full((50, 2), 0.5); oracle.calculate_occupancy(ctr, xyz, sg, b)
    assert np.array_equal(b, np.maximum(a, 0.5))


def test_dist_rawkernels_golden(oracle, g_raw):
    g = g_raw
    c, bx, ch, s1, s2 = g["coords"], g["box"], g["chains"], g["sel1"], g["sel2"]
    F = c.shape[2]
    r = np.zeros_like(g["dist_pbc"]); oracle.dist_trajectory(c, bx, s1, s2, ch, False, True, r)
    assert np.array_equal(r.view(np.uint32), g["dist_pbc"].view(np.uint32))
    r = np.zeros_like(g["dist_nopbc"]); oracle.dist_trajectory(c, bx, s1, s2, ch, False, False, r)
    assert np.array_equal(r.view(np.uint32), g["dist_nopbc"].view(np.uint32))
    r = np.zeros_like(g["dist_self_pbc"]); oracle.dist_trajectory(c, bx, s1, s1, ch, True, True, r)
    assert np.array_equal(r.view(np.uint32), g["dist_self_pbc"].view(np.uint32))
    ct = oracle.contacts_trajectory(c, bx, s1, s2, ch, False, True, 6.5)
    assert [len(x) // 2 for x in ct] == g["ct_cnt"].tolist()
    assert np.array_equal(np.concatenate([np.array(x, np.uint32) for x in ct]).reshape(-1, 2), g["ct_pairs"])
    ct = oracle.contacts_trajectory(c, bx, s1, s1, ch, True, True, 7.25)
    assert [len(x) // 2 for x in ct] == g["ct_self_cnt"].tolist()
    assert np.array_equal(np.concatenate([np.array(x, np.uint32) for x in ct]).reshape(-1, 2), g["ct_self_pairs"])

    def groups(off, atoms):
        return [atoms[off[i]:off[i + 1]].tolist() for i in range(len(off) - 1)]

    g1, g2 = groups(g["g1_off"], g["g1_atoms"]), groups(g["g2_off"], g["g2_atoms"])
    gc1 = np.array([ch[x[0]] for x in g1], np.uint32); gc2 = np.array([ch[x[0]] for x in g2], np.uint32)
    for r1 in (0, 1):
        for r2 in (0, 1):
            r = np.zeros((F, len(g1) * len(g2)), np.float32)
            oracle.dist_trajectory_reduction(c, bx, g1, g2, gc1, gc2, False, True, g["masses"], r1, r2, r)
            assert np.array_equal(r.view(np.uint32), g[f"red_{r1}{r2}"].view(np.uint32)), (r1, r2)
    r = np.zeros_like(g["red_self"])
    oracle.dist_trajectory_reduction(c, bx, g1, g1, gc1, gc1, True, True, g["masses"], 0, 0, r)
    assert np.array_equal(r.view(np.uint32), g["red_self"].view(np.uint32))
    r = np.zeros_like(g["red_pairs_01"])
    oracle.dist_trajectory_reduction_pairs(c, bx, g1[:6], g2, gc1[:6], gc2, True, g["masses"], 0, 1, r)
    assert np.array_equal(r.view(np.uint32), g["red_pairs_01"].view(np.uint32))
    for D in (1, 2, 3, 5):
        a, b = g[f"cd{D}_a"], g[f"cd{D}_b"]
        r = np.zeros((len(a), len(b)), np.float32); oracle.cdist(a, b, r)
        assert np.array_equal(r.view(np.uint32), g[f"cd{D}_out"].view(np.uint32))
        p = np.zeros(len(a) * (len(a) - 1) // 2, np.float32); oracle.pdist(a, p)
        assert np.array_equal(p.view(np.uint32), g[f"pd{D}_out"].view(np.uint32))
    assert np.array_equal(oracle.squareform(g["pd3_out"]), g["sq_out"])
    assert np.array_equal(np.array(oracle.get_collisions(g["cd3_a"], g["cd3_b"], 6.0), np.uint32).reshape(-1, 2),
                          g["coll_out"])


def test_dist_trajectory_fixture_golden(oracle, g_traj):
    """tests/test_metricdistance.py:182-193 on every 10th frame + exact output of today's kernel."""
    g = g_traj
    sel = {s: m for s, m in zip(g["sel_strings"].tolist(), g["sel_masks"])}
    s1 = np.where(sel["protein and name CA"])[0].astype(np.uint32)
    s2 = np.where(sel["resname MOL and noh"])[0].astype(np.uint32)
    ch = np.ones(g["coords"].shape[0], np.uint32); ch[s2] = 2
    r = np.zeros((g["coords"].shape[2], len(s1) * len(s2)), np.float32)
    oracle.dist_trajectory(g["coords"], g["box"], s1, s2, ch, False, True, r)
    assert np.allclose(r, g["gold_distances"], atol=1e-3)
    assert np.array_equal(r.view(np.uint32), g["ref_distances"].view(np.uint32))
    ct = oracle.contacts_trajectory(g["coords"], g["box"], s1, s2, ch, False, True, 8)
    assert [len(x) // 2 for x in ct] == g["ct_ca_lig_sel8_cnt"].tolist()
    assert np.array_equal(np.concatenate([np.array(x, np.uint32) for x in ct]).reshape(-1, 2), g["ct_ca_lig_sel8_pairs"])


def test_oracle_vs_live_reference(oracle, refmods):
    """When oracle/_ref is present (it is in the build container and travels to the GPU box),
    compare against the reference's own binaries on fresh random inputs."""
    live = refmods is not None
    occ_ref, dist_ref = refmods[:2] if live else (None, None)
    outs = []
    rng = np.random.default_rng(5)
    for trial in range(3):
        N, M, C = 30 + 10 * trial, 400, 1 + 3 * trial
        xyz = (rng.normal(size=(N, 3)) * 5).astype(np.float32)
        ctr = rng.normal(size=(M, 3)) * 6
        sg = rng.choice([0.0, 1.2, 1.7, 2.2], size=(N, C))
        b = np.zeros((M, C)); oracle.calculate_occupancy(ctr, xyz, sg, b)
        if live:
            a = np.zeros((M, C)); occ_ref.calculate_occupancy(ctr, xyz, sg, a)
            assert np.array_equal(a, b)
        outs.append(b)
    N, F = 64, 5
    c = (rng.normal(size=(N, 3, F)) * 12).astype(np.float32)
    bx = np.abs(rng.normal(size=(3, F)) * 2 + 15).astype(np.float32)
    ch = rng.integers(0, 4, N).astype(np.uint32)
    s1 = np.arange(0, 40, dtype=np.uint32); s2 = np.arange(20, 64, dtype=np.uint32)
    for pbc in (False, True):
        b = np.zeros((F, 40 * 44), np.float32); oracle.dist_trajectory(c, bx, s1, s2, ch, False, pbc, b)
        ct = oracle.contacts_trajectory(c, bx, s1, s2, ch, False, pbc, 9.0)
        if live:
            a = np.zeros((F, 40 * 44), np.float32); dist_ref.dist_trajectory(c, bx, s1, s2, ch, False, pbc, a)
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
            assert dist_ref.contacts_trajectory(c, bx, s1, s2, ch, False, pbc, 9.0) == ct
        outs += [b.view(np.uint32), _lists(ct)]
    _pin("occupancy_distances", outs, live)


def _canonical(b):
    b = np.sort(np.asarray(b, dtype=np.uint32).reshape(-1, 2), axis=1)
    b = np.unique(b, axis=0)
    return b


def test_bond_grid_search_golden(oracle, g_bonds):
    """Row a13: the reference's 15 csv goldens (tests/test_bondguesser.py:27-44), compared like the reference does
    (after calculateUniqueBonds).  The oracle's raw output ORDER was additionally checked identical to the reference's
    bond_grid_search in the build container (tests/golden/make_golden.py asserts the reference reproduces the csv)."""
    from moleculekit_b200 import bondguesser as bgm  # host-only use: the radii table and name rule

    g = g_bonds
    assert dict(zip(g["vdw_keys"].tolist(), g["vdw_vals"].tolist())) == {k: float(v) for k, v in bgm.vdw_radii.items()}
    for pid in g["pdbids"].tolist():
        coords = g[f"{pid}_coords"]
        radii = bgm.bond_radii(g[f"{pid}_element"], g[f"{pid}_name"])
        ish = (g[f"{pid}_element"] == "H").astype(np.uint32)
        got = oracle.bond_grid_search(coords, np.max(radii) * 1.2, ish, radii)
        assert np.array_equal(_canonical(got), g[f"{pid}_bonds"]), pid


def test_bond_kernel_vs_live_reference(oracle, refmods):
    """grid_bonds of the reference binary on one box pair vs the oracle's pair test (raw output order)."""
    live = refmods is not None
    rng = np.random.default_rng(3)
    n = 60
    coords = (rng.random((n, 3)) * 3.0).astype(np.float32)
    radii = rng.choice([1.0, 1.52, 1.7, 1.8], n).astype(np.float32)
    ish = (radii == 1.0).astype(np.uint32)
    got = oracle.bond_grid_search(coords, 4.0, ish, radii)           # range 3 < 4 -> a single box as well
    if live:
        bref = refmods[2]
        atoms_in_box = np.arange(n, dtype=np.uint32)[None, :]          # one box holding every atom
        gridlist = np.full((1, 14), 1, dtype=np.uint32)
        bref.make_grid_neighborlist_nonperiodic(gridlist, 1, 1, 1)
        want = np.array(bref.grid_bonds(coords, radii, ish, 4.0, 0, atoms_in_box, gridlist), dtype=np.uint32).reshape(-1, 2)
        assert np.array_equal(got, want)
    assert len(got) > 0
    _pin("bond_kernel", [np.ascontiguousarray(got, dtype=np.uint32)], live)


# ------------------------------------------------------------------------------------------------ K9: wrap_box
def _fbits(a):
    """float32 bit patterns with NaNs canonicalised (x86 and the GPU produce different NaN payloads)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = a.view(np.uint32).copy()
    b[np.isnan(a)] = 0x7FC00000
    return b


def test_wrap_box_oracle_vs_golden(oracle, g_wrap):
    """oracle_wrap_box against (a) the output of the reference's compiled wrap_box (bit-exact), (b) the reference's stored
    golden trajectory output_wrapped.xtc at the reference test's tolerance (tests/test_wrapping.py:16) and (c) the seeded
    reference outputs, incl. empty groups and a zero box component."""
    g = g_wrap
    zero = np.zeros(3, np.float32)
    out = g["coords"].copy()
    oracle.wrap_box(g["groups"], out, g["box"], g["centersel"], zero)
    assert np.array_equal(_fbits(out), _fbits(g["ref_wrapped"]))
    assert np.allclose(out, g["gold_wrapped_xtc"], atol=1e-2)
    assert not np.array_equal(out, g["coords"])
    out = g["coords"].copy()
    oracle.wrap_box(g["groups"], out, g["box"], np.zeros(0, np.uint32), g["center_fixed"])
    assert np.array_equal(_fbits(out), _fbits(g["ref_wrapped_fixed"]))
    for c in range(int(g["ncase"])):
        out = g[f"r{c}_coords"].copy()
        oracle.wrap_box(g[f"r{c}_groups"], out, g[f"r{c}_box"], g[f"r{c}_centersel"], g[f"r{c}_center"])
        assert np.array_equal(_fbits(out), _fbits(g[f"r{c}_ref"])), c


def test_wrap_box_oracle_vs_live_reference(oracle, refmods):
    live = refmods is not None
    outs = []
    rng = np.random.default_rng(5)
    for trial in range(12):
        N, F = int(rng.integers(1, 500)), int(rng.integers(1, 9))
        cuts = np.unique(np.concatenate([[0], rng.integers(0, N, size=int(rng.integers(0, 80))), [N]])).astype(np.uint32)
        box = rng.uniform(8, 30, size=(3, F)).astype(np.float32)
        xyz = rng.normal(0, 40, size=(N, 3, F)).astype(np.float32)
        cs = np.zeros(0, np.uint32) if trial % 3 == 0 else \
            np.sort(rng.choice(N, size=min(N, 23), replace=False)).astype(np.uint32)
        cen = rng.normal(0, 5, 3).astype(np.float32)
        b = xyz.copy()
        oracle.wrap_box(cuts, b, box, cs, cen)
        if live:
            a = xyz.copy()
            refmods[3].wrap_box(cuts, a, box, cs, cen)
            assert np.array_equal(_fbits(a), _fbits(b)), trial
        outs.append(_fbits(b))
    _pin("wrap_box", outs, live)



# ------------------------------------------------------------------------- K9b: triclinic / compact wrapping
TRIC_MODES = (("triclinic", None), ("compact", 1), ("rectangular", 0))


def _oracle_tric(oracle, name, mode, groups, coords, bv, cs, cen):
    if mode is None:
        oracle.wrap_triclinic_unitcell(groups, coords, bv, cs, cen)
    else:
        oracle.wrap_compact_unitcell(groups, coords, bv, cs, cen, mode)


def test_triclinic_wrapping_oracle_vs_golden(oracle, g_tric):
    """oracle_wrap_triclinic / oracle_wrap_compact against (a) the outputs of the reference's compiled kernels on the cut of
    its dodecahedral test system (bit-exact), (b) the reference's stored goldens output_{triclinic,compact,rectangular}_
    wrapped.xtc at the reference test's tolerance (tests/test_wrapping.py:31-44) and (c) seeded reference outputs."""
    g = g_tric
    zero = np.zeros(3, np.float32)
    for name, mode in TRIC_MODES:
        out = g["coords"].copy()
        _oracle_tric(oracle, name, mode, g["groups"], out, g["boxvectors"], g["centersel"], zero)
        assert np.array_equal(_fbits(out), _fbits(g[f"ref_{name}"])), name
        assert np.max(np.abs(out - g[f"gold_{name}_xtc"])) < 1e-2, name
        out = g["coords"].copy()
        _oracle_tric(oracle, name, mode, g["groups"], out, g["boxvectors"], np.zeros(0, np.uint32), g["center_fixed"])
        assert np.array_equal(_fbits(out), _fbits(g[f"ref_{name}_fixed"])), name
        for c in range(int(g["ncase"])):
            out = g[f"r{c}_coords"].copy()
            _oracle_tric(oracle, name, mode, g[f"r{c}_groups"], out, g[f"r{c}_boxvectors"], g[f"r{c}_centersel"],
                         g[f"r{c}_center"])
            assert np.array_equal(_fbits(out), _fbits(g[f"r{c}_ref_{name}"])), (name, c)


def test_triclinic_wrapping_oracle_vs_live_reference(oracle, refmods):
    live = refmods is not None
    outs = []
    rng = np.random.default_rng(6)
    for trial in range(9):
        N, F = int(rng.integers(1, 400)), int(rng.integers(1, 6))
        cuts = np.unique(np.concatenate([[0], rng.integers(0, N, size=int(rng.integers(0, 60))), [N]])).astype(np.uint32)
        L = rng.uniform(20, 40)
        vec = [[L, 0, 0], [0, L, 0], [L / 2, L / 2, L * np.sqrt(2) / 2]] if trial % 2 else \
            [[L, 0, 0], [L / 3, 2 * np.sqrt(2) * L / 3, 0], [-L / 3, np.sqrt(2) * L / 3, np.sqrt(6) * L / 3]]
        bv = np.repeat(np.array(vec)[:, :, None], F, axis=2) * (1 + 0.001 * rng.normal(size=(1, 1, F)))
        xyz = rng.normal(0, 60, size=(N, 3, F)).astype(np.float32)
        cs = np.zeros(0, np.uint32) if trial % 3 == 0 else \
            np.sort(rng.choice(N, size=min(N, 23), replace=False)).astype(np.uint32)
        cen = rng.normal(0, 5, 3).astype(np.float32)
        for name, mode in TRIC_MODES:
            b = xyz.copy()
            _oracle_tric(oracle, name, mode, cuts, b, bv, cs, cen)
            if live:
                a = xyz.copy()
                if mode is None:
                    refmods[3].wrap_triclinic_unitcell(cuts, a, bv, cs, cen)
                else:
                    refmods[3].wrap_compact_unitcell(cuts, a, bv, cs, cen, mode)
                assert np.array_equal(_fbits(a), _fbits(b)), (trial, name)
            outs.append(_fbits(b))
    _pin("triclinic_wrapping", outs, live)


def test_box_vectors_host_mirror(g_tric):
    """wrapping.box_vectors == Molecule.boxvectors of the reference on its dodecahedral system (stored in the fixture)."""
    from moleculekit_b200.wrapping import box_vectors

    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        got = box_vectors(g_tric["box"], g_tric["boxangles"])
    assert got.dtype == np.float64 and np.array_equal(got, g_tric["boxvectors"])


# ------------------------------------------------------------------------------------------- K12: hydrogen bonds
def _hb_arrays(res):
    return np.array([len(x) // 3 for x in res]), np.array([v for x in res for v in x], dtype=np.int32).reshape(-1, 3)


def test_hbonds_oracle_vs_golden(oracle, g_hbonds):
    """oracle_hbonds against the reference's hydrogen-bond test (tests/test_interactions.py:7-55; the fixture asserts its
    expected rows and its 178-row count when it is generated) and seeded outputs of the compiled hbonds.calculate incl. zero
    boxes, an overlapping donor pair and a NaN coordinate."""
    g = g_hbonds
    prot, ben = g["protein"].astype(np.uint32), g["ben"].astype(np.uint32)
    everything = np.ones_like(prot)

    def run(s1, s2, intra, ign=False, dth=2.5, ath=120):
        don, acc = g["donors"], g["acceptors"]
        sel_idx = np.where(s1.astype(bool) | s2.astype(bool))[0]           # interactions.py:439-447
        don = don[np.all(np.isin(don, sel_idx), axis=1)]
        acc = acc[np.isin(acc, sel_idx)]
        if ign:
            don = np.unique(don[:, 0])[:, None].astype(np.uint32)
        return oracle.hbonds_calculate(don, acc, g["coords"], g["box"], s1, s2, dth, ath, intra, ign)

    r = run(prot, ben, False)
    assert np.array_equal(np.array(r[0]).reshape(-1, 3), g["hb_prot_ben"]) and r[0] == r[1]
    assert np.array_equal(g["hb_prot_ben"], [[3414, 3421, 2471], [3414, 3422, 2789], [3415, 3423, 2472], [3415, 3424, 2482]])
    r = run(everything, everything, True)
    assert np.array_equal(np.array(r[0]).reshape(-1, 3), g["hb_all"]) and len(r[0]) == 3 * 178
    assert np.array_equal(np.array(run(everything, everything, True, ign=True)[0]).reshape(-1, 3), g["hb_all_nohs"])
    assert np.array_equal(np.array(run(everything, everything, True, dth=3.2, ath=100)[1]).reshape(-1, 3), g["hb_all_wide"])
    assert np.array_equal(np.array(run(prot, ben, False, ign=True, dth=3.5)[0]).reshape(-1, 3), g["hb_prot_ben_nohs"])
    for c in range(int(g["ncase"])):
        dth, ath = (float(x) for x in g[f"r{c}_thr"])
        for intra in (0, 1):
            for ign in (0, 1):
                dn = g[f"r{c}_donors"] if not ign else np.unique(g[f"r{c}_donors"][:, 0])[:, None].astype(np.uint32)
                res = oracle.hbonds_calculate(dn, g[f"r{c}_acceptors"], g[f"r{c}_coords"], g[f"r{c}_box"], g[f"r{c}_sel1"],
                                              g[f"r{c}_sel2"], dth, ath, bool(intra), bool(ign))
                counts, tri = _hb_arrays(res)
                assert np.array_equal(counts, g[f"r{c}_out_{intra}{ign}_counts"]), (c, intra, ign)
                assert np.array_equal(tri, g[f"r{c}_out_{intra}{ign}"]), (c, intra, ign)


def test_hbonds_oracle_vs_live_reference(oracle, refmods):
    live = refmods is not None
    outs = []
    rng = np.random.default_rng(8)
    for trial in range(10):
        N, F = int(rng.integers(20, 200)), int(rng.integers(1, 5))
        L = rng.uniform(8, 15, size=(3, F)).astype(np.float32)
        xyz = (rng.uniform(0, 1, size=(N, 3, F)) * 12).astype(np.float32)
        nd, na = int(rng.integers(1, 40)), int(rng.integers(1, 40))
        heavy, hyd = rng.integers(0, N, nd), rng.integers(0, N, nd)
        for k in range(nd):
            if hyd[k] != heavy[k]:
                v = rng.normal(size=(3, F)); v /= np.linalg.norm(v, axis=0)
                xyz[hyd[k]] = xyz[heavy[k]] + v.astype(np.float32)
        dn = np.stack([heavy, hyd], 1).astype(np.uint32)
        acc = rng.integers(0, N, na).astype(np.uint32)
        s1, s2 = (rng.random(N) < .6).astype(np.uint32), (rng.random(N) < .6).astype(np.uint32)
        dth, ath = float(rng.uniform(2, 6)), float(rng.uniform(60, 150))
        for intra in (False, True):
            for ign in (False, True):
                dd = dn if not ign else np.unique(dn[:, 0])[:, None].astype(np.uint32)
                got = oracle.hbonds_calculate(dd, acc, xyz, L, s1, s2, dth, ath, intra, ign)
                if live:
                    want = [list(x) for x in refmods[6].calculate(dd, acc, xyz, L, s1, s2, dist_threshold=dth,
                                                                  angle_threshold=ath, intra=intra, ignore_hs=ign)]
                    assert got == want, (trial, intra, ign)
                outs.append(_lists(got))
    _pin("hbonds", outs, live)



def _hb_dense_case(F, seed=7):
    """800 donor pairs x 800 acceptors in a ~9 A box with molecules displaced by up to 8 boxes (minimum-image integers up to
    8: box * n is inexact in float) and thresholds that let a third of the pairs through: every rounding of the wrap, the
    norms and the arc cosine gets exercised close to a decision boundary somewhere."""
    rng = np.random.default_rng(seed)
    N = 2400
    L = rng.uniform(7, 11, size=(3, F)).astype(np.float32)
    base = (rng.uniform(0, 1, size=(N, 3, F)) * 9).astype(np.float32)
    xyz = (base + rng.integers(-8, 9, size=(N, 3, 1)).astype(np.float32) * L[None]).astype(np.float32)
    heavy = np.arange(0, 1600, 2); hyd = heavy + 1
    v = rng.normal(size=(800, 3, F)); v /= np.linalg.norm(v, axis=1, keepdims=True)
    xyz[hyd] = xyz[heavy] + v.astype(np.float32)
    return np.stack([heavy, hyd], 1).astype(np.uint32), np.arange(1600, 2400).astype(np.uint32), xyz, L, np.ones(N, np.uint32)


def test_hbonds_float_overloads(oracle, refmods):
    """The reference is built as C++: round / sqrt / acos on float arguments are the float overloads.  On 2.6e7 pair tests
    (9.4e6 bonds) the oracle's float model equals the compiled reference exactly, while the model that goes through double
    (the .pyx read as C) does not -- index outputs alone rarely tell them apart, this case does."""
    import ctypes as C

    live = refmods is not None
    don, acc, xyz, L, ones = _hb_dense_case(40)
    got = oracle.hbonds_calculate(don, acc, xyz, L, ones, ones, 5.5, 95.0, True, False)
    if live:
        want = [list(x) for x in refmods[6].calculate(don, acc, xyz, L, ones, ones, dist_threshold=5.5,
                                                      angle_threshold=95.0, intra=True, ignore_hs=False)]
        assert got == want
    assert sum(map(len, got)) // 3 > 5_000_000
    _pin("hbonds_float_overloads", [_lists(got)], live)
    oracle.lib().oracle_hbonds_set_model(C.c_int(1))
    try:
        assert oracle.hbonds_calculate(don, acc, xyz, L, ones, ones, 5.5, 95.0, True, False) != got
    finally:
        oracle.lib().oracle_hbonds_set_model(C.c_int(0))



# ---------------------------------------------------------------------- K13: pi-pi, cation-pi, sigma-hole kernels
def _ring_arrays(res):
    pairs, da = res
    return (np.array([len(x) // 2 for x in pairs]), np.array([v for x in pairs for v in x], dtype=np.int32).reshape(-1, 2),
            np.array([v for x in da for v in x], dtype=np.float32).reshape(-1, 2))


def _ring_cases(g):
    """(name, mode, args) of every stored case: the protein of the reference's interaction tests + the seeded systems"""
    for f in range(2):
        c, b = np.ascontiguousarray(g["p_coords"][:, :, f:f + 1]), np.ascontiguousarray(g["p_box"][:, f:f + 1])
        # pipi_calculate concatenates the two ring lists (interactions.py:690-694): the same set twice is NOT "identical rings"
        ra2 = np.concatenate([g["p_ring_atoms"], g["p_ring_atoms"]])
        st2 = (g["p_ring_starts"] + g["p_ring_starts"].max()).astype(np.uint32)
        yield f"p_pipi_{f}", f"p_pipi_da_{f}", None, 0, (ra2, g["p_ring_starts"], st2, c, b, 6.0, 40.0, 7.0, 50.0)
        yield f"p_cat_{f}", f"p_cat_da_{f}", None, 1, (g["p_ring_atoms"], g["p_ring_starts"], g["p_cations"], c, b, 7.0, 30.0)
    for c in range(int(g["ncase"])):
        th = [float(x) for x in g[f"r{c}_th"]]
        xyz, L, ra = g[f"r{c}_coords"], g[f"r{c}_box"], g[f"r{c}_ring_atoms"]
        yield f"r{c}_pipi", f"r{c}_pipi_da", f"r{c}_pipi_counts", 0, (ra, g[f"r{c}_s1"], g[f"r{c}_s2"], xyz, L, *th[:4])
        yield f"r{c}_cat", f"r{c}_cat_da", f"r{c}_cat_counts", 1, (ra, g[f"r{c}_sa"], g[f"r{c}_cations"], xyz, L, th[4], th[5])
        yield f"r{c}_sig", f"r{c}_sig_da", f"r{c}_sig_counts", 2, (ra, g[f"r{c}_sa"], g[f"r{c}_hal"], xyz, L, th[4], th[5] / 4)


def test_ring_interactions_oracle_vs_golden(oracle, g_rings):
    """oracle_ring_interactions (pipi / cationpi / sigmahole .pyx) against the reference's outputs: pairs, distances AND
    angles bit for bit -- on the protein of the reference's interaction tests (rings of its get_protein_rings) and on the
    seeded periodic systems."""
    g = g_rings
    total = 0
    for name, da_name, cnt_name, mode, args in _ring_cases(g):
        counts, pairs, da = _ring_arrays(oracle.ring_interactions(mode, *args))
        assert np.array_equal(pairs, g[name]), name
        assert np.array_equal(_fbits(da), _fbits(g[da_name])), name
        if cnt_name:
            assert np.array_equal(counts, g[cnt_name]), name
        total += len(pairs)
    assert total > 300


def test_ring_interactions_oracle_vs_live_reference(oracle, refmods):
    live = refmods is not None
    outs = []
    rng = np.random.default_rng(12)
    hits = 0
    for trial in range(12):
        N, F = 120, int(rng.integers(1, 4))
        L = rng.uniform(10, 18, size=(3, F)).astype(np.float32)
        xyz = (rng.uniform(0, 1, size=(N, 3, F)) * 12).astype(np.float32)
        starts = np.arange(0, 61, 6, dtype=np.uint32)
        ra = np.arange(60, dtype=np.uint32)
        for r in range(10):
            ctr = rng.uniform(0, 12, size=(3, 1)); u = rng.normal(size=3); u /= np.linalg.norm(u)
            v = np.cross(u, rng.normal(size=3)); v /= np.linalg.norm(v)
            for j in range(6):
                xyz[6 * r + j] = (ctr + 1.39 * (np.cos(j * np.pi / 3) * u[:, None] + np.sin(j * np.pi / 3) * v[:, None])
                                  + rng.normal(0, .05, size=(3, F))).astype(np.float32)
        cations = rng.integers(60, N, size=9).astype(np.uint32)
        hal = np.stack([cations, rng.integers(60, N, size=9)], 1).astype(np.uint32)
        for mode, args in ((0, (ra, starts, starts, xyz, L, 6.5, 35.0, 8.0, 45.0)),
                           (1, (ra, starts, cations, xyz, L, 7.5, 15.0)),
                           (2, (ra, starts, hal, xyz, L, 7.5, 5.0))):
            got = _ring_arrays(oracle.ring_interactions(mode, *args))
            if live:
                want = _ring_arrays(refmods[7 + mode].calculate(*args))
                assert np.array_equal(want[0], got[0]) and np.array_equal(want[1], got[1]), (trial, mode)
                assert np.array_equal(_fbits(want[2]), _fbits(got[2])), (trial, mode)
            outs += [got[0].astype(np.int64), got[1].astype(np.int64), _fbits(got[2])]
            hits += len(got[1])
    assert hits > 100
    _pin("ring_interactions", outs, live)


def test_bonded_groups_host_mirror(g_wrap, refmods):
    """getBondedGroups (host logic of the wrap path) reproduces the reference's group offsets on the cut of its own
    test system, and the union-find keeps the reference's root identities on a scrambled bond list."""
    from moleculekit_b200 import wrapping as wr
    from moleculekit_b200.molecule_lite import MolLite

    g = g_wrap
    mol = MolLite(g["coords"], box=g["box"], bonds=g["bonds"])
    groups, group = wr.getBondedGroups(mol)
    assert groups.dtype == np.uint32 and np.array_equal(groups, g["groups"])
    assert group.shape == (mol.numAtoms,) and group[0] == 0 and group[-1] == len(groups) - 2
    if refmods is not None and len(refmods) >= 4:
        rng = np.random.default_rng(11)
        n = 400
        bonds = rng.integers(0, n, size=(500, 2)).astype(np.uint32)
        p1, s1 = np.arange(n, dtype=np.uint32), np.ones(n, np.uint32)
        p2, s2 = p1.copy(), s1.copy()
        refmods[3].get_bonded_groups(bonds, n, p1, s1)
        wr.get_bonded_groups(bonds, n, p2, s2)
        assert np.array_equal(p1, p2)


# ------------------------------------------------------------------------------------------------ K10: within_distance
def _within_cases(g):
    for pid, op, cutoff, src, origin, key in g["cases"].tolist():
        yield pid, op, float(cutoff), origin, g[f"{pid}_coords"], g[key + "_source"], g[key + "_expected"]


def test_within_oracle_vs_reference_goldens(oracle, g_within):
    """`within` / `exwithin` masks of the reference (8 of the 24 cases are its stored selections.pickle goldens) from the
    oracle's restatement of within_distance + the node logic of atomselect.py:231-254."""
    n_stored = 0
    for pid, op, cutoff, origin, coords, source, expected in _within_cases(g_within):
        n = coords.shape[0]
        mask = np.zeros(n, dtype=bool)
        if source.any():
            sc = coords[source]
            oracle.within_distance(coords, cutoff, np.arange(n, dtype=np.uint32), np.where(source)[0].astype(np.uint32),
                                   sc.min(axis=0), sc.max(axis=0), mask)
            if op == "exwithin":
                mask[source] = False
        assert np.array_equal(mask, expected), (pid, op, cutoff)
        n_stored += origin == "stored"
    assert n_stored == 8


def test_within_oracle_vs_live_reference(oracle, refmods):
    live = refmods is not None
    outs = []
    rng = np.random.default_rng(21)
    for t in range(12):
        N = int(rng.integers(2, 500))
        coords = rng.normal(0, 8, size=(N, 3)).astype(np.float32)
        cutoff = np.float32(rng.uniform(1, 6))
        if t % 3 == 0:  # atoms placed within a few ulps of the cutoff sphere of atom 0
            dirs = rng.normal(size=(N - 1, 3))
            dirs /= np.linalg.norm(dirs, axis=1)[:, None]
            coords[1:] = (coords[0] + dirs * (cutoff * (1 + rng.normal(0, 2e-7, size=(N - 1, 1))))).astype(np.float32)
            sel2 = np.array([0], np.uint32)
        else:
            sel2 = np.sort(rng.choice(N, int(rng.integers(1, min(N, 60) + 1)), replace=False)).astype(np.uint32)
        sel1 = np.sort(rng.choice(N, int(rng.integers(1, N + 1)), replace=False)).astype(np.uint32)
        a, b = np.zeros(len(sel1), bool), np.zeros(len(sel1), bool)
        a[0] = b[0] = True  # pre-set entries are never cleared
        mn, mx = coords[sel2].min(axis=0), coords[sel2].max(axis=0)
        oracle.within_distance(coords, float(cutoff), sel1, sel2, mn, mx, b)
        if live:
            refmods[4].within_distance(coords, float(cutoff), sel1, sel2, mn, mx, a)
            assert np.array_equal(a, b), t
        outs.append(b)
    _pin("within", outs, live)


# ------------------------------------------------------------------------------------------------ K11: XTC decoding
def test_xtc_oracle_and_header_walk_vs_reference_goldens(oracle, g_xtc):
    """The oracle's restatement of the XTC decompression and the product's header walk against arrays the reference's
    read_xtc returned for files written by the reference's write_xtc (tests/golden/xtc/)."""
    import os

    from moleculekit_b200 import xtc as px  # host-only use: the header walk

    g = g_xtc
    for name in g["names"].tolist():
        raw = open(os.path.join(g["_dir"], name + ".xtc"), "rb").read()
        coords, box, time, step = oracle.read_xtc(raw)
        assert np.array_equal(coords.view(np.uint32), g[f"{name}_coords"].view(np.uint32)), name
        assert np.array_equal(box, g[f"{name}_box"]) and np.array_equal(time, g[f"{name}_time"])
        assert np.array_equal(step, g[f"{name}_step"])
        idx = px.index_xtc(raw)
        assert idx["natoms"] == coords.shape[0] and len(idx["frames"]) == coords.shape[2]
        assert np.array_equal(idx["box"], g[f"{name}_box"]) and np.array_equal(idx["time"], g[f"{name}_time"])
        assert np.array_equal(idx["step"], g[f"{name}_step"])
        assert (idx["frames"]["smallidx"] < 0).all() == (coords.shape[0] <= 9)
    with pytest.raises(RuntimeError, match="bad magic"):
        px.index_xtc(b"\\x00" * 64)


def test_xtc_oracle_vs_live_reference(oracle, refmods, tmp_path):
    if refmods is None or len(refmods) < 6:
        pytest.skip("oracle/_ref not built")
    xr = refmods[5]
    rng = np.random.default_rng(77)
    for t in range(6):
        N, F = int(rng.integers(10, 400)), int(rng.integers(1, 5))
        xyz = (rng.normal(0, [0.05, 1.0, 30.0][t % 3], size=(N, 3, F)) + rng.normal(0, 3, 3)[None, :, None]).astype(np.float32)
        box = np.zeros((3, 3, F), np.float32)
        fn = str(tmp_path / f"t{t}.xtc")
        xr.write_xtc(fn.encode(), np.ascontiguousarray(xyz), box, np.zeros(F, np.float32), np.zeros(F, np.uint32))
        ref = xr.read_xtc(fn.encode())
        got = oracle.read_xtc(open(fn, "rb").read())
        assert np.array_equal(np.asarray(ref[0]).view(np.uint32), got[0].view(np.uint32)), t
