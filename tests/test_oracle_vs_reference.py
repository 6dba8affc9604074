"""CPU tier: the restatement oracle against the REAL reference run live (oracle/_ref), on seeds the golden fixtures
do not contain.  Where the reference install is absent, against the recorded results of tests/recorded.py."""
import numpy as np
import pytest

import cases
import recorded
from impl_oracle import OracleImpl


def _corners(h):
    corners = [h.crs2xyzCoord([c, r, s]) for c in [0, h.ncrs[0] - 1] for r in [0, h.ncrs[1] - 1] for s in [0, h.ncrs[2] - 1]]
    return [sorted(float(p[k]) for p in corners) for k in range(3)]


class _Atom:
    def __init__(self, coord):
        self.coord = coord


@pytest.mark.parametrize("name,seed", [("ortho", 23), ("perm", 29), ("hex", 31), ("tric", 37)])
def test_oracle_matches_live_reference(name, seed, request):
    from pdb_eda_b200 import ccp4 as my_ccp4, synthetic
    data, _ = cases.make_case(name, seed)
    ref = recorded.reference()
    if ref is None:
        mdm = cases.parse_with(my_ccp4, data)
        orc = OracleImpl(mdm)
        rng = np.random.default_rng(seed)
        atoms = cases.random_atoms(mdm, 8, seed=seed + 1)      # from the header, bit-identical to the reference's (test_oracle_golden)
        radii = rng.uniform(0.5, 2.4, len(atoms))
        mean, std = recorded.host_mean_std(mdm)
        cut, bcut = recorded.inputs(request.node.name, [mean + 1.3 * std, mean + 2.4 * std])
        out = [[orc.sphere_lists(atoms, radii, c) for c in (0.0, cut, -cut)], orc.sphere_sums(atoms[:4], np.full(4, 2.2), np.array([0, 4]), cut, -cut)[0],
               orc.full_blobs(bcut, -bcut)]
        ops = synthetic.cartesianOperators("P 21 21 21" if name != "hex" else "P 65 2 2", cases.GEOMETRIES[name]["cell"])
        xs, ys, zs = _corners(mdm.header)
        shift = np.array([np.dot(mdm.header.orthoMat, (i, j, k)) for i in (-1, 0, 1) for j in (-1, 0, 1) for k in (-1, 0, 1)])
        out.append(orc.symmetry(atoms.astype(np.float64), ops, shift, [xs[0] - 5, ys[0] - 5, zs[0] - 5], [xs[-1] + 5, ys[-1] + 5, zs[-1] + 5]))
        recorded.check(request.node.name, out, rtol=1e-12, atol=1e-10)
        return
    ref_ccp4, ref_da, ref_cutils, _ = ref
    rdm = cases.parse_with(ref_ccp4, data)
    mdm = cases.parse_with(my_ccp4, data)
    orc = OracleImpl(mdm)
    rng = np.random.default_rng(seed)
    atoms = cases.random_atoms(rdm, 8, seed=seed + 1)
    radii = rng.uniform(0.5, 2.4, len(atoms))
    cut = float(rdm.meanDensity + 1.3 * rdm.stdDensity)
    recorded.inputs(request.node.name, [cut, float(rdm.meanDensity + 2.4 * rdm.stdDensity)], live=True)
    for c in (0.0, cut, -cut):
        want = [rdm.getSphereCrsFromXyz(a, r, c) for a, r in zip(atoms, radii)]
        crs, off = orc.sphere_lists(atoms, radii, c)
        assert [len(w) for w in want] == np.diff(off).tolist()
        assert np.array_equal(crs.reshape(-1, 3), np.array([x for w in want for x in w], dtype=np.int32).reshape(-1, 3))
    union = ref_cutils.getSphereCrsFromXyzList(rdm, list(atoms[:4]), 2.2)
    got = orc.sphere_sums(atoms[:4], np.full(4, 2.2), np.array([0, 4]), cut, -cut)[0]
    assert int(got[0]) == len(union)
    assert np.isclose(got[1], sum(ref_cutils.getPointDensityFromCrs(rdm, c) for c in union), rtol=1e-9, atol=1e-12)
    assert bool(got[6]) == bool(ref_cutils.testValidXyzList(rdm, list(atoms[:4]), 2.2))
    bcut = float(rdm.meanDensity + 2.4 * rdm.stdDensity)
    for c, part in zip((bcut, -bcut), orc.full_blobs(bcut, -bcut)):
        blobs = rdm.createFullBlobList(c)
        crs, label, stats = part
        assert len(blobs) == len(stats)
        for b, blob in enumerate(blobs):
            assert set(map(tuple, crs[label == b].tolist())) == blob.crsList
            assert np.isclose(stats[b, 1], blob.totalDensity, rtol=1e-9)
    ops = synthetic.cartesianOperators("P 21 21 21" if name != "hex" else "P 65 2 2", cases.GEOMETRIES[name]["cell"])
    h = rdm.header
    corners = [h.crs2xyzCoord([c, r, s]) for c in [0, h.ncrs[0] - 1] for r in [0, h.ncrs[1] - 1] for s in [0, h.ncrs[2] - 1]]
    xs, ys, zs = (sorted(float(p[k]) for p in corners) for k in range(3))
    sym = ref_cutils.createSymmetryAtoms([_Atom(a) for a in atoms], ops, h.orthoMat, xs, ys, zs)
    shift = np.array([np.dot(h.orthoMat, (i, j, k)) for i in (-1, 0, 1) for j in (-1, 0, 1) for k in (-1, 0, 1)])
    a, img, xyz = orc.symmetry(atoms.astype(np.float64), ops, shift, [xs[0] - 5, ys[0] - 5, zs[0] - 5], [xs[-1] + 5, ys[-1] + 5, zs[-1] + 5])
    assert len(sym) == len(a)
    assert np.allclose(xyz, np.array([np.asarray(s.coord, dtype=np.float64) for s in sym]), rtol=1e-12, atol=1e-10)
    nops = len(ops)
    assert [s.symmetry for s in sym] == [(int(i // nops) // 9 - 1, (int(i // nops) // 3) % 3 - 1, int(i // nops) % 3 - 1, int(i % nops)) for i in img]


@pytest.mark.parametrize("seed", [1, 2, 5, 8])
def test_oracle_matches_live_reference_on_random_geometries(seed, request):
    """The geometries of the GPU fuzz test (tests/test_cuda_vs_oracle.py::test_fuzz_random_geometries), oracle vs reference."""
    from pdb_eda_b200 import ccp4 as my_ccp4
    data, _ = cases.random_geometry(seed)
    ref = recorded.reference()
    if ref is None:
        mdm = cases.parse_with(my_ccp4, data)
        orc = OracleImpl(mdm)
        rng = np.random.default_rng(seed)
        atoms = cases.random_atoms(mdm, 6, seed=seed + 50, margin=4.0)
        radii = rng.uniform(0.4, 2.6, len(atoms))
        mean, std = recorded.host_mean_std(mdm)
        cut, bcut = recorded.inputs(request.node.name, [mean + 1.1 * std, mean + 2.2 * std])
        out = [[orc.sphere_lists(atoms, radii, c) for c in (0.0, cut, -cut)], orc.full_blobs(bcut, -bcut)]
        pts = np.stack([rng.integers(-2 * mdm.header.crsInterval[k], 3 * mdm.header.crsInterval[k], 60) for k in range(3)], axis=1)
        out.append(orc.point_density(pts))
        recorded.check(request.node.name, out, rtol=0, atol=0)
        return
    ref_ccp4, _, ref_cutils, _ = ref
    rdm = cases.parse_with(ref_ccp4, data)
    mdm = cases.parse_with(my_ccp4, data)
    assert np.array_equal(np.asarray(rdm.header.origin, float), np.asarray(mdm.header.origin, float))
    assert np.array_equal(rdm.header.deOrthoMat, mdm.header.deOrthoMat) and rdm.header.uniqueNcrs == mdm.header.uniqueNcrs
    orc = OracleImpl(mdm)
    rng = np.random.default_rng(seed)
    atoms = cases.random_atoms(rdm, 6, seed=seed + 50, margin=4.0)
    radii = rng.uniform(0.4, 2.6, len(atoms))
    cut = float(rdm.meanDensity + 1.1 * rdm.stdDensity)
    recorded.inputs(request.node.name, [cut, float(rdm.meanDensity + 2.2 * rdm.stdDensity)], live=True)
    for c in (0.0, cut, -cut):
        want = [rdm.getSphereCrsFromXyz(a, r, c) for a, r in zip(atoms, radii)]
        crs, off = orc.sphere_lists(atoms, radii, c)
        assert [len(w) for w in want] == np.diff(off).tolist()
        assert np.array_equal(crs.reshape(-1, 3), np.array([x for w in want for x in w], dtype=np.int32).reshape(-1, 3))
    bcut = float(rdm.meanDensity + 2.2 * rdm.stdDensity)
    for c, part in zip((bcut, -bcut), orc.full_blobs(bcut, -bcut)):
        blobs = rdm.createFullBlobList(c)
        crs, label, stats = part
        assert len(blobs) == len(stats)
        for b, blob in enumerate(blobs):
            assert set(map(tuple, crs[label == b].tolist())) == blob.crsList
    pts = np.stack([rng.integers(-2 * rdm.header.crsInterval[k], 3 * rdm.header.crsInterval[k], 60) for k in range(3)], axis=1)
    val, ok = orc.point_density(pts)
    assert [float(ref_cutils.getPointDensityFromCrs(rdm, [int(v) for v in p])) for p in pts] == val.tolist()
    assert [bool(ref_cutils.testValidCrs(rdm, [int(v) for v in p])) for p in pts] == ok.astype(bool).tolist()
