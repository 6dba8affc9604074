"""GPU tier: the DensityAnalysis API of this package against the REAL reference (oracle/_ref: unmodified pdb_eda
2.7.1 + compiled Cython cutils, run on the host CPU of the same box) on identical synthetic CCP4 / PDB inputs.

Covers what no test of the reference pins (SURVEY.md section 8c): aggregateCloud (ratio, voxel / electron totals,
atom / residue / domain tables, overlap completeness, medians), symmetry atoms, green / red blob lists, blob
statistics, atom / residue / symmetry-atom region density and discrepancy incl. the atom-mask path.
Bars: counts, voxel sets, labels, orders bit-exact; float64 sums and statistics within 1e-9 relative.
"""
import io
import os

import numpy as np
import pytest

import golden_checks as gc
import recorded
from pdb_eda_b200 import synthetic, structure

pytestmark = pytest.mark.gpu

CASES = {
    # name: (grid n, cell, space group, residues, axis order, crsStart)
    "p212121": dict(n=(64, 64, 64), cell=(32.0, 32.0, 32.0, 90, 90, 90), sg="P 21 21 21", residues=110, axisOrder=(1, 2, 3), crsStart=(0, 0, 0)),
    "perm": dict(n=(60, 72, 66), cell=(30.0, 36.0, 33.0, 90, 90, 90), sg="P 1 21 1", residues=90, axisOrder=(2, 3, 1), crsStart=(-4, 7, 3)),
    "hex": dict(n=(60, 60, 80), cell=(30.0, 30.0, 40.0, 90, 90, 120), sg="P 65 2 2", residues=60, axisOrder=(1, 2, 3), crsStart=(0, 0, 0)),
}


def _build(name):
    c = CASES[name]
    omat = synthetic.orthoMatrix(c["cell"])
    # keep the chain inside the cell: walk in a box inscribed in the (possibly skewed) cell
    lo = (omat @ np.array([0.25, 0.25, 0.1])) if c["cell"][5] != 90 else np.zeros(3)
    hi = (omat @ np.array([0.6, 0.75, 0.9])) if c["cell"][5] != 90 else np.array(c["cell"][:3])
    lo, hi = np.minimum(lo, hi), np.maximum(lo, hi)
    st = synthetic.polyAlaStructure(c["residues"], lo - 3 * (c["cell"][5] != 90), hi + 3 * (c["cell"][5] != 90), seed=31, residuesPerChain=50, hetero=5)
    fofc2, fofc = synthetic.mapPair(st, c["n"], c["cell"], seed=37, crsStart=c["crsStart"], axisOrder=c["axisOrder"])
    d1 = synthetic.ccp4Bytes(fofc2, c["cell"], c["n"], crsStart=c["crsStart"], axisOrder=c["axisOrder"])
    d2 = synthetic.ccp4Bytes(fofc, c["cell"], c["n"], crsStart=c["crsStart"], axisOrder=c["axisOrder"])
    ops = synthetic.cartesianOperators(c["sg"], c["cell"])
    pdb_text = structure.formatPDB(st, remark290=ops, cell=c["cell"], spaceGroup=c["sg"])
    return st, d1, d2, pdb_text


@pytest.fixture(scope="module", params=list(CASES))
def pair(request):
    """(reference DensityAnalysis, this package's) on the same inputs; the first is None without the reference installed,
    and the tests then compare with the recorded results (tests/recorded.py)."""
    from pdb_eda_b200 import ccp4, densityAnalysis, pdbParser
    st, d1, d2, pdb_text = _build(request.param)
    ref = recorded.reference()
    if ref is None:
        densityAnalysis.setGlobals(densityAnalysis._loadDefaultParams())
        m = densityAnalysis.fromFile(io.StringIO(pdb_text), io.BytesIO(d1), io.BytesIO(d2))
        assert m != 0
        (m1, s1), (m2, s2) = recorded.host_mean_std(m.densityObj), recorded.host_mean_std(m.diffDensityObj)
        cuts = recorded.inputs("pair-" + request.param, [m1 + 1.5 * s1, m2 + 3 * s2])
        gc.close([m.densityObj.densityCutoff, m.diffDensityObj.diffDensityCutoff], cuts)
        m.densityObj.densityCutoff, m.diffDensityObj.diffDensityCutoff = cuts
        return None, m
    ref_ccp4, ref_da, ref_cutils, ref_pp = ref
    densityAnalysis.setGlobals(ref_da.paramsGlobal)
    # reference side
    r_dens = ref_ccp4.parse(io.BytesIO(d1), "t")
    r_diff = ref_ccp4.parse(io.BytesIO(d2), "t")
    r_dens.densityCutoff = r_dens.meanDensity + 1.5 * r_dens.stdDensity
    r_diff.diffDensityCutoff = r_diff.meanDensity + 3 * r_diff.stdDensity
    recorded.inputs("pair-" + request.param, [r_dens.densityCutoff, r_diff.diffDensityCutoff], live=True)
    r_pdb = ref_pp.readPDBfile(io.StringIO(pdb_text))
    r = ref_da.DensityAnalysis("t", r_dens, r_diff, st, r_pdb)
    # this package, through its own loader (exercises fromFile, the PDB reader and the header parser)
    m = densityAnalysis.fromFile(io.StringIO(pdb_text), io.BytesIO(d1), io.BytesIO(d2))
    assert m != 0
    # the parity tests hand both sides the identical float32-narrowed cutoffs (SURVEY.md App. A.12)
    gc.close([m.densityObj.densityCutoff, m.diffDensityObj.diffDensityCutoff], [r_dens.densityCutoff, r_diff.diffDensityCutoff])
    m.densityObj.densityCutoff = r_dens.densityCutoff
    m.diffDensityObj.diffDensityCutoff = r_diff.diffDensityCutoff
    return r, m


def _same_rows(a, b, float_from):
    assert len(a) == len(b)
    for ra, rb in zip(a, b):
        assert list(ra[:float_from]) == list(rb[:float_from]), (ra, rb)
        for xa, xb in zip(ra[float_from:], rb[float_from:]):
            if isinstance(xa, (bool, np.bool_, str, tuple)):
                assert xa == xb
            else:
                gc.close(np.asarray(xa, dtype=np.float64), np.asarray(xb, dtype=np.float64), rtol=1e-9, atol=1e-9)


def _blob(b):
    return [np.array(sorted(b.crsList), dtype=np.int64).reshape(-1, 3), b.totalDensity, b.volume, list(b.centroid), list(b.coordCenter)]


def _atom(a):
    return [a.name, a.parent.id, getattr(a, "symmetry", None), np.asarray(a.coord, dtype=np.float64)]


def test_loader_and_structure(pair, request):
    r, m = pair
    if r is None:
        h = m.pdbObj.header
        recorded.check(request.node.name, [[_atom(a) for a in m.biopdbObj.get_atoms()], list(h.rotationMats), h.spaceGroup, h.resolution],
                       rtol=0, atol=0)
        return
    ra, ma = list(r.biopdbObj.get_atoms()), list(m.biopdbObj.get_atoms())
    assert len(ra) == len(ma)
    assert all(np.array_equal(x.coord, y.coord) and x.name == y.name for x, y in zip(ra, ma))
    assert len(r.pdbObj.header.rotationMats) == len(m.pdbObj.header.rotationMats)
    assert all(np.array_equal(x, y) for x, y in zip(r.pdbObj.header.rotationMats, m.pdbObj.header.rotationMats))
    assert r.pdbObj.header.spaceGroup == m.pdbObj.header.spaceGroup and r.pdbObj.header.resolution == m.pdbObj.header.resolution


def test_aggregate_cloud(pair, request):
    r, m = pair
    m.aggregateCloud()
    if r is None:
        assert m.densityElectronRatio is not None
        recorded.check(request.node.name, [m.numVoxelsAggregated, m.densityElectronRatio, m.totalAggregatedDensity, m.totalAggregatedElectrons,
                                           dict(m.atomTypeOverlapCompleteness), dict(m.atomTypeOverlapIncompleteness),
                                           m.residueCloudDescriptions, m.domainCloudDescriptions, m.atomCloudDescriptions, m.medians])
        return
    r.aggregateCloud()
    assert r.densityElectronRatio is not None and m.densityElectronRatio is not None
    assert r.numVoxelsAggregated == m.numVoxelsAggregated
    gc.close([m.densityElectronRatio, m.totalAggregatedDensity, m.totalAggregatedElectrons],
             [r.densityElectronRatio, r.totalAggregatedDensity, r.totalAggregatedElectrons])
    assert dict(r.atomTypeOverlapCompleteness) == dict(m.atomTypeOverlapCompleteness)
    assert dict(r.atomTypeOverlapIncompleteness) == dict(m.atomTypeOverlapIncompleteness)
    _same_rows(m.residueCloudDescriptions, r.residueCloudDescriptions, 3)
    _same_rows(m.domainCloudDescriptions, r.domainCloudDescriptions, 3)
    ra, ma = r.atomCloudDescriptions, m.atomCloudDescriptions
    assert ra.dtype == ma.dtype and len(ra) == len(ma)
    for field in ra.dtype.names:
        if ra.dtype[field].kind in "US" or ra.dtype[field].kind == "i":
            assert np.array_equal(ra[field], ma[field]), field
        else:
            gc.close(ma[field], ra[field], rtol=1e-9, atol=1e-9)
    assert r.medians.keys() == m.medians.keys()
    for column in r.medians:
        assert r.medians[column].keys() == m.medians[column].keys()
        gc.close([m.medians[column][t] for t in r.medians[column]], [r.medians[column][t] for t in r.medians[column]], rtol=1e-9, atol=1e-9)


def test_symmetry_atoms(pair, request):
    r, m = pair
    if r is None:
        assert m.symmetryAtomCoords.dtype == np.float64
        recorded.check(request.node.name, [len(m.symmetryOnlyAtoms), len(m.asymmetryAtoms), [a.symmetry for a in m.symmetryAtoms],
                                           [(a.name, a.parent.id) for a in m.symmetryAtoms], m.symmetryAtomCoords], rtol=1e-12, atol=1e-10)
        return
    rs, ms = r.symmetryAtoms, m.symmetryAtoms
    assert len(rs) == len(ms) and len(r.symmetryOnlyAtoms) == len(m.symmetryOnlyAtoms) and len(r.asymmetryAtoms) == len(m.asymmetryAtoms)
    assert [a.symmetry for a in rs] == [a.symmetry for a in ms]
    assert [(a.name, a.parent.id) for a in rs] == [(a.name, a.parent.id) for a in ms]
    gc.close(m.symmetryAtomCoords, r.symmetryAtomCoords, rtol=1e-12, atol=1e-10)
    assert m.symmetryAtomCoords.dtype == r.symmetryAtomCoords.dtype


def test_blob_lists_and_statistics(pair, request):
    r, m = pair
    if r is None:
        assert len(m.greenBlobList) > 3 and len(m.redBlobList) > 3
        blobs = [[_blob(b) for b in getattr(m, tag)] for tag in ("greenBlobList", "redBlobList")]
        m.aggregateCloud()
        stats = [m.calculateAtomSpecificBlobStatistics(getattr(m, tag)) for tag in ("greenBlobList", "redBlobList")]
        recorded.check(request.node.name, [blobs, stats])
        return
    for tag in ("greenBlobList", "redBlobList"):
        rb, mb = getattr(r, tag), getattr(m, tag)
        assert len(rb) == len(mb) and len(rb) > 3
        for x, y in zip(rb, mb):
            assert x.crsList == y.crsList                      # membership and order of blobs bit-exact
            gc.close([y.totalDensity, y.volume] + list(y.centroid) + list(y.coordCenter),
                     [x.totalDensity, x.volume] + list(x.centroid) + list(x.coordCenter), rtol=1e-9, atol=1e-9)
    r.aggregateCloud()
    m.aggregateCloud()
    for tag in ("greenBlobList", "redBlobList"):
        rstats = r.calculateAtomSpecificBlobStatistics(getattr(r, tag))
        mstats = m.calculateAtomSpecificBlobStatistics(getattr(m, tag))
        assert len(rstats) == len(mstats)
        for x, y in zip(rstats, mstats):
            assert x[1] == y[1] and x[3] == y[3] and x[5:10] == y[5:10]
            gc.close([y[0], y[2], y[4]] + list(np.asarray(y[10], dtype=np.float64)) + list(y[11]),
                     [x[0], x[2], x[4]] + list(np.asarray(x[10], dtype=np.float64)) + list(x[11]), rtol=1e-9, atol=1e-9)


def test_region_density_and_discrepancy(pair, request):
    r, m = pair
    mask = {"ALA": ["N", "CA", "C"]}
    if r is None:
        m.aggregateCloud()
        out = [m.calculateResidueRegionDensity(3.5, 1.5, "", mask), m.calculateResidueRegionDensity(3.5, 1.5, "ALA", None, True)]
        assert len(m.calculateResidueRegionDensity(3.5, 1.5, "HOH", None, True)) == 5
        with pytest.raises(IndexError):
            m.calculateResidueRegionDiscrepancies(3.5, 3.0, "", mask)
        out += [m.calculateResidueRegionDiscrepancies(3.5, 3.0, "ALA", mask), m.calculateAtomRegionDensity(2.0, 1.5, "CA"),
                m.calculateAtomRegionDiscrepancies(2.0, 3.0, "O")]
        m._symmetryAtoms = m.symmetryAtoms[::23]
        try:
            out += [m.calculateSymmetryAtomRegionDensity(2.0, 1.5), m.calculateSymmetryAtomRegionDiscrepancies(2.0, 3.0, "CB")]
        finally:
            m._symmetryAtoms = None
        one = [a.coord for a in list(m.biopdbObj.get_atoms())[:4]]
        out += [m.calculateRegionDensity(one, 2.5), m.calculateRegionDiscrepancy(one, 2.5)]
        recorded.check(request.node.name, out)
        return
    r.aggregateCloud()
    m.aggregateCloud()
    _same_rows(m.calculateResidueRegionDensity(3.5, 1.5, "", mask), r.calculateResidueRegionDensity(3.5, 1.5, "", mask), 4)
    # per-atom optimised radii; restricted to ALA because the reference raises TypeError on single-atom residues here
    # (pdb_eda/ccp4.py:457 hands the radius list to a Cython float parameter) -- this package handles them
    _same_rows(m.calculateResidueRegionDensity(3.5, 1.5, "ALA", None, True), r.calculateResidueRegionDensity(3.5, 1.5, "ALA", None, True), 4)
    assert len(m.calculateResidueRegionDensity(3.5, 1.5, "HOH", None, True)) == 5
    # the discrepancy variant fails on residues the mask empties (HOH here), in the reference and here alike
    with pytest.raises(IndexError):
        r.calculateResidueRegionDiscrepancies(3.5, 3.0, "", mask)
    with pytest.raises(IndexError):
        m.calculateResidueRegionDiscrepancies(3.5, 3.0, "", mask)
    _same_rows(m.calculateResidueRegionDiscrepancies(3.5, 3.0, "ALA", mask), r.calculateResidueRegionDiscrepancies(3.5, 3.0, "ALA", mask), 4)
    _same_rows(m.calculateAtomRegionDensity(2.0, 1.5, "CA"), r.calculateAtomRegionDensity(2.0, 1.5, "CA"), 5)
    _same_rows(m.calculateAtomRegionDiscrepancies(2.0, 3.0, "O"), r.calculateAtomRegionDiscrepancies(2.0, 3.0, "O"), 5)
    # symmetry-atom variants on a subset (the reference needs ~30 ms per atom)
    rsub, msub = r.symmetryAtoms[::23], m.symmetryAtoms[::23]
    r._symmetryAtoms, m._symmetryAtoms = rsub, msub
    try:
        ra = r.calculateSymmetryAtomRegionDensity(2.0, 1.5)
        ma = m.calculateSymmetryAtomRegionDensity(2.0, 1.5)
        assert [x[:6] for x in ra] == [x[:6] for x in ma]
        assert [x[7] for x in ra] == [x[7] for x in ma]
        gc.close([x[8:] for x in ma], [x[8:] for x in ra], rtol=1e-9, atol=1e-9)
        rd = r.calculateSymmetryAtomRegionDiscrepancies(2.0, 3.0, "CB")
        md = m.calculateSymmetryAtomRegionDiscrepancies(2.0, 3.0, "CB")
        assert [x[:6] for x in rd] == [x[:6] for x in md] and [x[7] for x in rd] == [x[7] for x in md]
        gc.close([x[8:] for x in md], [x[8:] for x in rd], rtol=1e-9, atol=1e-9)
    finally:
        r._symmetryAtoms = m._symmetryAtoms = None
    one = [a.coord for a in list(m.biopdbObj.get_atoms())[:4]]
    gc.close(m.calculateRegionDensity(one, 2.5), r.calculateRegionDensity(one, 2.5), rtol=1e-9, atol=1e-12)
    gc.close(m.calculateRegionDiscrepancy(one, 2.5), r.calculateRegionDiscrepancy(one, 2.5), rtol=1e-9, atol=1e-12)


def test_rscc_rsr_metrics(pair, request):
    """residueMetrics / atomMetrics / calculateRsccRsrMetrics / medianAbsFoFc (SURVEY.md section 8f-3)."""
    import warnings
    r, m = pair
    if r is None:
        rres = m.residueMetrics()
        assert np.isfinite(np.array([x[3] for x in rres], dtype=np.float64)).sum() > len(rres) // 2
        crs = m.densityObj.getSphereCrsFromXyz(m.asymmetryAtoms[3].coord, 1.4, 0.0)
        recorded.check(request.node.name, [rres, m.atomMetrics(m.asymmetryAtoms[::7]), m.medianAbsFoFc(), m.calculateRsccRsrMetrics(crs),
                                           np.asarray(m.fc.density)], rtol=1e-8)
        return
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        rres = r.residueMetrics()
        ratoms = r.atomMetrics(r.asymmetryAtoms[::7])
        rmed = r.medianAbsFoFc()
        crs = r.densityObj.getSphereCrsFromXyz(r.asymmetryAtoms[3].coord, 1.4, 0.0)
        rone = r.calculateRsccRsrMetrics(crs)
    mres = m.residueMetrics()
    matoms = m.atomMetrics(m.asymmetryAtoms[::7])
    assert [x[:3] for x in rres] == [x[:3] for x in mres]
    ok = np.isfinite(np.array([x[3] for x in rres], dtype=np.float64))
    assert ok.sum() > len(rres) // 2
    gc.close(np.array([x[3:] for x in mres], dtype=np.float64)[ok], np.array([x[3:] for x in rres], dtype=np.float64)[ok], rtol=1e-8, atol=1e-9)
    assert [x[:5] for x in ratoms] == [x[:5] for x in matoms]
    gc.close([x[6:] for x in matoms], [x[6:] for x in ratoms], rtol=1e-8, atol=1e-9)
    gc.close(m.medianAbsFoFc(), rmed, rtol=1e-9)
    gc.close(m.calculateRsccRsrMetrics(crs), rone, rtol=1e-8, atol=1e-9)
    assert np.array_equal(np.asarray(m.fc.density), r.fc.density)


def test_blue_blob_list(pair, request):
    """blueBlobList: createFullBlobList(mean + 1.5 sigma) on the 2Fo-Fc map (pdb_eda/densityAnalysis.py:414-423) -- dense
    foreground (the reference warns that it "uses a LOT OF MEMORY at 1.5sd", pdb_eda/singleStructure.py:30)."""
    r, m = pair
    if r is None:
        mb = m.blueBlobList
        assert len(mb) >= 1 and sum(len(q.crsList) for q in mb) > 1000
        recorded.check(request.node.name, [_blob(b) for b in mb])
        return
    rb, mb = r.blueBlobList, m.blueBlobList
    assert len(rb) == len(mb) >= 1 and sum(len(p.crsList) for p in rb) > 1000
    assert all(p.crsList == q.crsList for p, q in zip(rb, mb))                       # membership and order
    gc.close([q.totalDensity for q in mb], [p.totalDensity for p in rb], rtol=1e-9)
    gc.close([q.volume for q in mb], [p.volume for p in rb], rtol=1e-12)
    gc.close([q.centroid for q in mb], [p.centroid for p in rb], rtol=1e-9, atol=1e-9)


def test_fc_object_and_single_coordinate_regions(pair, request):
    """ADVICE items: the public ``fc`` attribute answers the calls the reference's deep copy answers, and the region methods
    accept a single flat coordinate like findAberrantBlobs does (pdb_eda/ccp4.py:453)."""
    r, m = pair
    if r is None:
        cut = m.densityObj.densityCutoff
        assert m.fc.meanDensity == m.densityObj.meanDensity
        one = [float(v) for v in m.asymmetryAtoms[7].coord]
        gc.close(m.calculateRegionDiscrepancy(one, 2.5), m.calculateRegionDiscrepancy([one], 2.5), rtol=0, atol=0)
        recorded.check(request.node.name + "-exact", [[float(m.fc.getPointDensityFromCrs(crs)) for crs in ([3, 4, 5], [-2, 70, 1], [10 ** 3, 0, 0])],
                                                      m.fc.getTotalAbsDensity(cut), m.calculateRegionDensity(one, 2.5)], rtol=1e-9, atol=1e-12)
        blobs = m.fc.findAberrantBlobs(list(m.asymmetryAtoms[5].coord), 2.0, cut)       # float32-narrowed Fc on the device
        recorded.check(request.node.name + "-fc-blobs", sorted(b.totalDensity for b in blobs), rtol=1e-5, atol=0)
        return
    for crs in ([3, 4, 5], [-2, 70, 1], [10 ** 3, 0, 0]):
        assert float(m.fc.getPointDensityFromCrs(crs)) == float(r.fc.getPointDensityFromCrs(crs))
    cut = r.densityObj.densityCutoff
    gc.close(m.fc.getTotalAbsDensity(cut), r.fc.getTotalAbsDensity(cut), rtol=1e-9)
    assert m.fc.meanDensity == m.densityObj.meanDensity
    blobs_r = r.fc.findAberrantBlobs(list(r.asymmetryAtoms[5].coord), 2.0, cut)
    blobs_m = m.fc.findAberrantBlobs(list(m.asymmetryAtoms[5].coord), 2.0, cut)
    assert len(blobs_r) == len(blobs_m)                                              # float32-narrowed Fc on the device: counts agree,
    gc.close(sorted(b.totalDensity for b in blobs_m), sorted(b.totalDensity for b in blobs_r), rtol=1e-5)   # sums to float32 accuracy
    one = [float(v) for v in m.asymmetryAtoms[7].coord]
    gc.close(m.calculateRegionDensity(one, 2.5), r.calculateRegionDensity(one, 2.5), rtol=1e-9, atol=1e-12)
    # (the reference's calculateRegionDiscrepancy iterates the coordinate list at :1198 and fails on a flat one; here it works)
    gc.close(m.calculateRegionDiscrepancy(one, 2.5), m.calculateRegionDiscrepancy([one], 2.5), rtol=0, atol=0)


def test_from_pdbid_uses_the_cache(pair, tmp_path, monkeypatch):
    """fromPDBid with the files already in ./ccp4_data and ./pdb_data (no network), pdb_eda/densityAnalysis.py:88-179."""
    import gzip
    from pdb_eda_b200 import densityAnalysis
    name = [k for k in CASES][0]
    st, d1, d2, pdb_text = _build(name)
    monkeypatch.chdir(tmp_path)
    os.makedirs("ccp4_data")
    os.makedirs("pdb_data")
    open("ccp4_data/9xyz.ccp4", "wb").write(d1)
    open("ccp4_data/9xyz_diff.ccp4", "wb").write(d2)
    with gzip.open("pdb_data/pdb9xyz.ent.gz", "wt") as fh:
        fh.write(pdb_text)
    an = densityAnalysis.fromPDBid("9XYZ")
    assert an != 0 and an.pdbid == "9xyz"
    assert len(list(an.biopdbObj.get_atoms())) == len(list(st.get_atoms()))
    assert an.densityObj.densityCutoff > 0 and len(an.pdbObj.header.rotationMats) == 4
    assert densityAnalysis.fromPDBid("0000") == 0      # nothing cached, no network: the loader reports failure with 0
    assert densityAnalysis.cleanPDBid("9xyz") and not os.path.exists("ccp4_data/9xyz.ccp4")


def test_error_conventions(pair):
    r, m = pair
    from pdb_eda_b200 import densityAnalysis
    assert densityAnalysis.fromFile("/nonexistent/file.pdb") == 0
    empty = densityAnalysis.DensityAnalysis("x", m.densityObj, m.diffDensityObj, structure.Structure("e"), m.pdbObj)
    assert empty.aggregateCloud() is None and empty.densityElectronRatio is None
    with pytest.raises(RuntimeError):
        empty.calculateAtomSpecificBlobStatistics(m.greenBlobList)
    assert m.densityObj.createFullBlobList(0) is None
