"""GPU tier: the batched cloud aggregation (csrc/pe_aggregate.cu through ``CloudBatch``) against the C oracle, and against the
other pipeline of ``DensityAnalysis.aggregateCloud``.

Per-atom records: for every candidate atom the oracle lists the sphere voxels above the cutoff (``orc.sphere_list``), splits
them into 26-connected clouds (``orc.cluster_crs``, createCrsLists) and sums each cloud (``orc.blob_stats``, fromCrsList);
the record holds the number of clouds and, for the nearest cloud by centroid distance (the FIRST minimum,
pdb_eda/densityAnalysis.py:630-634), its voxel count, distance, total density and centroid.  The per-structure centroid cutoff
(:609) and the "contributes" flag (:623-634) are restated in numpy.

Batched vs full: ``_aggregateCloudFull`` merges residue / domain clouds with ``pe_overlap_pairs`` / ``pe_cluster_crs_grouped``
/ ``pe_crs_stats`` (held against host statements in test_set_algebra_vs_host.py); the batched path merges with its own pair or
hash-table kernels.  Equal totals, counts and medians from the two tie the batched merge to an independent check.
"""
import copy
import io

import numpy as np
import pytest

import golden_checks as gc
import recorded
import test_analysis_vs_reference as tar
from oracle import orc
from pdb_eda_b200 import _blas, ccp4, cloudBatch, densityAnalysis, synthetic

pytestmark = pytest.mark.gpu


def _params(scale):
    params = copy.deepcopy(densityAnalysis._loadDefaultParams())
    params["radii"] = {k: float(np.float32(v * scale)) for k, v in params["radii"].items()}
    return params


def _analysis(name, nsd=1.5):
    st, d1, d2, pdb_text = tar._build(name)
    m = densityAnalysis.fromFile(io.StringIO(pdb_text), io.BytesIO(d1), io.BytesIO(d2))
    mean, std = recorded.host_mean_std(m.densityObj)
    m.densityObj.densityCutoff = float(np.float32(mean + nsd * std))
    return m


def oracle_records(dm, xyz, radius, cutoff):
    """(n x 8) expected per-atom records (flags column left 0) and each atom's smallest centroid distance (NaN: no cloud)."""
    g = orc.geom(dm.header, dm.origin, mv=_blas.probe())
    rho = np.ascontiguousarray(dm.densityArray, dtype=np.float32)
    out = np.zeros((len(xyz), 8))
    best_dist = np.full(len(xyz), np.nan)
    for a in range(len(xyz)):
        crs = orc.sphere_list(g, rho, xyz[a], radius[a], cutoff)
        if len(crs) == 0:
            continue
        label, n = orc.cluster_crs(crs)
        st = orc.blob_stats(g, rho, crs, label, n)
        centroid = st[:, 2:5] / st[:, 1:2]
        dist = np.linalg.norm(xyz[a][None, :] - centroid, axis=1)
        b = int(np.argmin(dist))                                    # the first minimum
        out[a, :7] = [n, st[b, 0], dist[b], st[b, 1], *centroid[b]]
        best_dist[a] = dist[b]
    return out, best_dist


def _check_records(batch, rows, arr):
    xyz = batch.d_xyz.cpu().numpy()
    radius = batch.d_radius.cpu().numpy()
    no_cloud = 0
    for k, (dm, _) in enumerate(batch.items):
        a0, a1 = int(batch.atomStart[k]), int(batch.atomStart[k + 1])
        want, best = oracle_records(dm, xyz[a0:a1], radius[a0:a1], float(np.float32(dm.densityCutoff)))
        got = rows[a0:a1]
        assert np.array_equal(got[:, 0], want[:, 0]), k                    # number of clouds
        assert np.array_equal(got[:, 1], want[:, 1]), k                    # voxels of the best cloud
        has = want[:, 0] > 0
        gc.close(got[has, 2:7], want[has, 2:7], rtol=1e-9, atol=1e-12)
        # an atom without a cloud: the kernel writes an all-zero record (it never contributes)
        assert not got[~has].any(), k
        no_cloud += int((~has).sum())
        # centroid cutoff and the "contributes" flag (bit 0)
        with np.errstate(all="ignore"):
            cutoff = np.nanmedian(best) + 2.5 * np.nanstd(best) if has.any() else np.nan
        gc.close([arr["centroidCutoff"][k]], [cutoff], rtol=1e-9)
        nc = want[:, 0]
        accepted = (nc > 0) & ((nc == 1) | ~(best > cutoff))
        assert np.array_equal((got[:, 7].astype(np.int64) & 1) != 0, accepted), k
    return no_cloud


@pytest.mark.parametrize("radiusScale", [1.0, 1.8, 3.0])
def test_atom_records_match_the_oracle(radiusScale):
    """The three structures of test_analysis_vs_reference in one batch (orthogonal, axis-permuted with a non-zero start,
    hexagonal) plus the orthogonal one again at a high cutoff, which leaves atoms without a cloud.  The three radius scales
    select the 8-lane count / fill path with the bitmap hand-off, the warp-per-atom path and the hash-table fallback."""
    params = _params(radiusScale)
    densityAnalysis.setGlobals(params)
    try:
        items = []
        for name, nsd in [(name, 1.5) for name in tar.CASES] + [("p212121", 4.0)]:
            m = _analysis(name, nsd)
            items.append((m.densityObj, cloudBatch.AtomTable.fromStructure(m.biopdbObj, params)))
        batch = cloudBatch.CloudBatch(items, params)
        batch.launch()
        arr = batch.collectArrays()
        flags = batch.ws[:16].cpu().numpy().view(np.int32)
        assert flags[0] == 0
        assert flags[1] == (1 if radiusScale >= 3.0 else 0)                # which kernels merged the clouds
        no_cloud = _check_records(batch, batch.atomRows(), arr)
        if radiusScale == 1.0:
            assert no_cloud > 0
    finally:
        densityAnalysis.setGlobals(densityAnalysis._loadDefaultParams())


@pytest.mark.parametrize("radius", [1.2, 3.0])
def test_equidistant_clouds_pick_the_first(radius):
    """Each atom sits exactly halfway between two one-voxel clouds of equal density: both centroid distances are the same
    float64 number, and the record must describe the first cloud in createCrsLists order.  Radius 1.2 A keeps every candidate
    box within 256 voxels (8 lanes per atom); 3.0 A takes the one-warp-per-atom fill."""
    n = 32
    values = np.zeros((n, n, n), dtype=np.float32)
    sites = [(6, 6, 8, 0), (6, 22, 8, 1), (22, 6, 8, 2), (22, 22, 8, 0), (14, 14, 24, 1)]   # (c, r, s, axis of the pair)
    for c, r, s, ax in sites:
        for sign in (-2, 2):
            v = [c, r, s]
            v[ax] += sign
            values[v[2], v[1], v[0]] = 1.0
    cell = (16.0, 16.0, 16.0, 90, 90, 90)
    dm = ccp4.parse(io.BytesIO(synthetic.ccp4Bytes(values, cell, (n, n, n))), "ties")
    dm.densityCutoff = 0.5
    g = orc.geom(dm.header, dm.origin, mv=_blas.probe())
    coords = orc.crs2xyz(g, np.array([s[:3] for s in sites])).astype(np.float32)
    assert np.array_equal(coords.astype(np.float64), orc.crs2xyz(g, np.array([s[:3] for s in sites])))
    params = synthetic.defaultParams()
    params["radii"] = {t: radius for t in params["radii"]}
    table = synthetic.polyAlaTable(coords, np.full(len(coords), 20.0), params)
    batch = cloudBatch.CloudBatch([(dm, table)], params)
    batch.launch()
    rows = batch.atomRows()
    want, best = oracle_records(dm, coords.astype(np.float64), np.full(len(coords), radius, np.float32), 0.5)
    assert np.array_equal(want[:, 0], np.full(len(sites), 2.0)) and np.all(best == best[0])
    assert np.array_equal(rows[:, :7], want[:, :7])


@pytest.mark.parametrize("radiusScale", [1.0, 1.8])
@pytest.mark.parametrize("name", list(tar.CASES))
def test_batched_equals_full_pipeline(name, radiusScale, monkeypatch):
    params = _params(radiusScale)
    densityAnalysis.setGlobals(params)
    try:
        batched = _analysis(name)
        batched.aggregateCloud()
        monkeypatch.setattr(densityAnalysis, "BATCHED_CLOUD", False)
        full = _analysis(name)
        full.aggregateCloud()
        assert full._residueCloudDescriptions is not densityAnalysis._LAZY          # the full pipeline ran
        assert batched._residueCloudDescriptions is densityAnalysis._LAZY           # ... and the batched one
        assert batched.densityElectronRatio is not None
        assert batched.numVoxelsAggregated == full.numVoxelsAggregated
        gc.close([batched.totalAggregatedDensity, batched.totalAggregatedElectrons, batched.densityElectronRatio],
                 [full.totalAggregatedDensity, full.totalAggregatedElectrons, full.densityElectronRatio], rtol=1e-9)
        assert dict(batched.atomTypeOverlapCompleteness) == dict(full.atomTypeOverlapCompleteness)
        assert dict(batched.atomTypeOverlapIncompleteness) == dict(full.atomTypeOverlapIncompleteness)
        assert len(batched.atomCloudDescriptions) == len(full.atomCloudDescriptions)
        assert batched.numResidueCloudsAnalyzed == full.numResidueCloudsAnalyzed == len(full.residueCloudDescriptions)
        assert batched.numDomainCloudsAnalyzed == full.numDomainCloudsAnalyzed == len(full.domainCloudDescriptions)
        assert set(batched.medians) == set(full.medians)
        for column, per_type in full.medians.items():
            assert set(map(str, batched.medians[column])) == set(map(str, per_type)), column
            mine = {str(t): v for t, v in batched.medians[column].items()}
            for t, v in per_type.items():
                assert np.isnan(mine[str(t)]) == np.isnan(v), (column, t)
                gc.close([mine[str(t)]], [v], rtol=1e-9, atol=1e-12)
    finally:
        densityAnalysis.setGlobals(densityAnalysis._loadDefaultParams())
