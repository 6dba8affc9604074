"""Multiple-structures mode and the optimiser's inner loop against the REFERENCE's arithmetic.

The reference's drivers need the network (``fromPDBid``) and docopt, so the tests feed live reference ``DensityAnalysis``
objects (oracle/_ref, Cython cutils, on the host CPU) through the statements of
  * ``analyzePDBID``                 pdb_eda/multipleStructures.py:335-353   (per-structure row: diffs with 0 for a missing type)
  * ``processFunction``              pdb_eda/optimizeParams.py:434-436       (diffs / slopes: a missing or NaN type is omitted)
  * ``calculateMedianDiffsSlopes``   pdb_eda/optimizeParams.py:360-408       (gather over structures, medians, completeness)
restated line by line below, and compare with this package's per-structure path (``multi.analyzeStructure``), its batched
path (``multi.PoolShard`` -> ``packBatch`` -> ``gatherPacked``) and ``multi.OptimizeService``.  Without the reference
installed, the same paths are compared with each other and with the recorded results of tests/recorded.py.
"""
import io

import numpy as np
import pytest

import golden_checks as gc
import recorded
from pdb_eda_b200 import structure, synthetic


# ------------------------------------------------------------------------------------------------ the reference's statements
def ref_analyzePDBID(analyzer, radii):
    """pdb_eda/multipleStructures.py:335-346 (without F000 / header means, which need no voxel work)."""
    diffs = {atomType: ((analyzer.medians['corrected_density_electron_ratio'][atomType] - analyzer.densityElectronRatio) / analyzer.densityElectronRatio)
             if atomType in analyzer.medians['corrected_density_electron_ratio'] else 0 for atomType in sorted(radii)}
    atomOverlapCompleteness = sum(analyzer.atomTypeOverlapCompleteness.values())
    atomOverlapInCompleteness = sum(analyzer.atomTypeOverlapIncompleteness.values())
    if atomOverlapCompleteness > 0 or atomOverlapInCompleteness > 0:
        atomOverlapCompleteness = atomOverlapCompleteness / (atomOverlapCompleteness + atomOverlapInCompleteness)
    stats = {'density_electron_ratio': analyzer.densityElectronRatio, 'voxel_volume': analyzer.densityObj.header.unitVolume,
             'num_voxels_aggregated': analyzer.numVoxelsAggregated, 'total_aggregated_electrons': analyzer.totalAggregatedElectrons,
             'num_atoms_analyzed': len(analyzer.atomCloudDescriptions), 'num_residue_clouds_analyzed': len(analyzer.residueCloudDescriptions),
             'num_domain_clouds_analyzed': len(analyzer.domainCloudDescriptions), 'atom_overlap_completeness': atomOverlapCompleteness}
    return diffs, stats


def ref_processFunction(analyzer, params):
    """pdb_eda/optimizeParams.py:434-441."""
    diffs = {atomType: ((analyzer.medians['corrected_density_electron_ratio'][atomType] - analyzer.densityElectronRatio) / analyzer.densityElectronRatio)
             for atomType in params["radii"]
             if atomType in analyzer.medians['corrected_density_electron_ratio'] and not np.isnan(analyzer.medians['corrected_density_electron_ratio'][atomType])}
    newSlopes = {atomType: analyzer.medians['slopes'][atomType] for atomType in params["slopes"]
                 if atomType in analyzer.medians['slopes'] and not np.isnan(analyzer.medians['slopes'][atomType])}
    return {"diffs": diffs, "slopes": newSlopes, "atomtype_overlap_completeness": analyzer.atomTypeOverlapCompleteness,
            "atomtype_overlap_incompleteness": analyzer.atomTypeOverlapIncompleteness}


def ref_calculateMedianDiffsSlopes(results, currentParams):
    """pdb_eda/optimizeParams.py:360-408 on in-memory results (the reference passes them through temporary JSON files)."""
    diffs = {atomType: [] for atomType in currentParams["radii"]}
    slopes = {atomType: [] for atomType in currentParams["slopes"]}
    atomTypeOverlapCompleteness = {atomType: 0 for atomType in currentParams["radii"]}
    atomTypeOverlapIncompleteness = {atomType: 0 for atomType in currentParams["radii"]}
    for result in results:
        if result:
            for atomType, diff in result['diffs'].items():
                diffs[atomType].append(diff)
            for atomType, slope in result['slopes'].items():
                slopes[atomType].append(slope)
            for atomType, count in result['atomtype_overlap_completeness'].items():
                atomTypeOverlapCompleteness[atomType] += count
            for atomType, count in result['atomtype_overlap_incompleteness'].items():
                atomTypeOverlapIncompleteness[atomType] += count
    for atomType in atomTypeOverlapCompleteness.keys():
        if atomTypeOverlapCompleteness[atomType] > 0 or atomTypeOverlapIncompleteness[atomType] > 0:
            atomTypeOverlapCompleteness[atomType] = atomTypeOverlapCompleteness[atomType] / (atomTypeOverlapCompleteness[atomType] + atomTypeOverlapIncompleteness[atomType])
        else:
            atomTypeOverlapCompleteness[atomType] = 1
    with np.errstate(all="ignore"):
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            medianDiffs = {key: (np.nanmedian(value) if (value and not np.isnan(value).all()) else 0) for (key, value) in diffs.items()}
            meanDiffs = {key: (np.nanmean(value) if (value and not np.isnan(value).all()) else 0) for (key, value) in diffs.items()}
            sizeDiffs = {key: sum(~np.isnan(value)) for (key, value) in diffs.items()}
            squaredDiffs = [item ** 2 for values in diffs.values() for item in values if not np.isnan(item)]
            overallStdDevDiffs = np.sqrt(sum(squaredDiffs) / (len(squaredDiffs) - 1))
            medianSlopes = {key: np.nanmedian(value) for (key, value) in slopes.items()}
    medianSlopes = {key: value for (key, value) in medianSlopes.items() if not np.isnan(value)}
    return (medianDiffs, meanDiffs, overallStdDevDiffs, medianSlopes, sizeDiffs, atomTypeOverlapCompleteness)


# ------------------------------------------------------------------------------------------------ inputs
def _entries(n_structures=4):
    out = []
    for k in range(n_structures):
        n = (48, 56, 64, 52)[k % 4]
        cell = (n * 0.5,) * 3 + (90.0, 90.0, 90.0)
        st = synthetic.polyAlaStructure(36 + 7 * k, (0, 0, 0), cell[:3], seed=80 + k, residuesPerChain=30)
        if k == 1:                                   # one structure without CB atoms: its type is missing there
            for residue in st.get_residues():
                residue.child_list = [a for a in residue.child_list if a.name != "CB"]
        a, b = synthetic.mapPair(st, (n, n, n), cell, seed=90 + k)
        text = structure.formatPDB(st, remark290=synthetic.cartesianOperators("P 21 21 21", cell), cell=cell, spaceGroup="P 21 21 21")
        out.append((st, text, synthetic.ccp4Bytes(a, cell, (n, n, n)), synthetic.ccp4Bytes(b, cell, (n, n, n))))
    return out


def _tiny_entry():
    """Too few electrons: aggregateCloud yields nothing, the structure contributes no row (pdb_eda/densityAnalysis.py:726)."""
    n = 48
    cell = (24.0,) * 3 + (90.0, 90.0, 90.0)
    st = synthetic.polyAlaStructure(4, (0, 0, 0), cell[:3], seed=3)
    a, b = synthetic.mapPair(st, (n, n, n), cell, seed=4)
    text = structure.formatPDB(st, cell=cell, spaceGroup="P 1")
    return st, text, synthetic.ccp4Bytes(a, cell, (n, n, n)), synthetic.ccp4Bytes(b, cell, (n, n, n))


@pytest.fixture(scope="module")
def both():
    """(parameters, reference analyzers or None without the reference installed, this package's analyzers)."""
    from pdb_eda_b200 import densityAnalysis
    ref = recorded.reference()
    if ref is None:
        params = densityAnalysis._loadDefaultParams()
        densityAnalysis.setGlobals(params)
        mine = [densityAnalysis.fromFile(io.StringIO(text), io.BytesIO(d1), io.BytesIO(d2)) for _, text, d1, d2 in _entries() + [_tiny_entry()]]
        stats = [recorded.host_mean_std(m.densityObj) for m in mine]
        for m, cut in zip(mine, recorded.inputs("multi", [mean + 1.5 * std for mean, std in stats])):
            m.densityObj.densityCutoff = cut
        return params, None, mine
    ref_ccp4, ref_da, ref_cutils, ref_pp = ref
    params = ref_da.paramsGlobal
    densityAnalysis.setGlobals(params)
    refs, mine = [], []
    for st, text, d1, d2 in _entries() + [_tiny_entry()]:
        dens = ref_ccp4.parse(io.BytesIO(d1), "t")
        dens.densityCutoff = dens.meanDensity + 1.5 * dens.stdDensity
        r = ref_da.DensityAnalysis("t", dens, None, st, ref_pp.readPDBfile(io.StringIO(text)))
        r.aggregateCloud()
        refs.append(r)
        m = densityAnalysis.fromFile(io.StringIO(text), io.BytesIO(d1), io.BytesIO(d2))
        m.densityObj.densityCutoff = dens.densityCutoff
        mine.append(m)
    recorded.inputs("multi", [r.densityObj.densityCutoff for r in refs], live=True)
    assert refs[-1].densityElectronRatio is None and all(r.densityElectronRatio for r in refs[:-1])
    return params, refs, mine


@pytest.mark.gpu
def test_rows_of_analyzePDBID(both):
    """f2: the per-structure row of multiple-structures mode, per-structure path and batched path."""
    from pdb_eda_b200 import cloudBatch, multi
    params, refs, mine = both
    types = sorted(params["radii"])
    entries = [(k, m.densityObj, cloudBatch.AtomTable.fromStructure(m.biopdbObj, params)) for k, m in enumerate(mine)]
    shard = multi.PoolShard(entries, params)
    shard.launch()
    cumulative, rows = shard.pack(optimizer=False)
    assert rows[:, 0].tolist() == [0.0, 1.0, 2.0, 3.0]                      # the structure with too few electrons has no row
    ns = 1 + len(multi.STAT_COLUMNS)
    col = {c: 1 + k for k, c in enumerate(multi.STAT_COLUMNS)}
    if refs is None:
        singles = [multi.analyzeStructure(m, types) for m in mine[:-1]]
        for k, single in enumerate(singles):
            gc.close(rows[k, ns:ns + len(types)], [single["diffs"][t] for t in types], rtol=1e-9, atol=1e-12)
            for name in multi.STAT_COLUMNS[:-1]:                               # all but execution_time
                gc.close(rows[k, col[name]], single["stats"][name], rtol=1e-9)
        assert multi.analyzeStructure(mine[-1], types) == 0
        recorded.check("test_rows_of_analyzePDBID", [cumulative, np.delete(rows, col["execution_time"], axis=1),
                                                     [[single["diffs"], [single["stats"][c] for c in multi.STAT_COLUMNS[:-1]]] for single in singles]],
                       atol=1e-12)
        return
    for k, (r, m) in enumerate(zip(refs[:-1], mine[:-1])):
        diffs, stats = ref_analyzePDBID(r, params["radii"])
        single = multi.analyzeStructure(m, types)
        assert list(single["diffs"]) == list(diffs)
        gc.close([single["diffs"][t] for t in types], [diffs[t] for t in types], rtol=1e-9, atol=1e-12)
        gc.close(rows[k, ns:ns + len(types)], [diffs[t] for t in types], rtol=1e-9, atol=1e-12)
        for name, want in stats.items():
            gc.close(single["stats"][name], want, rtol=1e-9)
            gc.close(rows[k, col[name]], want, rtol=1e-9)
    assert multi.analyzeStructure(mine[-1], types) == 0
    assert cumulative[0] == 4 and cumulative[1] == sum(r.numVoxelsAggregated for r in refs[:-1])


@pytest.mark.gpu
def test_calculateMedianDiffsSlopes(both, tmp_path):
    """f4: one optimiser iteration -- the tuple of calculateMedianDiffsSlopes from the reference's own analyzers and arithmetic
    against the batched shard, the per-structure path and OptimizeService."""
    from pdb_eda_b200 import cloudBatch, multi
    params, refs, mine = both
    types = list(params["radii"])
    if refs is None:
        batched = multi.PoolShard([(k, m.densityObj, cloudBatch.AtomTable.fromStructure(m.biopdbObj, params)) for k, m in enumerate(mine)],
                                  params).analyze(optimizer=True)
        want = (batched["medianDiffs"], batched["meanDiffs"], batched["overallStdDevDiffs"], batched["medianSlopes"], batched["sizeDiffs"],
                batched["atomTypeOverlapCompleteness"])
        recorded.check("test_calculateMedianDiffsSlopes", list(want), atol=1e-12)
    else:
        want = ref_calculateMedianDiffsSlopes([ref_processFunction(r, params) if r.densityElectronRatio else 0 for r in refs], params)
    entries = [(k, m.densityObj, cloudBatch.AtomTable.fromStructure(m.biopdbObj, params)) for k, m in enumerate(mine)]
    batched = multi.PoolShard(entries, params).analyze(optimizer=True)
    single = multi.gatherResults({k: multi.analyzeStructure(m, types, optimizer=True) for k, m in enumerate(mine)}, list(range(len(mine))),
                                 len(mine), types, "cpu")
    service = multi.OptimizeService(list(range(len(mine))), lambda k: mine[k]).evaluate(params)
    for got in ((batched["medianDiffs"], batched["meanDiffs"], batched["overallStdDevDiffs"], batched["medianSlopes"], batched["sizeDiffs"],
                 batched["atomTypeOverlapCompleteness"]),
                (single["medianDiffs"], single["meanDiffs"], single["overallStdDevDiffs"], single["medianSlopes"], single["sizeDiffs"],
                 single["atomTypeOverlapCompleteness"]), service):
        for k in (0, 1, 4, 5):                                                  # medianDiffs, meanDiffs, sizeDiffs, completeness
            assert set(got[k]) == set(want[k])
            gc.close([got[k][t] for t in want[k]], [want[k][t] for t in want[k]], rtol=1e-9, atol=1e-12)
        gc.close(got[2], want[2], rtol=1e-9)
        assert set(got[3]) == set(want[3])                                      # medianSlopes: only types some structure has
        gc.close([got[3][t] for t in want[3]], [want[3][t] for t in want[3]], rtol=1e-9, atol=1e-12)
    cb = [t for t in types if want[4][t] == 3]                                  # the CB type: present in 3 of the 4 structures
    assert len(cb) == 1 and sum(1 for t in types if want[4][t] == 4) == 4


def test_pack_batch_equals_pack_of_dicts():
    """CPU tier: the vectorised packing of batch arrays gives the rows of the per-structure dicts, in both flavours."""
    from pdb_eda_b200 import multi
    rng = np.random.default_rng(2)
    types = ["a", "b", "c"]
    nS, T = 6, 3
    ok = np.array([True, True, False, True, True, True])
    present = rng.random((nS, T)) < 0.7
    present[ok, 0] = True
    arr = {"ok": ok, "ratio": rng.uniform(0.4, 0.6, nS), "numVoxels": rng.integers(1000, 5000, nS).astype(float),
           "totalElectrons": rng.uniform(500, 900, nS), "totalDensity": rng.uniform(200, 500, nS), "analysed": rng.integers(50, 90, nS).astype(float),
           "residueClouds": rng.integers(5, 20, nS).astype(float), "domainClouds": rng.integers(1, 5, nS).astype(float),
           "unitVolume": rng.uniform(0.1, 0.2, nS), "present": present & ok[:, None],
           "medians": {"corrected_density_electron_ratio": np.where(present, rng.uniform(0.4, 0.6, (nS, T)), np.nan),
                       "slopes": np.where(present, rng.normal(size=(nS, T)), np.nan)},
           "complete": rng.integers(0, 30, (nS, T)), "incomplete": rng.integers(0, 5, (nS, T))}
    arr["complete"][3] = 0
    arr["incomplete"][3] = 0
    indices = [10, 11, 12, 13, 14, 15]
    for optimizer in (False, True):
        results = {}
        for k, idx in enumerate(indices):
            if not ok[k]:
                results[idx] = 0
                continue
            missing = np.nan if optimizer else 0
            c, i = int(arr["complete"][k].sum()), int(arr["incomplete"][k].sum())
            results[idx] = {"pdbid": "x", "diffs": {t: (arr["medians"]["corrected_density_electron_ratio"][k, j] - arr["ratio"][k]) / arr["ratio"][k]
                                                   if present[k, j] else missing for j, t in enumerate(types)},
                            "slopes": {t: arr["medians"]["slopes"][k, j] if present[k, j] else np.nan for j, t in enumerate(types)},
                            "stats": {"density_electron_ratio": arr["ratio"][k], "voxel_volume": arr["unitVolume"][k],
                                      "num_voxels_aggregated": arr["numVoxels"][k], "total_aggregated_electrons": arr["totalElectrons"][k],
                                      "total_aggregated_density": arr["totalDensity"][k], "num_atoms_analyzed": arr["analysed"][k],
                                      "num_residue_clouds_analyzed": arr["residueClouds"][k], "num_domain_clouds_analyzed": arr["domainClouds"][k],
                                      "atom_overlap_completeness": c / (c + i) if (c > 0 or i > 0) else c, "execution_time": 0.0},
                            "atomtype_overlap_completeness": {t: int(arr["complete"][k, j]) for j, t in enumerate(types)},
                            "atomtype_overlap_incompleteness": {t: int(arr["incomplete"][k, j]) for j, t in enumerate(types)}}
        c1, r1 = multi._pack(results, indices, types)
        c2, r2 = multi.packBatch(arr, indices, types, optimizer)
        np.testing.assert_array_equal(c1, c2)
        np.testing.assert_array_equal(r1, r2)
