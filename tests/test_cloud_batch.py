"""Batched cloud aggregation (pdb_eda_b200/cloudBatch.py, csrc/pe_aggregate.cu).

CPU tier: the batch-wide statistics block against the per-structure restatement of pdb_eda/densityAnalysis.py:734-766
(``DensityAnalysis._atomTypeStatistics``, itself checked against the live reference in test_analysis_vs_reference.py).
GPU tier: ``CloudBatch`` over several structures in ONE batch against the REAL reference's ``aggregateCloud`` run on each
structure (oracle/_ref on the host CPU; without it, against the recorded results of tests/recorded.py): every number
``analyzePDBID`` (pdb_eda/multipleStructures.py:320-356) reads.
"""
import io

import numpy as np
import pytest

import golden_checks as gc
from pdb_eda_b200 import synthetic


def _fake_atoms(rng, n, types):
    rows = []
    for k in range(n):
        t = types[int(rng.integers(len(types)))]
        bf = float(rng.uniform(5, 60))
        if rng.random() < 0.08:
            bf = 0.0 if rng.random() < 0.5 else -1.0
        cd = float(abs(rng.normal(0.1, 0.05)))
        if rng.random() < 0.02:
            cd = float(rng.uniform(1, 2))          # outliers for the centroid filter
        rows.append(["A", k, "ALA", "X", t, float(rng.uniform(0.3, 0.8)), int(rng.integers(5, 40)), 7, bf, cd, [0.0, 0.0, 0.0]])
    return rows


def test_batch_statistics_match_per_structure():
    from pdb_eda_b200 import cloudBatch, densityAnalysis
    params = synthetic.defaultParams()
    types = sorted(params["radii"])
    params["slopes"] = {t: 0.01 * (k + 1) for k, t in enumerate(types)}
    saved = densityAnalysis.paramsGlobal
    densityAnalysis.setGlobals(params)
    try:
        rng = np.random.default_rng(5)
        sizes = [400, 37, 3, 150, 9, 0, 60]
        structures = [_fake_atoms(rng, n, types if k != 3 else types[:2]) for k, n in enumerate(sizes)]
        for row in structures[4]:
            row[8] = 20.0                              # all b-factors equal: slopes fall back to the current ones
        structures[4][0][9] = float("nan")
        ratios = [0.5, 0.45, 0.6, 0.52, 0.4, 0.5, 0.48]
        vols = [0.125, 0.1, 0.2, 0.125, 0.15, 0.1, 0.11]
        typeOf = {t: k for k, t in enumerate(types)}
        s = np.array([k for k, rows in enumerate(structures) for _ in rows])
        flat = [row for rows in structures for row in rows]
        keep, med, present = cloudBatch.batchAtomTypeStatistics(
            s, [typeOf[r[4]] for r in flat], len(types), [r[5] for r in flat], [r[6] for r in flat], [r[9] for r in flat],
            [r[8] for r in flat], ratios, vols, [params["slopes"][t] for t in types])
        for k, rows in enumerate(structures):
            with np.errstate(all="ignore"):
                import warnings
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    atoms, medians = densityAnalysis.DensityAnalysis._atomTypeStatistics([list(r) for r in rows], ratios[k], vols[k])
            assert len(atoms) == int(keep[s == k].sum())
            have = {types[j] for j in np.flatnonzero(present[k])}
            assert have == set(str(t) for t in medians["num_voxels"])
            for column in cloudBatch.MEDIAN_COLUMNS:
                for t in medians[column]:
                    gc.close(med[column][k, typeOf[str(t)]], medians[column][t], rtol=1e-11, atol=1e-12)
    finally:
        densityAnalysis.setGlobals(saved)


def test_segmented_median_and_std():
    from pdb_eda_b200 import cloudBatch
    rng = np.random.default_rng(3)
    group = rng.integers(0, 7, 500)
    values = rng.normal(size=500)
    values[rng.random(500) < 0.1] = np.nan
    group[group == 5] = 4                              # group 5 is empty
    med = cloudBatch._segmentedNanMedian(values, group, 8)
    std = cloudBatch._segmentedNanStd(values, group, 8)
    for g in range(8):
        sel = values[group == g]
        if np.isnan(sel).all():
            assert np.isnan(med[g])
            continue
        assert med[g] == np.nanmedian(sel)
        gc.close(std[g], np.nanstd(sel), rtol=1e-12)


@pytest.mark.gpu
def test_cloud_batch_matches_the_reference():
    """Without the reference installed: against the recorded results (tests/recorded.py)."""
    import recorded
    import test_analysis_vs_reference as tar
    from pdb_eda_b200 import cloudBatch, densityAnalysis, pdbParser
    ref = recorded.reference()
    params = ref[1].paramsGlobal if ref else densityAnalysis._loadDefaultParams()
    densityAnalysis.setGlobals(params)
    refs, items = [], []
    for name in tar.CASES:
        st, d1, d2, pdb_text = tar._build(name)
        if ref is None:
            m = densityAnalysis.fromFile(io.StringIO(pdb_text), io.BytesIO(d1), io.BytesIO(d2))
            mean, std = recorded.host_mean_std(m.densityObj)
            m.densityObj.densityCutoff = recorded.inputs("cloud_batch-" + name, [mean + 1.5 * std])[0]
            items.append((m.densityObj, cloudBatch.AtomTable.fromStructure(m.biopdbObj, params)))
            assert items[-1][1].supported
            continue
        ref_ccp4, ref_da, ref_cutils, ref_pp = ref
        r_dens = ref_ccp4.parse(io.BytesIO(d1), "t")
        r_dens.densityCutoff = r_dens.meanDensity + 1.5 * r_dens.stdDensity
        recorded.inputs("cloud_batch-" + name, [r_dens.densityCutoff], live=True)
        r = ref_da.DensityAnalysis("t", r_dens, None, st, ref_pp.readPDBfile(io.StringIO(pdb_text)))
        r.aggregateCloud()
        assert r.densityElectronRatio is not None
        refs.append(r)
        m = densityAnalysis.fromFile(io.StringIO(pdb_text), io.BytesIO(d1), io.BytesIO(d2))
        m.densityObj.densityCutoff = r_dens.densityCutoff
        table = cloudBatch.AtomTable.fromStructure(m.biopdbObj, params)
        assert table.supported
        items.append((m.densityObj, table))
    # one structure with too few electrons: no result, the others are unaffected (pdb_eda/densityAnalysis.py:726)
    st, d1, d2, pdb_text = tar._build("p212121")
    tiny = synthetic.polyAlaStructure(3, (0, 0, 0), (32.0, 32.0, 32.0), seed=5)
    m = densityAnalysis.fromFile(io.StringIO(__import__("pdb_eda_b200").structure.formatPDB(tiny, cell=tar.CASES["p212121"]["cell"], spaceGroup="P 1")),
                                 io.BytesIO(d1), io.BytesIO(d2))
    items.append((m.densityObj, cloudBatch.AtomTable.fromStructure(m.biopdbObj, params)))
    results = cloudBatch.CloudBatch(items, params).run()
    assert results[-1].densityElectronRatio is None
    if ref is None:
        assert all(res.densityElectronRatio is not None for res in results[:-1])
        recorded.check("test_cloud_batch_matches_the_reference",
                       [[res.numVoxelsAggregated, res.densityElectronRatio, res.totalAggregatedDensity, res.totalAggregatedElectrons,
                         dict(res.atomTypeOverlapCompleteness), dict(res.atomTypeOverlapIncompleteness), res.numAtomsAnalyzed,
                         res.numResidueClouds, res.numDomainClouds, res.medians] for res in results[:-1]])
        return
    for r, res in zip(refs, results):
        assert res.numVoxelsAggregated == r.numVoxelsAggregated
        gc.close([res.densityElectronRatio, res.totalAggregatedDensity, res.totalAggregatedElectrons],
                 [r.densityElectronRatio, r.totalAggregatedDensity, r.totalAggregatedElectrons], rtol=1e-9)
        assert dict(res.atomTypeOverlapCompleteness) == dict(r.atomTypeOverlapCompleteness)
        assert dict(res.atomTypeOverlapIncompleteness) == dict(r.atomTypeOverlapIncompleteness)
        assert res.numAtomsAnalyzed == len(r.atomCloudDescriptions)
        assert res.numResidueClouds == len(r.residueCloudDescriptions)
        assert res.numDomainClouds == len(r.domainCloudDescriptions)
        assert set(res.medians) == set(r.medians)
        for column in r.medians:
            assert set(res.medians[column]) == set(str(t) for t in r.medians[column])
            for t in r.medians[column]:
                gc.close(res.medians[column][str(t)], r.medians[column][t], rtol=1e-9, atol=1e-9)


@pytest.mark.gpu
def test_cloud_batch_is_deterministic_and_order_independent():
    """The same structures in another batch order / alone give identical numbers (no cross-structure leakage)."""
    import test_analysis_vs_reference as tar
    from pdb_eda_b200 import cloudBatch, densityAnalysis
    params = densityAnalysis._loadDefaultParams()
    densityAnalysis.setGlobals(params)
    items = []
    for name in ("p212121", "perm"):
        st, d1, d2, pdb_text = tar._build(name)
        m = densityAnalysis.fromFile(io.StringIO(pdb_text), io.BytesIO(d1), io.BytesIO(d2))
        items.append((m.densityObj, cloudBatch.AtomTable.fromStructure(m.biopdbObj, params)))
    both = cloudBatch.CloudBatch(items, params).run()
    again = cloudBatch.CloudBatch(items, params).run()
    swapped = cloudBatch.CloudBatch(items[::-1], params).run()[::-1]
    alone = [cloudBatch.CloudBatch([it], params).run()[0] for it in items]
    for a, others in zip(both, zip(again, swapped, alone)):
        for b in others:
            assert (a.numVoxelsAggregated, a.totalAggregatedDensity, a.totalAggregatedElectrons, a.numAtomsAnalyzed, a.numDomainClouds) == \
                   (b.numVoxelsAggregated, b.totalAggregatedDensity, b.totalAggregatedElectrons, b.numAtomsAnalyzed, b.numDomainClouds)


@pytest.mark.gpu
def test_statistics_kernel_matches_the_numpy_statement():
    """pe_cloud_statistics on hand-made per-atom records (b-factors <= 0, types with one or two atoms, equal b-factors, NaN
    and outlying centroid distances, a structure below minTotalElectrons) against batchAtomTypeStatistics."""
    import ctypes
    import torch
    from pdb_eda_b200 import cloudBatch, _lib
    from pdb_eda_b200._device import _ptr, _stream
    lib = _lib.load()
    rng = np.random.default_rng(8)
    nT = 6
    sizes = [700, 41, 3, 2500, 12, 0, 90, 260]
    slopes = np.array([0.01 * (k + 1) for k in range(nT)])
    atomMap, typeIndex, recs, static = [], [], [], []
    for k, n in enumerate(sizes):
        for _ in range(n):
            t = int(rng.integers(nT if k != 3 else 2))
            bf = float(rng.uniform(5, 60)) if k != 4 else 20.0
            if rng.random() < 0.08 and k != 4:
                bf = 0.0 if rng.random() < 0.5 else -1.0
            cd = float(abs(rng.normal(0.1, 0.05)))
            if rng.random() < 0.02:
                cd = float(rng.uniform(1, 2)) if rng.random() < 0.7 else float("nan")
            acc = rng.random() < 0.9
            recs.append([1.0, float(rng.integers(5, 40)), cd, float(rng.uniform(2, 7)), 0, 0, 0, (3.0 if rng.random() < 0.6 else 1.0) if acc else 0.0])
            static.append([float(rng.integers(6, 9)), float(rng.choice([1.0, 0.5, 0.37])), bf])
            atomMap.append(k)
            typeIndex.append(t)
    atomMap, typeIndex = np.array(atomMap, dtype=np.int32), np.array(typeIndex, dtype=np.int32)
    recs, static = np.array(recs), np.array(static)
    nS, nA = len(sizes), len(atomMap)
    start = np.concatenate(([0], np.cumsum(sizes)))
    maps = (_lib.PeBatchMap * nS)()
    for k in range(nS):
        maps[k].atom_begin, maps[k].atom_end = int(start[k]), int(start[k + 1])
    mapOut = np.zeros((nS, 8))
    mapOut[:, 1] = rng.uniform(400, 600, nS)
    mapOut[:, 2] = rng.uniform(900, 1100, nS)
    mapOut[6, 2] = 100.0                                   # below minTotalElectrons
    unitVolume = rng.uniform(0.1, 0.2, nS)
    perm = np.lexsort((typeIndex, atomMap)).astype(np.int32)
    gkey = atomMap[perm].astype(np.int64) * nT + typeIndex[perm]
    edge = np.flatnonzero(np.concatenate(([True], gkey[1:] != gkey[:-1])))
    segBegin, segEnd = edge.astype(np.int32), np.concatenate((edge[1:], [nA])).astype(np.int32)
    segMap, segType = (gkey[edge] // nT).astype(np.int32), (gkey[edge] % nT).astype(np.int32)
    dev = "cuda"
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d = dict(maps=torch.frombuffer(bytearray(bytes(maps)), dtype=torch.uint8).to(dev), recs=up(recs), mapOut=up(mapOut), static=up(static),
             perm=up(perm), sm=up(segMap), st=up(segType), sb=up(segBegin), se=up(segEnd), uv=up(unitVolume), sl=up(slopes))
    scratch = torch.empty((9, nA), dtype=torch.float64, device=dev)
    segOut = torch.empty((len(segBegin), 14), dtype=torch.float64, device=dev)
    mapStats = torch.empty((nS, 4), dtype=torch.float64, device=dev)
    _lib.check(lib.pe_cloud_statistics(nS, _ptr(d["maps"]), nA, _ptr(d["recs"]), _ptr(d["mapOut"]), _ptr(d["static"]), _ptr(d["perm"]),
                                       len(segBegin), _ptr(d["sm"]), _ptr(d["st"]), _ptr(d["sb"]), _ptr(d["se"]),
                                       int((segEnd - segBegin).max()), _ptr(d["uv"]), _ptr(d["sl"]),
                                       ctypes.c_double(400.0), _ptr(scratch), _ptr(segOut), _ptr(mapStats), _stream()), "pe_cloud_statistics")
    segOut, mapStats = segOut.cpu().numpy(), mapStats.cpu().numpy()
    rows = np.flatnonzero(recs[:, 7].astype(int) & 1)
    ratio = mapOut[:, 1] / mapOut[:, 2]
    der = recs[rows, 3] / static[rows, 0] / static[rows, 1]
    keep, med, present = cloudBatch.batchAtomTypeStatistics(atomMap[rows], typeIndex[rows], nT, der, recs[rows, 1], recs[rows, 2],
                                                            static[rows, 2], ratio, unitVolume, slopes)
    ok = mapOut[:, 2] >= 400.0
    analysed = np.bincount(atomMap[rows][keep], minlength=nS)
    assert np.array_equal(mapStats[:, 0], np.where(ok, analysed, 0))
    gc.close(mapStats[ok, 1], ratio[ok], rtol=1e-15)
    for s_ in range(len(segBegin)):
        k, t = int(segMap[s_]), int(segType[s_])
        sel = (atomMap == k) & (typeIndex == t)
        assert segOut[s_, 11] == (recs[sel, 7].astype(int) & 1).sum() and segOut[s_, 12] == ((recs[sel, 7].astype(int) >> 1) & 1).sum()
        if not ok[k] or not present[k, t]:
            assert segOut[s_, 0] == 0
            continue
        assert segOut[s_, 0] == (keep & (atomMap[rows] == k) & (typeIndex[rows] == t)).sum()
        for j, column in enumerate(cloudBatch.MEDIAN_COLUMNS):
            gc.close(segOut[s_, 1 + j], med[column][k, t], rtol=1e-10, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("radiusScale", [1.0, 1.8, 3.0])
def test_pair_path_equals_the_hash_table_path(radiusScale, monkeypatch):
    """pe_cloud_aggregate merges clouds through the atom grid + pair kernel and keeps the voxel hash table as the fallback for
    batches the pair kernel's frame cannot hold (a DEVICE flag decides; PE_CLOUD_FORCE_HASH=1 forces the fallback).  Both must give
    the same per-atom records and per-structure totals, bit for bit -- at the atom-type radii (candidate boxes of <= 256 voxels: 8
    lanes per atom in the count and fill passes), at 1.8 x the radii (boxes beyond 256 voxels: one warp per atom, no bitmap
    hand-off) and at 3 x (clouds wider than 15 voxels / atoms with more than 8 clouds: the device flag sends the batch to the
    hash-table kernels by itself), for orthogonal, axis-permuted and hexagonal cells in ONE batch."""
    import copy
    import test_analysis_vs_reference as tar
    from pdb_eda_b200 import cloudBatch, densityAnalysis
    params = copy.deepcopy(densityAnalysis._loadDefaultParams())
    params["radii"] = {k: float(np.float32(v * radiusScale)) for k, v in params["radii"].items()}
    densityAnalysis.setGlobals(params)
    try:
        items = []
        for name in tar.CASES:
            st, d1, d2, pdb_text = tar._build(name)
            m = densityAnalysis.fromFile(io.StringIO(pdb_text), io.BytesIO(d1), io.BytesIO(d2))
            items.append((m.densityObj, cloudBatch.AtomTable.fromStructure(m.biopdbObj, params)))
        out = {}
        for mode in ("0", "1"):
            monkeypatch.setenv("PE_CLOUD_FORCE_HASH", mode)
            batch = cloudBatch.CloudBatch(items, params)
            batch.launch()
            arr = batch.collectArrays()
            out[mode] = (batch.atomRows().copy(), arr, batch.ws[:16].cpu().numpy().view(np.int32).copy())
        rows0, arr0, flags0 = out["0"]
        rows1, arr1, flags1 = out["1"]
        assert flags0[0] == 0 and flags1[0] == 0 and flags1[1] == 1      # no error; the forced run took the hash-table kernels
        # the workspace's second flag says which kernels merged the clouds: the pair kernel at the first two scales, the hash
        # table at the third (the count pass's largest box and the atoms' cloud numbers decide on the device)
        assert flags0[1] == (1 if radiusScale >= 3.0 else 0), (radiusScale, flags0[:4], int(rows0[:, 0].max()))
        assert rows0.shape == rows1.shape and rows0.shape[0] > 0
        assert np.array_equal(rows0, rows1, equal_nan=True)
        for key in ("ok", "ratio", "numVoxels", "totalDensity", "totalElectrons", "analysed", "domainClouds", "residueClouds",
                    "centroidCutoff", "present", "complete", "incomplete"):
            assert np.array_equal(np.asarray(arr0[key]), np.asarray(arr1[key]), equal_nan=True), key
        for column in arr0["medians"]:
            assert np.array_equal(arr0["medians"][column], arr1["medians"][column], equal_nan=True), column
        assert arr0["numVoxels"].sum() > 0
    finally:
        densityAnalysis.setGlobals(densityAnalysis._loadDefaultParams())


@pytest.mark.gpu
def test_pair_path_equals_the_hash_table_path_on_a_pool(monkeypatch):
    """The same comparison over a pool of 24 synthetic structures drawn like bench.py's config-3 pool (64^3-192^3 maps, five space
    groups incl. the hexagonal cell, ~190,000 atoms, two batches): per-atom records and per-structure totals bit for bit."""
    import torch
    from pdb_eda_b200 import _device, ccp4, cloudBatch, multi
    params = synthetic.defaultParams()
    electronsOf = np.array([synthetic.ALA_ELECTRONS["ALA_" + a] for a, _, _ in synthetic._ALA_ATOMS])
    entries = []
    for sp in synthetic.poolSpec(24, sizes=(64, 96, 128, 192)):
        n, cell = sp["n"], sp["cell"]
        coords, bf = synthetic.fastPolyAla(sp["residues"], cell, sp["seed"])
        table = synthetic.polyAlaTable(coords, bf, params)
        rho = synthetic.densityMapDevice(coords, np.tile(electronsOf, sp["residues"]), n, cell, sp["seed"] + 1)
        hdr = ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((n, n, n), cell, (n, n, n)))
        dmap = _device.DeviceMap(_device.geom_from_header(hdr), rho.reshape(-1))
        m, s = dmap.mean_std()
        entries.append((sp["index"], cloudBatch.MapRef(dmap, m + 1.5 * s, hdr.unitVolume, "s%05d" % sp["index"]), table))
    shard = multi.PoolShard(entries, params, 1 << 17)
    assert len(shard.batches) >= 2

    def arrays():
        outs = []
        for b in shard.batches:
            b.launch()
            arr = b.collectArrays()
            outs.append((b.atomRows().copy(), {k: np.asarray(v).copy() for k, v in arr.items() if k not in ("medians", "unitVolume")},
                         b.ws[:16].cpu().numpy().view(np.int32).copy()))
        return outs

    monkeypatch.setenv("PE_CLOUD_FORCE_HASH", "0")
    pair = arrays()
    monkeypatch.setenv("PE_CLOUD_FORCE_HASH", "1")
    table = arrays()
    assert sum(len(x[0]) for x in pair) > 100000
    for x, y in zip(pair, table):
        assert x[2][0] == 0 and x[2][1] == 0 and y[2][1] == 1          # the pair kernel ran in the first pass, the hash table in the second
        assert np.array_equal(x[0], y[0], equal_nan=True)
        for k in x[1]:
            assert np.array_equal(x[1][k], y[1][k], equal_nan=True), k
        assert x[1]["numVoxels"].sum() > 0 and x[1]["ok"].all()
