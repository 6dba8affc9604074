"""Multiple-structures mode across GPUs: structures sharded over ranks, cumulative statistics all-reduced.

The reference runs one structure per ``multiprocessing.Pool`` task and gathers the per-structure results through
temporary JSON files (pdb_eda/multipleStructures.py:164-180, :320-356; pdb_eda/optimizeParams.py:341-408).  Here a
rank is one process per GPU (``torch.distributed``, NCCL over NVLink; gloo in the CPU tests): structures are dealt
out longest-first, every rank analyses its share on its own GPU, and two collectives replace the file gather:

  * one fused ``all_reduce(SUM)`` of the cumulative vector [structures analysed, voxels aggregated, electrons,
    density, per-atom-type complete / incomplete overlap counts] (pdb_eda/optimizeParams.py:376-379);
  * one ``all_gather`` of the fixed-width per-structure rows (ratio, counts, per-type diffs and slopes), because the
    medians over structures need every value (pdb_eda/optimizeParams.py:400-405).

A structure that fails to load or has too few electrons yields no row and contributes zeros, as in the reference
(``analyzePDBID`` returns 0, pdb_eda/multipleStructures.py:331-333).  There is no data-path collective: structures are
independent units.
"""
import time

import numpy as np
import torch
import torch.distributed as dist

STAT_COLUMNS = ("density_electron_ratio", "voxel_volume", "num_voxels_aggregated", "total_aggregated_electrons",
                "total_aggregated_density", "num_atoms_analyzed", "num_residue_clouds_analyzed",
                "num_domain_clouds_analyzed", "atom_overlap_completeness", "execution_time")


def shardStructures(costs, worldSize):
    """Longest-processing-time-first assignment (cf. the longest-job-first reordering of pdb_eda/optimizeParams.py:392-393).
    ``costs``: one number per structure (e.g. voxels x atoms).  Returns ``worldSize`` lists of structure indices; every
    rank computes the same assignment."""
    order = sorted(range(len(costs)), key=lambda i: (-float(costs[i]), i))
    loads = [0.0] * worldSize
    shards = [[] for _ in range(worldSize)]
    for i in order:
        r = min(range(worldSize), key=lambda k: (loads[k], k))
        shards[r].append(i)
        loads[r] += float(costs[i])
    return shards


def analyzeStructure(analyzer, atomTypes, optimizer=False):
    """The per-structure result of ``analyzePDBID`` (pdb_eda/multipleStructures.py:320-356), or 0 when the structure cannot
    be analysed.  ``optimizer=True`` gives the flavour of the optimiser's ``processFunction`` (pdb_eda/optimizeParams.py:410-448):
    an atom type the structure lacks (or whose median is NaN) is OMITTED there (:434-436) -- NaN here, which the medians over
    structures skip -- whereas analyzePDBID reports 0 for it (:335-336)."""
    start = time.process_time()
    if not analyzer or not analyzer.densityElectronRatio:
        return 0
    ratio = analyzer.densityElectronRatio
    corrected = analyzer.medians['corrected_density_electron_ratio']
    missing = np.nan if optimizer else 0
    diffs = {t: ((corrected[t] - ratio) / ratio) if t in corrected else missing for t in atomTypes}
    slopes = {t: analyzer.medians['slopes'][t] if t in analyzer.medians['slopes'] else np.nan for t in atomTypes}
    complete = sum(analyzer.atomTypeOverlapCompleteness.values())
    incomplete = sum(analyzer.atomTypeOverlapIncompleteness.values())
    completeness = complete / (complete + incomplete) if (complete > 0 or incomplete > 0) else complete
    stats = {'density_electron_ratio': ratio, 'voxel_volume': analyzer.densityObj.header.unitVolume,
             'num_voxels_aggregated': analyzer.numVoxelsAggregated, 'total_aggregated_electrons': analyzer.totalAggregatedElectrons,
             'total_aggregated_density': analyzer.totalAggregatedDensity, 'num_atoms_analyzed': len(analyzer.atomCloudDescriptions),
             'num_residue_clouds_analyzed': getattr(analyzer, "numResidueCloudsAnalyzed", None) if hasattr(analyzer, "numResidueCloudsAnalyzed")
             else len(analyzer.residueCloudDescriptions),
             'num_domain_clouds_analyzed': getattr(analyzer, "numDomainCloudsAnalyzed", None) if hasattr(analyzer, "numDomainCloudsAnalyzed")
             else len(analyzer.domainCloudDescriptions), 'atom_overlap_completeness': completeness}
    stats['execution_time'] = time.process_time() - start
    return {"pdbid": analyzer.pdbid, "diffs": diffs, "slopes": slopes, "stats": stats,
            "atomtype_overlap_completeness": dict(analyzer.atomTypeOverlapCompleteness),
            "atomtype_overlap_incompleteness": dict(analyzer.atomTypeOverlapIncompleteness)}


def _pack(results, indices, atomTypes):
    """Local results -> (cumulative vector, fixed-width row matrix)."""
    T = len(atomTypes)
    cumulative = np.zeros(4 + 2 * T, dtype=np.float64)
    rows = []
    for idx in indices:
        res = results.get(idx, 0)
        if not res:
            continue
        st = res["stats"]
        cumulative[0] += 1
        cumulative[1] += st["num_voxels_aggregated"]
        cumulative[2] += st["total_aggregated_electrons"]
        cumulative[3] += st["total_aggregated_density"]
        for k, t in enumerate(atomTypes):
            cumulative[4 + k] += res["atomtype_overlap_completeness"].get(t, 0)
            cumulative[4 + T + k] += res["atomtype_overlap_incompleteness"].get(t, 0)
        rows.append([float(idx)] + [float(st[c]) for c in STAT_COLUMNS] + [float(res["diffs"][t]) for t in atomTypes] +
                    [float(res["slopes"][t]) for t in atomTypes])
    width = 1 + len(STAT_COLUMNS) + 2 * T
    return cumulative, np.asarray(rows, dtype=np.float64).reshape(-1, width)


def packBatch(arr, indices, atomTypes, optimizer=False, executionTime=0.0):
    """``_pack`` for the arrays of ``CloudBatch.collectArrays`` (one entry per structure of the batch; ``indices`` their pool
    indices): no Python loop over structures.  Same row layout and the same two flavours as ``analyzeStructure``."""
    T = len(atomTypes)
    ok = np.asarray(arr["ok"], dtype=bool)
    idx = np.asarray(indices, dtype=np.float64)[ok]
    ratio = arr["ratio"][ok]
    complete, incomplete = arr["complete"][ok], arr["incomplete"][ok]
    cumulative = np.zeros(4 + 2 * T, dtype=np.float64)
    cumulative[0] = ok.sum()
    cumulative[1] = arr["numVoxels"][ok].sum()
    cumulative[2] = arr["totalElectrons"][ok].sum()
    cumulative[3] = arr["totalDensity"][ok].sum()
    cumulative[4:4 + T] = complete.sum(axis=0)
    cumulative[4 + T:] = incomplete.sum(axis=0)
    csum, isum = complete.sum(axis=1).astype(np.float64), incomplete.sum(axis=1).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        completeness = np.where((csum > 0) | (isum > 0), csum / (csum + isum), csum)
        corrected = arr["medians"]["corrected_density_electron_ratio"][ok]
        present = arr["present"][ok]
        diffs = (corrected - ratio[:, None]) / ratio[:, None]
    if optimizer:
        diffs = np.where(present, diffs, np.nan)                 # processFunction omits absent / NaN types (:434-436)
    else:
        diffs = np.where(present, diffs, 0.0)                    # analyzePDBID: 0 for a type the structure lacks (:335-336)
    slopes = np.where(present, arr["medians"]["slopes"][ok], np.nan)
    stats = np.stack((ratio, np.asarray(arr["unitVolume"], dtype=np.float64)[ok], arr["numVoxels"][ok], arr["totalElectrons"][ok],
                      arr["totalDensity"][ok], arr["analysed"][ok], arr["residueClouds"][ok], arr["domainClouds"][ok], completeness,
                      np.full(len(idx), float(executionTime))), axis=1)
    rows = np.concatenate((idx[:, None], stats, diffs, slopes), axis=1) if len(idx) else np.zeros((0, 1 + len(STAT_COLUMNS) + 2 * T))
    return cumulative, rows


def gatherResults(results, indices, nStructures, atomTypes, device="cpu", group=None):
    """Collective step of multiple-structures mode.  ``results``: {structure index: result dict or 0} of THIS rank's
    shard ``indices``.  Returns the same summary on every rank (see ``gatherPacked``)."""
    atomTypes = list(atomTypes)
    cumulative, rows = _pack(results, indices, atomTypes)
    return gatherPacked(cumulative, rows, atomTypes, device, group)


def gatherPacked(cumulative, rows, atomTypes, device="cpu", group=None, local=False):
    """The two collectives on a rank's packed results (``_pack`` / ``packBatch``).  Returns the same summary on every rank:
    ``cumulative`` (dict), ``rows`` (n_ok x width float64, ordered by structure index), ``medianDiffs``, ``meanDiffs``,
    ``overallStdDevDiffs``, ``medianSlopes``, ``sizeDiffs``, ``atomTypeOverlapCompleteness`` --
    the quantities of ``calculateMedianDiffsSlopes`` (pdb_eda/optimizeParams.py:400-408)."""
    atomTypes = list(atomTypes)
    T = len(atomTypes)
    world = dist.get_world_size(group) if (dist.is_initialized() and not local) else 1   # local: this rank's structures only
    width = 1 + len(STAT_COLUMNS) + 2 * T
    if world > 1:
        cum_t = torch.from_numpy(cumulative).to(device)
        dist.all_reduce(cum_t, op=dist.ReduceOp.SUM, group=group)       # ONE fused all-reduce of all cumulative counts
        cumulative = cum_t.cpu().numpy()
        # rows: pad every rank's block to the largest shard (an 8-byte MAX all-reduce), gather, drop the padding
        cap_t = torch.tensor([len(rows)], dtype=torch.int64, device=device)
        dist.all_reduce(cap_t, op=dist.ReduceOp.MAX, group=group)
        cap = max(int(cap_t.item()), 1)
        block = torch.full((cap, width), -1.0, dtype=torch.float64, device=device)
        if len(rows):
            block[:len(rows)] = torch.from_numpy(rows).to(device)
        gathered = [torch.empty_like(block) for _ in range(world)]
        dist.all_gather(gathered, block, group=group)
        allrows = torch.cat(gathered).cpu().numpy()
        allrows = allrows[allrows[:, 0] >= 0]
    else:
        allrows = rows
    allrows = allrows[np.argsort(allrows[:, 0], kind="stable")] if len(allrows) else allrows
    ns = 1 + len(STAT_COLUMNS)
    D = np.asarray(allrows[:, ns:ns + T], dtype=np.float64).reshape(-1, T)           # per-structure diffs, one column per type
    S = np.asarray(allrows[:, ns + T:ns + 2 * T], dtype=np.float64).reshape(-1, T)   # slopes
    complete = {t: cumulative[4 + k] for k, t in enumerate(atomTypes)}
    incomplete = {t: cumulative[4 + T + k] for k, t in enumerate(atomTypes)}
    completeness = {t: (complete[t] / (complete[t] + incomplete[t]) if (complete[t] > 0 or incomplete[t] > 0) else 1) for t in atomTypes}
    with np.errstate(all="ignore"):
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            haveD = (~np.isnan(D)).any(axis=0) if len(D) else np.zeros(T, dtype=bool)
            medD = np.nanmedian(D, axis=0) if len(D) else np.zeros(T)
            meanD = np.nanmean(D, axis=0) if len(D) else np.zeros(T)
            haveS = (~np.isnan(S)).any(axis=0) if len(S) else np.zeros(T, dtype=bool)
            medS = np.nanmedian(S, axis=0) if len(S) else np.zeros(T)
        medianDiffs = {t: (medD[k] if haveD[k] else 0) for k, t in enumerate(atomTypes)}
        meanDiffs = {t: (meanD[k] if haveD[k] else 0) for k, t in enumerate(atomTypes)}
        sizeDiffs = {t: int(np.sum(~np.isnan(D[:, k]))) for k, t in enumerate(atomTypes)}
        valid = D[~np.isnan(D)]
        overallStd = float(np.sqrt(np.sum(valid ** 2) / (len(valid) - 1))) if len(valid) > 1 else float("nan")
        medianSlopes = {t: medS[k] for k, t in enumerate(atomTypes) if haveS[k]}
    return {"cumulative": {"structures": int(cumulative[0]), "num_voxels_aggregated": cumulative[1],
                           "total_aggregated_electrons": cumulative[2], "total_aggregated_density": cumulative[3],
                           "density_electron_ratio": cumulative[3] / cumulative[2] if cumulative[2] else None,
                           "atomtype_overlap_completeness": complete, "atomtype_overlap_incompleteness": incomplete},
            "rows": allrows, "columns": ["index"] + list(STAT_COLUMNS) + ["diff:" + t for t in atomTypes] + ["slope:" + t for t in atomTypes],
            "medianDiffs": medianDiffs, "meanDiffs": meanDiffs, "overallStdDevDiffs": overallStd, "medianSlopes": medianSlopes,
            "sizeDiffs": sizeDiffs, "atomTypeOverlapCompleteness": completeness}


def _workerInit(deviceIndex, params):
    """Initialiser of a host worker process: its own CUDA context on the rank's GPU, the parent's parameter set."""
    from . import densityAnalysis
    if torch.cuda.is_available():
        torch.cuda.set_device(deviceIndex)
    densityAnalysis.setGlobals(params)


def _workerAnalyze(args):
    loader, item, atomTypes = args
    try:
        return analyzeStructure(loader(item), atomTypes)
    except Exception:
        return 0


def runMultipleStructures(items, loader, costs=None, atomTypes=None, device=None, group=None, workers=1):
    """Multiple-structures mode: ``loader(item)`` returns a DensityAnalysis (or 0); structures are sharded over the
    ranks of the default process group, analysed on this rank's GPU, and summarised collectively.

    ``workers`` > 1: the per-structure host work (file parsing, the reference's set-growth bookkeeping, the numpy
    statistics block) is what bounds throughput, not the kernels, so a rank may spread its share over a pool of
    host processes that all drive the rank's GPU -- the reference's ``multiprocessing.Pool`` (pdb_eda/multipleStructures.py:167)
    with the voxel loops on the device.  ``loader`` must then be picklable (a module-level function or functools.partial)."""
    from . import densityAnalysis
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    atomTypes = sorted(densityAnalysis.paramsGlobal["radii"]) if atomTypes is None else list(atomTypes)
    costs = [1.0] * len(items) if costs is None else costs
    mine = shardStructures(costs, world)[rank]
    results = {}
    if workers > 1 and len(mine) > 1:
        import torch.multiprocessing as mp
        index = torch.cuda.current_device() if torch.cuda.is_available() else 0
        order = sorted(mine, key=lambda i: -float(costs[i]))                       # longest first, one task per structure
        with mp.get_context("spawn").Pool(min(workers, len(mine)), initializer=_workerInit,
                                          initargs=(index, densityAnalysis.paramsGlobal)) as pool:
            for idx, res in zip(order, pool.map(_workerAnalyze, [(loader, items[i], atomTypes) for i in order], chunksize=1)):
                results[idx] = res
    else:
        for idx in mine:
            try:
                results[idx] = analyzeStructure(loader(items[idx]), atomTypes)
            except Exception:
                results[idx] = 0                     # a bad structure yields no row; the run continues
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
    return gatherResults(results, mine, len(items), atomTypes, device, group)


class OptimizeService:
    """The inner loop of parameter optimisation as a persistent service (pdb_eda/optimizeParams.py:341-448): the reference
    re-downloads nothing but re-parses and re-analyses every entry in a fresh Pool task per iteration; here every rank
    loads its share of the structures ONCE, the maps stay resident in HBM and the atoms on the device as one ``PoolShard``;
    an iteration only uploads the new radii / slopes and re-runs the batched cloud aggregation on the GPU, followed by the
    two collectives of ``gatherPacked``.  Structures the batched layout cannot express (``AtomTable.supported`` false) make
    the service fall back to ``DensityAnalysis.aggregateCloud`` per structure."""

    def __init__(self, items, loader, costs=None, device=None, group=None):
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.n = len(items)
        self.mine = shardStructures([1.0] * self.n if costs is None else costs, self.world)[self.rank]
        self.analyzers = {}
        for idx in self.mine:
            try:
                self.analyzers[idx] = loader(items[idx])
            except Exception:
                self.analyzers[idx] = 0
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
        self.device = device
        self.shard = None
        self._names = None

    def _shardFor(self, params):
        """The device-resident shard; rebuilt only when the set of known atom names changes (never during an optimisation)."""
        from .cloudBatch import AtomTable
        names = frozenset(params["full_atom_name_map_atom_type"])
        if self.shard is None or names != self._names:
            entries = []
            for idx, analyzer in self.analyzers.items():
                if not analyzer:
                    continue
                table = AtomTable.fromStructure(analyzer.biopdbObj, params)
                if not table.supported:
                    return None
                entries.append((idx, analyzer.densityObj, table))
            self.shard = PoolShard(entries, params, device=self.device)
            self._names = names
        else:
            self.shard.setRadii(params)
        return self.shard

    def evaluate(self, params):
        """One optimiser iteration: (medianDiffs, meanDiffs, overallStdDevDiffs, medianSlopes, sizeDiffs,
        atomTypeOverlapCompleteness), the tuple of ``calculateMedianDiffsSlopes``."""
        from . import densityAnalysis
        densityAnalysis.setGlobals(params)
        types = list(params["radii"])
        shard = self._shardFor(params) if torch.cuda.is_available() else None
        if shard is not None:
            s = shard.analyze(self.device, self.group, optimizer=True)
            order = {t: k for k, t in enumerate(types)}                         # the shard keeps its types sorted
            pick = lambda d: {t: d[t] for t in sorted(d, key=lambda t: order.get(t, 0))}
            return (pick(s["medianDiffs"]), pick(s["meanDiffs"]), s["overallStdDevDiffs"], s["medianSlopes"], pick(s["sizeDiffs"]),
                    pick(s["atomTypeOverlapCompleteness"]))
        results = {}
        for idx, analyzer in self.analyzers.items():
            if not analyzer:
                results[idx] = 0
                continue
            analyzer.resetCloud()
            try:
                results[idx] = analyzeStructure(analyzer, types, optimizer=True)
            except Exception:
                results[idx] = 0
        s = gatherResults(results, self.mine, self.n, types, self.device, self.group)
        return (s["medianDiffs"], s["meanDiffs"], s["overallStdDevDiffs"], s["medianSlopes"], s["sizeDiffs"], s["atomTypeOverlapCompleteness"])


class PoolShard:
    """One rank's share of a pool of structures, resident on its GPU and analysed in batches (``cloudBatch.CloudBatch``):
    the device-side form of the reference's Pool of ``analyzePDBID`` / ``processFunction`` tasks
    (pdb_eda/multipleStructures.py:164-180, pdb_eda/optimizeParams.py:355-358).  ``entries``: (pool index, 2Fo-Fc map
    (DensityMatrix or cloudBatch.MapRef), cloudBatch.AtomTable) of the structures this rank owns, e.g. the shard
    ``shardStructures`` assigns to it.  A batch holds at most ``maxAtoms`` atoms (its cloud voxels size one workspace)."""

    def __init__(self, entries, params, maxAtoms=1 << 21, device=None):
        from .cloudBatch import CloudBatch
        self.params = params
        self.atomTypes = sorted(params["radii"])
        self.batches, self.indices = [], []
        cur, curIdx, atoms = [], [], 0
        for idx, dm, table in entries:
            if cur and atoms + len(table) > maxAtoms:
                self.batches.append(CloudBatch(cur, params, device))
                self.indices.append(curIdx)
                cur, curIdx, atoms = [], [], 0
            cur.append((dm, table))
            curIdx.append(idx)
            atoms += len(table)
        if cur:
            self.batches.append(CloudBatch(cur, params, device))
            self.indices.append(curIdx)
        self.nStructures = sum(len(i) for i in self.indices)
        self.nAtoms = sum(b.nAtoms for b in self.batches)

    def setRadii(self, params):
        self.params = params
        for b in self.batches:
            b.setRadii(params)

    def launch(self, minCloudElectrons=25.0, minTotalElectrons=400.0):
        for b in self.batches:
            b.launch(minCloudElectrons, minTotalElectrons)

    def pack(self, optimizer=False):
        """(cumulative vector, rows) of this shard: the payload of the two collectives."""
        T = len(self.atomTypes)
        cumulative = np.zeros(4 + 2 * T, dtype=np.float64)
        rows = []
        for b, idx in zip(self.batches, self.indices):
            c, r = packBatch(b.collectArrays(), idx, self.atomTypes, optimizer)
            cumulative += c
            rows.append(r)
        width = 1 + len(STAT_COLUMNS) + 2 * T
        return cumulative, (np.concatenate(rows) if rows else np.zeros((0, width)))

    def analyze(self, device=None, group=None, optimizer=False, minCloudElectrons=25.0, minTotalElectrons=400.0, local=False):
        """One pass over the shard + the fused all-reduce and the all-gather; the same summary on every rank
        (``local=True``: no collectives, this rank's structures only)."""
        self.launch(minCloudElectrons, minTotalElectrons)
        cumulative, rows = self.pack(optimizer)
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
        return gatherPacked(cumulative, rows, self.atomTypes, device, group, local)


def summarizeMetrics(ok, failed, rows, device="cpu", group=None):
    """(entries ok, entries failed, rows) summed over the ranks with ONE all_reduce; the same dict on every rank."""
    counts = np.array([ok, failed, rows], dtype=np.float64)
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        t = torch.from_numpy(counts).to(device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        counts = t.cpu().numpy()
    return {"ok": int(counts[0]), "failed": int(counts[1]), "rows": int(counts[2])}


def runMultipleMetrics(items, loader, level, costs=None, write=None, device=None, group=None, maxBytes=8 << 30):
    """RSCC / RSR rows (``residueMetrics()`` or ``atomMetrics()``, ``level`` "residue" / "atom") of many entries:
    ``loader(item)`` returns a DensityAnalysis (or 0); the entries are sharded over the ranks of the default process group
    longest first, and every rank analyses its share in batches of at most ``maxBytes`` device bytes (both maps + atoms,
    ``metricsBatch.MetricsBatch``).  Rows are ragged and large, so they are not gathered: ``write(index, rows)`` is called
    on the owning rank for every entry that yields rows.  An entry that fails to load or on which the single-structure
    call would raise is counted as failed.  Returns the all-reduced counts (``summarizeMetrics``) on every rank."""
    from . import metricsBatch
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    costs = [1.0] * len(items) if costs is None else costs
    mine = shardStructures(costs, world)[rank]                 # longest first

    def loaded():
        for idx in mine:
            try:
                yield idx, loader(items[idx])
            except Exception:
                yield idx, 0                                   # a bad entry yields no rows; the run continues

    ok = failed = nrows = 0
    for idx, rows in metricsBatch.analyzeStream(loaded(), level, maxBytes, device):
        if rows is None:
            failed += 1
            continue
        ok += 1
        nrows += len(rows)
        if write is not None:
            write(idx, rows)
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
    return summarizeMetrics(ok, failed, nrows, device, group)
