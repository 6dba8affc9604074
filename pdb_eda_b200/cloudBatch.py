"""Cloud aggregation for a batch of structures -- the unit of work of multiple-structures mode.

The reference analyses one entry per ``multiprocessing.Pool`` task: ``analyzePDBID`` (pdb_eda/multipleStructures.py:320-356)
and the optimiser's ``processFunction`` (pdb_eda/optimizeParams.py:410-448) both boil down to ``aggregateCloud``
(pdb_eda/densityAnalysis.py:571-780) plus a handful of per-structure numbers.  Here the atoms of MANY structures are
laid out as one set of arrays (atoms of a structure contiguous, one ``pe_batch_map`` per structure) and the whole
aggregation -- per-atom clouds, centroid cutoff, residue / domain merging, completeness counters -- runs as one sequence
of CUDA launches over the batch (``pe_cloud_count`` + ``pe_cloud_aggregate``, csrc/pe_aggregate.cu), followed by the
per-atom-type statistics block (pdb_eda/densityAnalysis.py:734-766) as one more kernel (``pe_cloud_statistics``,
csrc/pe_cloudstats.cu: exact medians by radix select, the b-factor regression with its p-value test).  The host reads back
a few numbers per structure and per (structure, atom type).  ``batchAtomTypeStatistics`` is the numpy statement of the
same block over a batch; the tests hold the kernel against it and it against the per-structure code.

What this path does not produce are the order-dependent descriptions of merged clouds (the atom that names a domain
cloud depends on Python set iteration order, pdb_eda/densityAnalysis.py:717); ``DensityAnalysis.aggregateCloud`` keeps
the replay that yields those.  Structures this layout cannot express (atoms with identical coordinates, which share one
``allAtomClouds`` entry at pdb_eda/densityAnalysis.py:606; more than 64 candidate atoms or repeated atom names in one
residue) are flagged ``supported = False`` and must take ``DensityAnalysis.aggregateCloud``.
"""
import collections
import ctypes

import numpy as np
import torch
from scipy import special

from . import _device
from . import _lib
from ._device import _ptr, _stream
from ._lib import PeBatchMap, check
from ._gc import pausedGC

MEDIAN_COLUMNS = ("num_voxels", "density_electron_ratio", "centroid_distance", "adj_density_electron_ratio", "volume", "bfactor",
                  "slopes", "domain_fraction", "corrected_fraction", "corrected_density_electron_ratio")


class AtomTable:
    """The candidate atoms of one structure (pdb_eda/densityAnalysis.py:596-603: residues with id[0] == ' ', atoms with a
    known RES_ATOM type and non-zero occupancy) as arrays, in the reference's traversal order."""

    def __init__(self, coords32, names, nameIndex, occupancy, bfactor, residue, local, bonded, nResidues, labels=None,
                 supported=True, reason=""):
        self.coords32 = np.ascontiguousarray(coords32, dtype=np.float32).reshape(-1, 3)
        self.names = list(names)                      # distinct RES_ATOM names
        self.nameIndex = np.asarray(nameIndex, dtype=np.int32)
        self.occupancy = np.asarray(occupancy, dtype=np.float64)
        self.bfactor = np.asarray(bfactor, dtype=np.float64)
        self.residue = np.asarray(residue, dtype=np.int32)
        self.local = np.asarray(local, dtype=np.int32)
        self.bonded = np.asarray(bonded, dtype=np.uint64)
        self.nResidues = int(nResidues)
        self.labels = labels                          # optional (chain, residue number, residue name, atom name) per atom
        self.supported = bool(supported)
        self.reason = reason

    def __len__(self):
        return len(self.nameIndex)

    @classmethod
    @pausedGC
    def fromStructure(cls, biopdbObj, params):
        """Walks a (duck-typed) Biopython structure once."""
        types = params["full_atom_name_map_atom_type"]
        bondedAtoms = params["bonded_atoms"]
        coords, nameIdx, occ, bf, res, local, labels, bondedList = [], [], [], [], [], [], [], []
        names, nameOf = [], {}
        masksOf = {}                                  # RES_ATOM sequence of a residue -> bonded-atom mask of each of its atoms
        supported, reason = True, ""
        ridx = -1
        for residue in biopdbObj.get_residues():
            rid = residue.id
            if rid[0] != ' ':
                continue
            ridx += 1
            resname = residue.resname
            prefix = resname.strip() + "_"
            chainId, number = residue.parent.id, rid[1]
            present = {}                              # RES_ATOM -> local index
            sequence = []
            for atom in residue.child_list:
                owner = atom.parent
                if owner is residue:
                    resAtom, ownerName = prefix + atom.name, resname
                else:
                    ownerName = owner.resname
                    resAtom = ownerName.strip() + "_" + atom.name
                if resAtom not in types:
                    continue
                occupancy = atom.get_occupancy()
                if occupancy == 0:
                    continue
                k = len(present)
                if present.setdefault(resAtom, k) != k:
                    supported, reason = False, "residue with a repeated atom name (%s)" % resAtom
                index = nameOf.get(resAtom)
                if index is None:
                    index = nameOf[resAtom] = len(names)
                    names.append(resAtom)
                sequence.append(resAtom)
                coords.append(atom.coord)
                nameIdx.append(index)
                occ.append(occupancy)
                bf.append(atom.get_bfactor())
                res.append(ridx)
                local.append(k)
                labels.append((chainId, number, ownerName, atom.name))
            if len(present) > 64:
                supported, reason = False, "residue with more than 64 candidate atoms"
            key = tuple(sequence)
            masks = masksOf.get(key)
            if masks is None:
                masks = []
                for resAtom in sequence:
                    mask = 0
                    for other in bondedAtoms.get(resAtom, ()):
                        j = present.get(other)
                        if j is not None and j < 64:
                            mask |= 1 << j
                    masks.append(mask)
                masksOf[key] = masks
            bondedList.extend(masks)
        n = len(coords)
        bonded = np.array(bondedList, dtype=np.uint64) if n else np.zeros(0, dtype=np.uint64)
        coords32 = np.asarray(coords, dtype=np.float32).reshape(-1, 3)
        if n and _distinctRows(coords32) < n:
            supported, reason = False, "atoms with identical coordinates share one cloud entry"
        return cls(coords32, names, nameIdx, occ, bf, res, np.minimum(np.asarray(local, dtype=np.int64), 63), bonded, ridx + 1, labels,
                   supported, reason)


def _distinctRows(coords32):
    """Number of distinct coordinate triples (-0.0 and 0.0 are one key, like the tuple keys of pdb_eda/densityAnalysis.py:606)."""
    rows = np.ascontiguousarray(np.asarray(coords32, dtype=np.float32) + np.float32(0.0))
    return len(np.unique(rows.view(np.dtype((np.void, 12))).ravel()))


def _typeTables(table, params):
    """Per distinct RES_ATOM name of a table: radius, electrons, atom type."""
    types = params["full_atom_name_map_atom_type"]
    radii = params["radii"]
    electrons = params["full_atom_name_map_electrons"]
    t = [types[name] for name in table.names]
    return (np.array([radii[x] for x in t], dtype=np.float64), np.array([electrons[name] for name in table.names], dtype=np.float64), t)


# ---------------------------------------------------------------------------------------------------- statistics
def _segmentedNanMedian(values, group, nGroups, mask=None):
    """np.nanmedian(values[group == g]) for every g (NaN for an empty selection): one lexsort for all groups."""
    values = np.asarray(values, dtype=np.float64)
    if mask is not None:
        values, group = values[mask], group[mask]
    out = np.full(nGroups, np.nan)
    if len(values) == 0:
        return out
    order = np.lexsort((values, group))               # NaN sorts last inside its group
    v, g = values[order], group[order]
    valid = np.bincount(g[~np.isnan(v)], minlength=nGroups)
    start = np.concatenate(([0], np.cumsum(np.bincount(g, minlength=nGroups))))[:-1]
    has = valid > 0
    lo = start[has] + (valid[has] - 1) // 2
    hi = start[has] + valid[has] // 2
    out[has] = (v[lo] + v[hi]) / 2.0
    odd = has.copy()
    odd[has] = (valid[has] % 2) == 1
    out[odd] = v[start[odd] + valid[odd] // 2]        # the middle element itself for odd counts
    return out


def _segmentedNanStd(values, group, nGroups):
    """np.nanstd(values[group == g]) for every g (population, ddof 0)."""
    values = np.asarray(values, dtype=np.float64)
    ok = ~np.isnan(values)
    n = np.bincount(group[ok], minlength=nGroups).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        mean = np.bincount(group[ok], weights=values[ok], minlength=nGroups) / n
        dev = values[ok] - mean[group[ok]]
        return np.sqrt(np.bincount(group[ok], weights=dev * dev, minlength=nGroups) / n)


def batchAtomTypeStatistics(structure, typeIndex, nTypes, densityElectronRatio, numVoxels, centroidDistance, bfactor, ratio,
                            unitVolume, currentSlopes):
    """pdb_eda/densityAnalysis.py:734-766 for all structures of a batch at once.

    Rows = contributing atoms (the reference's ``atomList``), ``structure`` / ``typeIndex`` their structure and atom-type
    indices; ``ratio`` / ``unitVolume`` per structure; ``currentSlopes`` per type.  Returns (keep mask of the rows that
    survive the centroid filter, {column: (nStructures, nTypes) array of medians, NaN where a type is absent},
    present (nStructures, nTypes) bool)."""
    nS = len(ratio)
    structure = np.asarray(structure, dtype=np.int64)
    typeIndex = np.asarray(typeIndex, dtype=np.int64)
    cd = np.asarray(centroidDistance, dtype=np.float64)
    with np.errstate(all="ignore"):
        cutoff = _segmentedNanMedian(cd, structure, nS) + _segmentedNanStd(cd, structure, nS) * 2
        allNan = np.bincount(structure[~np.isnan(cd)], minlength=nS) == 0          # np.isnan(...).all(): no filter then
        keep = allNan[structure] | (cd < cutoff[structure])
    s, t = structure[keep], typeIndex[keep]
    der = np.asarray(densityElectronRatio, dtype=np.float64)[keep]
    nv = np.asarray(numVoxels, dtype=np.float64)[keep]
    cd = cd[keep]
    bf = np.asarray(bfactor, dtype=np.float64)[keep].copy()
    g = s * nTypes + t
    nG = nS * nTypes
    count = np.bincount(g, minlength=nG)
    present = (count > 0).reshape(nS, nTypes)
    med = {}
    with np.errstate(all="ignore"):
        med["num_voxels"] = _segmentedNanMedian(nv, g, nG)
        adj = der / nv * med["num_voxels"][g]
        volume = nv * np.asarray(unitVolume, dtype=np.float64)[s]
        med["density_electron_ratio"] = _segmentedNanMedian(der, g, nG)
        med["centroid_distance"] = _segmentedNanMedian(cd, g, nG)
        med["adj_density_electron_ratio"] = _segmentedNanMedian(adj, g, nG)
        med["volume"] = _segmentedNanMedian(volume, g, nG)
        med["bfactor"] = _segmentedNanMedian(bf, g, nG, mask=bf > 0)
        low = bf <= 0
        bf[low] = med["bfactor"][g][low]
        # slopes: linregress(log(bfactor), (adj - ratio) / ratio) per (structure, type) group
        r_s = np.asarray(ratio, dtype=np.float64)[s]
        x = np.log(bf)
        y = (adj - r_s) / r_s
        n = count.astype(np.float64)
        xm = np.bincount(g, weights=x, minlength=nG) / n
        ym = np.bincount(g, weights=y, minlength=nG) / n
        dx, dy = x - xm[g], y - ym[g]
        ssxm = np.bincount(g, weights=dx * dx, minlength=nG) / n
        ssym = np.bincount(g, weights=dy * dy, minlength=nG) / n
        ssxym = np.bincount(g, weights=dx * dy, minlength=nG) / n
        degenerate = (ssxm == 0.0) | (ssym == 0.0)
        rr = np.where(degenerate, np.where(ssxym == 0, np.nan, 0.0), np.clip(ssxym / np.sqrt(ssxm * ssym), -1.0, 1.0))
        fitSlope = ssxym / ssxm
        df = n - 2
        tt = rr * np.sqrt(df / ((1.0 - rr + 1.0e-20) * (1.0 + rr + 1.0e-20)))
        prob = 2 * special.stdtr(df, -np.abs(tt))
        # distinct b-factors per group (NaN counts as one value, like np.unique)
        order = np.lexsort((bf, g))
        bs, gs = bf[order], g[order]
        newValue = np.ones(len(bs), dtype=bool)
        if len(bs) > 1:
            same = (gs[1:] == gs[:-1]) & ((bs[1:] == bs[:-1]) | (np.isnan(bs[1:]) & np.isnan(bs[:-1])))
            newValue[1:] = ~same
        nUnique = np.bincount(gs[newValue], minlength=nG)
        current = np.tile(np.asarray(currentSlopes, dtype=np.float64), nS)
        useCurrent = (count <= 2) | (nUnique == 1) | (prob > 0.05)
        med["slopes"] = np.where(useCurrent, current, fitSlope)
        med["slopes"][count == 0] = np.nan
        domain = (adj - r_s) / r_s
        corrected = domain - (np.log(bf) - np.log(med["bfactor"][g])) * med["slopes"][g]
        correctedRatio = corrected * r_s + r_s
        med["domain_fraction"] = _segmentedNanMedian(domain, g, nG)
        med["corrected_fraction"] = _segmentedNanMedian(corrected, g, nG)
        med["corrected_density_electron_ratio"] = _segmentedNanMedian(correctedRatio, g, nG)
    return keep, {k: v.reshape(nS, nTypes) for k, v in med.items()}, present


# ---------------------------------------------------------------------------------------------------- results
class CloudResult:
    """What ``analyzePDBID`` / ``processFunction`` read from a DensityAnalysis after ``aggregateCloud``."""

    def __init__(self, pdbid=None):
        self.pdbid = pdbid
        self.densityElectronRatio = None
        self.numVoxelsAggregated = None
        self.totalAggregatedElectrons = None
        self.totalAggregatedDensity = None
        self.numAtomsAnalyzed = 0
        self.numResidueClouds = 0
        self.numDomainClouds = 0
        self.medians = None
        self.atomTypeOverlapCompleteness = None
        self.atomTypeOverlapIncompleteness = None
        self.centroidDistanceCutoff = None
        self.unitVolume = None


class MapRef:
    """The part of a 2Fo-Fc ``DensityMatrix`` the batch needs, for maps that only exist on the device (synthetic pools)."""

    def __init__(self, deviceMap, densityCutoff, unitVolume, pdbid=None):
        self.deviceMap = deviceMap
        self.densityCutoff = densityCutoff
        self.unitVolume = unitVolume
        self.pdbid = pdbid


class CloudBatch:
    """A batch of (2Fo-Fc DensityMatrix, AtomTable) pairs laid out for ``pe_cloud_aggregate``; the maps stay where they are
    in HBM (only pointers are gathered), the atom arrays are uploaded once."""

    def __init__(self, items, params, device=None, pdbids=None):
        self.items = list(items)
        self.params = params
        self.lib = _lib.load()
        _device.require_cuda()
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        self.pdbids = list(pdbids) if pdbids is not None else [getattr(dm, "pdbid", None) for dm, _ in self.items]
        self.atomTypes = sorted(params["radii"])
        typeOf = {t: k for k, t in enumerate(self.atomTypes)}
        nS = len(self.items)
        counts = np.array([len(t) for _, t in self.items], dtype=np.int64)
        self.atomStart = np.concatenate(([0], np.cumsum(counts)))
        nA = int(self.atomStart[-1])
        self.nAtoms, self.nStructures = nA, nS
        resStart = np.concatenate(([0], np.cumsum([t.nResidues for _, t in self.items])))
        self.nResidues = int(resStart[-1])
        xyz = np.empty((nA, 3), dtype=np.float64)
        radius = np.empty(nA, dtype=np.float32)
        self.atomMap = np.empty(nA, dtype=np.int32)
        residue = np.empty(nA, dtype=np.int32)
        local = np.empty(nA, dtype=np.int32)
        bonded = np.empty(nA, dtype=np.uint64)
        self.electrons = np.empty(nA, dtype=np.float64)          # electrons of the atom's RES_ATOM name
        self.occupancy = np.empty(nA, dtype=np.float64)
        self.bfactor = np.empty(nA, dtype=np.float64)
        self.typeIndex = np.empty(nA, dtype=np.int32)
        maps = (PeBatchMap * max(nS, 1))()
        self.unitVolume = np.empty(nS, dtype=np.float64)
        self._keepAlive = []
        for k, (dm, table) in enumerate(self.items):
            if not table.supported:
                raise ValueError("structure %d cannot take the batched path: %s" % (k, table.reason))
            a0, a1 = int(self.atomStart[k]), int(self.atomStart[k + 1])
            r, e, tnames = _typeTables(table, params)
            xyz[a0:a1] = table.coords32                           # float32 widened exactly
            radius[a0:a1] = r[table.nameIndex].astype(np.float32)
            self.atomMap[a0:a1] = k
            residue[a0:a1] = table.residue + resStart[k]
            local[a0:a1] = table.local
            bonded[a0:a1] = table.bonded
            self.electrons[a0:a1] = e[table.nameIndex]
            self.occupancy[a0:a1] = table.occupancy
            self.bfactor[a0:a1] = table.bfactor
            self.typeIndex[a0:a1] = np.array([typeOf[x] for x in tnames], dtype=np.int32)[table.nameIndex] if len(table) else 0
            dmap = dm.deviceMap
            self._keepAlive.append(dmap)
            maps[k].geom = dmap.geom
            maps[k].d_rho = dmap.rho.data_ptr()
            maps[k].cutoff = float(np.float32(dm.densityCutoff))
            maps[k].atom_begin, maps[k].atom_end = a0, a1
            self.unitVolume[k] = dm.unitVolume if isinstance(dm, MapRef) else dm.header.unitVolume
        # atoms type by type inside every structure: the (structure, type) groups of the statistics block are segments
        perm = np.lexsort((self.typeIndex, self.atomMap)).astype(np.int32)
        gkey = self.atomMap[perm].astype(np.int64) * len(self.atomTypes) + self.typeIndex[perm]
        edge = np.flatnonzero(np.concatenate(([True], gkey[1:] != gkey[:-1]))) if nA else np.zeros(0, dtype=np.int64)
        self.segBegin = edge.astype(np.int32)
        self.segEnd = np.concatenate((edge[1:], [nA])).astype(np.int32) if nA else np.zeros(0, dtype=np.int32)
        self.segMap = (gkey[edge] // len(self.atomTypes)).astype(np.int32) if nA else np.zeros(0, dtype=np.int32)
        self.segType = (gkey[edge] % len(self.atomTypes)).astype(np.int32) if nA else np.zeros(0, dtype=np.int32)
        self.nSegments = len(self.segBegin)
        self.maxSegment = int((self.segEnd - self.segBegin).max()) if self.nSegments else 0
        up = lambda arr: torch.from_numpy(np.ascontiguousarray(arr)).to(device)
        self.d_maps = torch.frombuffer(bytearray(bytes(maps)), dtype=torch.uint8).to(device)
        self.d_xyz, self.d_radius, self.d_atomMap = up(xyz), up(radius), up(self.atomMap)
        self.d_residue, self.d_local = up(residue), up(local)
        self.d_bonded = up(bonded.view(np.int64))
        self.d_electrons = up(self.electrons * self.occupancy)
        self.d_static = up(np.stack((self.electrons, self.occupancy, self.bfactor), axis=1))
        self.d_perm, self.d_segMap = up(perm), up(self.segMap)
        self.d_segType, self.d_segBegin, self.d_segEnd = up(self.segType), up(self.segBegin), up(self.segEnd)
        self.d_unitVolume = up(self.unitVolume)
        self.d_slopes = up(self._currentSlopes(params))
        self.d_offset = torch.empty(nA + 1, dtype=torch.int32, device=device)
        self.d_totals = torch.zeros(2, dtype=torch.int64, device=device)
        self.d_scan = torch.empty(256 + 4 * (nA // 1024 + 4), dtype=torch.uint8, device=device)
        self.d_boxBits = torch.empty((max(nA, 1), 8), dtype=torch.int32, device=device)  # count pass -> fill pass (pe_cloud_count)
        self.d_atomOut = torch.empty((nA, 8), dtype=torch.float64, device=device)
        self.d_mapOut = torch.empty((max(nS, 1), 8), dtype=torch.float64, device=device)
        self.d_scratch = torch.empty((9, max(nA, 1)), dtype=torch.float64, device=device)
        self.d_segOut = torch.empty((max(self.nSegments, 1), 14), dtype=torch.float64, device=device)
        self.d_mapStats = torch.empty((max(nS, 1), 4), dtype=torch.float64, device=device)
        pin = lambda t: torch.empty(t.shape, dtype=t.dtype).pin_memory()
        self.h_mapOut, self.h_segOut, self.h_mapStats = pin(self.d_mapOut), pin(self.d_segOut), pin(self.d_mapStats)
        self.ws = None
        self.nEntries = 0

    def _currentSlopes(self, params):
        slopes = params["slopes"]
        return np.array([slopes.get(x, np.nan) for x in self.atomTypes], dtype=np.float64)

    def setRadii(self, params):
        """New radii / slopes (one optimiser iteration, pdb_eda/optimizeParams.py:417-421); the atoms stay on the device."""
        self.params = params
        radius = np.empty(self.nAtoms, dtype=np.float32)
        for k, (_, table) in enumerate(self.items):
            a0, a1 = int(self.atomStart[k]), int(self.atomStart[k + 1])
            radius[a0:a1] = _typeTables(table, params)[0][table.nameIndex].astype(np.float32)
        self.d_radius.copy_(torch.from_numpy(radius))
        self.d_slopes.copy_(torch.from_numpy(self._currentSlopes(params)))

    # ---- device part: enqueue, then read back -------------------------------------------------------------------
    def launch(self, minCloudElectrons=25.0, minTotalElectrons=400.0):
        """Enqueues the whole aggregation and the statistics; one host synchronisation in between (the number of cloud
        voxels of the batch sizes the workspace), then asynchronous copies of the small result tables to pinned memory."""
        nS, nA = self.nStructures, self.nAtoms
        if nS == 0:
            return
        check(self.lib.pe_cloud_count(nS, _ptr(self.d_maps), nA, _ptr(self.d_atomMap), _ptr(self.d_xyz), _ptr(self.d_radius),
                                      _ptr(self.d_offset), _ptr(self.d_totals), _ptr(self.d_scan), _ptr(self.d_boxBits), _stream()),
              "pe_cloud_count")
        nEntries, maxBox = self.d_totals.tolist()
        self.nEntries = int(nEntries)
        need = int(self.lib.pe_cloud_workspace_bytes(nA, nEntries, self.nResidues, nS))
        if self.ws is None or self.ws.numel() < need:
            self.ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        check(self.lib.pe_cloud_aggregate(nS, _ptr(self.d_maps), nA, _ptr(self.d_atomMap), _ptr(self.d_xyz), _ptr(self.d_radius),
                                          _ptr(self.d_residue), _ptr(self.d_local), _ptr(self.d_bonded), _ptr(self.d_electrons),
                                          self.nResidues, _ptr(self.d_offset), nEntries, max(int(maxBox), 1),
                                          ctypes.c_double(minCloudElectrons), _ptr(self.d_boxBits), _ptr(self.d_atomOut), _ptr(self.d_mapOut),
                                          _ptr(self.ws), _stream()), "pe_cloud_aggregate")
        check(self.lib.pe_cloud_statistics(nS, _ptr(self.d_maps), nA, _ptr(self.d_atomOut), _ptr(self.d_mapOut), _ptr(self.d_static),
                                           _ptr(self.d_perm), self.nSegments, _ptr(self.d_segMap), _ptr(self.d_segType),
                                           _ptr(self.d_segBegin), _ptr(self.d_segEnd), self.maxSegment, _ptr(self.d_unitVolume), _ptr(self.d_slopes),
                                           ctypes.c_double(minTotalElectrons), _ptr(self.d_scratch), _ptr(self.d_segOut),
                                           _ptr(self.d_mapStats), _stream()), "pe_cloud_statistics")
        self.h_mapOut.copy_(self.d_mapOut, non_blocking=True)
        self.h_segOut.copy_(self.d_segOut, non_blocking=True)
        self.h_mapStats.copy_(self.d_mapStats, non_blocking=True)

    def collectArrays(self):
        """Synchronises and returns the batch's results as arrays: per structure ``ok`` (enough electrons, :726), ``ratio``,
        ``numVoxels``, ``totalElectrons``, ``totalDensity``, ``analysed`` (len(atomCloudDescriptions)), ``residueClouds`` /
        ``domainClouds`` (those with >= minCloudElectrons); per (structure, atom type) ``present``, ``medians[column]``,
        ``complete`` / ``incomplete`` (the overlap completeness counters, :653-659)."""
        nS, nT = self.nStructures, len(self.atomTypes)
        bad = ctypes.c_int32(0)
        if nS and self.nAtoms:
            check(self.lib.pe_cloud_status(_ptr(self.ws), _stream(), ctypes.byref(bad)), "pe_cloud_status")
        else:
            torch.cuda.current_stream().synchronize()
        if bad.value:
            raise _lib.PdbEdaLibError("pe_cloud_aggregate: voxel index outside the supported key range or inconsistent counts")
        mapOut = self.h_mapOut.numpy()[:nS]
        mapStats = self.h_mapStats.numpy()[:nS]
        seg = self.h_segOut.numpy()[:self.nSegments]
        ok = mapStats[:, 3] != 0
        out = {"ok": ok, "ratio": mapStats[:, 1].copy(), "numVoxels": mapOut[:, 0].copy(), "totalDensity": mapOut[:, 1].copy(),
               "totalElectrons": mapOut[:, 2].copy(), "analysed": mapStats[:, 0].copy(), "domainClouds": mapOut[:, 4].copy(),
               "residueClouds": mapOut[:, 6].copy(), "centroidCutoff": mapOut[:, 7].copy(), "centroidCutoff2": mapStats[:, 2].copy(),
               "unitVolume": self.unitVolume}
        sm, stp = self.segMap, self.segType
        present = np.zeros((nS, nT), dtype=bool)
        present[sm, stp] = (seg[:, 0] > 0) & ok[sm]
        medians = {}
        for j, column in enumerate(MEDIAN_COLUMNS):
            table = np.full((nS, nT), np.nan)
            table[sm, stp] = seg[:, 1 + j]
            medians[column] = table
        complete = np.zeros((nS, nT), dtype=np.int64)
        incomplete = np.zeros((nS, nT), dtype=np.int64)
        complete[sm, stp] = seg[:, 12].astype(np.int64)
        incomplete[sm, stp] = (seg[:, 11] - seg[:, 12]).astype(np.int64)
        out.update(present=present, medians=medians, complete=complete, incomplete=incomplete)
        return out

    def collect(self):
        """The same as objects, one ``CloudResult`` per structure (all fields None-like below minTotalElectrons)."""
        arr = self.collectArrays()
        results = []
        for k in range(self.nStructures):
            res = CloudResult(self.pdbids[k])
            res.centroidDistanceCutoff = arr["centroidCutoff"][k]
            res.unitVolume = self.unitVolume[k]
            if arr["ok"][k]:
                res.densityElectronRatio = float(arr["ratio"][k])
                res.numVoxelsAggregated = int(arr["numVoxels"][k])
                res.totalAggregatedElectrons = float(arr["totalElectrons"][k])
                res.totalAggregatedDensity = float(arr["totalDensity"][k])
                res.numAtomsAnalyzed = int(arr["analysed"][k])
                res.numResidueClouds = int(arr["residueClouds"][k])
                res.numDomainClouds = int(arr["domainClouds"][k])
                cols = np.flatnonzero(arr["present"][k])
                res.medians = {c: {self.atomTypes[j]: arr["medians"][c][k, j] for j in cols} for c in MEDIAN_COLUMNS}
                res.atomTypeOverlapCompleteness = collections.defaultdict(
                    int, {self.atomTypes[j]: int(arr["complete"][k, j]) for j in np.flatnonzero(arr["complete"][k])})
                res.atomTypeOverlapIncompleteness = collections.defaultdict(
                    int, {self.atomTypes[j]: int(arr["incomplete"][k, j]) for j in np.flatnonzero(arr["incomplete"][k])})
            results.append(res)
        return results

    def run(self, minCloudElectrons=25.0, minTotalElectrons=400.0):
        self.launch(minCloudElectrons, minTotalElectrons)
        return self.collect()

    def atomRows(self):
        """Device -> host read of the per-atom records (n_atoms x 8, see ``pe_cloud_aggregate``)."""
        return self.d_atomOut.cpu().numpy()
