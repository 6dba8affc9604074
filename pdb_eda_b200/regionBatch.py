"""Region density and region discrepancy per atom, residue or symmetry atom for a batch of structures -- ``density`` /
``difference`` with ``--atom`` / ``--residue`` / ``--symmetry-atom`` of many entries.

``DensityAnalysis.calculate*RegionDensity`` / ``calculate*RegionDiscrepancies`` (pdb_eda/densityAnalysis.py:948-1211) analyse
one structure: the density-electron ratio of its cloud aggregation, one ``pe_sphere_sums`` launch and one read-back.  Here the
atoms of MANY structures are laid out as one set of arrays (groups -- residues, or single atoms -- in CSR form across
structures), every structure's map stays where it is in HBM with its own cutoffs (only pointers are gathered into one
``pe_sums_map`` table), the ratios of the batch come from one ``CloudBatch``, and one launch of ``pe_batch_sphere_sums``
(csrc/pe_union.cu, csrc/pe_sphere.cu) yields the sums of every group; every row of it is bit-identical to the row
``pe_sphere_sums`` gives for that structure alone.  The rows are then built with numpy and are the rows, in the order and
with the types, that the single-structure calls return.
"""
import ctypes

import numpy as np
import torch

from . import _device
from . import _lib
from . import densityAnalysis
from ._device import _ptr, _stream
from ._lib import PE_SPHERE_NOUT, PeGeom, check

KINDS = ("density", "difference")
LEVELS = ("atom", "residue", "symmetry-atom")


class PeSumsMap(ctypes.Structure):
    """Mirror of ``struct pe_sums_map`` (include/pdbeda_b200.h)."""
    _fields_ = [("geom", PeGeom), ("d_rho", ctypes.c_void_p), ("cut_pos", ctypes.c_float), ("cut_neg", ctypes.c_float)]


def _f32(x):
    return float(np.float32(x))


# ---------------------------------------------------------------------------------------------------- rows from sums
def densityRows(sums, ratio):
    """``_regionDensityRows`` of (n, 8) sums: [sum of rho > cutoff, / ratio] per group, as np.float64 scalars."""
    pos = np.asarray(sums, dtype=np.float64).reshape(-1, PE_SPHERE_NOUT)[:, 3]
    return [list(r) for r in zip(pos, pos / ratio)]


def discrepancyRows(sums, ratio, avgAbsVoxel):
    """``_regionDiscrepancyRows`` of (n, 8) sums: the ten values per group.  ``avgAbsVoxel``: getTotalAbsDensity(cutoff) /
    number of voxels.  The expected columns are Python floats (a float times ``int(n)``), the others np.float64, as there."""
    sums = np.asarray(sums, dtype=np.float64).reshape(-1, PE_SPHERE_NOUT)
    pos, neg = sums[:, 3], sums[:, 5]
    actual = pos + neg
    actualAbs = np.abs(pos) + np.abs(neg)
    expected = (avgAbsVoxel * sums[:, 0]).tolist()          # n is an exact integer: the same product as avg * int(n)
    cols = (actualAbs, actualAbs / ratio, expected, [x / ratio for x in expected], actual, actual / ratio, pos, pos / ratio,
            neg, neg / ratio)
    return [list(r) for r in zip(*cols)]


# ---------------------------------------------------------------------------------------------------- entries
class RegionEntry:
    """One structure of a batch: its map and cutoffs, its atoms (float64 coordinates, float32 radii), its groups in CSR form
    (None: one group per atom), and ``finish(ratio, sums)`` that turns the sums into the rows of the single-structure call."""

    def __init__(self, analyzer, deviceMap, xyz, radius, groupStart, cutPos, cutNeg, finish):
        self.analyzer = analyzer
        self.map = deviceMap
        self.xyz = np.ascontiguousarray(np.asarray(xyz, dtype=np.float64).reshape(-1, 3))
        self.radius = np.ascontiguousarray(np.asarray(radius, dtype=np.float32).reshape(-1))
        self.groupStart = None if groupStart is None else np.asarray(groupStart, dtype=np.int64)
        self.cutPos, self.cutNeg = _f32(cutPos), _f32(cutNeg)
        if self.cutPos < 0 or self.cutNeg > 0:
            raise ValueError("cutoffs must satisfy cut_pos >= 0 >= cut_neg")
        self.finish = finish

    @property
    def nGroups(self):
        return len(self.xyz) if self.groupStart is None else len(self.groupStart) - 1

    def deviceBytes(self):
        """Bytes this entry holds on the device in a batch: the map, the atom arrays, the output rows and the cloud batch's
        per-atom tables."""
        return 4 * self.map.rho.numel() + len(self.xyz) * (24 + 4 + 4 + 32) + self.nGroups * (64 + 8) + \
            len(self.xyz) * 400


def _atoms(analyzer, level, type):
    atoms = analyzer.symmetryAtoms if level == "symmetry-atom" else list(analyzer.biopdbObj.get_atoms())
    if type:
        atoms = [atom for atom in atoms if atom.name == type]
    return atoms


def _atomPrefix(atom):
    return [atom.parent.parent.parent.id, atom.parent.parent.id, atom.parent.id[1], atom.parent.resname, atom.name]


def makeEntry(analyzer, kind, level, radius=3.5, numSD=None, type="", atomMask=None, useOptimizedRadii=False):
    """The call ``kind`` ("density" / "difference") x ``level`` ("atom" / "residue" / "symmetry-atom") of a DensityAnalysis as a
    batch entry, with that call's options (``useOptimizedRadii``: density only; ``atomMask``: residue level only).  Raises
    where the single-structure call raises before it needs the ratio."""
    if kind not in KINDS or level not in LEVELS:
        raise ValueError("kind must be one of %s and level one of %s" % (KINDS, LEVELS))
    if numSD is None:
        numSD = 1.5 if kind == "density" else 3.0
    density = kind == "density"
    dm = analyzer.densityObj if density else analyzer.diffDensityObj
    cutoff = dm.meanDensity + numSD * dm.stdDensity
    cutPos, cutNeg = (cutoff, 0.0) if density else (cutoff, -1.0 * cutoff)
    if level == "residue":
        residues = list(analyzer.biopdbObj.get_residues())
        if type:
            residues = [residue for residue in residues if residue.resname == type]
        kept, xyz, radii, start = [], [], [], [0]
        meanOf = {}
        for residue in residues:
            atoms = list(residue.get_atoms())
            if density:
                if atomMask and residue.resname in atomMask:
                    allowed = atomMask[residue.resname]
                    atoms = [atom for atom in atoms if atom.name in allowed]
                if not atoms:
                    continue
            else:
                if atomMask:
                    allowed = atomMask[residue.resname] if residue.resname in atomMask else ()
                    atoms = [atom for atom in atoms if atom.name in allowed]
                if not atoms:
                    raise IndexError("list index out of range")  # the reference fails on a residue left without atoms
            kept.append([residue.parent.parent.id, residue.parent.id, residue.id[1], residue.resname,
                         densityAnalysis._meanOccupancy(atoms, meanOf)])
            xyz.extend([atom.coord for atom in atoms])
            if density and useOptimizedRadii:
                radii.extend([analyzer._testRadius(atom, radius, True) for atom in atoms])
            else:
                radii.extend([radius] * len(atoms))
            start.append(len(xyz))
        prefixes, groupStart = kept, np.asarray(start)
    else:
        atoms = _atoms(analyzer, level, type)
        symmetry = level == "symmetry-atom"
        xyz = [np.asarray(atom.coord, dtype=np.float64) for atom in atoms] if symmetry else [atom.coord for atom in atoms]
        radii = [analyzer._testRadius(atom, radius, useOptimizedRadii) for atom in atoms] if density else [radius] * len(atoms)
        if symmetry:
            prefixes = [_atomPrefix(atom) + [atom.symmetry, atom.coord] for atom in atoms]
        else:
            prefixes = [_atomPrefix(atom) + [atom.get_occupancy()] for atom in atoms]
        groupStart = None
        xyz = np.asarray(xyz, dtype=np.float64).reshape(-1, 3)

    def finish(ratio, sums):
        if not ratio:
            raise RuntimeError("Failed to calculate densityElectronRatio, probably due to total aggregated electrons less than the minimum.")
        if not prefixes:
            return []
        if density:
            rows = densityRows(sums, ratio)
        else:
            rows = discrepancyRows(sums, ratio, dm.getTotalAbsDensity(cutoff) / dm.deviceMap.n_voxels)
        if level == "symmetry-atom":
            return [p + [bool(ok)] + r for p, r, ok in zip(prefixes, rows, (sums[:, 6] != 0).tolist())]
        return [p + r for p, r in zip(prefixes, rows)]

    # float64 radii narrowed to float32 as utils.sphereSums narrows them
    return RegionEntry(analyzer, dm.deviceMap, np.asarray(xyz, dtype=np.float64).reshape(-1, 3),
                       np.asarray(np.asarray(radii, dtype=np.float64), dtype=np.float32), groupStart, cutPos, cutNeg, finish)


# ---------------------------------------------------------------------------------------------------- the batch
class RegionBatch:
    """A batch of ``RegionEntry`` laid out for one ``pe_batch_sphere_sums`` launch, plus one ``CloudBatch`` for the ratios of
    the entries that need one.  All entries are grouped, or none is."""

    def __init__(self, entries, device=None):
        self.entries = list(entries)
        self.lib = _lib.load()
        _device.require_cuda()
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        nS = len(self.entries)
        grouped = {e.groupStart is not None for e in self.entries}
        if len(grouped) > 1:
            raise ValueError("a batch is all grouped or all per atom")
        self.grouped = grouped.pop() if grouped else False
        atomCounts = np.array([len(e.xyz) for e in self.entries], dtype=np.int64)
        groupCounts = np.array([e.nGroups for e in self.entries], dtype=np.int64)
        self.atomStart = np.concatenate(([0], np.cumsum(atomCounts)))
        self.groupBase = np.concatenate(([0], np.cumsum(groupCounts)))
        self.nAtoms, self.nGroups = int(self.atomStart[-1]), int(self.groupBase[-1])
        if self.nAtoms >= 2 ** 31 or self.nGroups >= 2 ** 31:
            raise ValueError("a batch holds fewer than 2^31 atoms and groups")
        xyz = np.concatenate([e.xyz for e in self.entries]) if nS else np.zeros((0, 3))
        radius = np.concatenate([e.radius for e in self.entries]) if nS else np.zeros(0, dtype=np.float32)
        groupMap = np.repeat(np.arange(nS, dtype=np.int32), groupCounts)
        maps = (PeSumsMap * max(nS, 1))()
        for k, e in enumerate(self.entries):
            maps[k].geom = e.map.geom
            maps[k].d_rho = e.map.rho.data_ptr()
            maps[k].cut_pos, maps[k].cut_neg = e.cutPos, e.cutNeg
        up = lambda arr: torch.from_numpy(np.ascontiguousarray(arr)).to(device)
        self.d_maps = torch.frombuffer(bytearray(bytes(maps)), dtype=torch.uint8).to(device)
        self.d_xyz = up(xyz if self.nAtoms else np.zeros((1, 3)))
        self.d_radius = up(radius if self.nAtoms else np.zeros(1, dtype=np.float32))
        self.d_groupMap = up(groupMap if self.nGroups else np.zeros(1, dtype=np.int32))
        self.d_atomStart = up(self.atomStart.astype(np.int32))
        self.d_groupStart = None
        if self.grouped:
            groupStart = np.empty(self.nGroups + 1, dtype=np.int32)
            groupStart[-1] = self.nAtoms
            for k, e in enumerate(self.entries):
                groupStart[self.groupBase[k]:self.groupBase[k + 1]] = e.groupStart[:-1] + self.atomStart[k]
            self.d_groupStart = up(groupStart)
        self.d_out = torch.empty((max(self.nGroups, 1), PE_SPHERE_NOUT), dtype=torch.float64, device=device)
        self.h_out = torch.empty(self.d_out.shape, dtype=torch.float64).pin_memory()
        self.ws = torch.empty(max(int(self.lib.pe_batch_sphere_sums_workspace_bytes(self.nAtoms)), 256), dtype=torch.uint8,
                              device=device)
        self.cloud, self.cloudOf = None, {}

    def launchSums(self):
        """Enqueues the sums of every group and the copy of the result rows to pinned memory."""
        check(self.lib.pe_batch_sphere_sums(len(self.entries), _ptr(self.d_maps), self.nAtoms, _ptr(self.d_xyz), _ptr(self.d_radius),
                                            self.nGroups, _ptr(self.d_groupMap), _ptr(self.d_groupStart), _ptr(self.d_atomStart),
                                            _ptr(self.d_out), _ptr(self.ws), _stream()), "pe_batch_sphere_sums")
        self.h_out.copy_(self.d_out, non_blocking=True)

    def launch(self):
        """Enqueues the cloud aggregation of the entries whose ratio is not known yet (the defaults of ``aggregateCloud``), then
        the sums.  Entries whose structure the batched cloud layout cannot express, or every entry when
        PDB_EDA_B200_FULL_CLOUD is set, take ``densityElectronRatio`` (the per-structure pipeline) in ``collect``."""
        items = []
        if densityAnalysis.BATCHED_CLOUD:
            from .cloudBatch import AtomTable, CloudBatch
            for k, e in enumerate(self.entries):
                an = e.analyzer
                if an._densityElectronRatio is not None:
                    continue
                table = AtomTable.fromStructure(an.biopdbObj, densityAnalysis.paramsGlobal)
                if table.supported:
                    self.cloudOf[k] = len(items)
                    items.append((an.densityObj, table))
            if items:
                self.cloud = CloudBatch(items, densityAnalysis.paramsGlobal, self.device)
                self.cloud.launch(25.0, 400.0)
        self.launchSums()

    def collect(self):
        """Synchronises; (ratio, (nGroups_k, 8) sums) of every entry."""
        arr = self.cloud.collectArrays() if self.cloud is not None else None
        torch.cuda.current_stream().synchronize()
        out = self.h_out.numpy()[:self.nGroups]
        res = []
        for k, e in enumerate(self.entries):
            j = self.cloudOf.get(k)
            if j is None:
                try:
                    ratio = e.analyzer.densityElectronRatio
                except Exception:
                    ratio = None                            # the single-structure call raises here too
            else:
                ratio = float(arr["ratio"][j]) if arr["ok"][j] and len(self.cloud.items[j][1]) else None
            res.append((ratio, out[self.groupBase[k]:self.groupBase[k + 1]].copy()))
        return res

    def run(self):
        self.launch()
        return self.collect()


def analyzeStream(pairs, kind, level, maxBytes=8 << 30, device=None, **options):
    """Yields (key, rows) for every (key, DensityAnalysis) of ``pairs``, in order: the rows of the single-structure call
    ``kind`` x ``level`` with ``options`` (``makeEntry``), or None for an analyzer that is missing (falsy) or on which that call
    would raise.  Analyzers are taken in batches of at most ``maxBytes`` device bytes (a larger entry forms a batch alone),
    so that only one batch of them is held at a time."""
    pending, used = [], 0                                   # (key, entry or None)

    def flush():
        entries = [e for _, e in pending if e is not None]
        results = iter(RegionBatch(entries, device).run() if entries else [])
        out = []
        for key, e in pending:
            rows = None
            if e is not None:
                ratio, sums = next(results)
                try:
                    rows = e.finish(ratio, sums)
                except Exception:
                    rows = None
            out.append((key, rows))
        pending.clear()
        return out

    for key, analyzer in pairs:
        entry = None
        if analyzer:
            try:
                entry = makeEntry(analyzer, kind, level, **options)
            except Exception:
                entry = None
        b = entry.deviceBytes() if entry is not None else 0
        if entry is not None and used and used + b > maxBytes:
            yield from flush()
            used = 0
        pending.append((key, entry))
        used += b
    yield from flush()


def analyzeRegions(analyzers, kind, level, maxBytes=8 << 30, device=None, **options):
    """``analyzeStream`` over a list: one list of rows (or None) per analyzer."""
    return [rows for _, rows in analyzeStream(enumerate(analyzers), kind, level, maxBytes, device, **options)]
