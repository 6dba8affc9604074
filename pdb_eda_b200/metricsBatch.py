"""Real-space correlation (RSCC) and R factor (RSR) per residue or per atom for a batch of structures -- ``statistics
--residue`` / ``--atom`` of many entries.

``DensityAnalysis.residueMetrics`` / ``atomMetrics`` (pdb_eda/densityAnalysis.py:803-858) analyse one structure through a
voxel-list chain (sphere lists -> grouped de-duplication -> two-pass sums).  Here the atoms of MANY structures are laid out
as one set of arrays with the groups (residues, or single atoms) in CSR form across structures, both maps of every
structure stay where they are in HBM (only pointers are gathered into one ``pe_pair_map`` table), and one launch of
``pe_pair_union_metrics`` (csrc/pe_metrics.cu) yields the eight sums of every group.  The rows are then built with numpy and
are the rows, in the order, that the single-structure calls return.
"""
import ctypes

import numpy as np
import torch

from . import _device
from . import _lib
from ._device import _ptr, _stream
from ._lib import PeGeom, check

LEVELS = ("residue", "atom")


class PePairMap(ctypes.Structure):
    """Mirror of ``struct pe_pair_map`` (include/pdbeda_b200.h)."""
    _fields_ = [("geom", PeGeom), ("d_fo", ctypes.c_void_p), ("d_diff", ctypes.c_void_p)]


def metricsRadius(resolution):
    """Sphere radius of the metrics from the resolution (pdb_eda/densityAnalysis.py:809-814)."""
    radius = 0.7
    if 0.6 <= resolution <= 3:
        radius = (resolution - 0.6) / 3 + 0.7
    elif resolution > 3:
        radius = resolution * 0.5
    return radius


def rsccRsr(sums):
    """(RSCC, RSR) per row of an (n, 8) array of pair sums (``pe_pair_metrics`` layout): RSCC clipped to [-1, 1], NaN where
    a denominator is 0 (pdb_eda/densityAnalysis.py:876-882)."""
    sums = np.asarray(sums, dtype=np.float64).reshape(-1, 8)
    with np.errstate(divide="ignore", invalid="ignore"):
        rscc = np.clip(sums[:, 7] / np.sqrt(sums[:, 5] * sums[:, 6]), -1.0, 1.0)
        rsr = sums[:, 3] / sums[:, 4]
    return rscc, rsr


class MetricsEntry:
    """One structure of a batch: its two device maps, its atoms (float32 coordinates) grouped in CSR form, the metrics radius,
    and what the rows need besides RSCC / RSR (``finish``)."""

    def __init__(self, foMap, diffMap, coords32, groupStart, radius, finish=None):
        if foMap.rho.numel() != diffMap.rho.numel():
            raise ValueError("the 2Fo-Fc and Fo-Fc maps must share one grid")
        self.foMap, self.diffMap = foMap, diffMap
        self.coords32 = np.ascontiguousarray(coords32, dtype=np.float32).reshape(-1, 3)
        self.groupStart = np.asarray(groupStart, dtype=np.int64)
        self.radius = radius
        self.finish = finish

    @property
    def nGroups(self):
        return len(self.groupStart) - 1

    def deviceBytes(self):
        """Bytes this entry holds on the device in a batch: both maps, the atom arrays and the output rows."""
        return 4 * (self.foMap.rho.numel() + self.diffMap.rho.numel()) + len(self.coords32) * (24 + 4 + 32) + self.nGroups * (64 + 8)


class MetricsBatch:
    """A batch of ``MetricsEntry`` laid out for one ``pe_pair_union_metrics`` launch."""

    def __init__(self, entries, device=None):
        self.entries = list(entries)
        self.lib = _lib.load()
        _device.require_cuda()
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        nS = len(self.entries)
        atomCounts = np.array([len(e.coords32) for e in self.entries], dtype=np.int64)
        groupCounts = np.array([e.nGroups for e in self.entries], dtype=np.int64)
        atomBase = np.concatenate(([0], np.cumsum(atomCounts)))
        self.groupBase = np.concatenate(([0], np.cumsum(groupCounts)))
        self.nAtoms, self.nGroups = int(atomBase[-1]), int(self.groupBase[-1])
        if self.nAtoms >= 2 ** 31 or self.nGroups >= 2 ** 31:
            raise ValueError("a batch holds fewer than 2^31 atoms and groups")
        xyz = np.concatenate([e.coords32 for e in self.entries]).astype(np.float64) if nS else np.zeros((0, 3))
        radius = np.repeat(np.array([np.float32(e.radius) for e in self.entries], dtype=np.float32), atomCounts)
        groupMap = np.repeat(np.arange(nS, dtype=np.int32), groupCounts)
        groupStart = np.empty(self.nGroups + 1, dtype=np.int32)
        groupStart[-1] = self.nAtoms
        maps = (PePairMap * max(nS, 1))()
        for k, e in enumerate(self.entries):
            groupStart[self.groupBase[k]:self.groupBase[k + 1]] = e.groupStart[:-1] + atomBase[k]
            maps[k].geom = e.foMap.geom
            maps[k].d_fo = e.foMap.rho.data_ptr()
            maps[k].d_diff = e.diffMap.rho.data_ptr()
        up = lambda arr: torch.from_numpy(np.ascontiguousarray(arr)).to(device)
        self.d_maps = torch.frombuffer(bytearray(bytes(maps)), dtype=torch.uint8).to(device)
        self.d_xyz = up(xyz.reshape(-1, 3) if self.nAtoms else np.zeros((1, 3)))
        self.d_radius = up(radius if self.nAtoms else np.zeros(1, dtype=np.float32))
        self.d_groupMap, self.d_groupStart = up(groupMap), up(groupStart)
        self.d_out = torch.empty((max(self.nGroups, 1), 8), dtype=torch.float64, device=device)
        self.h_out = torch.empty(self.d_out.shape, dtype=torch.float64).pin_memory()
        self.ws = torch.empty(int(self.lib.pe_pair_union_workspace_bytes(self.nAtoms)), dtype=torch.uint8, device=device)

    def launch(self):
        """Enqueues the sums of every group and the copy of the result rows to pinned memory."""
        check(self.lib.pe_pair_union_metrics(len(self.entries), _ptr(self.d_maps), self.nGroups, _ptr(self.d_groupMap),
                                             _ptr(self.d_groupStart), _ptr(self.d_xyz), _ptr(self.d_radius), _ptr(self.d_out),
                                             _ptr(self.ws), _stream()), "pe_pair_union_metrics")
        self.h_out.copy_(self.d_out, non_blocking=True)

    def collect(self):
        """Synchronises; the (nGroups_k, 8) sums of every entry."""
        torch.cuda.current_stream().synchronize()
        out = self.h_out.numpy()[:self.nGroups]
        return [out[self.groupBase[k]:self.groupBase[k + 1]].copy() for k in range(len(self.entries))]

    def run(self):
        self.launch()
        return self.collect()


# ---------------------------------------------------------------------------------------------------- entries of analyzers
def residueEntry(analyzer):
    """``residueMetrics()`` of a DensityAnalysis as a batch entry: every residue of ``get_residues()`` with all its atoms.
    Raises where ``residueMetrics()`` raises (no resolution, a residue whose occupancies sum to 0, maps on different grids)."""
    radius = metricsRadius(analyzer.biopdbObj.header['resolution'])
    labels, counts, coords, occ, bf = [], [], [], [], []
    for residue in analyzer.biopdbObj.get_residues():
        atoms = residue.child_list
        labels.append((residue.parent.id, residue.id[1], residue.resname))
        counts.append(len(atoms))
        for atom in atoms:
            coords.append(atom.coord)
            occ.append(atom.get_occupancy())
            bf.append(atom.get_bfactor())
    nRes = len(labels)
    group = np.repeat(np.arange(nRes), counts)
    occ, bf = np.asarray(occ, dtype=np.float64), np.asarray(bf, dtype=np.float64)
    if coords:
        occupancySum = np.bincount(group, weights=occ, minlength=nRes)            # in atom order, as the Python loop adds
        weighted = np.bincount(group, weights=bf * occ, minlength=nRes)
        if not np.all(occupancySum != 0):
            raise ZeroDivisionError("a residue's occupancies sum to 0")
        meanOccupancy = occupancySum / np.asarray(counts, dtype=np.float64)
        weightedB = weighted / occupancySum

    def finish(rscc, rsr):
        if not coords:
            return []                                                              # residueMetrics() of an entry without atoms
        return [[c, n, r, a, b, o, w] for (c, n, r), a, b, o, w in
                zip(labels, rscc.tolist(), rsr.tolist(), meanOccupancy.tolist(), weightedB.tolist())]

    groupStart = np.concatenate(([0], np.cumsum(counts))) if coords else np.zeros(1)   # no atoms: no groups
    return MetricsEntry(analyzer.densityObj.deviceMap, analyzer.diffDensityObj.deviceMap, np.asarray(coords, dtype=np.float32),
                        groupStart, radius, finish)


def atomEntry(analyzer):
    """``atomMetrics()`` of a DensityAnalysis as a batch entry: one group per atom of ``asymmetryAtoms`` (symmetry (0,0,0,0)),
    none when the entry has no REMARK 290 operator."""
    radius = metricsRadius(analyzer.biopdbObj.header['resolution'])
    atoms = analyzer.asymmetryAtoms
    coords = np.asarray([atom.coord for atom in atoms], dtype=np.float32).reshape(-1, 3)

    def finish(rscc, rsr):
        return [[atom.parent.parent.id, atom.parent.id[1], atom.parent.resname, atom.name, atom.symmetry, atom.coord, a, b,
                 atom.get_occupancy(), atom.get_bfactor()] for atom, a, b in zip(atoms, rscc.tolist(), rsr.tolist())]

    return MetricsEntry(analyzer.densityObj.deviceMap, analyzer.diffDensityObj.deviceMap, coords, np.arange(len(atoms) + 1), radius,
                        finish)


def makeEntry(analyzer, level):
    if level not in LEVELS:
        raise ValueError("level must be one of %s" % (LEVELS,))
    return residueEntry(analyzer) if level == "residue" else atomEntry(analyzer)


def analyzeStream(pairs, level, maxBytes=8 << 30, device=None):
    """Yields (key, rows) for every (key, DensityAnalysis) of ``pairs``, in order: the rows of ``residueMetrics()`` /
    ``atomMetrics()``, or None for an analyzer that is missing (falsy) or on which the single-structure call would raise.
    Analyzers are taken in batches of at most ``maxBytes`` device bytes (a larger entry forms a batch alone), so that only
    one batch of them is held at a time."""
    pending, used = [], 0                                   # (key, entry or None)

    def flush():
        entries = [e for _, e in pending if e is not None]
        sums = iter(MetricsBatch(entries, device).run() if entries else [])
        out = [(key, None if e is None else e.finish(*rsccRsr(next(sums)))) for key, e in pending]
        pending.clear()
        return out

    for key, analyzer in pairs:
        entry = None
        if analyzer:
            try:
                entry = makeEntry(analyzer, level)
            except Exception:
                entry = None
        b = entry.deviceBytes() if entry is not None else 0
        if entry is not None and used and used + b > maxBytes:
            yield from flush()
            used = 0
        pending.append((key, entry))
        used += b
    yield from flush()


def analyzeMetrics(analyzers, level, maxBytes=8 << 30, device=None):
    """``analyzeStream`` over a list: one list of rows (or None) per analyzer."""
    return [rows for _, rows in analyzeStream(enumerate(analyzers), level, maxBytes, device)]
