"""Real-space correlation (RSCC) and R factor (RSR) per residue or per atom -- ``statistics --residue`` / ``--atom`` -- of one
structure or of a batch of structures.

``residueEntry`` / ``atomEntry`` state what ``DensityAnalysis.residueMetrics`` / ``atomMetrics``
(pdb_eda/densityAnalysis.py:803-858) select and return: the groups (residues, or single atoms), the metrics radius and the
columns besides RSCC / RSR.  ``MetricsBatch`` lays the entries of one or MANY structures out with their groups across
structures (``groupBatch``); both maps of every structure stay where they are in HBM (only pointers are gathered into one
``pe_pair_map`` table), and one launch of ``pe_pair_union_metrics`` (csrc/pe_metrics.cu) yields the eight sums of every
group in a fixed summation order.  The single-structure calls run a batch of one; the rows are built with numpy.
"""
import numpy as np
import torch

from . import groupBatch
from ._device import _ptr, _stream
from ._lib import PePairMap, check

LEVELS = ("residue", "atom")


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
    """One structure of a batch: its two device maps, its atoms (float64 coordinates) grouped in CSR form, the metrics radius,
    and what the rows need besides RSCC / RSR (``finish``)."""

    def __init__(self, foMap, diffMap, xyz, groupStart, radius, finish=None):
        if foMap.rho.numel() != diffMap.rho.numel():
            raise ValueError("the 2Fo-Fc and Fo-Fc maps must share one grid")
        self.foMap, self.diffMap = foMap, diffMap
        self.xyz = np.ascontiguousarray(np.asarray(xyz, dtype=np.float64).reshape(-1, 3))
        self.radius = np.full(len(self.xyz), radius, dtype=np.float32)
        self.groupStart = np.asarray(groupStart, dtype=np.int64)
        self.finish = finish

    @property
    def nGroups(self):
        return len(self.groupStart) - 1

    def deviceBytes(self):
        """Bytes this entry holds on the device in a batch: both maps, the atom arrays and the output rows."""
        return 4 * (self.foMap.rho.numel() + self.diffMap.rho.numel()) + len(self.xyz) * (24 + 4 + 32) + self.nGroups * (64 + 8)


class MetricsBatch(groupBatch.GroupBatch):
    """A batch of ``MetricsEntry`` laid out for one ``pe_pair_union_metrics`` launch."""

    def __init__(self, entries, device=None):
        entries = list(entries)
        maps = (PePairMap * max(len(entries), 1))()
        for m, e in zip(maps, entries):
            m.geom, m.d_fo, m.d_diff = e.foMap.geom, e.foMap.rho.data_ptr(), e.diffMap.rho.data_ptr()
        super().__init__(entries, maps, device)
        self.ws = torch.empty(int(self.lib.pe_pair_union_workspace_bytes(self.nAtoms)), dtype=torch.uint8, device=self.device)

    def launch(self):
        """Enqueues the sums of every group and the copy of the result rows to pinned memory."""
        check(self.lib.pe_pair_union_metrics(len(self.entries), _ptr(self.d_maps), self.nGroups, _ptr(self.d_groupMap),
                                             _ptr(self.d_groupStart), _ptr(self.d_xyz), _ptr(self.d_radius), _ptr(self.d_out),
                                             _ptr(self.ws), _stream()), "pe_pair_union_metrics")
        self.h_out.copy_(self.d_out, non_blocking=True)


def entryRows(entry, device=None):
    """The rows of one entry: a batch of one, none without groups."""
    if not entry.nGroups:
        return []
    sums, = MetricsBatch([entry], device).run()
    return entry.finish(*rsccRsr(sums))


# ---------------------------------------------------------------------------------------------------- entries of analyzers
def residueEntry(analyzer, residueList=None):
    """``residueMetrics(residueList)`` of a DensityAnalysis as a batch entry: every residue (default: of ``get_residues()``)
    with all its atoms.  Raises where ``residueMetrics()`` raises (no resolution, a residue whose occupancies sum to 0, maps
    on different grids)."""
    radius = metricsRadius(analyzer.biopdbObj.header['resolution'])
    if residueList is None:
        residueList = analyzer.biopdbObj.get_residues()
    labels, counts, coords, occ, bf = [], [], [], [], []
    for residue in residueList:
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
    return MetricsEntry(analyzer.densityObj.deviceMap, analyzer.diffDensityObj.deviceMap, np.asarray(coords, dtype=np.float64),
                        groupStart, radius, finish)


def atomEntry(analyzer, atomList=None):
    """``atomMetrics(atomList)`` of a DensityAnalysis as a batch entry: one group per atom (default: of ``asymmetryAtoms``,
    symmetry (0,0,0,0); none when the entry has no REMARK 290 operator).  The coordinates stay float64: symmetry images
    need not be float32 values."""
    radius = metricsRadius(analyzer.biopdbObj.header['resolution'])
    atoms = analyzer.asymmetryAtoms if atomList is None else atomList
    coords = np.asarray([atom.coord for atom in atoms], dtype=np.float64).reshape(-1, 3)

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
    """``groupBatch.stream`` of ``residueMetrics()`` / ``atomMetrics()`` (``level`` "residue" / "atom"): (key, rows or None)
    for every (key, DensityAnalysis) of ``pairs``, in order; None where the single-structure call would raise."""
    return groupBatch.stream(pairs, lambda analyzer: makeEntry(analyzer, level),
                             lambda entries: [rsccRsr(sums) for sums in MetricsBatch(entries, device).run()], maxBytes)


def analyzeMetrics(analyzers, level, maxBytes=8 << 30, device=None):
    """``analyzeStream`` over a list: one list of rows (or None) per analyzer."""
    return [rows for _, rows in analyzeStream(enumerate(analyzers), level, maxBytes, device)]
