"""Region density and region discrepancy per atom, residue or symmetry atom -- ``density`` / ``difference`` with ``--atom`` /
``--residue`` / ``--symmetry-atom`` -- of one structure or of a batch of structures.

``makeEntry`` states what the six ``DensityAnalysis.calculate*RegionDensity`` / ``calculate*RegionDiscrepancies`` calls
(pdb_eda/densityAnalysis.py:948-1211) select and return: the atoms or residues, the ``type`` filter and atom mask, the radii,
the cutoffs and the row prefixes; ``finish`` turns the sums of its groups into the rows, built with numpy.  Those calls run
their entry through one ``pe_sphere_sums`` launch.  ``RegionBatch`` runs the entries of MANY structures: their groups laid
out across structures (``groupBatch``), every structure's map where it is in HBM with its own cutoffs (only pointers are
gathered into one ``pe_sums_map`` table), the ratios of the batch from one ``CloudBatch``, and one launch of
``pe_batch_sphere_sums`` (csrc/pe_union.cu, csrc/pe_sphere.cu) for the sums of every group; every row of it is bit-identical
to the row ``pe_sphere_sums`` gives for that structure alone, so the rows equal those of the single-structure calls in
value, type and order.
"""
import numpy as np
import torch

from . import groupBatch
from ._device import _ptr, _stream
from ._lib import PE_SPHERE_NOUT, PeSumsMap, check

KINDS = ("density", "difference")
LEVELS = ("atom", "residue", "symmetry-atom")


def _f32(x):
    return float(np.float32(x))


def _meanOccupancy(atoms, cache):
    """np.mean of the atoms' occupancies (pdb_eda/densityAnalysis.py:1031), computed once per distinct occupancy tuple: most
    residues are all 1.0, and 8,000 np.mean calls on five-element lists cost more than the kernel that follows."""
    occupancies = tuple([atom.get_occupancy() for atom in atoms])
    mean = cache.get(occupancies)
    if mean is None:
        mean = cache[occupancies] = np.mean(occupancies)
    return mean


# ---------------------------------------------------------------------------------------------------- rows from sums
def densityRows(sums, ratio):
    """Region density rows of (n, 8) sums: [sum of rho > cutoff, / ratio] per group, as np.float64 scalars."""
    pos = np.asarray(sums, dtype=np.float64).reshape(-1, PE_SPHERE_NOUT)[:, 3]
    return [list(r) for r in zip(pos, pos / ratio)]


def discrepancyRows(sums, ratio, avgAbsVoxel):
    """Region discrepancy rows of (n, 8) sums: the ten values per group.  ``avgAbsVoxel``: getTotalAbsDensity(cutoff) /
    number of voxels.  The expected columns are Python floats (the reference's float times ``int(n)``), the others
    np.float64."""
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
                         _meanOccupancy(atoms, meanOf)])
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
class RegionBatch(groupBatch.GroupBatch):
    """A batch of ``RegionEntry`` laid out for one ``pe_batch_sphere_sums`` launch, plus one ``CloudBatch`` for the ratios of
    the entries that need one.  All entries are grouped, or none is."""

    def __init__(self, entries, device=None):
        entries = list(entries)
        maps = (PeSumsMap * max(len(entries), 1))()
        for m, e in zip(maps, entries):
            m.geom, m.d_rho = e.map.geom, e.map.rho.data_ptr()
            m.cut_pos, m.cut_neg = e.cutPos, e.cutNeg
        super().__init__(entries, maps, device)
        self.ws = torch.empty(max(int(self.lib.pe_batch_sphere_sums_workspace_bytes(self.nAtoms)), 256), dtype=torch.uint8,
                              device=self.device)
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
        from . import densityAnalysis
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
        sums = super().collect()
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
            res.append((ratio, sums[k]))
        return res


def analyzeStream(pairs, kind, level, maxBytes=8 << 30, device=None, **options):
    """``groupBatch.stream`` of the single-structure call ``kind`` x ``level`` with ``options`` (``makeEntry``): (key, rows or
    None) for every (key, DensityAnalysis) of ``pairs``, in order; None where that call would raise."""
    return groupBatch.stream(pairs, lambda analyzer: makeEntry(analyzer, kind, level, **options),
                             lambda entries: RegionBatch(entries, device).run(), maxBytes)


def analyzeRegions(analyzers, kind, level, maxBytes=8 << 30, device=None, **options):
    """``analyzeStream`` over a list: one list of rows (or None) per analyzer."""
    return [rows for _, rows in analyzeStream(enumerate(analyzers), kind, level, maxBytes, device, **options)]
