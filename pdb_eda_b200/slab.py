"""Slab-decomposed blob labelling of one very large map across GPUs (BASELINE.json config 4: 1024^3 Fo-Fc).

The reference holds a whole map in one process and clusters with an N x N distance matrix
(pdb_eda/ccp4.py:123-124, :337-338; pdb_eda/cutils.pyx:55), so it cannot run such maps at all.  Here the section axis
(the slowest-varying axis in memory, pdb_eda/ccp4.py:338) is cut into one slab per rank:

  1. every rank labels its slab with the same fused threshold + CCL kernels as a whole map (``pe_blob_label``);
  2. ``pe_slab_boundary`` packs one exchange buffer per rank (blob counts, every local blob's smallest whole-map key, the
     voxels of the slab's first and last section) and ONE ``all_gather`` moves them over NVLink -- the halo exchange;
  3. ``pe_slab_merge`` (every rank, redundantly): 26-adjacency across each cut, union-find over all ranks' blobs, and the
     whole-map number of each local blob by binary searches in the gathered key arrays -- the reference's blob order
     (pdb_eda/cutils.pyx:59-69, SURVEY.md App. A.5) without a global sort;
  4. ``pe_slab_relabel`` rewrites the labels and accumulates the per-blob sums (DensityBlob.fromCrsList,
     pdb_eda/ccp4.py:522-545) with the whole map's geometry; ONE ``all_reduce`` completes them.

Two collectives and one host synchronisation (to size the all-reduce) per call: ``SlabLabeller``.  The exchange buffers'
layout follows the capacities, so these are per decomposition (``slabCapacities`` of the largest slab), never per slab.
``labelSlabsEmulated`` runs all "ranks" one after another on a single GPU through the same kernels (no kernel ever waits
on another), which is how the merge is verified against the whole-map labelling on one device.
``mergeBlobIds`` / ``mergeDistributed`` state the same merge in device-agnostic torch with ragged all-gathers: the gloo
tests on CPU run them, and they are what the CUDA merge replaced (5 collectives, 3 host round trips).
"""
import ctypes

import numpy as np
import torch
import torch.distributed as dist

from . import _device
from . import cutils as utils
from ._device import _ptr, _stream
from ._lib import PeGeom, check


def slabRanges(nSections, world):
    """[s0, s1) of every rank: contiguous, as equal as possible."""
    base, extra = divmod(nSections, world)
    out, s = [], 0
    for r in range(world):
        n = base + (1 if r < extra else 0)
        out.append((s, s + n))
        s += n
    return out


def checkRanges(ranges, nSections):
    """Rejects a decomposition that is not contiguous, non-empty [s0, s1) slabs covering [0, nSections) in order."""
    ranges = [(int(s0), int(s1)) for s0, s1 in ranges]
    if not ranges:
        raise ValueError("slab ranges: no slab")
    at = 0
    for s0, s1 in ranges:
        if s0 != at:
            raise ValueError("slab ranges %s: [%d, %d) does not start where the previous slab ends (%d)" % (ranges, s0, s1, at))
        if s1 <= s0:
            raise ValueError("slab ranges %s: [%d, %d) is empty" % (ranges, s0, s1))
        at = s1
    if at != nSections:
        raise ValueError("slab ranges %s: cover [0, %d), the map has %d sections" % (ranges, at, nSections))
    return ranges


def coveredSections(s0, s1, u2):
    """Sections of the slab [s0, s1) inside the unique volume (0 when it lies entirely in the repeated part of the map)."""
    return max(min(int(s1), int(u2)) - int(s0), 0)


def slabCapacities(u0, u1, maxCovered, capVoxels=None, capBlobs=None, capPlane=None):
    """(capVoxels, capBlobs, capPlane) of one decomposition: the explicit values where given, else a function of the plane
    size and the LARGEST slab's covered sections only.  The exchange buffer layout and ``pe_slab_merge``'s reading of the
    gathered buffers follow capBlobs and capPlane, so they must be equal on every rank; sizing them from each rank's own
    slab breaks that whenever slabs cover different numbers of sections (uneven splits, over-sampled maps)."""
    capVoxels = int(capVoxels or max(4096, u0 * u1 * max(int(maxCovered), 1) // 64))
    return capVoxels, int(capBlobs or max(1024, capVoxels // 4)), int(capPlane or max(4096, u0 * u1 // 16))


def agreedCapacities(u0, u1, covered, world=1, group=None, device=None, capVoxels=None, capBlobs=None, capPlane=None):
    """``slabCapacities`` of the decomposition as one rank sees it (``covered``: its own slab's covered sections).  With
    ``world > 1`` and no ``capVoxels``, one all_reduce(MAX) over ``group`` (a tensor on ``device``) finds the largest slab."""
    maxCovered = int(covered)
    if int(world) > 1 and not capVoxels:
        t = torch.tensor([maxCovered], dtype=torch.int64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        maxCovered = int(t.item())
    return slabCapacities(u0, u1, maxCovered, capVoxels, capBlobs, capPlane)


def _slabGeom(full, s0, s1):
    """Geometry of the slab [s0, s1) as a map of its own: same columns / rows, its own section count."""
    g = PeGeom.from_buffer_copy(bytes(full))
    u2 = full.unique_ncrs[2]
    g.ncrs[2] = s1 - s0
    g.unique_ncrs[2] = max(min(s1, u2) - s0, 1)
    return g


def boundaryPairs(lastPlane, firstPlaneNext, offsetHere, offsetNext):
    """Equivalences across one cut: blobs of this slab's last plane that are 26-adjacent to blobs of the next slab's
    first plane.  Planes are (column, row, local blob) lists; returns (m, 2) global blob ids.  CUDA (pe_overlap_pairs)."""
    if len(lastPlane) == 0 or len(firstPlaneNext) == 0:
        return torch.zeros((0, 2), dtype=torch.int64, device=lastPlane.device)
    crs = torch.cat((torch.cat((lastPlane[:, :2], torch.zeros_like(lastPlane[:, :1])), dim=1),
                     torch.cat((firstPlaneNext[:, :2], torch.ones_like(firstPlaneNext[:, :1])), dim=1))).to(torch.int32)
    owner = torch.cat((lastPlane[:, 2] + offsetHere, firstPlaneNext[:, 2] + offsetNext)).to(torch.int32)
    pairs = utils.overlapPairs(crs, owner, None, device=crs.device)
    return torch.from_numpy(pairs.astype(np.int64)).to(lastPlane.device)


def mergeBlobIds(nTotal, pairs, minKeys):
    """Min-id union of the blob ids joined by ``pairs`` and the reference's numbering of the merged blobs.
    Returns (new blob number of every old id, number of merged blobs).  Pure torch; runs on any device."""
    dev = minKeys.device
    root = torch.arange(nTotal, dtype=torch.int64, device=dev)
    if len(pairs):
        a, b = pairs[:, 0], pairs[:, 1]
        while True:
            m = torch.minimum(root[a], root[b])
            new = root.clone()
            new.scatter_reduce_(0, a, m, reduce="amin")
            new.scatter_reduce_(0, b, m, reduce="amin")
            new = new[new]                                   # pointer jumping
            if torch.equal(new, root):
                break
            root = new
    compKey = torch.full((nTotal,), torch.iinfo(torch.int64).max, dtype=torch.int64, device=dev)
    if nTotal:
        compKey.scatter_reduce_(0, root, minKeys, reduce="amin")
    isRoot = root == torch.arange(nTotal, device=dev)
    roots = torch.nonzero(isRoot)[:, 0]
    order = torch.argsort(compKey[roots], stable=True)       # blobs in the order of their smallest canonical key
    number = torch.empty(nTotal, dtype=torch.int64, device=dev)
    number[roots[order]] = torch.arange(len(roots), device=dev)
    return number[root], int(len(roots))


def _allGatherRagged(t, group):
    """all_gather of tensors whose first dimension differs per rank (pad to the maximum, trim after)."""
    world = dist.get_world_size(group)
    n = torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device)
    sizes = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(sizes, n, group=group)
    sizes = [int(s.item()) for s in sizes]
    cap = max(max(sizes), 1)
    pad = torch.zeros((cap,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    pad[:t.shape[0]] = t
    out = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(out, pad, group=group)
    return [o[:s] for o, s in zip(out, sizes)]


def mergeDistributed(nLocalBlobs, firstPlane, lastPlane, minKeys, pairFn=boundaryPairs, group=None):
    """Steps 2-3 for one sign on this rank.  ``firstPlane`` / ``lastPlane``: (column, row, local blob) of this slab's
    boundary sections; ``minKeys``: smallest canonical key per local blob.  Returns (new number of every local blob,
    total number of merged blobs)."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    counts = _allGatherRagged(torch.tensor([[nLocalBlobs]], dtype=torch.int64, device=minKeys.device), group)
    counts = [int(c[0, 0].item()) for c in counts]
    offsets = np.concatenate(([0], np.cumsum(counts)))
    firsts = _allGatherRagged(firstPlane, group)             # the halo exchange: one boundary plane per slab
    if rank + 1 < world:
        pairs = pairFn(lastPlane, firsts[rank + 1], int(offsets[rank]), int(offsets[rank + 1]))
    else:
        pairs = torch.zeros((0, 2), dtype=torch.int64, device=minKeys.device)
    allPairs = torch.cat(_allGatherRagged(pairs, group))
    allKeys = torch.cat(_allGatherRagged(minKeys, group))
    number, nMerged = mergeBlobIds(int(offsets[-1]), allPairs, allKeys)
    return number[int(offsets[rank]):int(offsets[rank + 1])], nMerged


class SlabLabeller:
    """One rank's side of the slab-decomposed labelling with every buffer pre-allocated; ``label`` can be called repeatedly
    (e.g. on the slabs of successive maps of one geometry) without allocating.

    ``fullHeader``: the whole map's DensityHeader; [s0, s1): this rank's sections; ``world`` / ``rank`` / ``group``: the
    ranks that hold the slabs in section order (``group=None``: the default process group; ``world == 1`` needs none).

    Capacities are per decomposition, not per slab: by default ``slabCapacities`` of the largest slab, which the ranks agree
    on with one all-reduce here (``world > 1`` and no ``capVoxels``).  Explicit ``capVoxels`` / ``capBlobs`` / ``capPlane``
    must be the same on every rank; ``pe_slab_merge`` flags buffers packed with other capacities and ``label`` raises."""

    def __init__(self, fullHeader, s0, s1, world=1, rank=0, device=None, origin=None, group=None, capVoxels=None, capBlobs=None,
                 capPlane=None):
        from ._lib import load
        self.lib = load()
        _device.require_cuda()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.world, self.rank, self.group = int(world), int(rank), group
        self.s0, self.s1 = int(s0), int(s1)
        self.geom = _device.geom_from_header(fullHeader, origin)
        U = (self.geom.unique_ncrs[0], self.geom.unique_ncrs[1], self.geom.unique_ncrs[2])
        self.U = U
        if not 0 <= self.s0 < self.s1 <= self.geom.ncrs[2]:
            raise ValueError("slab [%d, %d) of a map of %d sections" % (self.s0, self.s1, self.geom.ncrs[2]))
        self.covered = coveredSections(self.s0, self.s1, U[2])
        self.slabGeom = _slabGeom(self.geom, self.s0, self.s1)
        self.capVoxels, self.capBlobs, self.capPlane = agreedCapacities(U[0], U[1], self.covered, self.world, group, self.device,
                                                                        capVoxels, capBlobs, capPlane)
        self.capMerged = self.capBlobs * self.world
        dev = self.device
        self.counts = torch.zeros(5, dtype=torch.int64, device=dev)
        self.key = torch.empty(2 * self.capVoxels, dtype=torch.int32, device=dev)
        self.value = torch.empty(2 * self.capVoxels, dtype=torch.float32, device=dev)
        self.labelBuf = torch.empty(2 * self.capVoxels, dtype=torch.int32, device=dev)
        self.localStats = torch.empty((2 * self.capBlobs, 8), dtype=torch.float64, device=dev)
        self.blobWs = torch.empty(max(int(self.lib.pe_blob_workspace_bytes(ctypes.byref(self.slabGeom), self.capVoxels)), 256),
                                  dtype=torch.uint8, device=dev)
        self.exchange = torch.zeros(int(self.lib.pe_slab_exchange_bytes(self.capBlobs, self.capPlane)), dtype=torch.uint8, device=dev)
        self.gathered = torch.zeros(self.world * self.exchange.numel(), dtype=torch.uint8, device=dev) if self.world > 1 else self.exchange
        self.mergeWs = torch.empty(int(self.lib.pe_slab_workspace_bytes(self.world, self.capBlobs, U[0], U[1])), dtype=torch.uint8,
                                   device=dev)
        self.newNumber = torch.zeros(2 * self.capBlobs, dtype=torch.int32, device=dev)
        self.tail = torch.zeros(8, dtype=torch.int64, device=dev)    # [0:2] blobs of the whole map per sign
        self.stats = torch.empty((2, self.capMerged, 8), dtype=torch.float64, device=dev)
        self.hostTail = torch.zeros(13, dtype=torch.int64).pin_memory()

    # ---- the stages; each only enqueues on torch's current stream ------------------------------------------------------
    def _labelLocal(self, rhoSlab, cutPos, cutNeg):
        if self.covered <= 0:                                        # the slab lies entirely in the repeated part of the map
            self.counts.zero_()
            return
        rho = rhoSlab.reshape(-1)
        check(self.lib.pe_blob_label(ctypes.byref(self.slabGeom), _ptr(rho), ctypes.c_float(float(np.float32(cutPos))),
                                     ctypes.c_float(float(np.float32(cutNeg))), self.capVoxels, self.capBlobs, _ptr(self.counts),
                                     _ptr(self.key), _ptr(self.value), _ptr(self.labelBuf), _ptr(self.localStats), _ptr(self.blobWs),
                                     _stream()), "pe_blob_label")

    def _boundary(self):
        lastIsCut = 1 if (self.rank + 1 < self.world and self.s1 <= self.U[2]) else 0
        check(self.lib.pe_slab_boundary(ctypes.byref(self.slabGeom), self.U[2], self.s0, lastIsCut, _ptr(self.counts), self.capVoxels,
                                        _ptr(self.key), _ptr(self.labelBuf), self.capBlobs, self.capPlane, _ptr(self.exchange),
                                        _ptr(self.mergeWs), _stream()), "pe_slab_boundary")

    def _mergeAndRelabel(self, gathered):
        check(self.lib.pe_slab_merge(self.world, self.rank, _ptr(gathered), self.capBlobs, self.capPlane, self.U[0], self.U[1],
                                     _ptr(self.newNumber), _ptr(self.tail), _ptr(self.mergeWs), _stream()), "pe_slab_merge")
        check(self.lib.pe_slab_relabel(ctypes.byref(self.geom), max(self.covered, 1), self.s0, _ptr(self.counts), self.capVoxels,
                                       _ptr(self.key), _ptr(self.value), _ptr(self.labelBuf), self.capBlobs, _ptr(self.newNumber),
                                       _ptr(self.tail), self.capMerged, _ptr(self.stats), _ptr(self.mergeWs), _stream()),
              "pe_slab_relabel")

    def _readCounts(self):
        """The one host synchronisation: voxel / blob counts of this slab, blobs of the whole map, overflow flags."""
        self.hostTail[:5].copy_(self.counts, non_blocking=True)
        self.hostTail[5:13].copy_(self.tail, non_blocking=True)
        bad = ctypes.c_int32(0)
        check(self.lib.pe_slab_status(_ptr(self.mergeWs), _stream(), ctypes.byref(bad)), "pe_slab_status")
        c = self.hostTail.tolist()
        if c[4] or bad.value:
            raise RuntimeError("slab labelling: a capacity was exceeded here or on another rank, or the ranks' capacities differ "
                               "(voxels %d / %d of %d, blobs %d / %d of %d, plane %d)"
                               % (c[0], c[2], self.capVoxels, c[1], c[3], self.capBlobs, self.capPlane))
        return c

    def _result(self, c, stats):
        U, out = self.U, []
        uslab = max(self.covered, 1)
        for k in range(2):
            nfg, nMerged = int(c[2 * k]), int(c[5 + k])
            v0 = k * self.capVoxels
            kk = self.key[v0:v0 + nfg].long() & 0xFFFFFFFF
            colrow = kk // uslab
            crs = torch.stack((colrow // U[1], colrow % U[1], kk % uslab + self.s0), dim=1)
            out.append({"crs": crs, "value": self.value[v0:v0 + nfg], "label": self.labelBuf[v0:v0 + nfg].long(), "n_blobs": nMerged,
                        "stats": stats[k][:nMerged]})
        return out

    def label(self, rhoSlab, cutPos, cutNeg):
        """Labels this rank's slab (``rhoSlab``: float32 CUDA tensor of its sections) and merges across the ranks.  Returns per
        sign a dict with this rank's voxels (global crs, value, whole-map blob number) and the all-reduced per-blob sums."""
        self._labelLocal(rhoSlab, cutPos, cutNeg)
        self._boundary()
        if self.world > 1:
            dist.all_gather_into_tensor(self.gathered, self.exchange, group=self.group)      # the halo exchange
        self._mergeAndRelabel(self.gathered)
        c = self._readCounts()
        n0, n1 = int(c[5]), int(c[6])
        if self.world > 1:
            packed = torch.cat((self.stats[0, :n0], self.stats[1, :n1]))
            dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=self.group)
            stats = (packed[:n0], packed[n0:])
        else:
            stats = (self.stats[0], self.stats[1])
        return self._result(c, stats)


_labellers = {}


def labelSlabDistributed(fullHeader, rhoSlab, s0, s1, cutPos, cutNeg, origin=None, group=None):
    """One rank's call: label this rank's slab [s0, s1) of the map and merge across ranks (a cached ``SlabLabeller`` per
    geometry: the ranks agree on its capacities once, when a geometry is new).  Returns per sign a dict with this rank's
    voxels (global crs, value, global blob number) and the all-reduced per-blob statistics."""
    rank, world = (dist.get_rank(group), dist.get_world_size(group)) if dist.is_initialized() else (0, 1)
    keyOf = (tuple(fullHeader.ncrs), tuple(fullHeader.crsStart), tuple(fullHeader.xyzInterval), int(s0), int(s1), world, rank,
             rhoSlab.device.index, id(group))
    lab = _labellers.get(keyOf)
    if lab is None:
        _labellers.clear()                       # one geometry at a time: the buffers of a 1024^3 slab are large
        lab = _labellers[keyOf] = SlabLabeller(fullHeader, s0, s1, world, rank, rhoSlab.device, origin, group)
    return lab.label(rhoSlab, cutPos, cutNeg)


def labelSlabsEmulated(fullHeader, rho, world, cutPos, cutNeg, origin=None, ranges=None, capVoxels=None, capBlobs=None,
                       capPlane=None):
    """All ranks of ``SlabLabeller.label`` executed one after another on ONE GPU (``rho``: the whole map on the device) through
    the same kernels; the exchange buffers are concatenated instead of all-gathered and the partial sums added instead of
    all-reduced.  ``ranges``: the slabs [s0, s1) (default ``slabRanges(ns, world)``; ``world`` may then be None); capacities
    as in ``SlabLabeller``, the same for every slab.  Returns per sign the complete voxel list in canonical order with
    whole-map blob numbers and statistics."""
    geom = _device.geom_from_header(fullHeader, origin)
    ns, nr, nc = geom.ncrs[2], geom.ncrs[1], geom.ncrs[0]
    if ranges is None:
        ranges = slabRanges(ns, world)
    elif world is not None and int(world) != len(ranges):
        raise ValueError("slab ranges: %d slabs for world %d" % (len(ranges), world))
    ranges = checkRanges(ranges, ns)
    world = len(ranges)
    vol = rho.reshape(ns, nr, nc)
    U = geom.unique_ncrs
    caps = slabCapacities(U[0], U[1], max(coveredSections(s0, s1, U[2]) for s0, s1 in ranges), capVoxels, capBlobs, capPlane)
    labs = [SlabLabeller(fullHeader, s0, s1, world, r, rho.device, origin, None, *caps) for r, (s0, s1) in enumerate(ranges)]
    for lab, (s0, s1) in zip(labs, ranges):
        lab._labelLocal(vol[s0:s1].contiguous(), cutPos, cutNeg)
        lab._boundary()
    gathered = torch.cat([lab.exchange for lab in labs]) if world > 1 else labs[0].exchange
    parts, total = [], None
    for lab in labs:
        lab._mergeAndRelabel(gathered)
        c = lab._readCounts()
        stats = lab.stats[:, :max(int(c[5]), int(c[6]), 1)].clone()
        total = stats if total is None else total + stats
        parts.append((lab, c))
    out = []
    U = labs[0].U
    for k in range(2):
        res = [lab._result(c, (total[0], total[1]))[k] for lab, c in parts]
        crs = torch.cat([r["crs"] for r in res])
        value = torch.cat([r["value"] for r in res])
        label = torch.cat([r["label"] for r in res])
        key = (crs[:, 0] * U[1] + crs[:, 1]) * U[2] + crs[:, 2]
        order = torch.argsort(key)
        nLocal = sum(int(c[2 * k + 1]) for _, c in parts)
        out.append({"crs": crs[order], "value": value[order], "label": label[order], "n_blobs": res[0]["n_blobs"],
                    "stats": res[0]["stats"], "n_pairs": nLocal - res[0]["n_blobs"]})
    return out
