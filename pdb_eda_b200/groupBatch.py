"""Groups of atoms of many structures laid out for one batched launch, and the stream of such batches.

Region density / discrepancy (``regionBatch``, ``pe_batch_sphere_sums``) and RSCC / RSR (``metricsBatch``,
``pe_pair_union_metrics``) take the same input: per structure its atoms (float64 coordinates, float32 radii), its groups
(residues, or single atoms) in CSR form and a table entry that names its map(s) in HBM.  ``GroupBatch`` lays the entries of a
batch out as one set of arrays -- atoms and groups concatenated across structures, the owning structure of every group -- and
holds the (n, 8) float64 result rows of every group; ``stream`` takes many structures through such batches, bounded by
device bytes.
"""
import numpy as np
import torch

from . import _device
from . import _lib

NOUT = 8                                                    # float64 sums per group of both kernels


class GroupBatch:
    """The layout of a batch of entries.  Every entry provides ``xyz`` ((n, 3) float64), ``radius`` ((n,) float32),
    ``groupStart`` (CSR offsets into its atoms, or None: one group per atom) and ``nGroups``; ``maps`` is the ctypes table
    with one struct per entry (at least one element).  All entries are grouped, or none is.  A subclass allocates its
    workspace and enqueues its launch into ``d_out`` and the copy to ``h_out`` (``launch``)."""

    def __init__(self, entries, maps, device=None):
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
        up = lambda arr: torch.from_numpy(np.ascontiguousarray(arr)).to(device)
        self.d_maps = torch.frombuffer(bytearray(bytes(maps)), dtype=torch.uint8).to(device)
        self.d_xyz = up(np.concatenate([e.xyz for e in self.entries]) if self.nAtoms else np.zeros((1, 3)))
        self.d_radius = up(np.concatenate([e.radius for e in self.entries]) if self.nAtoms else np.zeros(1, dtype=np.float32))
        self.d_groupMap = up(np.repeat(np.arange(nS, dtype=np.int32), groupCounts) if self.nGroups else np.zeros(1, dtype=np.int32))
        self.d_atomStart = up(self.atomStart.astype(np.int32))
        self.d_groupStart = None
        if self.grouped:
            groupStart = np.empty(self.nGroups + 1, dtype=np.int32)
            groupStart[-1] = self.nAtoms
            for k, e in enumerate(self.entries):
                groupStart[self.groupBase[k]:self.groupBase[k + 1]] = e.groupStart[:-1] + self.atomStart[k]
            self.d_groupStart = up(groupStart)
        self.d_out = torch.empty((max(self.nGroups, 1), NOUT), dtype=torch.float64, device=device)
        self.h_out = torch.empty(self.d_out.shape, dtype=torch.float64).pin_memory()

    def collect(self):
        """Synchronises; the (nGroups_k, 8) sums of every entry."""
        torch.cuda.current_stream().synchronize()
        out = self.h_out.numpy()[:self.nGroups]
        return [out[self.groupBase[k]:self.groupBase[k + 1]].copy() for k in range(len(self.entries))]

    def run(self):
        self.launch()
        return self.collect()


def stream(pairs, makeEntry, runBatch, maxBytes):
    """Yields (key, rows) for every (key, analyzer) of ``pairs``, in order.  ``makeEntry(analyzer)`` builds an entry;
    ``runBatch(entries)`` returns, per entry, the arguments of its ``finish``, which returns the rows.  Rows are None for an
    analyzer that is missing (falsy) and where ``makeEntry`` or ``finish`` raises.  Entries are taken in batches of at most
    ``maxBytes`` device bytes (``entry.deviceBytes()``; a larger entry forms a batch alone), so that only one batch of them
    is held at a time."""
    pending, used = [], 0                                   # (key, entry or None)

    def flush():
        entries = [e for _, e in pending if e is not None]
        results = iter(runBatch(entries) if entries else [])
        out = []
        for key, e in pending:
            rows = None
            if e is not None:
                args = next(results)
                try:
                    rows = e.finish(*args)
                except Exception:
                    rows = None
            out.append((key, rows))
        pending.clear()
        return out

    for key, analyzer in pairs:
        entry = None
        if analyzer:
            try:
                entry = makeEntry(analyzer)
            except Exception:
                entry = None
        b = entry.deviceBytes() if entry is not None else 0
        if entry is not None and used and used + b > maxBytes:
            yield from flush()
            used = 0
        pending.append((key, entry))
        used += b
    yield from flush()
