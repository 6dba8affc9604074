"""Allocation-free batched pass of the voxel path over one structure.

One :class:`VoxelPass` holds every device buffer a structure needs (atoms, radii, residue offsets, outputs,
workspaces) and enqueues, without host synchronisation, the three voxel workloads the reference runs per structure:

  cloud    per-atom sphere gather-sums at the atom-type radii with the 2Fo-Fc cutoff
           (findAberrantBlobs per atom, pdb_eda/densityAnalysis.py:605)
  region   per-residue set-union sphere sums at a fixed radius (calculateResidueRegionDensity /
           calculateRegionDensity, pdb_eda/densityAnalysis.py:1001-1068)
  blobs    green + red blob lists of the Fo-Fc map in one pass (pdb_eda/densityAnalysis.py:392-412)

It is what ``bench.py`` times and what ``DensityAnalysis`` uses for its batched queries.
"""
import atexit
import ctypes
import os
import warnings

import numpy as np
import torch

from . import _device, _lib
from ._device import _ptr, _stream
from ._lib import PE_SPHERE_NOUT, check

# SMs the blob pass gets in VoxelPass.step, the other SMs running the sphere kernel (profiles/r05_partitioned_step.md);
# PDB_EDA_B200_BLOB_SMS overrides it, 0 shares all SMs between the two passes.
BLOB_SMS = 48
_partitions = {}   # (device index, blob SMs) -> (blob stream, sphere stream) of a live SM partition, or None where there is none


def blobSms():
    """The blob pass's SM count for VoxelPass.step: PDB_EDA_B200_BLOB_SMS when set, else BLOB_SMS."""
    text = os.environ.get("PDB_EDA_B200_BLOB_SMS")
    if text is None:
        return BLOB_SMS
    try:
        return int(text)
    except ValueError:
        return -1                                   # not a count: smPartition refuses it and says so once


def smPartition(device, blobSms):
    """(blob stream, sphere stream) of a partition of ``device`` into ``blobSms`` SMs and the rest (pe_sm_partition_create), as
    torch streams, made once per process, device and count; None for 0, and None with one warning when the count is not one the
    driver splits exactly or the driver has no green contexts."""
    index = device.index if device.index is not None else torch.cuda.current_device()
    key = (index, blobSms)
    if key in _partitions:
        return _partitions[key]
    part = None
    if blobSms != 0:
        lib = _lib.load()
        sb, sr, nb, nr = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_int32(), ctypes.c_int32()
        rc = lib.pe_sm_partition_create(index, blobSms, ctypes.byref(sb), ctypes.byref(sr), ctypes.byref(nb), ctypes.byref(nr))
        if rc == 0:
            dev = torch.device("cuda", index)
            part = (torch.cuda.ExternalStream(sb.value, device=dev), torch.cuda.ExternalStream(sr.value, device=dev))
        else:
            warnings.warn("VoxelPass.step: no partition of %d SMs for the blob pass on cuda:%d (%s); the blob and sphere passes "
                          "share the SMs" % (blobSms, index, lib.pe_last_error().decode("utf-8", "replace")), RuntimeWarning, stacklevel=3)
    _partitions[key] = part
    return part


@atexit.register
def releasePartitions():
    """Destroys every SM partition made so far (their streams are synchronised first); the next step makes them again."""
    lib = _lib.load() if _partitions else None
    for key in list(_partitions):
        part = _partitions.pop(key)
        if part is not None:
            check(lib.pe_sm_partition_destroy(ctypes.c_void_p(part[0].cuda_stream), ctypes.c_void_p(part[1].cuda_stream)),
                  "pe_sm_partition_destroy")


class VoxelPass:
    def __init__(self, densityDev, diffDev, xyz, radii, residueStart, regionRadius=3.5, densityCutoff=None,
                 diffCutoff=None, capVoxels=None, capBlobs=None):
        self.dens = densityDev
        self.diff = diffDev
        dev = densityDev.device
        self.device = dev
        self.lib = densityDev.lib
        self.xyz = _device._as_dev(xyz, torch.float64, dev, (-1, 3))
        self.n_atoms = self.xyz.shape[0]
        self.radii = _device._as_dev(radii, torch.float32, dev, (-1,))
        self.max_radius = float(self.radii.max().item()) if self.n_atoms else 0.0
        self.region_radii = torch.full((self.n_atoms,), float(np.float32(regionRadius)), dtype=torch.float32, device=dev)
        self.res_start = _device._as_dev(residueStart, torch.int32, dev, (-1,))
        self.n_res = self.res_start.numel() - 1
        if densityCutoff is None:
            m, s = densityDev.mean_std()
            densityCutoff = m + 1.5 * s
        if diffCutoff is None:
            m, s = diffDev.mean_std()
            diffCutoff = m + 3.0 * s
        self.density_cut = float(np.float32(densityCutoff))
        self.diff_cut = float(np.float32(diffCutoff))
        self.cloud_out = torch.empty((self.n_atoms, PE_SPHERE_NOUT), dtype=torch.float64, device=dev)
        self.region_out = torch.empty((self.n_res, PE_SPHERE_NOUT), dtype=torch.float64, device=dev)
        self.sphere_ws = torch.empty(max(int(self.lib.pe_sphere_workspace_bytes(self.n_atoms)), 256), dtype=torch.uint8, device=dev)
        g = diffDev.geom
        nvox = g.unique_ncrs[0] * g.unique_ncrs[1] * g.unique_ncrs[2]
        self.n_blob_voxels = nvox
        self.cap_voxels = int(capVoxels or max(4096, nvox // 64))
        self.cap_blobs = int(capBlobs or max(1024, self.cap_voxels // 4))
        self.blob_counts = torch.zeros(5, dtype=torch.int64, device=dev)
        self.blob_key = torch.empty(2 * self.cap_voxels, dtype=torch.int32, device=dev)
        self.blob_value = torch.empty(2 * self.cap_voxels, dtype=torch.float32, device=dev)
        self.blob_label = torch.empty(2 * self.cap_voxels, dtype=torch.int32, device=dev)
        self.blob_stats = torch.empty((2 * self.cap_blobs, 8), dtype=torch.float64, device=dev)
        self.blob_ws = torch.empty(max(int(self.lib.pe_blob_workspace_bytes(ctypes.byref(g), self.cap_voxels)), 256),
                                   dtype=torch.uint8, device=dev)

    # ---- the workloads; each only enqueues kernels on torch's current stream -----------------------------------------
    def spheres(self):
        """The cloud and the region pass in one call (one kernel at the cloud pass's atom-type radii)."""
        check(self.lib.pe_sphere_sums_atoms_and_groups(
            ctypes.byref(self.dens.geom), _ptr(self.dens.rho), self.n_atoms, _ptr(self.xyz), _ptr(self.radii),
            ctypes.c_float(self.max_radius), _ptr(self.region_radii), self.n_res, _ptr(self.res_start),
            ctypes.c_float(self.density_cut), ctypes.c_float(0.0), _ptr(self.cloud_out), _ptr(self.region_out),
            _ptr(self.sphere_ws), _stream()), "pe_sphere_sums_atoms_and_groups")

    def blobs(self):
        check(self.lib.pe_blob_label(ctypes.byref(self.diff.geom), _ptr(self.diff.rho), ctypes.c_float(self.diff_cut),
                                     ctypes.c_float(-self.diff_cut), self.cap_voxels, self.cap_blobs, _ptr(self.blob_counts),
                                     _ptr(self.blob_key), _ptr(self.blob_value), _ptr(self.blob_label), _ptr(self.blob_stats),
                                     _ptr(self.blob_ws), _stream()), "pe_blob_label")

    def step(self):
        """One pass.  The blob pass reads only the Fo-Fc map and the sphere passes only the 2Fo-Fc map, so the two run on two
        streams forked from and joined back to torch's current stream by events.  Each kernel fills every SM it is given up to
        its occupancy, so on shared SMs the block scheduler runs them nearly one after the other; by default the blob pass
        therefore runs on its own partition of blobSms() SMs and the sphere kernel on the other SMs, each at its full per-SM
        occupancy (profiles/r05_partitioned_step.md).  With 0 SMs, or where no partition can be made, both share all SMs."""
        part = smPartition(self.device, blobSms())
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream(device=self.device)
            self._fork, self._join, self._join_rest = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
        main = torch.cuda.current_stream()
        self._fork.record(main)
        blob_stream = part[0] if part is not None else self._side
        blob_stream.wait_event(self._fork)
        with torch.cuda.stream(blob_stream):
            self.blobs()
        if part is not None:
            part[1].wait_event(self._fork)
            with torch.cuda.stream(part[1]):
                self.spheres()
            self._join_rest.record(part[1])
            main.wait_event(self._join_rest)
        else:
            self.spheres()
        self._join.record(blob_stream)
        main.wait_event(self._join)

    def stepFromHost(self, hostDensity, hostDiff, hostXyz=None):
        """One pass with HOST inputs (pinned float32 map payloads as read from the CCP4 files, optional float64 atom
        coordinates) and host results: the uploads run on a copy stream, the sphere passes start as soon as the 2Fo-Fc map
        has landed and overlap the upload of the Fo-Fc map, which the blob pass then waits for.  Returns ``results()``."""
        if getattr(self, "_copy", None) is None:
            self._copy = torch.cuda.Stream(device=self.device)
            self._ev = [torch.cuda.Event() for _ in range(3)]
        ev_free, ev_dens, ev_diff = self._ev
        main = torch.cuda.current_stream()
        ev_free.record(main)                       # the previous pass no longer reads the device maps
        self._copy.wait_event(ev_free)
        with torch.cuda.stream(self._copy):
            self.dens.rho.copy_(hostDensity.view(-1), non_blocking=True)
            if hostXyz is not None:
                self.xyz.copy_(hostXyz, non_blocking=True)
            ev_dens.record(self._copy)
            self.diff.rho.copy_(hostDiff.view(-1), non_blocking=True)
            ev_diff.record(self._copy)
        main.wait_event(ev_dens)
        self.spheres()
        main.wait_event(ev_diff)
        self.blobs()
        return self.results()

    # ---- results (synchronise) ----------------------------------------------------------------------------------------
    def _host_buffers(self):
        if getattr(self, "_h", None) is None:
            pin = lambda t: torch.empty(t.shape, dtype=t.dtype).pin_memory()
            self._h = {"cloud": pin(self.cloud_out), "region": pin(self.region_out), "counts": pin(self.blob_counts),
                       "key": pin(self.blob_key), "label": pin(self.blob_label), "stats": pin(self.blob_stats)}
        return self._h

    def results(self):
        """Device -> host read of everything one step produced: asynchronous copies into page-locked buffers, two
        synchronisations (the blob counts decide how much of the blob arrays is read)."""
        h = self._host_buffers()
        h["cloud"].copy_(self.cloud_out, non_blocking=True)
        h["region"].copy_(self.region_out, non_blocking=True)
        h["counts"].copy_(self.blob_counts, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        counts = h["counts"].numpy().copy()
        if counts[4]:
            raise RuntimeError("blob capacities too small: %s voxels / %s blobs needed" % (max(counts[0], counts[2]), max(counts[1], counts[3])))
        spans = []
        for k in range(2):
            nfg, nb = int(counts[2 * k]), int(counts[2 * k + 1])
            v0, b0 = k * self.cap_voxels, k * self.cap_blobs
            h["key"][v0:v0 + nfg].copy_(self.blob_key[v0:v0 + nfg], non_blocking=True)
            h["label"][v0:v0 + nfg].copy_(self.blob_label[v0:v0 + nfg], non_blocking=True)
            h["stats"][b0:b0 + nb].copy_(self.blob_stats[b0:b0 + nb], non_blocking=True)
            spans.append((v0, nfg, b0, nb))
        torch.cuda.current_stream().synchronize()
        out = {"cloud": h["cloud"].numpy(), "region": h["region"].numpy(), "blob_counts": counts}
        for (v0, nfg, b0, nb), tag in zip(spans, ("green", "red")):
            out[tag] = {"key": h["key"].numpy()[v0:v0 + nfg], "label": h["label"].numpy()[v0:v0 + nfg], "stats": h["stats"].numpy()[b0:b0 + nb]}
        return out

    def unit_counts(self):
        """(atom-sphere voxels of the cloud pass, of the region pass, blob-CCL voxels) of the last step."""
        cloud = float(self.cloud_out[:, 0].sum().item())
        region = float(self.region_out[:, 0].sum().item())
        return cloud, region, float(self.n_blob_voxels)
