#!/usr/bin/env python3
"""Multi-GPU check, launched with torchrun (one rank per GPU, NCCL):
  (a) multiple-structures mode: synthetic structures sharded over the ranks, cumulative statistics all-reduced and
      rows all-gathered, compared on rank 0 with a single-process pass over all structures;
  (b) slab-decomposed blob labelling of one map across the ranks (halo exchange over NCCL), compared on every rank
      with the whole-map labelling;
  (c) the same on a non-cubic, permuted, shifted map whose section count splits into unequal slabs.
Prints DIST_CHECK_OK on success."""
import io
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pdb_eda_b200 import _device, ccp4, densityAnalysis, multi, slab, structure, synthetic  # noqa: E402


def make_item(i):
    n = (48, 56, 64)[i % 3]
    cell = (n * 0.5,) * 3 + (90.0, 90.0, 90.0)
    st = synthetic.polyAlaStructure(40 + 6 * i, (0, 0, 0), cell[:3], seed=50 + i, residuesPerChain=30)
    a, b = synthetic.mapPair(st, (n, n, n), cell, seed=70 + i)
    text = structure.formatPDB(st, remark290=synthetic.cartesianOperators("P 21 21 21", cell), cell=cell, spaceGroup="P 21 21 21")
    return (text, synthetic.ccp4Bytes(a, cell, (n, n, n)), synthetic.ccp4Bytes(b, cell, (n, n, n)), n ** 3 * (40 + 6 * i))


def loader(item):
    if item is None:
        return 0                                   # a structure that fails to load
    return densityAnalysis.fromFile(io.StringIO(item[0]), io.BytesIO(item[1]), io.BytesIO(item[2]))


def main():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=device)
    densityAnalysis.setGlobals(synthetic.defaultParams())
    types = sorted(densityAnalysis.paramsGlobal["radii"])
    # ---- (a)
    items = [make_item(i) for i in range(7)]
    items.insert(3, None)
    costs = [it[3] if it else 1 for it in items]
    summary = multi.runMultipleStructures(items, loader, costs, types, device)
    if rank == 0:
        results = {i: multi.analyzeStructure(loader(it), types) for i, it in enumerate(items)}
        single = multi.gatherResults(results, list(range(len(items))), len(items), types, "cpu") if False else None
        cumulative, rows = multi._pack(results, list(range(len(items))), types)
        assert summary["cumulative"]["structures"] == 7 == int(cumulative[0])
        assert summary["cumulative"]["num_voxels_aggregated"] == cumulative[1]
        np.testing.assert_allclose(summary["cumulative"]["total_aggregated_density"], cumulative[3], rtol=1e-12)
        keep = [c for c in range(rows.shape[1]) if c != 1 + multi.STAT_COLUMNS.index("execution_time")]
        np.testing.assert_allclose(summary["rows"][:, keep], rows[:, keep], rtol=1e-12, atol=0)
        assert 3.0 not in summary["rows"][:, 0]
    # ---- (b)
    n = 192
    vol = synthetic.smoothNoiseMapDevice(n, seed=9, device=device)
    hdr = ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((n, n, n), (n * 0.5,) * 3 + (90, 90, 90), (n, n, n)))
    s0, s1 = slab.slabRanges(n, world)[rank]
    parts = slab.labelSlabDistributed(hdr, vol[s0:s1].contiguous(), s0, s1, 2.3, -2.3)
    whole = _device.DeviceMap(_device.geom_from_header(hdr), vol.reshape(-1)).blob_label(2.3, -2.3)
    for w, p in zip(whole, parts):
        sel = (w["crs"][:, 2] >= s0) & (w["crs"][:, 2] < s1)
        wc, wl = w["crs"][sel].long(), w["label"][sel].long()
        key = (p["crs"][:, 0] * n + p["crs"][:, 1]) * n + p["crs"][:, 2]
        order = torch.argsort(key)
        assert torch.equal(wc, p["crs"][order]) and torch.equal(wl, p["label"][order])
        assert w["n_blobs"] == p["n_blobs"]
        torch.testing.assert_close(p["stats"], w["stats"], rtol=1e-9, atol=1e-9)
    # ---- (c) a non-cubic, permuted, shifted map of 67 sections (a prime: every world > 1 gives unequal slabs), slabs above
    # the capacity floors, so the ranks must agree on one exchange layout
    import cases
    shape = (67, 120, 160)                                   # (sections, rows, columns)
    host = cases._noise(shape, 17)
    hdr2 = ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header(shape[::-1], (64.0, 40.0, 90.0, 90, 90, 90), (128, 80, 180),
                                                                  crsStart=(5, -7, 3), axisOrder=(3, 1, 2)))
    vol2 = torch.from_numpy(host).to(device)
    s0, s1 = slab.slabRanges(shape[0], world)[rank]
    parts2 = slab.labelSlabDistributed(hdr2, vol2[s0:s1].contiguous(), s0, s1, 2.5, -2.5)
    whole2 = _device.DeviceMap(_device.geom_from_header(hdr2), vol2.reshape(-1)).blob_label(2.5, -2.5)
    U = hdr2.uniqueNcrs
    for w, p in zip(whole2, parts2):
        sel = (w["crs"][:, 2] >= s0) & (w["crs"][:, 2] < s1)
        key = (p["crs"][:, 0] * U[1] + p["crs"][:, 1]) * U[2] + p["crs"][:, 2]
        order = torch.argsort(key)
        assert torch.equal(w["crs"][sel].long(), p["crs"][order]) and torch.equal(w["label"][sel].long(), p["label"][order])
        assert w["n_blobs"] == p["n_blobs"] > 100
        torch.testing.assert_close(p["stats"], w["stats"], rtol=1e-9, atol=1e-9)
    dist.barrier()
    if rank == 0:
        print("DIST_CHECK_OK world=%d structures=%d blobs=%d/%d" % (world, summary["cumulative"]["structures"], parts[0]["n_blobs"], parts[1]["n_blobs"]))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
