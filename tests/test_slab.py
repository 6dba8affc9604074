"""Slab-decomposed blob labelling: CPU tier = the cross-rank merge over gloo (world_size 2 and 3) against a
single-process merge, the ranks' agreement on one set of capacities (gloo) and the host checks of slab ranges; GPU tier =
all slabs emulated on one GPU against the whole-map labelling (tests/test_slab_vs_host.py: against host references)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp


def _pairs_cpu(lastPlane, firstNext, offHere, offNext):
    """Device-agnostic stand-in for the CUDA pair finder: 26-adjacency across the cut = |dc| <= 1 and |dr| <= 1."""
    if len(lastPlane) == 0 or len(firstNext) == 0:
        return torch.zeros((0, 2), dtype=torch.int64)
    dc = (lastPlane[:, None, 0] - firstNext[None, :, 0]).abs() <= 1
    dr = (lastPlane[:, None, 1] - firstNext[None, :, 1]).abs() <= 1
    i, j = torch.nonzero(dc & dr, as_tuple=True)
    pairs = torch.stack((lastPlane[i, 2] + offHere, firstNext[j, 2] + offNext), dim=1)
    return torch.unique(pairs, dim=0)


def _toy(world, seed=3, n=24):
    """A random binary volume cut into slabs; per slab: scipy labels (local blobs in canonical order), planes, keys."""
    from scipy import ndimage
    from pdb_eda_b200 import slab
    rng = np.random.default_rng(seed)
    vol = ndimage.gaussian_filter(rng.standard_normal((n, n, n)), 1.2) > 0.12      # [s][r][c]
    out = []
    for s0, s1 in slab.slabRanges(n, world):
        lab, nb = ndimage.label(vol[s0:s1], np.ones((3, 3, 3)))
        s, r, c = np.nonzero(lab)
        key = (c * n + r) * n + (s + s0)
        order = np.argsort(key)
        s, r, c, key = s[order], r[order], c[order], key[order]
        raw = lab[s, r, c]
        first = {}
        for x in raw:                      # renumber blobs by first appearance in canonical order
            first.setdefault(int(x), len(first))
        local = np.array([first[int(x)] for x in raw], dtype=np.int64)
        out.append(dict(s0=s0, s1=s1, c=c, r=r, s=s + s0, key=key, label=local, n=nb))
    lab, nb = ndimage.label(vol, np.ones((3, 3, 3)))
    s, r, c = np.nonzero(lab)
    key = (c * n + r) * n + s
    order = np.argsort(key)
    raw = lab[s[order], r[order], c[order]]
    first = {}
    for x in raw:
        first.setdefault(int(x), len(first))
    truth = {int(k): first[int(x)] for k, x in zip(key[order], raw)}
    return out, truth, nb


def _rank_inputs(part):
    t = lambda a: torch.from_numpy(np.asarray(a, dtype=np.int64))
    sel0, sel1 = part["s"] == part["s0"], part["s"] == part["s1"] - 1
    first = torch.stack((t(part["c"][sel0]), t(part["r"][sel0]), t(part["label"][sel0])), dim=1)
    last = torch.stack((t(part["c"][sel1]), t(part["r"][sel1]), t(part["label"][sel1])), dim=1)
    minkeys = torch.full((part["n"],), torch.iinfo(torch.int64).max, dtype=torch.int64)
    minkeys.scatter_reduce_(0, t(part["label"]), t(part["key"]), reduce="amin")
    return first, last, minkeys


def _worker(rank, world, port, out):
    import torch.distributed as dist
    from pdb_eda_b200 import slab
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    parts, truth, nb = _toy(world)
    first, last, minkeys = _rank_inputs(parts[rank])
    number, merged = slab.mergeDistributed(parts[rank]["n"], first, last, minkeys, pairFn=_pairs_cpu)
    got = number[torch.from_numpy(parts[rank]["label"])].numpy()
    want = np.array([truth[int(k)] for k in parts[rank]["key"]])
    out[rank] = (bool(np.array_equal(got, want)), merged, nb)
    dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


@pytest.mark.timeout(180)
@pytest.mark.parametrize("world", [2, 3])
def test_merge_over_gloo(world):
    manager = mp.Manager()
    out = manager.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    for rank in range(world):
        ok, merged, nb = out[rank]
        assert ok and merged == nb


def test_merge_blob_ids_single_process():
    from pdb_eda_b200 import slab
    # ids 0..5; 1-4 and 4-5 joined; keys decide the numbering
    keys = torch.tensor([50, 40, 30, 20, 10, 60])
    number, n = slab.mergeBlobIds(6, torch.tensor([[1, 4], [4, 5]]), keys)
    assert n == 4 and number.tolist() == [3, 0, 2, 1, 0, 0]
    number, n = slab.mergeBlobIds(3, torch.zeros((0, 2), dtype=torch.int64), torch.tensor([3, 1, 2]))
    assert n == 3 and number.tolist() == [2, 0, 1]
    assert slab.slabRanges(10, 4) == [(0, 3), (3, 6), (6, 8), (8, 10)]


def _own_slab_rule(u0, u1, covered):
    """The capacities a slab would get if it were sized for itself (the rule, applied to one slab)."""
    capVoxels = max(4096, u0 * u1 * max(covered, 1) // 64)
    return capVoxels, max(1024, capVoxels // 4), max(4096, u0 * u1 // 16)


# (U0, U1, U2, stored sections, ranges): three ranks each
CAPACITY_LAYOUTS = {
    "1024^3": (1024, 1024, 1024, 1024, None),
    "1000^3": (1000, 1000, 1000, 1000, None),
    "over-sampled": (1024, 1024, 512, 600, None),                   # 200 / 200 / 112 covered sections
    "thin": (160, 120, 67, 67, [(0, 1), (1, 33), (33, 67)]),
    "beyond": (256, 192, 40, 67, [(0, 34), (34, 40), (40, 67)]),    # the last slab lies beyond the unique volume
}


def _capacity_worker(rank, world, port, out):
    import torch.distributed as dist
    from pdb_eda_b200 import _lib, slab
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lib = _lib.load()
    res = {}
    for name, (u0, u1, u2, ns, ranges) in CAPACITY_LAYOUTS.items():
        s0, s1 = (ranges or slab.slabRanges(ns, world))[rank]
        caps = slab.agreedCapacities(u0, u1, slab.coveredSections(s0, s1, u2), world, device="cpu")
        res[name] = caps + (int(lib.pe_slab_exchange_bytes(caps[1], caps[2])),)
    out[rank] = res
    dist.destroy_process_group()


@pytest.mark.timeout(180)
def test_every_rank_gets_the_same_capacities():
    """The ranks of uneven, thin, over-sampled and beyond-the-unique-volume decompositions agree (one all-reduce over gloo) on
    capacities and exchange bytes, those of the largest slab; sizing each slab for itself would give them different layouts."""
    from pdb_eda_b200 import _lib, slab
    world = 3
    manager = mp.Manager()
    out = manager.dict()
    mp.spawn(_capacity_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    lib = _lib.load()
    for name, (u0, u1, u2, ns, ranges) in CAPACITY_LAYOUTS.items():
        ranges = ranges or slab.slabRanges(ns, world)
        got = {out[r][name] for r in range(world)}
        assert len(got) == 1, (name, got)
        capVoxels, capBlobs, capPlane, nbytes = got.pop()
        own = [_own_slab_rule(u0, u1, slab.coveredSections(s0, s1, u2)) for s0, s1 in ranges]
        assert len({o[1] for o in own}) > 1, name                     # the case the agreement exists for
        assert (capVoxels, capBlobs, capPlane) == max(own)             # the largest slab's
        assert nbytes == lib.pe_slab_exchange_bytes(capBlobs, capPlane) >= max(lib.pe_slab_exchange_bytes(o[1], o[2]) for o in own)
    # the rule as a function: largest slab of slabRanges(1024, 6) and of an explicit override
    own = [_own_slab_rule(1024, 1024, s1 - s0) for s0, s1 in slab.slabRanges(1024, 6)]
    assert slab.slabCapacities(1024, 1024, 171) == max(own) and own[0][1] != own[-1][1]
    assert slab.slabCapacities(1024, 1024, 171, capVoxels=8192) == (8192, 2048, 65536)
    assert slab.agreedCapacities(160, 120, 0) == (4096, 1024, 4096)


def test_slab_ranges_are_checked_before_any_device_work():
    """A gap, an overlap, an empty slab, ranges that stop short or run past the map, more slabs than sections and a world that
    contradicts the ranges are rejected on the host (ValueError) before a labeller or a device buffer exists: the map here is
    a CPU tensor and there may be no GPU at all."""
    from pdb_eda_b200 import ccp4, slab, synthetic
    hdr = ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((20, 16, 12), (10.0, 8.0, 6.0, 90, 90, 90), (20, 16, 12)))
    rho = torch.zeros(20 * 16 * 12)
    for ranges in ([(0, 5), (6, 12)], [(0, 6), (5, 12)], [(0, 6), (6, 6), (6, 12)], [(0, 6), (6, 11)], [(0, 6), (6, 13)],
                   [(1, 6), (6, 12)], [(6, 12), (0, 6)], []):
        with pytest.raises(ValueError):
            slab.labelSlabsEmulated(hdr, rho, None, 1.0, -1.0, ranges=ranges)
    with pytest.raises(ValueError):
        slab.labelSlabsEmulated(hdr, rho, 13, 1.0, -1.0)
    with pytest.raises(ValueError):
        slab.labelSlabsEmulated(hdr, rho, 3, 1.0, -1.0, ranges=[(0, 6), (6, 12)])
    assert slab.checkRanges([(0, 1), (1, 12)], 12) == [(0, 1), (1, 12)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,world", [(96, 2), (160, 4), (160, 8)])
def test_emulated_slabs_match_whole_map(n, world):
    from pdb_eda_b200 import _device, ccp4, slab, synthetic
    import golden_checks as gc
    vol = synthetic.smoothNoiseMapDevice(n, seed=n + world)
    hdr = ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((n, n, n), (n * 0.5,) * 3 + (90, 90, 90), (n, n, n)))
    whole = _device.DeviceMap(_device.geom_from_header(hdr), vol.reshape(-1)).blob_label(2.2, -2.2)
    parts = slab.labelSlabsEmulated(hdr, vol, world, 2.2, -2.2)
    for w, p in zip(whole, parts):
        assert p["n_pairs"] > 0 and w["n_blobs"] > 50
        assert torch.equal(w["crs"].long(), p["crs"])
        assert torch.equal(w["label"].long(), p["label"])
        assert w["n_blobs"] == p["n_blobs"]
        gc.close(p["stats"].cpu().numpy(), w["stats"].cpu().numpy(), rtol=1e-9, atol=1e-9)
