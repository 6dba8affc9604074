#!/usr/bin/env python3
"""Region density and region discrepancy per residue of the synthetic config-3 pool: one pe_batch_sphere_sums launch for the
whole pool against a loop of per-structure pe_sphere_sums launches on the same inputs, then ``multiple --single-mode`` batched
against entry by entry, in one run.

Kernel part -- pool: synthetic.poolSpec (grid sizes 64-256 on a 0.5 A grid, five space groups), a 2Fo-Fc map
(synthetic.densityMapDevice) and a Fo-Fc map (smoothed noise at 0.1 x the 2Fo-Fc sigma) resident in HBM per structure, one
group per residue (5 atoms) at 3.5 A.  ``density --residue``: 2Fo-Fc map, cutoffs (mean + 1.5 sigma, 0); ``difference
--residue``: Fo-Fc map, cutoffs (c, -c) with c = mean + 3 sigma.  Times are CUDA events (warm-up, repeats, median / min /
max); the two paths' outputs must be bit-identical.  Union voxels/s and algorithmic bytes (4 B per union voxel + atom inputs
+ group outputs) over the device-to-device copy rate measured in the same run.  The discrepancy rows also need
getTotalAbsDensity of every map (DeviceMap.sum_abs, one reduction over the map): its time is reported beside the batch's.

End-to-end part: ``multiple --single-mode "density --residue"`` over a directory of synthetic entries (poly-ALA with waters,
REMARK 290, CCP4 map pairs), batched (multipleStructures.runSingleMode) against the ``single`` path entry by entry
(singleStructure.analyze + writeResult), host clock around work that ends in a device synchronisation; the result files
must be byte-identical.

    python profiles/region_pool.py [--structures 256] [--repeats 20] [--entries 48] [--out region_pool.json]
"""
import argparse
import filecmp
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pdb_eda_b200 import _device, ccp4, regionBatch, synthetic  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "profiles"))
from metrics_pool import copy_rate  # noqa: E402


def build_pool(n, seed):
    """[(2Fo-Fc DeviceMap, Fo-Fc DeviceMap, coords float64, groupStart)] of the config-3 pool."""
    out = []
    for sp in synthetic.poolSpec(n, seed=seed):
        m, cell = sp["n"], sp["cell"]
        coords, _ = synthetic.fastPolyAla(sp["residues"], cell, sp["seed"])
        electrons = np.tile([7.0, 6.0, 6.0, 8.0, 6.0], sp["residues"])
        fo = synthetic.densityMapDevice(coords, electrons, m, cell, sp["seed"] + 1).reshape(-1)
        diff = synthetic.smoothNoiseMapDevice(m, seed=sp["seed"] + 2).reshape(-1) * (0.1 * float(fo.std()))
        geom = _device.geom_from_header(ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((m, m, m), cell, (m, m, m))))
        out.append((_device.DeviceMap(geom, fo.contiguous()), _device.DeviceMap(geom, diff.contiguous()),
                    np.asarray(coords, dtype=np.float32).astype(np.float64), np.arange(0, len(coords) + 1, 5)))
    torch.cuda.synchronize()
    return out


def timed(fn, warmup, repeats):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(repeats):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        times.append(s.elapsed_time(e))
    return {"median": float(np.median(times)), "min": float(min(times)), "max": float(max(times)), "repeats": repeats, "warmup": warmup}


def kernel_part(pool, kind, args, peak):
    entries = []
    for fo, diff, xyz, gs in pool:
        dm = fo if kind == "density" else diff
        m, s = dm.mean_std()
        c = m + (1.5 if kind == "density" else 3.0) * s
        cp, cn = (c, 0.0) if kind == "density" else (c, -1.0 * c)
        entries.append(regionBatch.RegionEntry(None, dm, xyz, np.full(len(xyz), 3.5, dtype=np.float32), gs, cp, cn, None))
    b = regionBatch.RegionBatch(entries)
    batched_t = timed(b.launchSums, args.warmup, args.repeats)
    torch.cuda.synchronize()
    batched = b.d_out.cpu().numpy()[:b.nGroups]
    outs = [torch.empty((e.nGroups, 8), dtype=torch.float64, device="cuda") for e in entries]

    def loop():
        for e, o in zip(entries, outs):
            e.map.sphere_sums(e.xyz, e.radius, e.groupStart, e.cutPos, e.cutNeg, out=o)
    loop_t = timed(loop, args.warmup, max(3, args.repeats // 4))
    ref = torch.cat(outs).cpu().numpy()
    rec = {"batched_ms": batched_t, "per_structure_loop_ms": loop_t, "speedup": loop_t["median"] / batched_t["median"],
           "bit_identical": bool(batched.tobytes() == ref.tobytes())}
    assert rec["bit_identical"], "batched and per-structure sums differ"
    voxels = float(batched[:, 0].sum())
    alg = 4 * voxels + b.nAtoms * (24 + 4) + b.nGroups * (8 * 8 + 8 + 4)
    med = batched_t["median"] / 1e3
    rec.update(union_voxels=voxels, union_voxels_per_s=voxels / med, residues_per_s=b.nGroups / med, algorithmic_bytes=alg,
               fraction_of_copy_rate=alg / med / peak)
    if kind == "difference":
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for e, (_, diff, _, _) in zip(entries, pool):
            diff.invalidate()
            diff.sum_abs(e.cutPos)
        torch.cuda.synchronize()
        rec["sum_abs_all_maps_ms"] = (time.perf_counter() - t0) * 1e3
    return rec, b.nAtoms, b.nGroups


def write_entries(folder, n, seed):
    from pdb_eda_b200 import structure
    ids = []
    for k in range(n):
        cell = (40.0 + 4 * (k % 5), 44.0, 48.0, 90, 90, 90)
        grid = tuple(int(round(c / 0.5)) for c in cell[:3])
        st = synthetic.polyAlaStructure(60 + 20 * (k % 7), np.zeros(3), np.array(cell[:3]), seed=seed + k, residuesPerChain=30, hetero=5)
        a, b = synthetic.mapPair(st, grid, cell, seed=seed + 100 + k)
        ops = synthetic.cartesianOperators("P 21 21 21", cell)
        text = structure.formatPDB(st, remark290=ops, cell=cell, spaceGroup="P 21 21 21", resolution=2.0)
        pdbid = "%d%03d" % (1 + k // 1000, k % 1000)
        open(os.path.join(folder, "pdb" + pdbid + ".ent"), "w").write(text)
        open(os.path.join(folder, pdbid + ".ccp4"), "wb").write(synthetic.ccp4Bytes(a, cell, grid))
        open(os.path.join(folder, pdbid + "_diff.ccp4"), "wb").write(synthetic.ccp4Bytes(b, cell, grid))
        ids.append(pdbid)
    return ids


def end_to_end(n, seed):
    from pdb_eda_b200 import multipleStructures, singleStructure
    with tempfile.TemporaryDirectory() as tmp:
        data = os.path.join(tmp, "data")
        os.makedirs(data)
        ids = write_entries(data, n, seed)
        single = multipleStructures.parseSingleMode("density --residue --out-format csv")
        outB, outS = os.path.join(tmp, "batched"), os.path.join(tmp, "single")
        os.makedirs(outS)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        summary = multipleStructures.runSingleMode(ids, outB, single, data)
        torch.cuda.synchronize()
        batched_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        for pdbid in ids:
            a = multipleStructures._entryArgs(single, pdbid, outS, data)
            singleStructure.writeResult(a, *singleStructure.analyze(a))
        torch.cuda.synchronize()
        single_s = time.perf_counter() - t0
        same = all(filecmp.cmp(os.path.join(outB, i + ".result"), os.path.join(outS, i + ".result"), shallow=False) for i in ids)
    assert same, "batched and per-entry result files differ"
    return {"entries": n, "summary": summary, "batched_s": batched_s, "per_entry_s": single_s, "speedup": single_s / batched_s,
            "files_byte_identical": same}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--structures", type=int, default=256)
    p.add_argument("--seed", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--repeats", type=int, default=20)
    p.add_argument("--entries", type=int, default=48)
    p.add_argument("--out", default="")
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("region_pool.py measures on a CUDA device; there is none")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout
    gpu = gpu.strip().splitlines()[torch.cuda.current_device()] if gpu.strip() else torch.cuda.get_device_name()
    peak = copy_rate()
    pool = build_pool(args.structures, args.seed)
    rec = {"device": gpu, "structures": len(pool), "radius": 3.5, "copy_rate_bytes_per_s": peak,
           "map_bytes_resident": int(sum(4 * (fo.rho.numel() + diff.rho.numel()) for fo, diff, _, _ in pool))}
    for kind in ("density", "difference"):
        rec[kind + "_residue"], rec["atoms"], rec["residues"] = kernel_part(pool, kind, args, peak)
    del pool
    torch.cuda.empty_cache()
    rec["end_to_end_density_residue"] = end_to_end(args.entries, args.seed)
    line = json.dumps(rec, sort_keys=True)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(rec, indent=2, sort_keys=True) + "\n")


if __name__ == "__main__":
    main()
