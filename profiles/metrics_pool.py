#!/usr/bin/env python3
"""Per-residue RSCC / RSR of the synthetic config-3 pool: the batched kernel (pe_pair_union_metrics, one launch for the whole
pool) against the per-structure voxel-list chain (sphere lists -> grouped de-duplication -> pe_pair_metrics), on the same
structures, in one run.

Pool: synthetic.poolSpec (grid sizes 64-256 on a 0.5 A grid, five space groups), a 2Fo-Fc map (synthetic.densityMapDevice)
and a Fo-Fc map (smoothed noise at 0.1 x the 2Fo-Fc sigma) resident in HBM per structure, resolutions drawn in 0.6-3.0 A so
that the metrics radii span 0.7-1.5 A.  Prints and writes (--out) one JSON record: device name and power limit (nvidia-smi),
batched times (CUDA events; warm-up, repeats, median / min / max), chain time, structures/s, residues/s, union voxels/s,
algorithmic bytes (8 B per union voxel + atom inputs + group outputs) over the measured device-to-device copy rate, and the
largest difference between the two paths' outputs.

    python profiles/metrics_pool.py [--structures 256] [--repeats 20] [--out metrics_pool.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pdb_eda_b200 import _device, _lib, ccp4, cutils, metricsBatch, synthetic  # noqa: E402
from pdb_eda_b200._device import _ptr, _stream  # noqa: E402


class _Dm:
    """The part of a DensityMatrix the chain's calls read."""

    def __init__(self, deviceMap):
        self.deviceMap = deviceMap


def build_pool(n, seed):
    spec = synthetic.poolSpec(n, seed=seed)
    rng = np.random.default_rng(seed)
    entries = []
    for sp in spec:
        m, cell = sp["n"], sp["cell"]
        coords, _ = synthetic.fastPolyAla(sp["residues"], cell, sp["seed"])
        electrons = np.tile([7.0, 6.0, 6.0, 8.0, 6.0], sp["residues"])
        fo = synthetic.densityMapDevice(coords, electrons, m, cell, sp["seed"] + 1).reshape(-1)
        diff = synthetic.smoothNoiseMapDevice(m, seed=sp["seed"] + 2).reshape(-1) * (0.1 * float(fo.std()))
        hdr = ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((m, m, m), cell, (m, m, m)))
        geom = _device.geom_from_header(hdr)
        radius = metricsBatch.metricsRadius(float(rng.uniform(0.6, 3.0)))
        entries.append(metricsBatch.MetricsEntry(_device.DeviceMap(geom, fo.contiguous()), _device.DeviceMap(geom, diff.contiguous()),
                                                 coords, np.arange(0, len(coords) + 1, 5), radius))
    torch.cuda.synchronize()
    return entries


def chain(entry):
    """The voxel-list chain on one structure: sphere lists -> grouped de-duplication -> pe_pair_metrics."""
    fo, diff = _Dm(entry.foMap), _Dm(entry.diffMap)
    lists = cutils.sphereLists(fo, entry.xyz, entry.radius, 0.0)
    group = torch.from_numpy(np.repeat(np.arange(entry.nGroups, dtype=np.int32), np.diff(entry.groupStart))).cuda()[lists["atom"].long()]
    _, first, _ = cutils.clusterCrs(lists["crs"], group, wantFirst=True)
    return cutils.pairMetrics(fo, diff, lists["crs"], group, first, entry.nGroups)


def copy_rate():
    """Device-to-device copy of 4 GiB (read + write), bytes moved per second: the HBM yardstick of this run."""
    a = torch.empty(1 << 30, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    for _ in range(2):
        b.copy_(a)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(10):
        b.copy_(a)
    e.record()
    e.synchronize()
    rate = 10 * 2 * a.numel() * 4 / (s.elapsed_time(e) / 1e3)
    del a, b
    torch.cuda.empty_cache()
    return rate


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--structures", type=int, default=256)
    p.add_argument("--seed", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--repeats", type=int, default=20)
    p.add_argument("--out", default="")
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("metrics_pool.py measures on a CUDA device; there is none")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    gpu = gpu.strip().splitlines()[torch.cuda.current_device()] if gpu.strip() else torch.cuda.get_device_name()
    lib = _lib.load()
    peak = copy_rate()
    entries = build_pool(args.structures, args.seed)
    b = metricsBatch.MetricsBatch(entries)

    def launch():
        _lib.check(lib.pe_pair_union_metrics(len(b.entries), _ptr(b.d_maps), b.nGroups, _ptr(b.d_groupMap), _ptr(b.d_groupStart),
                                             _ptr(b.d_xyz), _ptr(b.d_radius), _ptr(b.d_out), _ptr(b.ws), _stream()), "pe_pair_union_metrics")

    for _ in range(args.warmup):
        launch()
    times = []
    for _ in range(args.repeats):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        launch()
        e.record()
        e.synchronize()
        times.append(s.elapsed_time(e))
    batched = b.d_out.cpu().numpy()
    # the chain, structure after structure (its calls synchronise inside), warm then timed
    for entry in entries[:4]:
        chain(entry)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    outs = [chain(entry) for entry in entries]
    torch.cuda.synchronize()
    chain_ms = (time.perf_counter() - t0) * 1e3
    ref = torch.cat(outs).cpu().numpy()
    n_equal = bool(np.array_equal(batched[:, 0], ref[:, 0]))
    diffs = {}
    for name, x, y in zip(("rscc", "rsr"), metricsBatch.rsccRsr(batched), metricsBatch.rsccRsr(ref)):
        same_nan = bool(np.array_equal(np.isnan(x), np.isnan(y)))
        ok = ~np.isnan(x) & ~np.isnan(y)
        diffs[name] = {"nan_positions_equal": same_nan, "max_abs_diff": float(np.max(np.abs(x[ok] - y[ok]))) if ok.any() else 0.0}
    med = float(np.median(times))
    voxels = float(batched[:, 0].sum())
    alg_bytes = 8 * voxels + b.nAtoms * (24 + 4) + b.nGroups * (8 * 8 + 8)
    rec = {
        "device": gpu, "structures": len(entries), "residues": b.nGroups, "atoms": b.nAtoms, "union_voxels": voxels,
        "map_bytes_resident": int(sum(4 * (e.foMap.rho.numel() + e.diffMap.rho.numel()) for e in entries)),
        "radius_range": [float(min(e.radius[0] for e in entries)), float(max(e.radius[0] for e in entries))],
        "batched_ms": {"median": med, "min": float(min(times)), "max": float(max(times)), "repeats": len(times), "warmup": args.warmup},
        "chain_ms": chain_ms, "speedup": chain_ms / med,
        "batched_structures_per_s": len(entries) / (med / 1e3), "batched_residues_per_s": b.nGroups / (med / 1e3),
        "batched_union_voxels_per_s": voxels / (med / 1e3),
        "algorithmic_bytes": alg_bytes, "copy_rate_bytes_per_s": peak,
        "fraction_of_copy_rate": alg_bytes / (med / 1e3) / peak,
        "n_equal": n_equal, "compare": diffs,
    }
    line = json.dumps(rec, sort_keys=True)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(rec, indent=2, sort_keys=True) + "\n")


if __name__ == "__main__":
    main()
