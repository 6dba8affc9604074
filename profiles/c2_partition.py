#!/usr/bin/env python3
"""The C2 step (bench.py's N = 1 workload, seed 2) with the blob pass on its own partition of k SMs and the sphere kernel on the
others (VoxelPass.step, PDB_EDA_B200_BLOB_SMS = k; k = 0 shares all SMs), swept over k.

  step     ms/step over --steps steps per setting, the settings alternated within each of --repeats rounds (order rotated)
  kernels  per-kernel device times (pe_profile_*) of --profile-steps profiled steps per setting
  alone    each path by itself on its partition's stream (and on all SMs for k = 0): SM scaling without the other path's
           HBM traffic, so that the step time minus max(alone) is the interference of the two paths
  results  one step's results per k against k = 0: cloud / region rows, blob keys, labels and counts must be identical; the
           float64 blob sums are reported as bit-identical or as their largest relative difference

usage: python profiles/c2_partition.py [--out FILE.md] [--steps 2000] [--repeats 3]"""
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
import bench  # noqa: E402
from pdb_eda_b200 import _device, _lib, ccp4, pipeline, synthetic  # noqa: E402

KS = (0, 16, 24, 32, 40, 48, 56)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:
        out = "nvidia-smi unavailable (%s)" % exc
    return "%s; nvidia-smi: %s" % (torch.cuda.get_device_name(0), out)


def build_pass():
    work = bench.build_workload(bench.FULL, seed=2)
    n, cell = work["n"], work["cell"]
    geom = _device.geom_from_header(ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((n, n, n), cell, (n, n, n))))
    dens = _device.DeviceMap(geom, torch.from_numpy(work["fofc2"].reshape(-1)).cuda())
    diff = _device.DeviceMap(geom, torch.from_numpy(work["fofc"].reshape(-1)).cuda())
    return pipeline.VoxelPass(dens, diff, work["xyz"].astype(np.float64), work["radii"], work["res_start"], bench.REGION_RADIUS)


def per_step_ms(fn, steps, stream, warmup=20):
    """ms per call of fn enqueued on stream, by events on that stream."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        for _ in range(warmup):
            fn()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def compare(a, b):
    """'identical', 'sums within <rel>' (blob sums only) or 'DIFFERENT: <what>' for two results() of a step."""
    bad = [k for k in ("cloud", "region", "blob_counts") if not np.array_equal(a[k], b[k])]
    bad += ["%s %s" % (t, k) for t in ("green", "red") for k in ("key", "label") if not np.array_equal(a[t][k], b[t][k])]
    if bad:
        return "DIFFERENT: " + ", ".join(bad)
    rel = 0.0
    for t in ("green", "red"):
        x, y = a[t]["stats"], b[t]["stats"]
        if not np.array_equal(x, y):
            rel = max(rel, float(np.max(np.abs(x - y) / np.maximum(np.abs(y), 1e-300))))
    return "identical" if rel == 0.0 else "sums within %.1e relative" % rel


def snapshot(res):
    return {k: (v.copy() if isinstance(v, np.ndarray) else {kk: vv.copy() for kk, vv in v.items()}) for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="markdown report (default: stdout only)")
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--profile-steps", type=int, default=300)
    ap.add_argument("--alone-steps", type=int, default=1000)
    args = ap.parse_args()
    _device.require_cuda()
    torch.cuda.set_device(0)
    t0 = time.time()
    vp = build_pass()
    setup_s = time.time() - t0
    main_stream = torch.cuda.current_stream()
    sms_total = _lib.require_device()[0]
    results, same = {}, {}
    for k in KS:
        os.environ["PDB_EDA_B200_BLOB_SMS"] = str(k)
        vp.step()
        results[k] = snapshot(vp.results())
        assert k == 0 or pipeline.smPartition(vp.device, k) is not None, "no partition of %d SMs" % k
        same[k] = compare(results[k], results[0])

    # ---- the step, settings alternated
    step_ms = {k: [] for k in KS}
    for r in range(args.repeats):
        order = KS[r % len(KS):] + KS[:r % len(KS)]
        for k in order:
            os.environ["PDB_EDA_B200_BLOB_SMS"] = str(k)
            step_ms[k].append(per_step_ms(vp.step, args.steps, main_stream))

    # ---- per-kernel device times (a run of its own: the events add work to every launch)
    kernels = {}
    for k in KS:
        os.environ["PDB_EDA_B200_BLOB_SMS"] = str(k)
        per_step_ms(vp.step, 20, main_stream)
        _lib.profile(True, reset=True)
        prof_ms = per_step_ms(vp.step, args.profile_steps, main_stream, warmup=0)
        prof = _lib.profile()
        _lib.profile(False)
        kernels[k] = {"ms_per_step_profiled": prof_ms,
                      "us_per_launch": {name: ms * 1e3 / max(c, 1) for name, (c, ms) in prof.items()}}

    # ---- each path alone on its SMs
    alone = {}
    for k in KS:
        part = pipeline.smPartition(vp.device, k) if k else None
        bs, rs = (part[0], part[1]) if part else (main_stream, main_stream)
        alone[k] = {"blobs_ms": per_step_ms(vp.blobs, args.alone_steps, bs), "spheres_ms": per_step_ms(vp.spheres, args.alone_steps, rs)}
    os.environ.pop("PDB_EDA_B200_BLOB_SMS")

    result = {"card": card(), "sms": sms_total, "steps": args.steps, "repeats": args.repeats, "setup_s": round(setup_s, 1),
              "step_ms": step_ms, "kernels": kernels, "alone": alone, "results_vs_k0": same}
    print(json.dumps(result))
    lines = ["# C2 step on SM partitions (blob pass on k SMs, sphere kernel on the other %d - k)" % sms_total, "",
             "Measured by `profiles/c2_partition.py` on %s." % result["card"], "",
             "C2 workload of bench.py (384^3 map pair, %d atoms / %d residues, seed 2). ms/step by CUDA events over %d steps per "
             "setting, settings alternated in %d rounds; k = 0 is the shared-SM two-stream schedule. Blob / sphere alone: that path "
             "by itself on its partition's stream (%d calls)." % (vp.n_atoms, vp.n_res, args.steps, args.repeats, args.alone_steps), "",
             "| k | ms/step (rounds) | median | blobs alone ms | spheres alone ms | max(alone) | threshold us | sparse us | sphere us | results vs k = 0 |",
             "|---:|---|---:|---:|---:|---:|---:|---:|---:|---|"]
    for k in KS:
        u = kernels[k]["us_per_launch"]
        lines.append("| %d | %s | %.4f | %.4f | %.4f | %.4f | %.1f | %.1f | %.1f | %s |" % (
            k, " / ".join("%.4f" % x for x in step_ms[k]), float(np.median(step_ms[k])), alone[k]["blobs_ms"], alone[k]["spheres_ms"],
            max(alone[k].values()), u.get("threshold_bitmap_kernel", float("nan")), u.get("blob_sparse_kernel", float("nan")),
            u.get("sphere_union_kernel", float("nan")), same[k]))
    lines += ["", "Per-kernel times are event pairs on each kernel's own stream in a profiled run; with two paths in flight they "
              "include the time a kernel shares the GPU with the other path.", ""]
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)
        with open(os.path.splitext(args.out)[0] + ".json", "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
