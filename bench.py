#!/usr/bin/env python3
"""bench.py -- the voxel hot path on BASELINE.json's configurations (one line of JSON on stdout).

N = 1  ("config.workload": "C2"): a ~40k-atom synthetic poly-ALA structure (8,000 residues) on a 384^3 P1 map pair
(cell 192 A, 0.5 A grid).  One step = one pass of the hot path over that structure:
  cloud   per-atom sphere gather-sums at the atom-type radii (2Fo-Fc, cutoff mean + 1.5 sigma)
  region  per-residue set-union sphere sums at 3.5 A (2Fo-Fc)
  blobs   green + red blob lists of the Fo-Fc map at +-(mean + 3 sigma): threshold, 26-connected labelling in the
          reference's blob order, per-blob sums
Units: atom-sphere voxels ((atom, voxel) pairs passing the distance test; cloud + region) + blob-CCL voxels (voxels
of the scanned unique volume).  `value` = units / device time, inputs resident in HBM.  `e2e` = the same through the
public API with HOST buffers (maps + atoms copied in, results copied out, every step).  The line also carries `c3`
(the multiple-structures pool of the N > 1 runs on this one GPU) and `e2e_api` (the DensityAnalysis calls a user makes).

N > 1  ("config.workload": "C3", BASELINE.json configs[2]): multiple-structures mode.  A fixed pool of synthetic
structures (mixed space groups, 64^3 - 256^3 maps, atoms ~ n^3 / 350; --pool, default 1,024 of the 4,096 so that the
whole pool also fits ONE GPU for the strong-scaling reference) is sharded over the ranks longest-first
(multi.shardStructures); one step = every rank analyses its share (cloud aggregation = analyzePDBID,
pdb_eda/multipleStructures.py:320-356, batched: cloudBatch / pe_cloud_*) + the fused all-reduce of the cumulative
statistics + the all-gather of the per-structure rows (multi.gatherPacked), all inside the timed region.  STRONG
scaling: the same pool at every N.  Units: atom-sphere voxels of the pool (multiple-structures mode computes no blobs).
`pool_on_one_gpu` = the same pool on rank 0 alone, timed in the same run (the denominator for scaling at fixed work);
`c4` = BASELINE.json configs[3]: one 1024^3 Fo-Fc map slab-partitioned over the ranks vs the whole map on one GPU.

--impl reference: the UNMODIFIED reference (oracle/_ref: pdb_eda 2.7.1 + its compiled Cython cutils) on the host CPU,
one core (its single-structure path is single threaded), on a bounded sample of the C2 workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from pdb_eda_b200 import synthetic  # noqa: E402

METRIC = "voxels/s (atom-sphere voxels + blob-CCL voxels per pass of the voxel hot path)"
UNIT = "voxels/s"
REGION_RADIUS = 3.5
FULL = dict(n=384, cell=192.0, residues=8000)
SAMPLE = dict(n=64, cell=32.0, residues=37)   # same grid spacing and atom density as FULL (1/216 of the volume)


def build_workload(spec, seed):
    """Synthetic structure + (2Fo-Fc, Fo-Fc) volumes + per-atom radii + residue offsets."""
    n, cell_len = spec["n"], spec["cell"]
    cell = (cell_len, cell_len, cell_len, 90.0, 90.0, 90.0)
    st = synthetic.polyAlaStructure(spec["residues"], (0, 0, 0), (cell_len,) * 3, seed=seed, residuesPerChain=1000)
    fofc2, fofc = synthetic.mapPair(st, (n, n, n), cell, seed=seed + 6)
    params = synthetic.defaultParams()
    atoms, radii, res_start = [], [], [0]
    for residue in st.get_residues():
        for atom in residue:
            key = residue.resname + "_" + atom.name
            atoms.append(atom.coord)
            radii.append(params["radii"][params["full_atom_name_map_atom_type"][key]])
        res_start.append(len(atoms))
    return dict(structure=st, cell=cell, n=n, fofc2=fofc2, fofc=fofc, xyz=np.asarray(atoms, dtype=np.float32),
                radii=np.asarray(radii, dtype=np.float32), res_start=np.asarray(res_start, dtype=np.int32))


def dump_outputs(out, directory, limit=64 << 20):
    """Writes the arrays one step returns to a caller (``VoxelPass.results()``) as ``directory/<name>.npy`` in float64, so that
    two builds can be compared output for output on the same seeded inputs.  An array larger than its share of ``limit``
    bytes is cut to a fixed seeded sample of its rows (written as ``<name>_rows.npy`` beside it)."""
    arrays = {"cloud": out["cloud"], "region": out["region"], "blob_counts": out["blob_counts"]}
    for tag in ("green", "red"):
        for k in ("key", "label", "stats"):
            arrays[tag + "_" + k] = out[tag][k]
    os.makedirs(directory, exist_ok=True)
    share = limit // (2 * len(arrays))              # an array and its row indices
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.nbytes > share:
            keep = max(1, share // (a.nbytes // len(a)) - 1)
            rows = np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))
            np.save(os.path.join(directory, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(directory, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, smax, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in self.samples:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arm
def load_reference():
    from oracle import refload
    if refload.available():
        return refload.load()
    return None


def reference_step(ref_mods, work):
    """One pass of the three sub-workloads through the reference's own public methods."""
    import io
    ref_ccp4 = ref_mods[0]
    cell, n = work["cell"], work["n"]
    dens = ref_ccp4.parse(io.BytesIO(synthetic.ccp4Bytes(work["fofc2"], cell, (n, n, n))), "bench")
    diff = ref_ccp4.parse(io.BytesIO(synthetic.ccp4Bytes(work["fofc"], cell, (n, n, n))), "bench")
    t0 = time.perf_counter()
    dcut = dens.meanDensity + 1.5 * dens.stdDensity
    fcut = diff.meanDensity + 3.0 * diff.stdDensity
    xyz, radii, rs = work["xyz"], work["radii"], work["res_start"]
    cloud = [dens.findAberrantBlobs(xyz[i], float(radii[i]), dcut) for i in range(len(xyz))]
    region = [dens.findAberrantBlobs([xyz[i] for i in range(rs[k], rs[k + 1])], REGION_RADIUS, dcut) for k in range(len(rs) - 1)]
    green = diff.createFullBlobList(fcut)
    red = diff.createFullBlobList(-fcut)
    dt = time.perf_counter() - t0
    return dt, (len(cloud), len(region), len(green), len(red))


def oracle_units(work):
    """Unit counts of a workload by the CPU oracle (outside any timed region)."""
    import io
    from oracle import orc
    from pdb_eda_b200 import ccp4
    cell, n = work["cell"], work["n"]
    dm = ccp4.parse(io.BytesIO(synthetic.ccp4Bytes(work["fofc2"], cell, (n, n, n))), "bench")
    g = orc.geom(dm.header, dm.origin)
    xyz = work["xyz"].astype(np.float64)
    cloud = orc.sphere_sums_batch(g, work["fofc2"], xyz, work["radii"])[:, 0].sum()
    region = orc.sphere_sums_batch(g, work["fofc2"], xyz, np.full(len(xyz), REGION_RADIUS, np.float32))[:, 0].sum()
    return float(cloud), float(region), float(n) ** 3


def oracle_step(work):
    """The oracle port of the same pass (used only when oracle/_ref is absent)."""
    import io
    from oracle import orc
    from pdb_eda_b200 import ccp4
    cell, n = work["cell"], work["n"]
    dm = ccp4.parse(io.BytesIO(synthetic.ccp4Bytes(work["fofc2"], cell, (n, n, n))), "bench")
    g = orc.geom(dm.header, dm.origin)
    xyz = work["xyz"].astype(np.float64)
    t0 = time.perf_counter()
    v2 = work["fofc2"].astype(np.float64)
    v1 = work["fofc"].astype(np.float64)
    dcut = v2.mean() + 1.5 * v2.std()
    fcut = v1.mean() + 3.0 * v1.std()
    orc.sphere_sums_batch(g, work["fofc2"], xyz, work["radii"], dcut)
    rs = work["res_start"]
    for k in range(len(rs) - 1):
        orc.sphere_union_sums(g, work["fofc2"], xyz[rs[k]:rs[k + 1]], np.full(rs[k + 1] - rs[k], REGION_RADIUS, np.float32), dcut, 0.0)
    orc.full_blobs(g, work["fofc"], fcut)
    orc.full_blobs(g, work["fofc"], -fcut)
    return time.perf_counter() - t0, None


def run_cpu_sample(steps, warmup):
    work = build_workload(SAMPLE, seed=2)
    units = sum(oracle_units(work))
    ref_mods = load_reference()
    kind = "reference" if ref_mods is not None else "port"
    times = []
    for i in range(warmup + steps):
        dt, _ = reference_step(ref_mods, work) if ref_mods is not None else oracle_step(work)
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    value = units * len(times) / total
    sample = ("%d^3 P1 map pair (cell %.0f A), %d atoms / %d residues, same grid spacing and atom density as C2; cloud + region "
              "(3.5 A) + green/red blobs via DensityMatrix.findAberrantBlobs / createFullBlobList; %d steps, %.1f s/step"
              % (SAMPLE["n"], SAMPLE["cell"], len(work["xyz"]), SAMPLE["residues"], len(times), total / len(times)))
    return value, {"value": value, "unit": UNIT, "cores": 1, "kind": kind, "sample": sample}, total / len(times) * 1e3


WORK_C2 = {
    "cloud": {"b200": "pe_sphere_sums per atom: sphere enumeration + wrapped density gather + sums (all, > cutoff, < -cutoff), valid flag",
              "reference": "DensityMatrix.findAberrantBlobs(atom.coord, radius, cutoff): the same enumeration and gather, then 26-connected "
                           "clustering of the voxels into DensityBlobs (centroids, totals) -- more than the B200 leg; ~1 % of the reference's step"},
    "region": {"b200": "pe_sphere_sums per residue (set-union of its atoms' 3.5 A spheres): sums, counts, valid flag",
               "reference": "DensityMatrix.findAberrantBlobs(list of coords, 3.5, cutoff): set-union enumeration + clustering into blobs, whose "
                            "totals the caller adds up (calculateRegionDensity) -- the sum is what both legs deliver"},
    "blobs": {"b200": "pe_blob_label: +-cutoff threshold of the whole Fo-Fc map, 26-connected labelling in createCrsLists order, per-blob sums",
              "reference": "createFullBlobList(+cutoff) and createFullBlobList(-cutoff): createFullCrsList + createCrsLists (N x N cdist) + "
                           "DensityBlob.fromCrsList"}}


def reference_c1_full_pass(ref_mods):
    """BASELINE.json configs[0] at full size through the reference's public methods, once: 96^3 P2(1)2(1)2(1), 2,500 atoms."""
    work = build_workload(dict(n=96, cell=48.0, residues=500), seed=1)
    units = sum(oracle_units(work))
    dt, counts = reference_step(ref_mods, work)
    return {"workload": "C1: 96^3 map pair, 2,500 atoms / 500 residues; cloud + region (3.5 A) + green/red blobs, one pass", "seconds": round(dt, 2),
            "units": units, "value": units / dt, "unit": UNIT, "cores": 1, "green_red_blobs": [counts[2], counts[3]]}


# ---- config 3 on the host: the reference's multiple-structures mode on a bounded sample of the pool, all host cores
_REF_C3 = {}


def _ref_c3_init():
    from oracle import refload
    _REF_C3["mods"] = refload.load()
    _REF_C3["mods"][1].setGlobals(synthetic.defaultParams())


def _ref_c3_analyze(item):
    """analyzePDBID's voxel work on one entry (pdb_eda/multipleStructures.py:320-346): parse the map, aggregateCloud, read the ratio."""
    import io
    ref_ccp4, ref_da = _REF_C3["mods"][0], _REF_C3["mods"][1]
    st, data = item
    dens = ref_ccp4.parse(io.BytesIO(data), "pool")
    dens.densityCutoff = dens.meanDensity + 1.5 * dens.stdDensity
    an = ref_da.DensityAnalysis("pool", dens, None, st, None)
    an.aggregateCloud()
    return (an.densityElectronRatio or 0.0, an.numVoxelsAggregated or 0)


def structure_from_arrays(coords32, bfactor):
    """A poly-ALA Structure (the duck-typed Biopython surface) from the arrays of synthetic.fastPolyAla."""
    from pdb_eda_b200 import structure as _st
    st = _st.Structure("pool")
    st.header["resolution"] = 2.0
    chain = st.add(_st.Model(0)).add(_st.Chain("A"))
    names = [(a, e) for a, _, e in synthetic._ALA_ATOMS]
    for k in range(len(coords32) // 5):
        res = chain.add(_st.Residue((" ", k + 1, " "), "ALA"))
        for j, (name, element) in enumerate(names):
            res.add(_st.Atom(name, coords32[5 * k + j], float(bfactor[5 * k + j]), 1.0, element=element))
    return st


def run_cpu_c3_sample(steps, warmup, cores):
    """The 64^3 structures of the pool, `cores` of them per step, one per worker of a multiprocessing.Pool like
    pdb_eda/multipleStructures.py:167-168.  Returns (value, cpu_baseline dict, ms per step)."""
    import multiprocessing as mp
    from oracle import orc
    from pdb_eda_b200 import ccp4
    import io
    params = synthetic.defaultParams()
    spec = [sp for sp in synthetic.poolSpec(4096) if sp["n"] == 64 and sp["cell"][5] == 90.0][:cores]
    items, units = [], 0.0
    electronsOf = np.array([synthetic.ALA_ELECTRONS["ALA_" + a] for a, _, _ in synthetic._ALA_ATOMS])
    for sp in spec:
        coords, bf = synthetic.fastPolyAla(sp["residues"], sp["cell"], sp["seed"])
        st = structure_from_arrays(coords, bf)
        n = sp["n"]
        fofc2, _ = synthetic.mapPair(st, (n, n, n), sp["cell"], seed=sp["seed"] + 1)
        data = synthetic.ccp4Bytes(fofc2, sp["cell"], (n, n, n))
        dm = ccp4.parse(io.BytesIO(data), "pool")
        radii = np.array([params["radii"][params["full_atom_name_map_atom_type"]["ALA_" + a]] for a, _, _ in synthetic._ALA_ATOMS] * sp["residues"],
                         dtype=np.float32)
        units += float(orc.sphere_sums_batch(orc.geom(dm.header, dm.origin), fofc2, coords.astype(np.float64), radii)[:, 0].sum())
        items.append((st, data))
    times = []
    with mp.get_context("fork").Pool(cores, initializer=_ref_c3_init) as pool:
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            out = pool.map(_ref_c3_analyze, items, chunksize=1)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    total = sum(times)
    value = units * len(times) / total
    sample = ("%d structures of the pool per step (64^3 maps, %d atoms each on average), one per worker of a multiprocessing.Pool(%d): parse + "
              "aggregateCloud (analyzePDBID, pdb_eda/multipleStructures.py:320-346); %d steps, %.1f s/step, %d structures with a ratio"
              % (len(items), int(np.mean([5 * sp["residues"] for sp in spec])), cores, len(times), total / len(times), sum(1 for r in out if r[0])))
    return value, {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample,
                   "structures_per_s": len(items) * len(times) / total}, total / len(times) * 1e3


def api_timing(work):
    """Wall-clock of the public DensityAnalysis calls on the full C2 structure (context for the kernel-level numbers;
    not part of the timed step): the reference cannot run these at this size at all (SURVEY.md section 3.3)."""
    import io
    import torch
    from pdb_eda_b200 import ccp4, densityAnalysis, pdbParser, structure
    cell, n = work["cell"], work["n"]
    densityAnalysis.setGlobals(synthetic.defaultParams())
    out = {}

    def timed(label, fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        res = fn()
        torch.cuda.synchronize()
        out[label] = round(time.perf_counter() - t, 4)
        return res

    # the files a user would hold: CCP4 bytes of both maps and the PDB text (synthesised outside the timed calls)
    b1 = synthetic.ccp4Bytes(work["fofc2"], cell, (n, n, n))
    b2 = synthetic.ccp4Bytes(work["fofc"], cell, (n, n, n))
    text = structure.formatPDB(work["structure"], remark290=synthetic.cartesianOperators("P 1", cell), cell=cell, spaceGroup="P 1")

    def load():
        an = densityAnalysis.fromFile(io.StringIO(text), io.BytesIO(b1), io.BytesIO(b2))
        an.densityObj.meanDensity, an.diffDensityObj.meanDensity      # the cutoffs are part of loading (pdb_eda/densityAnalysis.py:131,148)
        return an

    an = timed("load_parse_upload_meanstd_s", load)
    timed("aggregateCloud_s", an.aggregateCloud)
    blobs = timed("green_red_blob_lists_s", lambda: (an.greenBlobList, an.redBlobList))
    timed("blob_statistics_s", lambda: an.calculateAtomSpecificBlobStatistics(blobs[0] + blobs[1]))
    timed("residue_region_density_s", lambda: an.calculateResidueRegionDensity(REGION_RADIUS))
    out.update({"atoms_analysed": len(an.atomCloudDescriptions), "residue_clouds": an.numResidueCloudsAnalyzed,
                "domain_clouds": an.numDomainCloudsAnalyzed, "green_blobs": len(blobs[0]), "red_blobs": len(blobs[1]),
                "density_electron_ratio": an.densityElectronRatio})
    return out


def main_reference(args, rank, world):
    if rank != 0:
        return
    if world > 1 or args.gpus > 1:
        # the N > 1 arm runs config 3: the reference's multiple-structures mode on all host cores
        cores = max(1, len(os.sched_getaffinity(0)))
        value, cpu, ms = run_cpu_c3_sample(args.steps, min(args.warmup, 1), cores)   # ~10 s per step: one warm-up pass is enough
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": {"workload": "C3 (bounded sample: %s)" % cpu["sample"]},
                "structures_per_s": cpu["structures_per_s"],
                "cpu_baseline": cpu, "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return
    value, cpu, ms = run_cpu_sample(args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": {"workload": "C2 (bounded sample: %s)" % cpu["sample"]},
            "work": {k: v["reference"] for k, v in WORK_C2.items()},
            "cpu_baseline": cpu, "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    ref_mods = load_reference()
    if ref_mods is not None and not args.no_c1:
        line["c1_full_size"] = reference_c1_full_pass(ref_mods)       # BASELINE.json configs[0] as it stands, one pass (~70 s)
    print(json.dumps(line))


def bind_to_gpu(local_rank):
    """Pins this process to the CPU cores NVML reports as local to its GPU (same NUMA node / PCIe root), BEFORE any pinned host
    buffer is allocated, so that the staging memory of a rank lives next to its GPU.  Returns a short description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"cores": len(allowed or os.sched_getaffinity(0)), "first": min(allowed) if allowed else None,
                "last": max(allowed) if allowed else None, "bound": bool(allowed)}
    except Exception as exc:                      # NVML absent or not permitted: run unbound and say so
        return {"bound": False, "error": str(exc)[:80]}


# ------------------------------------------------------------------------------------------------ GPU arm
def main_gpu(args, rank, world, local_rank):
    import io
    import torch
    import torch.distributed as dist
    from pdb_eda_b200 import _device, _lib, ccp4
    from pdb_eda_b200.pipeline import VoxelPass

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries the one JSON line only
        dist.init_process_group("nccl", device_id=device)
    _device.require_cuda()

    work = build_workload(FULL, seed=2 + rank)
    n, cell = work["n"], work["cell"]
    hdr_dens = ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((n, n, n), cell, (n, n, n)))
    # pinned host copies of the inputs (what a caller holds after reading the CCP4 / PDB files)
    h_dens = torch.from_numpy(work["fofc2"].reshape(-1)).pin_memory()
    h_diff = torch.from_numpy(work["fofc"].reshape(-1)).pin_memory()
    h_xyz = torch.from_numpy(work["xyz"].astype(np.float64)).pin_memory()
    geom = _device.geom_from_header(hdr_dens)
    d_dens = torch.empty(n ** 3, dtype=torch.float32, device=device)
    d_diff = torch.empty(n ** 3, dtype=torch.float32, device=device)
    d_dens.copy_(h_dens, non_blocking=True)
    d_diff.copy_(h_diff, non_blocking=True)
    dens = _device.DeviceMap(geom, d_dens)
    diff = _device.DeviceMap(geom, d_diff)
    vp = VoxelPass(dens, diff, work["xyz"].astype(np.float64), work["radii"], work["res_start"], REGION_RADIUS)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- unit counts (outside the timed region)
    vp.step()
    torch.cuda.synchronize()
    res = vp.results()
    cloud_units = float(res["cloud"][:, 0].sum())
    cloud_candidates = float(res["cloud"][:, 7].sum())          # box voxels examined (SURVEY.md section 8d asks for both)
    region_per_atom = dens.sphere_sums(vp.xyz, vp.region_radii)
    region_pairs = float(region_per_atom[:, 0].sum().item())
    region_candidates = float(region_per_atom[:, 7].sum().item())
    blob_units = float(vp.n_blob_voxels)
    units = cloud_units + region_pairs + blob_units

    # ---- device-resident timing
    for _ in range(max(args.warmup, 3)):
        vp.step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    lib = _lib.load()
    launches0 = lib.pe_launch_count()
    _lib.profile(True, reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        vp.step()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = lib.pe_launch_count() - launches0
    prof = _lib.profile()
    _lib.profile(False)

    # an un-instrumented repeat (no per-kernel events) for the headline device number
    barrier()
    e0.record()
    for _ in range(args.steps):
        vp.step()
    e1.record()
    barrier()
    ms_plain = e0.elapsed_time(e1)

    # ---- end to end through the public API with host buffers
    def e2e_step():
        """The public end-to-end call: pinned host maps + atoms in, host results out (VoxelPass.stepFromHost)."""
        return vp.stepFromHost(h_dens, h_diff, h_xyz)

    for _ in range(2):
        out = e2e_step()
    barrier()
    e0.record()
    for _ in range(args.steps):
        out = e2e_step()
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    h2d = h_dens.numel() * 4 + h_diff.numel() * 4 + h_xyz.numel() * 8
    d2h = (out["cloud"].nbytes + out["region"].nbytes + out["blob_counts"].nbytes +
           sum(out[t][k].nbytes for t in ("green", "red") for k in ("key", "label", "stats")))

    # ---- max over ranks, sum of units
    stats = torch.tensor([ms_plain, ms_e2e, ms_total], dtype=torch.float64, device=device)
    tot_units = torch.tensor([units], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot_units, op=dist.ReduceOp.SUM)
    ms_plain, ms_e2e, ms_total = stats.tolist()
    all_units = tot_units.item()

    if rank == 0:
        value = all_units * args.steps / (ms_plain * 1e-3)
        e2e_value = all_units * args.steps / (ms_e2e * 1e-3)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        n_fg = float(res["blob_counts"][0] + res["blob_counts"][2])
        n_blob = float(res["blob_counts"][1] + res["blob_counts"][3])
        region_union = float(res["region"][:, 0].sum())
        # algorithmic bytes per launch (DESIGN.md section 3; SURVEY.md section 8d)
        algo = {"threshold_bitmap_kernel": 4.0 * blob_units,                               # 4 N_vox
                "sphere_union_kernel": 4.0 * region_union + 52.0 * vp.n_atoms,            # 4 V_in + 52 A (region pass)
                "sphere_sums_kernel": 4.0 * cloud_units + 52.0 * vp.n_atoms}              # 4 V_in + 52 A (cloud pass)
        # what actually limits each kernel (profiles/r02_union_phases.md, profiles/r01_v10_c2_step.md): the HBM fraction is the
        # contract number; kernels that are not HBM-bound also carry the ceiling that applies to them
        bounds = {"threshold_bitmap_kernel": "hbm", "sphere_union_kernel": "latency", "sphere_sums_kernel": "latency", "blob_sparse_kernel": "latency"}
        notes = {"sphere_union_kernel": "one warp per residue: exact row chords -> bitmap -> compaction -> sector-granular gathers; bound by the "
                                        "length of each warp's dependent instruction chains at 28 warps / SM, not by HBM (issue slots 64 % busy; "
                                        "ALU 38 %, LSU 32 %, XU 20 %, FP64 12 %); V_in = union voxels",
                 "sphere_sums_kernel": "bound by latency of the per-atom chain (box, tables, exact row chords, 32-byte gathers), not by HBM",
                 "blob_sparse_kernel": "sparse union-find over the bit planes with 3 grid barriers: latency of dependent 4-byte L2 transactions"}
        kernels = []
        for name, (count, ms) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
            kernels.append({"kernel": name, "launches": count, "ms_total": round(ms, 4), "us_per_launch": round(ms * 1e3 / max(count, 1), 2)})
        try:  # DRAM traffic and warp instructions per launch from the committed ncu capture of this workload (profiles/)
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        except Exception:
            traffic = {}
        inst = traffic.get("_warp_instructions", {})
        sm_mhz = float(peaks.get("sm_max_mhz", 1965.0))
        issue_peak = 148 * 4 * sm_mhz * 1e6                         # warp instructions / s: 148 SMs x 4 schedulers x clock
        algo["blob_sparse_kernel"] = 8.0 * n_fg + 64.0 * n_blob      # 8 N_fg + 64 N_blob (SURVEY.md section 8d)
        roofs = []
        for k in kernels:
            if k["kernel"] in algo:
                t = k["ms_total"] / max(k["launches"], 1) * 1e-3
                ach = algo[k["kernel"]] / t / 1e9
                r = {"kernel": k["kernel"], "bound": bounds.get(k["kernel"], "hbm"), "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(ach / peak, 4), "traffic": traffic.get(k["kernel"]), "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": algo[k["kernel"]], "us_per_launch": k["us_per_launch"]}
                if k["kernel"] in inst:
                    r["issue_roofline"] = {"warp_instructions_per_launch": inst[k["kernel"]], "achieved": round(inst[k["kernel"]] / t, 1),
                                           "peak": issue_peak, "unit": "warp instructions/s", "frac": round(inst[k["kernel"]] / t / issue_peak, 4),
                                           "source": "smsp__inst_executed.sum of the committed ncu capture (profiles/traffic.json)"}
                    if k["kernel"] == "sphere_union_kernel":
                        r["issue_roofline"]["warp_instructions_per_32_voxels"] = round(inst[k["kernel"]] / (region_union / 32.0), 1)
                if k["kernel"] in notes:
                    r["note"] = notes[k["kernel"]]
                roofs.append(r)
        dominant = roofs[0] if roofs else None      # kernels are sorted by total device time
        others = roofs[1:]
        # whole paths (north_star quotes its targets per path): every kernel of the path, algorithmic bytes of the path
        us = {k["kernel"]: k["us_per_launch"] * k["launches"] / args.steps for k in kernels}
        paths = []
        for label, names, nbytes in (
                ("blob_ccl (threshold + sparse labelling, both signs)", ("threshold_bitmap_kernel", "blob_sparse_kernel"),
                 4.0 * blob_units + 8.0 * n_fg + 64.0 * n_blob),
                ("atom_spheres (cloud + region passes)", ("sphere_sums_kernel", "sphere_union_kernel"),
                 algo["sphere_union_kernel"] + algo["sphere_sums_kernel"])):
            t_us = sum(us.get(nm, 0.0) for nm in names)
            if t_us > 0:
                ach = nbytes / (t_us * 1e-6) / 1e9
                paths.append({"path": label, "kernels": list(names), "us_per_step": round(t_us, 2), "algorithmic_bytes_per_step": nbytes,
                              "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4)})
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_plain / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": "C2: 384^3 P1 map pair, %d atoms / %d residues per GPU; cloud + region(3.5 A) + green/red blobs"
                                       % (vp.n_atoms, vp.n_res),
                           "parallelism": "replicas x%d (single structure does not shard)" % world,
                           "l2": "inputs larger than L2 (2 x 226 MB maps per pass); no explicit flush"},
                "work": {k: v["b200"] for k, v in WORK_C2.items()},
                "units_per_step": {"cloud_atom_sphere_voxels": cloud_units, "cloud_box_candidates": cloud_candidates,
                                   "region_atom_sphere_voxels": region_pairs, "region_box_candidates": region_candidates,
                                   "region_union_voxels": region_union, "blob_ccl_voxels": blob_units,
                                   "foreground_voxels": n_fg, "blobs": n_blob},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                        "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "roofline": dominant, "roofline_other": others, "roofline_paths": paths,
                "kernels": kernels[:12], "ms_per_step_profiled": ms_total / args.steps, "clocks": clocks}
        if world == 1 and not args.no_cpu:
            _, cpu, _ = run_cpu_sample(1, 0)
            line["cpu_baseline"] = cpu
            api_first = api_timing(work)        # first use in the process: kernel images are loaded, workspaces allocated, buffers pinned
            api = api_timing(work)              # the same calls on a fresh DensityAnalysis object, warm process
            line["api_c2"] = api
            calls = ("load_parse_upload_meanstd_s", "aggregateCloud_s", "green_red_blob_lists_s", "blob_statistics_s", "residue_region_density_s")
            line["e2e_api"] = {"seconds": round(sum(api[c] for c in calls), 4), "calls": {c: api[c] for c in calls},
                               "seconds_first_use": round(sum(api_first[c] for c in calls), 4),
                               "what": "pdb_eda_b200.densityAnalysis on the C2 structure, host CCP4 / PDB bytes in, Python rows out: fromFile-equivalent "
                                       "load -> aggregateCloud -> greenBlobList + redBlobList -> calculateAtomSpecificBlobStatistics -> "
                                       "calculateResidueRegionDensity(3.5)"}
        if world == 1 and not args.no_c3:
            # BASELINE.json configs[2] on this one GPU: the pool the N > 1 runs shard (their strong-scaling reference point)
            del vp, dens, diff, d_dens, d_diff
            torch.cuda.empty_cache()
            line["c3"] = run_c3_one_gpu(args.pool, args.steps, device, synthetic.defaultParams())[0]
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ config 3: structure pool
def _pool_units(entries, params):
    """Atom-sphere voxels ((atom, voxel) pairs passing the distance test, SURVEY.md section 8d) of a list of pool entries."""
    from pdb_eda_b200 import cloudBatch
    units = 0.0
    for _, mref, table in entries:
        radii = cloudBatch._typeTables(table, params)[0][table.nameIndex].astype(np.float32)
        out = mref.deviceMap.sphere_sums(table.coords32.astype(np.float64), radii)
        units += float(out[:, 0].sum().item())
    return units


def _time_passes(shard, steps, warmup, barrier, **kw):
    """(ms per pass by CUDA events, ms per pass by the host clock, last summary)."""
    import torch
    summary = None
    for _ in range(warmup):
        summary = shard.analyze(**kw)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        summary = shard.analyze(**kw)
    e1.record()
    barrier()
    wall = (time.perf_counter() - t0) * 1e3 / steps
    return e0.elapsed_time(e1) / steps, wall, summary


def _summary_digest(summary):
    c = summary["cumulative"]
    return {"structures": c["structures"], "num_voxels_aggregated": c["num_voxels_aggregated"],
            "total_aggregated_electrons": c["total_aggregated_electrons"], "total_aggregated_density": c["total_aggregated_density"],
            "density_electron_ratio": c["density_electron_ratio"],
            "median_diffs": {k.split("#")[0]: float(v) for k, v in summary["medianDiffs"].items()}}


def run_c3_one_gpu(pool, steps, device, params):
    """The whole pool on this GPU alone (no collectives): {ms_per_pass, structures_per_s, value, summary digest}."""
    import torch
    from pdb_eda_b200 import multi
    spec = synthetic.poolSpec(pool)
    t0 = time.perf_counter()
    entries = synthetic.buildPoolEntries(spec, params, device)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t0
    units = _pool_units(entries, params)
    shard = multi.PoolShard(entries, params, device=device)
    ms, wall, summary = _time_passes(shard, steps, 2, torch.cuda.synchronize, device=device, local=True)
    return {"structures": pool, "atoms": shard.nAtoms, "batches": len(shard.batches), "atom_sphere_voxels": units,
            "cloud_voxels": int(sum(b.nEntries for b in shard.batches)), "ms_per_pass": ms, "ms_per_pass_host_clock": wall,
            "structures_per_s": pool / (ms * 1e-3), "value": units / (ms * 1e-3), "unit": UNIT, "setup_s": round(setup_s, 1),
            "summary": _summary_digest(summary)}, summary


def main_c3(args, rank, world, local_rank):
    """N > 1: BASELINE.json configs[2], strong scaling over a fixed pool (see the module docstring)."""
    import torch
    import torch.distributed as dist
    from pdb_eda_b200 import _device, _lib, multi

    affinity = bind_to_gpu(local_rank)
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries the one JSON line only
    dist.init_process_group("nccl", device_id=device)
    _device.require_cuda()
    params = synthetic.defaultParams()
    spec = synthetic.poolSpec(args.pool)
    costs = synthetic.poolCosts(spec)
    mine = multi.shardStructures(costs, world)[rank]
    t0 = time.perf_counter()
    entries = synthetic.buildPoolEntries([spec[i] for i in mine], params, device)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t0
    units = _pool_units(entries, params)
    shard = multi.PoolShard(entries, params, device=device)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    warmup = max(args.warmup, 3)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    lib = _lib.load()
    # ---- device-resident timing: K passes over the pool, collectives inside
    ms, wall, summary = _time_passes(shard, args.steps, warmup, barrier, device=device)
    # ---- instrumented repeat: per-kernel device times + launch count
    launches0 = lib.pe_launch_count()
    _lib.profile(True, reset=True)
    ms_prof, _, _ = _time_passes(shard, args.steps, 0, barrier, device=device)
    launches = lib.pe_launch_count() - launches0
    prof = _lib.profile()
    _lib.profile(False)
    # ---- end to end: every step uploads the shard's maps from pinned host memory first
    host_maps = []
    for _, mref, _ in entries:
        h = torch.empty(mref.deviceMap.rho.shape, dtype=torch.float32).pin_memory()
        h.copy_(mref.deviceMap.rho)
        host_maps.append(h)
    torch.cuda.synchronize()

    class _E2E:
        def analyze(self, **kw):
            for (_, mref, _), h in zip(entries, host_maps):
                mref.deviceMap.rho.copy_(h, non_blocking=True)
            return shard.analyze(**kw)

    e2e_steps = args.steps
    ms_e2e, _, _ = _time_passes(_E2E(), e2e_steps, 1, barrier, device=device)
    clocks = sampler.stop() if rank == 0 else None
    h2d = sum(h.numel() * 4 for h in host_maps)
    d2h = sum(b.h_mapOut.numel() + b.h_segOut.numel() + b.h_mapStats.numel() for b in shard.batches) * 8

    stats = torch.tensor([ms, ms_e2e, ms_prof, wall], dtype=torch.float64, device=device)
    sums = torch.tensor([units, float(shard.nAtoms), float(sum(b.nEntries for b in shard.batches)), float(h2d), float(d2h),
                         float(len(shard.batches))], dtype=torch.float64, device=device)
    dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    ms, ms_e2e, ms_prof, wall = stats.tolist()
    all_units, all_atoms, all_entries, all_h2d, all_d2h, all_batches = sums.tolist()
    del host_maps

    one = None
    if rank == 0 and not args.no_single:
        # strong-scaling denominator measured in the same run: the same pool on this GPU alone
        del shard, entries
        torch.cuda.empty_cache()
        one, one_summary = run_c3_one_gpu(args.pool, args.steps, device, params)
        a, b = _summary_digest(summary), one["summary"]
        close = lambda x, y: abs(x - y) <= 1e-9 * max(abs(x), abs(y), 1e-300)
        one["same_results_as_%d_gpus" % world] = bool(
            a["structures"] == b["structures"] and a["num_voxels_aggregated"] == b["num_voxels_aggregated"] and
            close(a["total_aggregated_density"], b["total_aggregated_density"]) and
            close(a["total_aggregated_electrons"], b["total_aggregated_electrons"]) and
            all(close(a["median_diffs"][k], b["median_diffs"][k]) for k in a["median_diffs"]) and
            np.array_equal(np.asarray(summary["rows"])[:, 0], np.asarray(one_summary["rows"])[:, 0]))
    c4 = run_c4(args, rank, world, device) if not args.no_c4 else None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        kernels = []
        for name, (count, kms) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
            kernels.append({"kernel": name, "launches": count, "ms_total": round(kms, 4), "us_per_launch": round(kms * 1e3 / max(count, 1), 2)})
        # rank 0's share of the pool for the per-kernel lines (kernel times are rank 0's)
        dominant = kernels[0] if kernels else None
        roof = None
        # algorithmic bytes per launch on rank 0 (DESIGN.md section 3.6): (bytes per pool voxel, per atom, per sphere voxel)
        c3_bytes = {
            "cloud_pair_kernel": (11.0, 48.0, 0.0, "latency",
                                  "one warp per atom: its clouds as byte masks in shared memory, neighbour atoms from the per-structure "
                                  "cell grid, their voxels tested against the masks, (cloud, cloud) pairs united in two union-find "
                                  "forests: dependent random loads (cell slot -> chain -> entries -> parents), bound by their latency; "
                                  "algorithmic bytes = key + cloud number (10 B) read and first flag (1 B) written per pool voxel, "
                                  "48 B of records per atom"),
            "cloud_fill_kernel": (22.0, 132.0, 0.0, "issue",
                                  "one warp per atom: bitmap from the count pass -> ordered voxel list -> bit-parallel flood fill -> "
                                  "entries (key, density, owner, cloud: 18 B written + 4 B gathered per pool voxel) -> per-cloud sums; "
                                  "issue slots 60 % busy (profiles/r02_c3_pool.md), not a streaming kernel"),
            "cloud_count_kernel": (0.0, 64.0, 4.0, "issue",
                                   "one warp per atom: sphere enumeration with exact float64 distance tests + one 4-byte gather per "
                                   "in-sphere voxel; 64 B per atom (coordinates, radius, count, bitmap for the fill pass)"),
            "cloud_merge_kernel": (30.0, 16.0, 0.0, "latency",
                                   "hash-table path (batches the pair kernel cannot hold): 14 table probes per pool voxel + union-find"),
        }
        if dominant is not None:
            r0_entries = all_entries / world
            r0_atoms = all_atoms / world
            r0_sphere = all_units / world
            pe, pa, ps, bound, note = c3_bytes.get(dominant["kernel"], (0.0, 0.0, 0.0, "latency", "no algorithmic byte model for this kernel"))
            per_launch = (pe * r0_entries + pa * r0_atoms + ps * r0_sphere) / max(dominant["launches"] / args.steps, 1)
            t = dominant["ms_total"] / max(dominant["launches"], 1) * 1e-3
            ach = per_launch / t / 1e9
            roof = {"kernel": dominant["kernel"], "bound": bound, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                    "frac": round(ach / peak, 4), "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": per_launch,
                    "us_per_launch": dominant["us_per_launch"],
                    "note": note + "; rank 0's share of the pool (an even share is assumed)"}
        value = all_units / (ms * 1e-3)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "C3: multiple-structures mode, pool of %d synthetic structures (64^3-256^3 maps, P1 / P2(1) / P2(1)2(1)2(1) / "
                                       "P4(3)2(1)2 / P6(5)22, %d atoms), cloud aggregation per structure (analyzePDBID) in batches + fused "
                                       "all-reduce of the cumulative statistics + all-gather of the rows inside the timed region"
                                       % (args.pool, int(all_atoms)),
                           "parallelism": "structures sharded over %d GPUs longest-first (multi.shardStructures); no data-path collective" % world,
                           "pool": args.pool, "pool_of_baseline": 4096,
                           "l2": "inputs larger than L2 (%.1f GB of maps per pass over the pool); no explicit flush" % (all_h2d / 1e9)},
                "units_per_step": {"atom_sphere_voxels": all_units, "cloud_voxels": all_entries, "atoms": all_atoms, "structures": args.pool,
                                   "blob_ccl_voxels": 0.0},
                "structures_per_s": args.pool / (ms * 1e-3),
                "e2e": {"value": all_units / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": all_h2d, "d2h_bytes_per_step": all_d2h,
                        "ms_per_step": ms_e2e, "structures_per_s": args.pool / (ms_e2e * 1e-3), "steps": e2e_steps,
                        "h2d_gb_per_s_per_rank": round(all_h2d / world / (ms_e2e * 1e-3) / 1e9, 2), "cpu_affinity_rank0": affinity},
                "gpu_launches": int(launches), "roofline": roof, "kernels": kernels[:14], "ms_per_step_profiled": ms_prof,
                "ms_per_step_host_clock": wall, "gpu_busy_frac_rank0": round(sum(k["ms_total"] for k in kernels) / (ms_prof * args.steps), 3),
                "batches": int(all_batches), "setup_s_rank0": round(setup_s, 1), "summary": _summary_digest(summary),
                "pool_on_one_gpu": one, "c4": c4, "clocks": clocks}
        print(json.dumps(line))
    dist.barrier()
    dist.destroy_process_group()


def run_c4(args, rank, world, device):
    """BASELINE.json configs[3]: one n^3 Fo-Fc map (n = --c4-n, default 1024) slab-partitioned over the ranks with halo label
    merge (slab.SlabLabeller: pe_blob_label per slab, one all-gather, CUDA merge, one all-reduce), against the whole map on one
    GPU (rank 0, the same pre-allocated calling pattern), timed in the same run; results compared on rank 0."""
    import torch
    import torch.distributed as dist
    from pdb_eda_b200 import ccp4, slab
    n = args.c4_n
    hdr = ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((n, n, n), (n * 0.5,) * 3 + (90, 90, 90), (n, n, n)))
    s0, s1 = slab.slabRanges(n, world)[rank]
    vol = synthetic.smoothNoiseMapDevice(n, seed=4, device=device)           # every rank generates the same map, keeps its slab
    mine = vol[s0:s1].contiguous()
    if rank != 0:
        del vol
        torch.cuda.empty_cache()
    cut = 3.0
    lab = slab.SlabLabeller(hdr, s0, s1, world, rank, device)
    for _ in range(3):
        parts = lab.label(mine, cut, -cut)
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = args.steps
    e0.record()
    for _ in range(reps):
        parts = lab.label(mine, cut, -cut)
    e1.record()
    dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out = None
    if rank == 0:
        keep = [{"n_blobs": p["n_blobs"], "stats": p["stats"].clone()} for p in parts]
        del lab, parts
        torch.cuda.empty_cache()
        one_ms = ok = None
        if n ** 3 < 2 ** 31:                                                 # one pe_blob_label call takes fewer than 2^31 voxels
            whole_lab = slab.SlabLabeller(hdr, 0, n, 1, 0, device)          # world = 1: the whole map, no collective
            for _ in range(3):
                whole = whole_lab.label(vol, cut, -cut)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps):
                whole = whole_lab.label(vol, cut, -cut)
            e1.record()
            torch.cuda.synchronize()
            ok = bool(all(w["n_blobs"] == p["n_blobs"] and torch.allclose(w["stats"], p["stats"], rtol=1e-9, atol=1e-9)
                          for w, p in zip(whole, keep)))
            one_ms = e0.elapsed_time(e1) / reps
        out = {"workload": "C4: %d^3 Fo-Fc map, +-3 sigma blobs, %d slabs along the section axis, halo label merge over NCCL" % (n, world),
               "blob_ccl_voxels": float(n) ** 3, "ms_slabs": t.item(), "value_slabs": float(n) ** 3 / (t.item() * 1e-3),
               "ms_whole_map_one_gpu": one_ms, "value_whole_map_one_gpu": float(n) ** 3 / (one_ms * 1e-3) if one_ms else None,
               "unit": "blob-CCL voxels/s", "green_blobs": int(keep[0]["n_blobs"]), "red_blobs": int(keep[1]["n_blobs"]),
               "same_blobs_and_sums_as_whole_map": ok, "collectives_per_call": 2}
        if one_ms is None:
            out["note"] = "the whole map (%d voxels) is beyond one call's 2^31: slabs only (tests/test_baseline_configs.py checks such a map)" % n ** 3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--pool", type=int, default=1024, help="structures in the config-3 pool (BASELINE.json: 4,096)")
    ap.add_argument("--c4-n", type=int, default=1024, help="edge of the config-4 map")
    ap.add_argument("--no-single", action="store_true", help="N > 1: skip timing the pool on one GPU")
    ap.add_argument("--no-c4", action="store_true", help="N > 1: skip the config-4 slab run")
    ap.add_argument("--no-c3", action="store_true", help="N = 1: skip the config-3 pool key")
    ap.add_argument("--no-c1", action="store_true", help="reference arm: skip the full-size config-1 pass")
    ap.add_argument("--dump-outputs", metavar="DIR", help="N = 1: write what the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl != "b200" or world > 1):
        ap.error("--dump-outputs writes the outputs of the one-GPU B200 run (--impl b200 without torchrun)")
    if args.impl == "reference":
        main_reference(args, rank, world)
    elif world > 1:
        main_c3(args, rank, world, local_rank)
    else:
        main_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
