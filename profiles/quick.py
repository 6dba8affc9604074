#!/usr/bin/env python3
"""Fast kernel-level timing of the C2-shaped workload with device-generated inputs (no 25 s host map synthesis):
smoothed-noise maps made in HBM, residues placed at random.  Used for ncu captures and tuning; bench.py is the
number that counts.   usage: python profiles/quick.py [steps] [n] [residues]"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pdb_eda_b200 import _device, _lib, ccp4, synthetic  # noqa: E402
from pdb_eda_b200.pipeline import VoxelPass  # noqa: E402

if os.environ.get("PE_LIB"):  # A/B runs of two builds of the library (tuning only)
    _lib.LIB_PATH = os.path.abspath(os.environ["PE_LIB"])

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
n = int(sys.argv[2]) if len(sys.argv) > 2 else 384
nres = int(sys.argv[3]) if len(sys.argv) > 3 else 8000
cell = n * 0.5
hdr = ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((n, n, n), (cell,) * 3 + (90, 90, 90), (n, n, n)))
geom = _device.geom_from_header(hdr)
dens = _device.DeviceMap(geom, synthetic.smoothNoiseMapDevice(n, seed=1).reshape(-1))
diff = _device.DeviceMap(geom, synthetic.smoothNoiseMapDevice(n, seed=2).reshape(-1))
rng = np.random.default_rng(0)
ca = rng.uniform(4, cell - 4, (nres, 3))
offs = np.array([o for _, o, _ in synthetic._ALA_ATOMS])
xyz = np.round((ca[:, None, :] + offs[None, :, :]).reshape(-1, 3), 3).astype(np.float32).astype(np.float64)
radii = np.tile(np.array([0.78, 0.72, 0.66, 0.81, 0.84], dtype=np.float32), nres)
start = np.arange(0, 5 * nres + 1, 5, dtype=np.int32)
vp = VoxelPass(dens, diff, xyz, radii, start, 3.5)
for _ in range(3):
    vp.step()
torch.cuda.synchronize()
_lib.profile(True, reset=True)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(steps):
    vp.step()
e1.record()
torch.cuda.synchronize()
prof = _lib.profile()
_lib.profile(False)
print("ms/step (profiled): %.4f" % (e0.elapsed_time(e1) / steps))
e0.record()
for _ in range(steps):
    vp.step()
e1.record()
torch.cuda.synchronize()
print("ms/step: %.4f" % (e0.elapsed_time(e1) / steps))
for name, (count, ms) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
    print("%-28s %4d launches %9.2f us/launch" % (name, count, ms * 1e3 / count))
print("units:", vp.unit_counts(), "blob counts:", vp.blob_counts.tolist())
import ctypes
t = (ctypes.c_ulonglong * 12)()
_lib.load().pe_blob_stage_times(t)
t = list(t)
print("blob sparse phases P1..P4 (us):", [round((t[i + 1] - t[i]) / 1e3, 1) for i in range(4)])
u = (ctypes.c_ulonglong * 5)()
_lib.load().pe_sphere_union_warp_cycles(u)
if sum(u):
    tot = float(sum(u))
    print("warp-per-group union kernel, warp cycles by phase (boxes, offsets + tables, membership, gather, reduce): %s; "
          "cycles per group %.0f" % ([round(x / tot, 3) for x in u], tot / (13 + steps * 2) / nres))
