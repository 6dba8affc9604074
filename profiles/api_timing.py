#!/usr/bin/env python3
"""Wall-clock of the public DensityAnalysis API on BASELINE.json's configs 1, 2 and 5 (synthetic inputs).
usage: python profiles/api_timing.py [c1|c2|c5 ...]"""
import io
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pdb_eda_b200 import densityAnalysis, structure, synthetic  # noqa: E402

CONFIGS = {
    "c1": dict(n=(96, 96, 96), cell=(48.0, 48.0, 48.0, 90, 90, 90), sg="P 21 21 21", residues=500),
    "c2": dict(n=(384, 384, 384), cell=(192.0, 192.0, 192.0, 90, 90, 90), sg="P 1", residues=8000),
    "c5": dict(n=(120, 120, 240), cell=(60.0, 60.0, 120.0, 90, 90, 120), sg="P 65 2 2", residues=400),
}


def run(name):
    c = CONFIGS[name]
    t0 = time.perf_counter()
    if c["cell"][5] == 90:
        lo, hi = (0, 0, 0), c["cell"][:3]
    else:
        omat = synthetic.orthoMatrix(c["cell"])
        a, b = omat @ np.array([0.3, 0.3, 0.1]), omat @ np.array([0.6, 0.7, 0.9])
        lo, hi = np.minimum(a, b) - 3, np.maximum(a, b) + 3
    st = synthetic.polyAlaStructure(c["residues"], lo, hi, seed=1, residuesPerChain=250)
    d1, d2 = synthetic.mapPair(st, c["n"], c["cell"], seed=7)
    b1, b2 = synthetic.ccp4Bytes(d1, c["cell"], c["n"]), synthetic.ccp4Bytes(d2, c["cell"], c["n"])
    text = structure.formatPDB(st, remark290=synthetic.cartesianOperators(c["sg"], c["cell"]), cell=c["cell"], spaceGroup=c["sg"])
    print("%s: inputs built in %.1f s (%d atoms, %s grid)" % (name, time.perf_counter() - t0, 5 * c["residues"], "x".join(map(str, c["n"]))))
    densityAnalysis.setGlobals(synthetic.defaultParams())

    def timed(label, fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        print("  %-46s %8.3f s" % (label, time.perf_counter() - t))
        return out

    an = timed("fromFile (parse + H2D + mean/std)", lambda: densityAnalysis.fromFile(io.StringIO(text), io.BytesIO(b1), io.BytesIO(b2)))
    assert an != 0
    timed("aggregateCloud", an.aggregateCloud)
    print("    ratio %.6g, %d voxels, %d atom rows, %d residue clouds, %d domain clouds" % (
        an.densityElectronRatio, an.numVoxelsAggregated, len(an.atomCloudDescriptions), len(an.residueCloudDescriptions), len(an.domainCloudDescriptions)))
    green = timed("greenBlobList + redBlobList (one pass)", lambda: (an.greenBlobList, an.redBlobList))
    print("    %d green, %d red blobs" % (len(green[0]), len(green[1])))
    sym = timed("symmetryAtoms", lambda: an.symmetryAtoms)
    print("    %d symmetry atoms" % len(sym))
    timed("calculateAtomSpecificBlobStatistics (green+red)", lambda: an.calculateAtomSpecificBlobStatistics(green[0] + green[1]))
    timed("calculateResidueRegionDensity (3.5 A, mask N,CA,C)", lambda: an.calculateResidueRegionDensity(3.5, 1.5, "", {"ALA": ["N", "CA", "C"]}))
    timed("calculateResidueRegionDiscrepancies (3.5 A)", lambda: an.calculateResidueRegionDiscrepancies(3.5, 3.0))
    timed("calculateAtomRegionDensity (3.5 A)", lambda: an.calculateAtomRegionDensity(3.5))
    if name != "c2":
        timed("calculateSymmetryAtomRegionDensity (3.5 A)", lambda: an.calculateSymmetryAtomRegionDensity(3.5))
    for k in range(3):                                      # the first call includes one-time set-up
        timed("residueMetrics (call %d)" % (k + 1), an.residueMetrics)
    for k in range(3):
        timed("atomMetrics (call %d)" % (k + 1), an.atomMetrics)


if __name__ == "__main__":
    for name in (sys.argv[1:] or ["c1", "c5", "c2"]):
        run(name)
