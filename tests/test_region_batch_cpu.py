"""CPU tier of the batched region density / discrepancy path (pdb_eda_b200/regionBatch.py, pe_batch_sphere_sums): argument
errors without a device, which ``--single-mode`` options run batched, and the numpy row builders against the per-row
arithmetic of the single-structure calls."""
import types

import numpy as np
import pytest

from pdb_eda_b200 import _lib, densityAnalysis, multipleStructures, regionBatch


def test_argument_errors_without_a_device():
    lib = _lib.load()
    assert lib.pe_batch_sphere_sums_workspace_bytes(10) >= 10 * 32
    assert lib.pe_batch_sphere_sums(-1, None, 0, None, None, 1, None, None, None, None, None, None) == -1   # negative size
    assert b"negative size" in lib.pe_last_error()
    assert lib.pe_batch_sphere_sums(1, None, -2, None, None, 1, None, None, None, None, None, None) == -1
    assert lib.pe_batch_sphere_sums(1, None, 0, None, None, 0, None, None, None, None, None, None) == 0     # nothing to do
    assert lib.pe_batch_sphere_sums(0, None, 4, None, None, 2, None, None, None, None, None, None) == -1    # groups without maps
    assert b"groups without maps" in lib.pe_last_error()
    assert lib.pe_batch_sphere_sums(1, None, 4, None, None, 2, None, None, None, None, None, None) == -1    # null pointers
    assert b"null pointer" in lib.pe_last_error()
    p = 16                                                                                                # any non-null address
    # per-atom sums: one group per atom, and the structures' atom offsets are required
    assert lib.pe_batch_sphere_sums(1, p, 4, p, p, 3, p, None, p, p, p, None) == -1
    assert b"n_groups must equal n_atoms" in lib.pe_last_error()
    assert lib.pe_batch_sphere_sums(1, p, 4, p, p, 4, p, None, None, p, p, None) == -1
    assert b"d_atom_start" in lib.pe_last_error()


def test_host_table_rejects_bad_cutoffs():
    dm = types.SimpleNamespace(rho=types.SimpleNamespace(numel=lambda: 8))
    with pytest.raises(ValueError):
        regionBatch.RegionEntry(None, dm, np.zeros((1, 3)), np.ones(1), None, -1.0, 0.0, None)
    with pytest.raises(ValueError):
        regionBatch.RegionEntry(None, dm, np.zeros((1, 3)), np.ones(1), None, 1.0, 0.5, None)


@pytest.mark.parametrize("opts,path", [
    ("density --residue", "region"), ("density --atom --optimized-radii --type CA", "region"),
    ("density --symmetry-atom --num-sd 2", "region"), ("difference --residue --atom-mask m.json", "region"),
    ("difference --atom --radius 2.5", "region"), ("difference --symmetry-atom --include-pdbid", "region"),
    ("statistics --residue", "metrics"), ("statistics --atom", "metrics"), ("statistics --residue --print-validation", None),
    ("map --density", None), ("cloud --residue", None), ("blob --green", None)])
def test_which_single_mode_options_run_batched(opts, path):
    assert multipleStructures.batchedPath(multipleStructures.parseSingleMode(opts)) == path


class _Fake:
    """What ``_regionDensityRows`` / ``_regionDiscrepancyRows`` read of a DensityAnalysis."""

    def __init__(self, ratio, totalAbs, nVoxels):
        dm = types.SimpleNamespace(meanDensity=0.1, stdDensity=0.5, getTotalAbsDensity=lambda c: totalAbs,
                                   deviceMap=types.SimpleNamespace(n_voxels=nVoxels))
        self.densityObj = self.diffDensityObj = dm
        self._ratio = ratio

    def _requireRatio(self):
        return self._ratio


def _random_sums(rng, n):
    s = rng.standard_normal((n, 8)) * 10.0 ** rng.integers(-3, 6, (n, 1))
    s[:, 0] = rng.integers(0, 5000, n)
    s[:, 5] = -np.abs(s[:, 5])
    s[:, 6] = rng.integers(0, 2, n)
    return s


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_row_builders_equal_the_per_row_arithmetic(monkeypatch, seed):
    rng = np.random.default_rng(seed)
    sums = _random_sums(rng, 400)
    ratio = float(rng.uniform(0.05, 3.0))
    fake = _Fake(ratio, float(rng.uniform(1e3, 1e6)), int(rng.integers(10 ** 4, 10 ** 7)))
    monkeypatch.setattr(densityAnalysis.utils, "sphereSums", lambda *a, **k: sums)
    want, _ = densityAnalysis.DensityAnalysis._regionDensityRows(fake, np.zeros((400, 3)), np.ones(400), None, 1.5)
    got = regionBatch.densityRows(sums, ratio)
    want2, _ = densityAnalysis.DensityAnalysis._regionDiscrepancyRows(fake, np.zeros((400, 3)), 3.5, None, 3.0)
    got2 = regionBatch.discrepancyRows(sums, ratio, fake.diffDensityObj.getTotalAbsDensity(0) / fake.diffDensityObj.deviceMap.n_voxels)
    for g, w in list(zip(got, want)) + list(zip(got2, want2)):
        assert len(g) == len(w)
        for x, y in zip(g, w):
            assert type(x) is type(y) and x == y, (x, y)
