"""CPU tier of the batched region density / discrepancy path (pdb_eda_b200/regionBatch.py, pe_batch_sphere_sums): argument
errors without a device, which ``--single-mode`` options run batched, and the numpy row builders against the per-row
arithmetic of the reference (pdb_eda/densityAnalysis.py:1037-1068, :1160-1211)."""
import types

import numpy as np
import pytest

from pdb_eda_b200 import _lib, multipleStructures, regionBatch


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


def _random_sums(rng, n):
    s = rng.standard_normal((n, 8)) * 10.0 ** rng.integers(-3, 6, (n, 1))
    s[:, 0] = rng.integers(0, 5000, n)
    s[:, 5] = -np.abs(s[:, 5])
    s[:, 6] = rng.integers(0, 2, n)
    return s


def _density_rows(sums, ratio):
    """The reference's region density per row: [sum of rho > cutoff, / ratio]."""
    return [[row[3], row[3] / ratio] for row in sums]


def _discrepancy_rows(sums, ratio, avg_abs_vox):
    """The reference's region discrepancy per row: the ten values, the expected count as a float times ``int(n)``."""
    rows = []
    for row in sums:
        pos, neg = row[3], row[5]
        actual = pos + neg
        actual_abs = abs(pos) + abs(neg)
        expected = avg_abs_vox * int(row[0])
        rows.append([actual_abs, actual_abs / ratio, expected, expected / ratio, actual, actual / ratio, pos, pos / ratio, neg, neg / ratio])
    return rows


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_row_builders_equal_the_reference_row_arithmetic(seed):
    rng = np.random.default_rng(seed)
    sums = _random_sums(rng, 400)
    ratio = float(rng.uniform(0.05, 3.0))
    avg_abs_vox = float(rng.uniform(1e3, 1e6)) / int(rng.integers(10 ** 4, 10 ** 7))
    want = _density_rows(sums, ratio)
    got = regionBatch.densityRows(sums, ratio)
    want2 = _discrepancy_rows(sums, ratio, avg_abs_vox)
    got2 = regionBatch.discrepancyRows(sums, ratio, avg_abs_vox)
    assert len(got) == len(want) and len(got2) == len(want2)
    for g, w in list(zip(got, want)) + list(zip(got2, want2)):
        assert len(g) == len(w)
        for x, y in zip(g, w):
            assert type(x) is type(y) and x == y, (x, y)
