"""GPU tier of the batched RSCC / RSR path: ``pe_pair_union_metrics`` (csrc/pe_metrics.cu) against an independent host
statement and against the per-structure chain, its determinism, ``metricsBatch`` rows against ``residueMetrics()`` /
``atomMetrics()``, and ``multiple --single-mode`` end to end on one and on two ranks."""
import csv
import io
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import cases
from oracle import orc
from pdb_eda_b200 import _blas, _device, ccp4, cutils, metricsBatch, synthetic

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = ["ortho", "perm", "over", "hex", "tric"]


# ---------------------------------------------------------------------------------------------------- kernel inputs
def _pair(name, shift=0.0):
    """(2Fo-Fc DensityMatrix, Fo-Fc DeviceMap, host geometry, host fo, host diff) of a geometry of tests/cases.py."""
    g = cases.GEOMETRIES[name]
    fo = cases._noise(g["shape"], 11) + np.float32(shift)
    diff = (cases._noise(g["shape"], 12) * np.float32(0.3)).astype(np.float32)
    dm = ccp4.parse(io.BytesIO(synthetic.ccp4Bytes(fo, g["cell"], g["intervals"], crsStart=g["crsStart"],
                                                   axisOrder=g["axisOrder"])), name)
    dd = _device.DeviceMap(dm.deviceMap.geom, torch.from_numpy(diff.reshape(-1).copy()).cuda())
    return dm, dd, orc.geom(dm.header, dm.origin, mv=_blas.probe()), fo.reshape(-1), diff.reshape(-1)


def _groups(dm, seed, nGroups=14, margin=4.0):
    """Groups of 1-40 atoms in and beyond the stored map (a 40-atom group spans several tiles), two of them empty, with
    per-atom radii of 0.5-3.5 A."""
    rng = np.random.default_rng(seed)
    sizes = rng.integers(1, 41, nGroups)
    sizes[[3, 9]] = 0
    sizes[5] = 40
    coords = cases.random_atoms(dm, int(sizes.sum()), seed, margin=margin)
    radii = rng.uniform(0.5, 3.5, len(coords)).astype(np.float32)
    return coords, np.concatenate(([0], np.cumsum(sizes))), radii


def _batch(items):
    """One MetricsBatch over items (dm, dd, coords, groupStart, radii), per-atom radii set on the device."""
    entries = [metricsBatch.MetricsEntry(dm.deviceMap, dd, c, gs, 1.0) for dm, dd, c, gs, _ in items]
    b = metricsBatch.MetricsBatch(entries)
    b.d_radius.copy_(torch.from_numpy(np.concatenate([r for *_, r in items]).astype(np.float32)))
    return b


def _host_sums(g, fo, diff, coords, gs, radii):
    """orc.sphere_list per atom -> set-union per group -> orc.point_density on both maps -> float64 two-pass sums.
    Returns (sums (G, 8), magnitudes (G, 8), [(fo, fc) per group])."""
    sums, mags, values = [], [], []
    for k in range(len(gs) - 1):
        voxels = set()
        for a in range(gs[k], gs[k + 1]):
            voxels.update(map(tuple, orc.sphere_list(g, fo, coords[a], radii[a]).tolist()))
        crs = np.array(sorted(voxels), dtype=np.int32).reshape(-1, 3)
        f, _ = orc.point_density(g, fo, crs)
        d, _ = orc.point_density(g, diff, crs)
        c = f - d * 2
        n = len(crs)
        mf, mc = (f.sum() / n, c.sum() / n) if n else (0.0, 0.0)
        x, y = f - mf, c - mc
        terms = [f, c, np.abs(f - c), np.abs(f + c), x * x, y * y, x * y]
        sums.append([n] + [t.sum() for t in terms])
        mags.append([n] + [np.abs(t).sum() + 1e-3 * n for t in terms])
        values.append((f, c))
    return np.array(sums), np.array(mags), values


def _close_sums(got, want, mag, rtol=1e-12):
    """tests/test_set_algebra_vs_host.py::_close_sums: |got - want| <= rtol x (sum of the magnitudes of the terms)."""
    bad = np.abs(np.asarray(got) - np.asarray(want)) > rtol * np.asarray(mag) + 1e-300
    assert not bad.any(), np.argwhere(bad)[:5].tolist()


@pytest.fixture(scope="module")
def five():
    out = []
    for k, name in enumerate(CASES):
        dm, dd, g, fo, diff = _pair(name)
        coords, gs, radii = _groups(dm, 100 + k)
        out.append((name, dm, dd, g, fo, diff, coords, gs, radii))
    return out


def test_kernel_against_host_statement(five):
    from scipy import stats
    b = _batch([(dm, dd, c, gs, r) for _, dm, dd, _, _, _, c, gs, r in five])
    got = b.run()
    multi_tile = 0
    for (name, dm, dd, g, fo, diff, coords, gs, radii), out in zip(five, got):
        want, mag, values = _host_sums(g, fo, diff, coords, gs, radii)
        np.testing.assert_array_equal(out[:, 0], want[:, 0], err_msg=name)                      # n exact
        _close_sums(out[:, 1:], want[:, 1:], mag[:, 1:])
        assert (out[[3, 9]] == 0).all()                                                      # empty groups: zero rows
        rscc, rsr = metricsBatch.rsccRsr(out)
        for k, (f, c) in enumerate(values):
            if len(f) > 2 and f.std() > 0 and c.std() > 0:
                assert abs(rscc[k] - stats.pearsonr(f, c)[0]) <= 1e-10 * max(1.0, abs(rscc[k])), (name, k)
            if len(f):
                np.testing.assert_allclose(rsr[k], np.abs(f - c).sum() / np.abs(f + c).sum(), rtol=1e-12)
        boxes = [orc.sphere_box(g, coords[a], radii[a]) for a in range(gs[5], gs[6])]
        lo = np.min([b0 for b0, _ in boxes], axis=0)
        hi = np.max([b0 + d for b0, d in boxes], axis=0)
        multi_tile += int((hi - lo > 32).any())
    assert multi_tile >= 3                       # the 40-atom groups span several tiles


def test_offset_fo_map_does_not_cancel():
    """A 2Fo-Fc map offset by 1,000 (covered voxels only): centred moments keep RSCC to 1e-10; a one-pass sum of squares
    minus n x mean^2 would lose about six digits here."""
    from scipy import stats
    dm, dd, g, fo, diff = _pair("ortho", shift=1000.0)
    coords, gs, radii = _groups(dm, 7, margin=-4.0)
    out = _batch([(dm, dd, coords, gs, radii)]).run()[0]
    want, mag, values = _host_sums(g, fo, diff, coords, gs, radii)
    np.testing.assert_array_equal(out[:, 0], want[:, 0])
    _close_sums(out[:, 1:], want[:, 1:], mag[:, 1:])
    rscc, _ = metricsBatch.rsccRsr(out)
    checked = 0
    for k, (f, c) in enumerate(values):
        if len(f) > 2:
            assert abs(rscc[k] - stats.pearsonr(f, c)[0]) <= 1e-10, k
            checked += 1
    assert checked >= 10


def test_same_inputs_through_the_existing_chain(five):
    got = _batch([(dm, dd, c, gs, r) for _, dm, dd, _, _, _, c, gs, r in five]).run()
    for (name, dm, dd, g, fo, diff, coords, gs, radii), out in zip(five, got):
        lists = cutils.sphereLists(dm, coords, radii, 0.0)
        group = torch.from_numpy(np.repeat(np.arange(len(gs) - 1), np.diff(gs)).astype(np.int32)).cuda()[lists["atom"].long()]
        _, first, _ = cutils.clusterCrs(lists["crs"], group, wantFirst=True)
        diffDm = type("M", (), {"deviceMap": dd})()
        chain = cutils.pairMetrics(dm, diffDm, lists["crs"], group, first, len(gs) - 1).cpu().numpy()
        np.testing.assert_array_equal(out[:, 0], chain[:, 0], err_msg=name)
        for a, b in zip(metricsBatch.rsccRsr(out), metricsBatch.rsccRsr(chain)):
            np.testing.assert_array_equal(np.isnan(a), np.isnan(b))
            ok = ~np.isnan(a)
            np.testing.assert_allclose(a[ok], b[ok], rtol=1e-10, atol=1e-10)


def test_determinism(five):
    items = [(dm, dd, c, gs, r) for _, dm, dd, _, _, _, c, gs, r in five]
    b = _batch(items)
    first = [x.copy() for x in b.run()]
    second = b.run()
    for x, y in zip(first, second):
        assert x.tobytes() == y.tobytes()
    perm = [3, 0, 4, 2, 1]
    for k, out in zip(perm, _batch([items[k] for k in perm]).run()):
        assert out.tobytes() == first[k].tobytes()


# ---------------------------------------------------------------------------------------------------- rows of analyzers
STRUCTS = {
    "p212121": dict(n=(64, 64, 64), cell=(32.0, 32.0, 32.0, 90, 90, 90), sg="P 21 21 21", residues=70, axisOrder=(1, 2, 3),
                    crsStart=(0, 0, 0)),
    "perm": dict(n=(60, 72, 66), cell=(30.0, 36.0, 33.0, 90, 90, 90), sg="P 1 21 1", residues=60, axisOrder=(2, 3, 1),
                 crsStart=(-4, 7, 3)),
    "hex": dict(n=(60, 60, 80), cell=(30.0, 30.0, 40.0, 90, 90, 120), sg="P 65 2 2", residues=40, axisOrder=(1, 2, 3),
                crsStart=(0, 0, 0)),
}


def _entry_files(name, resolution, seed=31, remark290=True, zeroResidue=None):
    """(pdb text, 2Fo-Fc bytes, Fo-Fc bytes) of a synthetic poly-ALA entry with waters (HETATM)."""
    from pdb_eda_b200 import structure
    c = STRUCTS[name]
    omat = synthetic.orthoMatrix(c["cell"])
    skew = c["cell"][5] != 90
    lo = (omat @ np.array([0.25, 0.25, 0.1])) if skew else np.zeros(3)
    hi = (omat @ np.array([0.6, 0.75, 0.9])) if skew else np.array(c["cell"][:3])
    lo, hi = np.minimum(lo, hi), np.maximum(lo, hi)
    st = synthetic.polyAlaStructure(c["residues"], lo - 3 * skew, hi + 3 * skew, seed=seed, residuesPerChain=30, hetero=5)
    if zeroResidue is not None:
        for atom in list(st.get_residues())[zeroResidue].child_list:
            atom.occupancy = 0.0
    a, b = synthetic.mapPair(st, c["n"], c["cell"], seed=seed + 6, crsStart=c["crsStart"], axisOrder=c["axisOrder"])
    ops = synthetic.cartesianOperators(c["sg"], c["cell"]) if remark290 else None
    text = structure.formatPDB(st, remark290=ops, cell=c["cell"], spaceGroup=c["sg"], resolution=resolution)
    return (text, synthetic.ccp4Bytes(a, c["cell"], c["n"], crsStart=c["crsStart"], axisOrder=c["axisOrder"]),
            synthetic.ccp4Bytes(b, c["cell"], c["n"], crsStart=c["crsStart"], axisOrder=c["axisOrder"]))


def _analyzer(files):
    from pdb_eda_b200 import densityAnalysis
    return densityAnalysis.fromFile(io.StringIO(files[0]), io.BytesIO(files[1]), io.BytesIO(files[2]))


def _same_rows(got, want, metricColumns):
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert len(g) == len(w)
        for j, (x, y) in enumerate(zip(g, w)):
            if j in metricColumns:
                assert (math.isnan(x) and math.isnan(y)) or abs(x - y) <= 1e-10 * max(1.0, abs(y)), (j, x, y)
            elif isinstance(y, np.ndarray):
                np.testing.assert_array_equal(x, y)
            else:
                assert x == y, (j, x, y)


@pytest.fixture(scope="module")
def analyzers():
    from pdb_eda_b200 import densityAnalysis
    densityAnalysis.setGlobals(densityAnalysis._loadDefaultParams())
    out = []
    for name, res in [("p212121", 1.0), ("perm", 2.0), ("hex", 3.3), ("p212121", 7.0), ("hex", 2.0)]:
        out.append(_analyzer(_entry_files(name, res, seed=31 + len(out))))
    out.append(_analyzer(_entry_files("perm", 2.0, seed=40, zeroResidue=3)))     # residue with zero occupancy: fails
    out.append(_analyzer(_entry_files("p212121", 2.0, seed=41, remark290=False)))  # no REMARK 290: no atom rows
    out.append(0)                                                                   # an entry that did not load
    return out


@pytest.mark.parametrize("level", ["residue", "atom"])
def test_rows_against_single_structure_calls(analyzers, level):
    got = metricsBatch.analyzeMetrics(analyzers, level, maxBytes=40 << 20)         # several batches
    for k, an in enumerate(analyzers):
        if not an:
            assert got[k] is None
            continue
        try:
            want = an.residueMetrics() if level == "residue" else an.atomMetrics()
        except Exception:
            assert got[k] is None, k
            continue
        _same_rows(got[k], want, {3, 4} if level == "residue" else {6, 7})
    if level == "residue":
        assert got[5] is None and any(r[2] == "HOH" for r in got[0])
    else:
        assert got[6] == [] and got[5] is not None and len(got[0]) > 0


# ---------------------------------------------------------------------------------------------------- command line
def _write_dir(folder, ids):
    for k, pdbid in enumerate(ids):
        text, a, b = _entry_files(["p212121", "perm", "hex"][k], [1.5, 2.0, 3.3][k], seed=50 + k)
        open(os.path.join(folder, pdbid + ".ccp4"), "wb").write(a)
        open(os.path.join(folder, pdbid + "_diff.ccp4"), "wb").write(b)
        open(os.path.join(folder, "pdb" + pdbid + ".ent"), "w").write(text)


def _read(path, fmt):
    text = open(path).read()
    if fmt == "json":
        return json.loads(text)
    return list(csv.reader(io.StringIO(text)))


def _same_result(got, want, fmt):
    assert len(got) == len(want) > 1
    for g, w in zip(got, want):
        if fmt == "json":
            assert sorted(g) == sorted(w)
            g, w = [g[k] for k in sorted(g)], [w[k] for k in sorted(w)]
        for x, y in zip(g, w):
            try:
                fx, fy = float(x), float(y)
            except (TypeError, ValueError):
                assert x == y
                continue
            assert (math.isnan(fx) and math.isnan(fy)) or abs(fx - fy) <= 1e-10 * max(1.0, abs(fy)), (x, y)


IDS = ["1aaa", "2bbb", "3ccc"]


@pytest.fixture(scope="module")
def data_dir(tmp_path_factory):
    folder = str(tmp_path_factory.mktemp("entries"))
    _write_dir(folder, IDS)
    ids = os.path.join(folder, "ids.txt")
    open(ids, "w").write(" ".join(IDS + ["9zzz"]))
    return folder, ids


@pytest.mark.parametrize("fmt", ["json", "csv"])
def test_cli_single_mode_statistics(data_dir, tmp_path, fmt, capsys):
    from pdb_eda_b200 import densityAnalysis, multipleStructures, singleStructure
    densityAnalysis.setGlobals(densityAnalysis._loadDefaultParams())
    folder, ids = data_dir
    out = str(tmp_path / "out")
    opts = "statistics --residue --include-pdbid --out-format " + fmt
    multipleStructures.main([ids, out, "--single-mode", opts, "--data-dir", folder])
    summary = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert summary["ok"] == 3 and summary["failed"] == 1 and summary["rows"] > 0
    assert sorted(os.listdir(out)) == [i + ".result" for i in IDS]                 # the missing entry writes nothing
    for pdbid in IDS:
        ref = str(tmp_path / (pdbid + ".single"))
        singleStructure.main([pdbid, ref, "statistics", "--residue", "--include-pdbid", "--out-format", fmt, "--pdb-file",
                              os.path.join(folder, "pdb" + pdbid + ".ent"), "--density-file", os.path.join(folder, pdbid + ".ccp4"),
                              "--diff-file", os.path.join(folder, pdbid + "_diff.ccp4")])
        _same_result(_read(os.path.join(out, pdbid + ".result"), fmt), _read(ref, fmt), fmt)


def test_cli_single_mode_other_submode(data_dir, tmp_path, capsys):
    from pdb_eda_b200 import densityAnalysis, multipleStructures, singleStructure
    densityAnalysis.setGlobals(densityAnalysis._loadDefaultParams())
    folder, ids = data_dir
    out = str(tmp_path / "out")
    multipleStructures.main([ids, out, "--single-mode", "density --residue --out-format csv", "--data-dir", folder])
    assert json.loads(capsys.readouterr().out.strip().splitlines()[-1])["failed"] == 1
    ref = str(tmp_path / "ref.csv")
    singleStructure.main(["2bbb", ref, "density", "--residue", "--out-format", "csv", "--pdb-file", os.path.join(folder, "pdb2bbb.ent"),
                          "--density-file", os.path.join(folder, "2bbb.ccp4"), "--diff-file", os.path.join(folder, "2bbb_diff.ccp4")])
    assert open(os.path.join(out, "2bbb.result")).read() == open(ref).read()


def test_cli_two_ranks_under_torchrun(data_dir, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    folder, ids = data_dir
    env = dict(os.environ, PYTHONPATH=ROOT)
    outs = []
    for nproc in (1, 2):
        out = str(tmp_path / ("out%d" % nproc))
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr", "127.0.0.1",
               "--master-port", "29647", "-m", "pdb_eda_b200", "multiple", ids, out, "--single-mode",
               "statistics --atom --include-pdbid", "--data-dir", folder]
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
        assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
        assert '"failed": 1' in res.stdout and '"ok": 3' in res.stdout
        outs.append(out)
    assert sorted(os.listdir(outs[0])) == sorted(os.listdir(outs[1])) == [i + ".result" for i in IDS]
    for name in os.listdir(outs[0]):
        assert open(os.path.join(outs[0], name)).read() == open(os.path.join(outs[1], name)).read()
