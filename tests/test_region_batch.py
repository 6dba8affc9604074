"""GPU tier of the batched region density / discrepancy path: ``pe_batch_sphere_sums`` (csrc/pe_union.cu, csrc/pe_sphere.cu)
against ``pe_sphere_sums`` per structure bit for bit, ``regionBatch`` rows against the single-structure calls exactly, and
``multiple --single-mode "density | difference ..."`` against ``single`` byte for byte."""
import io
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import cases
import test_metrics_batch as tmb
from pdb_eda_b200 import _lib, ccp4, synthetic, regionBatch
from pdb_eda_b200._device import _ptr

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = ["ortho", "perm", "over", "hex", "tric"]


# ---------------------------------------------------------------------------------------------------- kernel
def _map(name):
    g = cases.GEOMETRIES[name]
    return ccp4.parse(io.BytesIO(synthetic.ccp4Bytes(cases._noise(g["shape"], 11), g["cell"], g["intervals"], crsStart=g["crsStart"],
                                                     axisOrder=g["axisOrder"])), name)


@pytest.fixture(scope="module")
def structures():
    """Structures on the five geometries, with atoms in and beyond the stored map and per-atom radii of 0.5-3.5 A: grouped
    (14 groups of 1-40 atoms, two empty, one of 40 atoms) and per atom (4k+1, 4k+2, 4k+3 atoms, and an empty structure
    between others).  Returns [(DeviceMap, xyz float64, radii float32, groupStart, cut scale)] per mode."""
    maps = {name: _map(name) for name in CASES}
    grouped, atoms = [], []
    for k, name in enumerate(CASES):
        coords, gs, radii = tmb._groups(maps[name], 100 + k)
        grouped.append((maps[name].deviceMap, coords.astype(np.float64), radii, gs))
    for k, (name, n) in enumerate([("ortho", 37), ("perm", 0), ("over", 42), ("hex", 51), ("tric", 60), ("perm", 33), ("over", 1)]):
        rng = np.random.default_rng(200 + k)
        coords = cases.random_atoms(maps[name], n, 200 + k, margin=4.0).reshape(-1, 3)
        atoms.append((maps[name].deviceMap, coords.astype(np.float64), rng.uniform(0.5, 3.5, n).astype(np.float32), None))
    return {"grouped": grouped, "atom": atoms}


def _cuts(dm, which):
    m, s = dm.mean_std()
    c = float(np.float32(m + s))
    return {"none": (0.0, 0.0), "pos": (c, 0.0), "both": (c, -c)}[which]


def _batch_sums(items, which, mapIndex=None):
    """pe_batch_sphere_sums over items [(dm, xyz, radii, groupStart or None)]; returns the rows of every item.  mapIndex:
    per item the map index its groups name (default: its own)."""
    lib = _lib.load()
    n = len(items)
    grouped = items[0][3] is not None
    maps = (_lib.PeSumsMap * n)()
    atomStart, groupStart, groupMap, nG = [0], [], [], []
    for k, (dm, xyz, r, gs) in enumerate(items):
        maps[k].geom, maps[k].d_rho = dm.geom, dm.rho.data_ptr()
        maps[k].cut_pos, maps[k].cut_neg = _cuts(dm, which)
        g = len(xyz) if gs is None else len(gs) - 1
        if gs is not None:
            groupStart.extend((np.asarray(gs[:-1]) + atomStart[-1]).tolist())
        groupMap.extend([k if mapIndex is None else mapIndex[k]] * g)
        nG.append(g)
        atomStart.append(atomStart[-1] + len(xyz))
    nA, nGroups = atomStart[-1], sum(nG)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    d_maps = torch.frombuffer(bytearray(bytes(maps)), dtype=torch.uint8).cuda()
    d_xyz = up(np.concatenate([it[1] for it in items]).reshape(-1, 3))
    d_r = up(np.concatenate([it[2] for it in items]).astype(np.float32))
    d_gm = up(np.asarray(groupMap, dtype=np.int32))
    d_gs = up(np.asarray(groupStart + [nA], dtype=np.int32)) if grouped else None
    d_as = up(np.asarray(atomStart, dtype=np.int32))
    out = torch.full((max(nGroups, 1), 8), -7.0, dtype=torch.float64, device="cuda")
    ws = torch.empty(int(lib.pe_batch_sphere_sums_workspace_bytes(nA)), dtype=torch.uint8, device="cuda")
    _lib.check(lib.pe_batch_sphere_sums(n, _ptr(d_maps), nA, _ptr(d_xyz), _ptr(d_r), nGroups, _ptr(d_gm), _ptr(d_gs), _ptr(d_as),
                                        _ptr(out), _ptr(ws), None), "pe_batch_sphere_sums")
    h = out.cpu().numpy()[:nGroups]
    base = np.concatenate(([0], np.cumsum(nG)))
    return [h[base[k]:base[k + 1]] for k in range(n)]


def _alone(item, which):
    dm, xyz, r, gs = item
    cp, cn = _cuts(dm, which)
    if len(xyz) == 0:
        return np.zeros((0, 8))
    return dm.sphere_sums(xyz, r, gs, cp, cn).cpu().numpy()


@pytest.mark.parametrize("mode", ["grouped", "atom"])
@pytest.mark.parametrize("which", ["none", "pos", "both"])
def test_bit_identical_to_the_single_structure_launch(structures, mode, which):
    items = structures[mode]
    got = _batch_sums(items, which)
    for k, item in enumerate(items):
        want = _alone(item, which)
        assert got[k].shape == want.shape
        assert got[k].tobytes() == want.tobytes(), (mode, which, k)
    flags = np.concatenate([g[:, 6] for g in got])
    assert (flags == 0).any() and (flags == 1).any()                # atoms beyond the stored map occur
    if mode == "grouped":
        assert any((g[:, 0] == 0).any() for g in got)                 # empty groups: zero rows


def test_small_and_large_quads_both_occur(structures):
    """The per-atom items reach both quad_sums (boxes at most 8 wide) and the one-warp-per-atom path."""
    dims = []
    for dm, xyz, r, gs in structures["atom"]:
        if len(xyz):
            dims.append(dm.sphere_lists(xyz, r)["box"][:, 3:].max(dim=1).values.cpu().numpy())
    d = np.concatenate(dims)
    assert (d <= 8).any() and (d > 8).any()


@pytest.mark.parametrize("mode", ["grouped", "atom"])
def test_out_of_range_map_index_gives_nan_rows(structures, mode):
    items = structures[mode]
    n = len(items)
    bad = [k if k != 2 else n for k in range(n)]                     # item 2 names no map of the table
    bad[4] = -1
    got = _batch_sums(items, "both", bad)
    for k, item in enumerate(items):
        if k in (2, 4):
            assert np.isnan(got[k]).all()
        else:
            assert got[k].tobytes() == _alone(item, "both").tobytes()


@pytest.mark.parametrize("mode", ["grouped", "atom"])
def test_deterministic_and_independent_of_batch_order(structures, mode):
    items = structures[mode]
    a = _batch_sums(items, "both")
    b = _batch_sums(items, "both")
    perm = np.random.default_rng(5).permutation(len(items))
    c = _batch_sums([items[i] for i in perm], "both")
    for k in range(len(items)):
        assert a[k].tobytes() == b[k].tobytes()
    for j, i in enumerate(perm):
        assert c[j].tobytes() == a[i].tobytes()


# ---------------------------------------------------------------------------------------------------- rows
CALLS = [("density", "atom"), ("density", "residue"), ("density", "symmetry-atom"),
         ("difference", "atom"), ("difference", "residue"), ("difference", "symmetry-atom")]


def _single(an, kind, level, radius=3.5, numSD=None, type="", atomMask=None, useOptimizedRadii=False):
    numSD = (1.5 if kind == "density" else 3.0) if numSD is None else numSD
    if kind == "density":
        if level == "atom":
            return an.calculateAtomRegionDensity(radius, numSD, type, useOptimizedRadii)
        if level == "residue":
            return an.calculateResidueRegionDensity(radius, numSD, type, atomMask, useOptimizedRadii)
        return an.calculateSymmetryAtomRegionDensity(radius, numSD, type, useOptimizedRadii)
    if level == "atom":
        return an.calculateAtomRegionDiscrepancies(radius, numSD, type)
    if level == "residue":
        return an.calculateResidueRegionDiscrepancies(radius, numSD, type, atomMask)
    return an.calculateSymmetryAtomRegionDiscrepancies(radius, numSD, type)


def _same(got, want):
    """Exact equality, value and type, of two row lists."""
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert len(g) == len(w)
        for x, y in zip(g, w):
            assert type(x) is type(y), (x, y)
            if isinstance(y, np.ndarray):
                np.testing.assert_array_equal(x, y)
                assert x.dtype == y.dtype
            else:
                assert x == y or (x != x and y != y), (x, y)


@pytest.fixture(scope="module")
def analyzers():
    from pdb_eda_b200 import densityAnalysis
    from pdb_eda_b200.cloudBatch import AtomTable
    densityAnalysis.setGlobals(densityAnalysis._loadDefaultParams())
    tmb.STRUCTS.setdefault("tiny", dict(tmb.STRUCTS["p212121"], residues=1))

    def fresh():
        out = []
        for name, res in [("p212121", 1.0), ("perm", 2.0), ("hex", 3.3)]:
            out.append(tmb._analyzer(tmb._entry_files(name, res, seed=61 + len(out))))
        out.append(tmb._analyzer(tmb._entry_files("tiny", 2.0, seed=70)))                   # too few electrons: no ratio
        out.append(tmb._analyzer(tmb._entry_files("p212121", 2.0, seed=71, remark290=False)))  # no REMARK 290
        an = tmb._analyzer(tmb._entry_files("perm", 2.0, seed=72))                       # ratio through the full pipeline
        atoms = list(an.biopdbObj.get_atoms())
        atoms[5].coord = atoms[4].coord.copy()
        assert not AtomTable.fromStructure(an.biopdbObj, densityAnalysis.paramsGlobal).supported
        out.append(an)
        out.append(0)                                                                   # an entry that did not load
        return out
    return fresh


OPTIONS = [dict(), dict(radius=2.25, numSD=0.8, type="CA"), dict(numSD=2.0, useOptimizedRadii=True),
           dict(radius=3.0, atomMask={"ALA": ["N", "CA", "C", "O"], "HOH": ["O"]}, useOptimizedRadii=True),
           dict(atomMask={"ALA": ["CA", "CB"]}), dict(type="HOH")]


@pytest.mark.parametrize("kind,level", CALLS)
def test_rows_equal_the_single_structure_calls(analyzers, kind, level):
    ans = analyzers()
    for k, options in enumerate(OPTIONS):
        if kind == "difference":
            options = {o: v for o, v in options.items() if o != "useOptimizedRadii"}
        if level != "residue":
            options = {o: v for o, v in options.items() if o != "atomMask"}
        got = regionBatch.analyzeRegions(ans, kind, level, maxBytes=3 << 20, **options)   # several batches
        for j, an in enumerate(ans):
            if not an:
                assert got[j] is None
                continue
            try:
                want = _single(an, kind, level, **options)
            except Exception:
                assert got[j] is None, (k, j)
                continue
            assert got[j] is not None, (k, j)
            _same(got[j], want)
        assert got[3] is None                                                          # no ratio, even without rows
        if k == 0:
            assert all(got[j] for j in (0, 1, 2, 5))
            if level == "symmetry-atom":
                assert got[4] == []
        if kind == "difference" and level == "residue" and "atomMask" in options and "HOH" not in options["atomMask"]:
            assert all(r is None for r in got)                                         # a residue left without atoms


# ---------------------------------------------------------------------------------------------------- command line
def _single_cli(folder, pdbid, ref, opts):
    from pdb_eda_b200 import singleStructure
    singleStructure.main([pdbid, ref] + opts + ["--pdb-file", os.path.join(folder, "pdb" + pdbid + ".ent"), "--density-file",
                                                os.path.join(folder, pdbid + ".ccp4"), "--diff-file", os.path.join(folder, pdbid + "_diff.ccp4")])


@pytest.fixture(scope="module")
def data_dir(tmp_path_factory):
    folder = str(tmp_path_factory.mktemp("entries"))
    tmb._write_dir(folder, tmb.IDS)
    ids = os.path.join(folder, "ids.txt")
    open(ids, "w").write(" ".join(tmb.IDS + ["9zzz"]))
    return folder, ids


@pytest.mark.parametrize("fmt", ["json", "csv"])
@pytest.mark.parametrize("kind,level", CALLS)
def test_cli_files_are_byte_identical_to_single(data_dir, tmp_path, capsys, kind, level, fmt):
    from pdb_eda_b200 import densityAnalysis, multipleStructures
    densityAnalysis.setGlobals(densityAnalysis._loadDefaultParams())
    folder, ids = data_dir
    out = str(tmp_path / "out")
    opts = [kind, "--" + level, "--out-format", fmt, "--radius", "3.0"] + (["--include-pdbid"] if level != "atom" else [])
    multipleStructures.main([ids, out, "--single-mode", " ".join(opts), "--data-dir", folder])
    summary = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert sorted(os.listdir(out)) == [i + ".result" for i in tmb.IDS]
    rows = 0
    for pdbid in tmb.IDS:
        ref = str(tmp_path / (pdbid + ".single"))
        _single_cli(folder, pdbid, ref, opts)
        text = open(ref).read()
        assert open(os.path.join(out, pdbid + ".result")).read() == text
        rows += len(json.loads(text)) if fmt == "json" else len(text.strip().splitlines()) - 1
    assert summary == {"ok": 3, "failed": 1, "rows": rows} and rows > 0


def test_cli_two_ranks_under_torchrun(data_dir, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    folder, ids = data_dir
    env = dict(os.environ, PYTHONPATH=ROOT)
    outs = []
    for nproc in (1, 2):
        out = str(tmp_path / ("out%d" % nproc))
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr", "127.0.0.1",
               "--master-port", "29648", "-m", "pdb_eda_b200", "multiple", ids, out, "--single-mode",
               "difference --symmetry-atom --include-pdbid", "--data-dir", folder]
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
        assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
        assert '"failed": 1' in res.stdout and '"ok": 3' in res.stdout
        outs.append(out)
    assert sorted(os.listdir(outs[0])) == sorted(os.listdir(outs[1])) == [i + ".result" for i in tmb.IDS]
    for name in os.listdir(outs[0]):
        assert open(os.path.join(outs[0], name)).read() == open(os.path.join(outs[1], name)).read()
