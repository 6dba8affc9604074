"""VoxelPass.step -- the C2 step bench.py times -- against host references that do not use CUDA, at full size (384^3, 40,000
atoms, 8,000 residues), on shared SMs and on every SM partition the driver grants: every cloud row (C oracle, one atom at a
time), every region row (C oracle, set-union per residue), every blob voxel, label and sum (C oracle flood fill, scipy for the
dense foreground).  Counts, keys, labels, valid flags and candidates match exactly; float64 sums within 1e-12 of the sum of
the magnitudes of their terms.

Also the paths the full-size workload does not take: boxes wider than 8 (two sphere launches), more than 2 M foreground voxels
(P4's chunk prefix in global memory), a voxel exactly at a cutoff (blobs keep rho >= cut, sphere sums keep rho > cut) in each
copy of the threshold test, partially stored maps, an empty red class and an empty foreground."""
import functools
import types
import warnings

import numpy as np
import pytest
import scipy.ndimage as ndi

import bench
from oracle import orc
from pdb_eda_b200 import _blas, ccp4, pipeline, synthetic

EXACT = (0, 2, 4, 6, 7)       # counts, valid flag, candidates
SUMS = (1, 3, 5)              # float64 density sums
C2_SMS = sorted({0, pipeline.BLOB_SMS, *range(8, 137, 8)})
MUST_PARTITION = {8, 48, 96, pipeline.BLOB_SMS} | set(range(8, 57, 8))   # counts the B200 has been seen to split exactly
SMALL_SMS = (0, 8, pipeline.BLOB_SMS)
ATOM_TYPE_RADII = np.array([0.78, 0.72, 0.66, 0.81, 0.84], dtype=np.float32)


def _close_sums(got, want, mag, rtol=1e-12):
    """Sums that differ only in their addition order: |got - want| <= rtol x (sum of the magnitudes of the terms)."""
    got, want, mag = (np.asarray(x, dtype=np.float64) for x in (got, want, mag))
    bad = ~(np.abs(got - want) <= rtol * mag + 1e-300)         # a NaN is bad too
    assert not bad.any(), np.argwhere(bad)[:5].tolist()


def _header(ncrs, cell, intervals, crsStart=(0, 0, 0), axisOrder=(1, 2, 3)):
    return ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header(ncrs, cell, intervals, crsStart, axisOrder))


def _host_geom(hdr):
    return orc.geom(hdr, hdr.origin, mv=_blas.probe())


def _device_map(hdr, values):
    import torch
    from pdb_eda_b200 import _device
    return _device.DeviceMap(_device.geom_from_header(hdr), torch.from_numpy(np.ascontiguousarray(values, np.float32).reshape(-1)).cuda())


def _xyz(g, crs):
    """crs2xyzCoord of an orthogonal cell, vectorised in the oracle's arithmetic (one product, one sum per coordinate)."""
    assert g.orthogonal
    crs = np.asarray(crs, dtype=np.float64)
    return np.stack([crs[:, g.map2xyz[i]] * g.grid_length[i] + g.origin[i] for i in range(3)], axis=1)


def _blob_terms(d, xyz):
    """The 8 terms one voxel adds to its blob's row: n, rho, rho x, rho y, rho z, x, y, z."""
    return np.concatenate((np.ones((len(d), 1)), d[:, None], d[:, None] * xyz, xyz), axis=1)


def _blob_ref(g, rho, cut):
    """createFullBlobList(cut) by the oracle: keys (c U1 + r) U2 + s, labels, rows and the magnitudes of the rows' terms."""
    crs, label, nb = orc.full_blobs(g, rho, cut)
    u = [int(g.unique_ncrs[a]) for a in range(3)]
    key = (crs[:, 0].astype(np.int64) * u[1] + crs[:, 1]) * u[2] + crs[:, 2]
    d, _ = orc.point_density(g, rho, crs)
    mag = np.stack([np.bincount(label, t, minlength=nb) for t in np.abs(_blob_terms(d, _xyz(g, crs))).T], axis=1)
    return {"key": key, "label": label, "stats": orc.blob_stats(g, rho, crs, label, nb), "mag": mag.reshape(nb, 8)}


def _sphere_refs(g, rho, xyz, radii, start, region_radius, cut, full_cell, cut_neg=0.0):
    """Cloud rows (one atom at a time) and region rows (set-union per group) with the magnitudes of their sums' terms."""
    rho = np.ascontiguousarray(rho, np.float32).reshape(-1)
    mag_rho = np.abs(rho)
    n, ng = len(xyz), len(start) - 1
    rr = np.float32(region_radius)
    cloud, cloud_mag = np.zeros((n, 8)), np.zeros((n, 8))
    if cut_neg == 0.0 and full_cell:
        cloud[:, :4] = orc.sphere_sums_batch(g, rho, xyz, radii, cut)
        cloud[:, 6] = 1.0
    else:
        cloud[:, :7] = [orc.sphere_union_sums(g, rho, p[None], r, cut, cut_neg) for p, r in zip(xyz, radii)]
    cloud[:, 7] = [np.prod(orc.sphere_box(g, p, r)[1]) for p, r in zip(xyz, radii)]
    cloud_mag[:, 1] = orc.sphere_sums_batch(g, mag_rho, xyz, radii, 0.0)[:, 1]
    box = np.array([np.prod(orc.sphere_box(g, p, rr)[1]) for p in xyz], dtype=np.float64)
    region, region_mag = np.zeros((ng, 8)), np.zeros((ng, 8))
    for k in range(ng):
        a0, a1 = int(start[k]), int(start[k + 1])
        region[k, :7] = orc.sphere_union_sums(g, rho, xyz[a0:a1], rr, cut, cut_neg)
        region[k, 7] = box[a0:a1].sum()
        region_mag[k, 1] = orc.sphere_union_sums(g, mag_rho, xyz[a0:a1], rr)[1]
    for rows, mag in ((cloud, cloud_mag), (region, region_mag)):
        mag[:, 3] = rows[:, 3]               # terms above cut > 0: all positive
        mag[:, 5] = -rows[:, 5]              # terms below cut_neg < 0: all negative
    return {"cloud": cloud, "cloud_mag": cloud_mag, "region": region, "region_mag": region_mag}


def _host_refs(hdr, rho2, rhof, xyz, radii, start, region_radius, density_cut, diff_cut):
    g = _host_geom(hdr)
    full = all(int(g.ncrs[a]) >= int(g.crs_interval[a]) for a in range(3))
    ref = _sphere_refs(g, rho2, xyz, radii, start, region_radius, density_cut, full)
    rhof = np.ascontiguousarray(rhof, np.float32).reshape(-1)
    ref["green"] = _blob_ref(g, rhof, diff_cut)
    ref["red"] = _blob_ref(g, rhof, -diff_cut)
    return ref


def _step(vp, blob_sms, monkeypatch):
    """One step with PDB_EDA_B200_BLOB_SMS = blob_sms into outputs filled with garbage first; its results (deep copies) and the
    warnings it raised."""
    monkeypatch.setenv("PDB_EDA_B200_BLOB_SMS", str(blob_sms))
    for t in (vp.cloud_out, vp.region_out, vp.blob_stats):
        t.fill_(float("nan"))
    vp.blob_key.fill_(-7)
    vp.blob_label.fill_(-7)
    with warnings.catch_warnings(record=True) as said:
        warnings.simplefilter("always")
        vp.step()
    res = vp.results()
    return {"cloud": res["cloud"].copy(), "region": res["region"].copy(), "blob_counts": res["blob_counts"].copy(),
            **{tag: {k: v.copy() for k, v in res[tag].items()} for tag in ("green", "red")},
            "warnings": [str(w.message) for w in said]}


def _assert_rows(got, want, mag, name):
    assert np.array_equal(got[:, EXACT], want[:, EXACT]), (name, np.argwhere(got[:, EXACT] != want[:, EXACT])[:5].tolist())
    _close_sums(got[:, SUMS], want[:, SUMS], mag[:, SUMS])


def _assert_matches(res, ref):
    counts = res["blob_counts"]
    assert counts[4] == 0                                       # no overflow, no placement failure
    _assert_rows(res["cloud"], ref["cloud"], ref["cloud_mag"], "cloud")
    _assert_rows(res["region"], ref["region"], ref["region_mag"], "region")
    for k, tag in enumerate(("green", "red")):
        got, want = res[tag], ref[tag]
        assert (counts[2 * k], counts[2 * k + 1]) == (len(want["key"]), len(want["stats"])), tag
        assert np.array_equal(got["key"].astype(np.int64) & 0xFFFFFFFF, want["key"]), tag
        assert np.array_equal(got["label"], want["label"]), tag
        assert np.array_equal(got["stats"][:, 0], want["stats"][:, 0]), tag
        _close_sums(got["stats"], want["stats"], want["mag"])


def _assert_same(a, b):
    """Two steps of one pass: the same sphere rows bit for bit, the same blob keys, labels and counts."""
    assert np.array_equal(a["cloud"], b["cloud"]) and np.array_equal(a["region"], b["region"])
    assert np.array_equal(a["blob_counts"], b["blob_counts"])
    for tag in ("green", "red"):
        assert np.array_equal(a[tag]["key"], b[tag]["key"]) and np.array_equal(a[tag]["label"], b[tag]["label"])


@pytest.fixture
def partitions():
    """Destroys the SM partitions a test made, so that green contexts do not accumulate over the module."""
    yield
    pipeline.releasePartitions()


# ------------------------------------------------------------------------------------------------ the C2 workload
@pytest.fixture(scope="module")
def c2():
    """The 384^3 workload bench.py times (seed 2) on the device, its VoxelPass and its host references."""
    from pdb_eda_b200.pipeline import VoxelPass
    work = bench.build_workload(bench.FULL, seed=2)
    n, cell = work["n"], work["cell"]
    hdr = _header((n, n, n), cell, (n, n, n))
    dens, diff = _device_map(hdr, work["fofc2"]), _device_map(hdr, work["fofc"])
    xyz = work["xyz"].astype(np.float64)
    vp = VoxelPass(dens, diff, xyz, work["radii"], work["res_start"], bench.REGION_RADIUS)
    ref = _host_refs(hdr, work["fofc2"], work["fofc"], xyz, work["radii"], work["res_start"], bench.REGION_RADIUS,
                     vp.density_cut, vp.diff_cut)
    return types.SimpleNamespace(work=work, hdr=hdr, dens=dens, diff=diff, xyz=xyz, vp=vp, ref=ref, first={})


@pytest.mark.gpu
def test_cutoffs_from_float64_statistics(c2):
    for dm, name, sigmas, cut in ((c2.dens, "fofc2", 1.5, c2.vp.density_cut), (c2.diff, "fofc", 3.0, c2.vp.diff_cut)):
        v = c2.work[name].astype(np.float64)
        m, s = float(np.mean(v)), float(np.std(v))
        got_m, got_s = dm.mean_std()
        assert abs(got_m - m) <= 1e-12 * s and abs(got_s - s) <= 1e-12 * s, name
        assert cut == float(np.float32(m + sigmas * s)), name


@pytest.mark.gpu
@pytest.mark.parametrize("k", C2_SMS)
def test_c2_step_against_host(c2, k, monkeypatch, partitions):
    got = _step(c2.vp, k, monkeypatch)
    if k:
        part = pipeline.smPartition(c2.vp.device, k)
        if part is None:
            assert k not in MUST_PARTITION, got["warnings"]
            pytest.skip("the driver refuses a partition of %d SMs: %s" % (k, "; ".join(got["warnings"])))
    assert len(got["green"]["key"]) > 50_000 and len(got["red"]["key"]) > 10_000
    _assert_matches(got, c2.ref)
    _assert_same(got, c2.first.setdefault("step", got))


@pytest.mark.gpu
def test_step_from_host_against_host(c2):
    import torch
    vp = c2.vp
    for t in (vp.cloud_out, vp.region_out, vp.blob_stats):
        t.fill_(float("nan"))
    vp.dens.rho.zero_()
    vp.diff.rho.zero_()                                         # the host call brings the maps back itself
    h_dens = torch.from_numpy(np.ascontiguousarray(c2.work["fofc2"]).reshape(-1)).pin_memory()
    h_diff = torch.from_numpy(np.ascontiguousarray(c2.work["fofc"]).reshape(-1)).pin_memory()
    res = vp.stepFromHost(h_dens, h_diff, torch.from_numpy(c2.xyz).pin_memory())
    _assert_matches(res, c2.ref)


@pytest.mark.gpu
def test_wide_radii_take_two_launches_on_a_partition(c2, monkeypatch, partitions):
    """Every 7th atom at 2.0 A: its box is 2 round(2.0 / 0.5) + 2 = 10 wide, so the cloud rows leave the fused kernel for
    sphere_sums_kernel, launched on the sphere partition's stream."""
    import torch
    from pdb_eda_b200 import _lib
    from pdb_eda_b200.pipeline import VoxelPass
    radii = c2.work["radii"].copy()
    radii[::7] = 2.0
    vp = VoxelPass(c2.dens, c2.diff, c2.xyz, radii, c2.work["res_start"], bench.REGION_RADIUS)
    ref = dict(c2.ref)
    g = _host_geom(c2.hdr)
    wide = np.arange(0, len(radii), 7)
    part = _sphere_refs(g, c2.work["fofc2"], c2.xyz[wide], radii[wide], np.arange(len(wide) + 1), bench.REGION_RADIUS,
                        vp.density_cut, True)
    for name in ("cloud", "cloud_mag"):
        ref[name] = ref[name].copy()
        ref[name][wide] = part[name]
    first = None
    for k in (0, pipeline.BLOB_SMS):
        torch.cuda.synchronize()
        _lib.profile(True, reset=True)
        try:
            got = _step(vp, k, monkeypatch)
            torch.cuda.synchronize()
            kernels = set(_lib.profile())
        finally:
            _lib.profile(False)
        if k:
            assert pipeline.smPartition(vp.device, k) is not None
        assert {"sphere_sums_kernel", "sphere_union_kernel", "blob_sparse_kernel"} <= kernels, kernels
        _assert_matches(got, ref)
        _assert_same(got, first or got)
        first = first or got


@pytest.mark.gpu
def test_dense_foreground_on_partitions(c2, monkeypatch, partitions):
    """The C2 Fo-Fc map at +-1 sigma: ~9 M voxels per class, beyond the 4,096 ranking chunks of P4's shared-memory prefix, so
    P4 ranks the roots through the chunk prefix in global memory -- on 24- and 144-block cooperative grids as well.  Checked
    against scipy.ndimage.label (26-connectivity) renumbered by first voxel in createFullCrsList order."""
    from pdb_eda_b200.pipeline import VoxelPass
    _, s = c2.diff.mean_std()
    cut = np.float32(1.0 * s)
    args = (c2.dens, c2.diff, c2.xyz, c2.work["radii"], c2.work["res_start"], bench.REGION_RADIUS)
    counting = VoxelPass(*args, diffCutoff=cut)
    counting.step()
    counts = counting.blob_counts.cpu().numpy()
    assert counts[4] == 1                                       # the default capacities overflow, the totals are there
    del counting
    vp = VoxelPass(*args, diffCutoff=cut, capVoxels=int(max(counts[0], counts[2])))
    assert counts[0] + counts[2] > 4096 * 512
    g = _host_geom(c2.hdr)
    crs_order = np.ascontiguousarray(c2.work["fofc"].transpose(2, 1, 0))  # [c][r][s]: C order = createFullCrsList order
    ref = {}
    for tag, mask in (("green", crs_order >= cut), ("red", crs_order <= -cut)):
        lab, nlab = ndi.label(mask, structure=np.ones((3, 3, 3), dtype=bool))
        flat = lab[mask]
        _, first = np.unique(flat, return_index=True)
        remap = np.empty(nlab + 1, dtype=np.int64)
        remap[1 + np.argsort(first)] = np.arange(nlab)
        label = remap[flat]
        del lab, flat
        crs = np.stack(np.nonzero(mask), axis=1)
        terms = _blob_terms(crs_order[mask].astype(np.float64), _xyz(g, crs))
        ref[tag] = {"key": np.flatnonzero(mask.reshape(-1)), "label": label,
                    "stats": np.stack([np.bincount(label, t, minlength=nlab) for t in terms.T], axis=1),
                    "mag": np.stack([np.bincount(label, t, minlength=nlab) for t in np.abs(terms).T], axis=1)}
        del terms, crs
    ref.update({name: c2.ref[name] for name in ("cloud", "cloud_mag", "region", "region_mag")})
    first = None
    for k in SMALL_SMS:
        got = _step(vp, k, monkeypatch)
        if k:
            assert pipeline.smPartition(vp.device, k) is not None
        _assert_matches(got, ref)
        _assert_same(got, first or got)
        first = first or got


# ------------------------------------------------------------------------------------------------ ties at the cutoffs
DENSITY_CUT, DIFF_CUT = np.float32(0.75), np.float32(0.5)
TIE_SHAPES = {"vec4": ((64, 64, 64), (1, 2, 3)),              # 64 columns: 16-byte loads, 64 sections: two whole words
              "vec1": ((150, 97, 61), (3, 1, 2))}             # 150 columns: scalar loads, 61 sections: a partial last word


def _ulps(x):
    x = np.float32(x)
    return x, np.nextafter(x, np.float32(np.inf)), np.nextafter(x, np.float32(-np.inf))


@functools.lru_cache(maxsize=None)
def _tie_case(name):
    """A structure and a map pair with planted ties (float32 cell values; 0.5 A grid):
      2Fo-Fc  the voxel nearest every third atom (inside its sphere) holds +-DENSITY_CUT or one ulp either side;
      Fo-Fc   lines of three voxels, v, b, v with v = +-1 in an otherwise empty 7^3 box, along the column, row or section axis,
              whose middle voxel b is +-DIFF_CUT (one blob of 3) or one ulp towards 0 (two blobs of 1); the lines cross word
              boundaries of the section axis and start at every column residue mod 4."""
    ncrs, order = TIE_SHAPES[name]
    nxyz = [0, 0, 0]
    for k, axis in enumerate(order):
        nxyz[axis - 1] = ncrs[k]
    cell = tuple(0.5 * v for v in nxyz) + (90.0, 90.0, 90.0)
    st = synthetic.polyAlaStructure(int(np.prod(nxyz) / 4400), (0, 0, 0), cell[:3], seed=21, residuesPerChain=60)
    a, b = synthetic.mapPair(st, tuple(nxyz), cell, seed=22, axisOrder=order)
    assert a.shape == (ncrs[2], ncrs[1], ncrs[0])
    a = (a * np.float32(0.5 / a.std())).astype(np.float32)
    b = (b * np.float32(0.2 / b.std())).astype(np.float32)
    hdr = _header(ncrs, cell, tuple(nxyz), axisOrder=order)
    g = _host_geom(hdr)
    xyz = np.array([at.coord for at in st.get_atoms()], dtype=np.float64)
    n = len(xyz) // 5 * 5
    xyz = xyz[:n]
    radii = np.tile(ATOM_TYPE_RADII, n // 5)
    start = np.arange(0, n + 1, 5, dtype=np.int32)
    values = _ulps(DENSITY_CUT) + _ulps(-DENSITY_CUT)
    sphere_ties = []
    for j, i in enumerate(range(0, n, 3)):
        c, r, s = orc.xyz2crs(g, xyz[i])[0]
        a[s, r, c] = values[j % 6]
        sphere_ties.append((i, (c, r, s)))
    for i, (c, r, s) in sphere_ties:                            # the last value planted at a shared voxel is the one that counts
        assert a[s, r, c] in values
    line_ties = []
    cs = range(6, ncrs[0] - 8, (ncrs[0] - 14) // 6 + 1)
    rs = range(6, ncrs[1] - 8, 14)
    ss = (4, 30, 44, ncrs[2] - 8)                               # a line along the sections at 30, 31, 32 crosses a word boundary
    j = 0
    for c0 in cs:
        for r0 in rs:
            for s0 in ss:
                axis, sign, joins = j % 3, 1 if (j // 3) % 2 == 0 else -1, (j // 6) % 2 == 0
                j += 1
                step = np.eye(3, dtype=int)[axis]
                b[s0 - 2:s0 + 5, r0 - 2:r0 + 5, c0 - 2:c0 + 5] = 0.0
                p = [np.array((c0, r0, s0)) + t * step for t in range(3)]
                bridge = np.float32(sign * DIFF_CUT) if joins else np.nextafter(np.float32(sign * DIFF_CUT), np.float32(0))
                for q, v in zip(p, (sign * 1.0, bridge, sign * 1.0)):
                    b[q[2], q[1], q[0]] = v
                line_ties.append((tuple(p[1]), bridge, joins))
    return types.SimpleNamespace(hdr=hdr, g=g, rho2=a, rhof=b, xyz=xyz, radii=radii, start=start, sphere_ties=sphere_ties,
                                 line_ties=line_ties)


@functools.lru_cache(maxsize=None)
def _tie_refs(name):
    t = _tie_case(name)
    return _host_refs(t.hdr, t.rho2, t.rhof, t.xyz, t.radii, t.start, 3.5, DENSITY_CUT, DIFF_CUT)


@pytest.mark.gpu
@pytest.mark.parametrize("k", sorted({0, pipeline.BLOB_SMS}))
def test_ties_at_the_cutoffs(k, monkeypatch, partitions):
    from pdb_eda_b200.pipeline import VoxelPass
    for name in TIE_SHAPES:
        t = _tie_case(name)
        dens, diff = _device_map(t.hdr, t.rho2), _device_map(t.hdr, t.rhof)
        vp = VoxelPass(dens, diff, t.xyz, t.radii, t.start, 3.5, densityCutoff=DENSITY_CUT, diffCutoff=DIFF_CUT)
        got = _step(vp, k, monkeypatch)
        if k:
            assert pipeline.smPartition(vp.device, k) is not None
        ref = _tie_refs(name)
        _assert_matches(got, ref)
        # the negative class of the sphere sums (HASNEG gather sites), per atom and per residue
        r35 = np.full(len(t.xyz), 3.5, np.float32)
        want = _sphere_refs(t.g, t.rho2, t.xyz, t.radii, t.start, 3.5, DENSITY_CUT, True, cut_neg=-DENSITY_CUT)
        cloud = dens.sphere_sums(t.xyz, t.radii, None, float(DENSITY_CUT), float(-DENSITY_CUT)).cpu().numpy()
        region = dens.sphere_sums(t.xyz, r35, t.start, float(DENSITY_CUT), float(-DENSITY_CUT)).cpu().numpy()
        _assert_rows(cloud, want["cloud"], want["cloud_mag"], name + " cloud")
        _assert_rows(region, want["region"], want["region_mag"], name + " region")
        assert want["cloud"][:, 4].sum() > 0 and want["region"][:, 4].sum() > 0


# ------------------------------------------------------------------------------------------------ odd geometries
def _odd_case(order, seed, crop=None, diff=None):
    """A 200-residue structure in a 48 A cell on a 96^3 grid whose z axis the column / row / section axis carries (order);
    crop = (crsStart, (nc, nr, ns)) stores only part of the cell; diff(b) -> (Fo-Fc map, diffCutoff or None)."""
    cell, n = (48.0, 48.0, 48.0, 90.0, 90.0, 90.0), (96, 96, 96)
    st = synthetic.polyAlaStructure(200, (0, 0, 0), cell[:3], seed=seed)
    a, b = synthetic.mapPair(st, n, cell, seed=seed + 1, axisOrder=order)
    start, ncrs = (0, 0, 0), n
    if crop is not None:
        start, ncrs = crop
        sl = (slice(start[2], start[2] + ncrs[2]), slice(start[1], start[1] + ncrs[1]), slice(start[0], start[0] + ncrs[0]))
        a, b = np.ascontiguousarray(a[sl]), np.ascontiguousarray(b[sl])
    cut = None
    if diff is not None:
        b, cut = diff(b)
    xyz = np.array([at.coord for at in st.get_atoms()], dtype=np.float64)
    return dict(hdr=_header(ncrs, cell, n, start, order), rho2=a, rhof=b, xyz=xyz, diffCutoff=cut)


ODD_CASES = {
    "z on rows": dict(order=(1, 3, 2), seed=31),
    "z on sections": dict(order=(1, 2, 3), seed=33),
    "z on columns": dict(order=(3, 1, 2), seed=35),
    "partial map": dict(order=(1, 2, 3), seed=37, crop=((10, 20, 30), (60, 50, 40))),
    "no red voxel": dict(order=(1, 3, 2), seed=39, diff=lambda b: (b - b.min() + np.float32(0.01), None)),
    "no foreground": dict(order=(3, 1, 2), seed=41, diff=lambda b: (b, float(np.abs(b).max()) * 1.5)),
}


@pytest.mark.gpu
def test_odd_geometries_on_partitions(monkeypatch, partitions):
    from pdb_eda_b200.pipeline import VoxelPass
    for name, spec in ODD_CASES.items():
        c = _odd_case(**spec)
        n = len(c["xyz"])
        radii = np.resize(ATOM_TYPE_RADII, n)
        start = np.arange(0, n + 1, 5, dtype=np.int32)
        vp = VoxelPass(_device_map(c["hdr"], c["rho2"]), _device_map(c["hdr"], c["rhof"]), c["xyz"], radii, start, 3.5,
                       diffCutoff=c["diffCutoff"])
        ref = _host_refs(c["hdr"], c["rho2"], c["rhof"], c["xyz"], radii, start, 3.5, vp.density_cut, vp.diff_cut)
        ng, nr = len(ref["green"]["key"]), len(ref["red"]["key"])
        if name == "partial map":
            assert (ref["cloud"][:, 6] == 0).any() and (ref["region"][:, 6] == 0).any() and (ref["cloud"][:, 6] == 1).any()
        assert (ng == 0) == (name == "no foreground") and (nr == 0) == (name in ("no foreground", "no red voxel")), name
        first = None
        for k in SMALL_SMS:
            got = _step(vp, k, monkeypatch)
            if k:
                assert pipeline.smPartition(vp.device, k) is not None
            try:
                _assert_matches(got, ref)
            except AssertionError as e:
                raise AssertionError("%s, %d blob SMs: %s" % (name, k, e)) from e
            _assert_same(got, first or got)
            first = first or got


# ------------------------------------------------------------------------------------------------ the references themselves
def test_host_references_agree():
    """Without a GPU: the oracle's blobs equal scipy's labelling renumbered by first voxel; its set-union of one sphere equals
    its one-atom sums; and on the tie maps a voxel exactly at the cut is blob foreground but not sphere-sum foreground."""
    work = bench.build_workload(bench.SAMPLE, seed=2)
    n, cell = work["n"], work["cell"]
    hdr = _header((n, n, n), cell, (n, n, n))
    g = _host_geom(hdr)
    fofc = work["fofc"]
    v = fofc.astype(np.float64)
    cut = np.float32(v.mean() + 3.0 * v.std())
    crs_order = np.ascontiguousarray(fofc.transpose(2, 1, 0))
    for c, mask in ((cut, crs_order >= cut), (-cut, crs_order <= -cut)):
        want = _blob_ref(g, fofc, c)
        lab, nlab = ndi.label(mask, structure=np.ones((3, 3, 3), dtype=bool))
        flat = lab[mask]
        _, first = np.unique(flat, return_index=True)
        remap = np.empty(nlab + 1, dtype=np.int64)
        remap[1 + np.argsort(first)] = np.arange(nlab)
        assert nlab > 3 and len(want["stats"]) == nlab
        assert np.array_equal(want["key"], np.flatnonzero(mask.reshape(-1)))
        assert np.array_equal(want["label"], remap[flat])
        terms = _blob_terms(crs_order[mask].astype(np.float64), _xyz(g, np.stack(np.nonzero(mask), axis=1)))
        _close_sums(want["stats"], np.stack([np.bincount(remap[flat], t, minlength=nlab) for t in terms.T], axis=1), want["mag"])
    # one-atom unions == the batched one-atom sums
    xyz, radii = work["xyz"].astype(np.float64), work["radii"]
    dcut = np.float32(work["fofc2"].astype(np.float64).mean() + 1.5 * work["fofc2"].astype(np.float64).std())
    batch = orc.sphere_sums_batch(g, work["fofc2"], xyz, radii, dcut)
    single = np.array([orc.sphere_union_sums(g, work["fofc2"], p[None], r, dcut, 0.0) for p, r in zip(xyz, radii)])
    assert batch[:, 2].sum() > 0 and np.array_equal(single[:, :4], batch) and (single[:, 4:6] == 0).all() and (single[:, 6] == 1).all()
    # ties: rho >= cut for blobs, rho > cut for sphere sums
    for name in TIE_SHAPES:
        t = _tie_case(name)
        rho2 = t.rho2.reshape(-1)
        for i, crs in t.sphere_ties:
            val = t.rho2[crs[2], crs[1], crs[0]]
            for cutoff in (DENSITY_CUT, -DENSITY_CUT):
                taken = {tuple(p) for p in orc.sphere_list(t.g, rho2, t.xyz[i], t.radii[i], cutoff)}
                inside = {tuple(p) for p in orc.sphere_list(t.g, rho2, t.xyz[i], t.radii[i], 0.0)}
                assert tuple(crs) in inside
                assert (tuple(crs) in taken) == (val > cutoff if cutoff > 0 else val < cutoff)
        assert len({float(t.rho2[s, r, c]) for _, (c, r, s) in t.sphere_ties} & {float(x) for x in _ulps(DENSITY_CUT) + _ulps(-DENSITY_CUT)}) == 6
        fg = {tuple(p) for p in orc.threshold_list(t.g, t.rhof, DIFF_CUT)} | {tuple(p) for p in orc.threshold_list(t.g, t.rhof, -DIFF_CUT)}
        assert {tuple(int(x) for x in p) for p, _, joins in t.line_ties if joins} <= fg
        assert not {tuple(int(x) for x in p) for p, _, joins in t.line_ties if not joins} & fg
        # a joining bridge makes one blob of three voxels, a voxel one ulp short leaves two blobs of one
        for c, sign in ((DIFF_CUT, 1), (-DIFF_CUT, -1)):
            ref = _blob_ref(t.g, t.rhof, c)
            blob_of = dict(zip(ref["key"].tolist(), ref["label"].tolist()))
            u = [int(t.g.unique_ncrs[a]) for a in range(3)]
            for p, bridge, joins in t.line_ties:
                if np.sign(bridge) != sign:
                    continue
                ends = []                                       # the line's two ends: p's only foreground neighbours
                for axis in range(3):
                    e0, e1 = np.array(p), np.array(p)
                    e0[axis] -= 1
                    e1[axis] += 1
                    k0, k1 = [(int(e[0]) * u[1] + int(e[1])) * u[2] + int(e[2]) for e in (e0, e1)]
                    if k0 in blob_of and k1 in blob_of:
                        ends.append((blob_of[k0], blob_of[k1]))
                assert len(ends) == 1, (name, p)
                assert (ends[0][0] == ends[0][1]) == joins, (name, p)
                sizes = ref["stats"][list(ends[0]), 0]
                assert (sizes == (3.0 if joins else 1.0)).all(), (name, p, sizes)
