"""GPU tier: the voxel-list set algebra of csrc/pe_cluster.cu against plain float64 / integer host statements.

``pe_cluster_crs`` / ``pe_cluster_crs_grouped`` (labels, cluster count, ``first[]``), ``pe_overlap_pairs``, ``pe_crs_stats``
and ``pe_pair_metrics`` serve the full ``aggregateCloud`` pipeline, ``blobFromCrsList`` and the RSCC / RSR metrics.  The
references here are vectorised numpy / scipy (sorted int64 keys, ``searchsorted`` over the 13 backward neighbour offsets,
``connected_components``), with voxel densities and coordinates taken from the C oracle (``orc.point_density``,
``orc.crs2xyz``), which tests/golden pins to the reference.  The adjacency helper is itself checked against
``orc.cluster_crs`` (the createCrsLists restatement) on small lists.
"""
import io

import numpy as np
import pytest
import torch
from scipy import ndimage, sparse, stats
from scipy.sparse import csgraph

import cases
import golden_checks as gc
from oracle import orc
from pdb_eda_b200 import _blas, _device, _lib, ccp4, cutils, synthetic
from pdb_eda_b200._device import _ptr, _stream

pytestmark = pytest.mark.gpu

# the 13 neighbours that precede a voxel in (c, r, s) order; with their negations and (0, 0, 0) all 27
BACK = np.array([(-1, q // 3 - 1, q % 3 - 1) for q in range(9)] + [(0, -1, -1), (0, -1, 0), (0, -1, 1), (0, 0, -1)],
                dtype=np.int64)
GMAX = (1 << 22) - 1          # largest group id of the grouped key
IMAX_G = (1 << 13) - 1        # largest |index| with groups
IMAX = (1 << 20) - 1          # largest |index| without groups


# ---------------------------------------------------------------------------------------------------- host statements
class _Keys:
    """Dense int64 keys of (group, c, r, s) rows: every axis (and the group) is ranked over the values it takes, with +-1
    around each index so that every neighbour query has a rank too."""

    def __init__(self, crs, group=None):
        crs = np.asarray(crs, dtype=np.int64).reshape(-1, 3)
        self.group = np.zeros(len(crs), np.int64) if group is None else np.asarray(group, dtype=np.int64)
        self.crs = crs
        self.axes = [np.unique(np.concatenate((crs[:, a] - 1, crs[:, a], crs[:, a] + 1))) for a in range(3)]
        self.groups = np.unique(self.group)
        span = [len(self.groups)] + [len(v) for v in self.axes]
        assert span[0] * span[1] * span[2] * span[3] < 2 ** 62
        self.span = span

    def key(self, d=(0, 0, 0)):
        k = np.searchsorted(self.groups, self.group)
        for a in range(3):
            k = k * self.span[a + 1] + np.searchsorted(self.axes[a], self.crs[:, a] + d[a])
        return k


def host_clusters(crs, group=None):
    """createCrsLists on a list with repeats, per group: (label numbered by smallest member index, count, first[])."""
    n = len(crs)
    keys = _Keys(crs, group)
    uk, first_idx, inv = np.unique(keys.key(), return_index=True, return_inverse=True)
    inv = inv.reshape(-1)
    rows, cols = [], []
    for d in BACK:
        nk = keys.key(d)
        j = np.minimum(np.searchsorted(uk, nk), len(uk) - 1)
        hit = uk[j] == nk
        rows.append(inv[hit])
        cols.append(j[hit])
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    graph = sparse.coo_matrix((np.ones(len(rows), np.int8), (rows, cols)), shape=(len(uk), len(uk)))
    ncomp, comp = csgraph.connected_components(graph, directed=False)
    comp_of = comp[inv]
    smallest = np.full(ncomp, n, np.int64)
    np.minimum.at(smallest, comp_of, np.arange(n))
    rank = np.empty(ncomp, np.int64)
    rank[np.argsort(smallest, kind="stable")] = np.arange(ncomp)
    first = np.zeros(n, np.uint8)
    first[first_idx] = 1
    return rank[comp_of], int(ncomp), first


def host_pairs(crs, owner, group=None):
    """{(a, b): a < b, some entry of a and some entry of b in one group with all |delta| <= 1}."""
    owner = np.asarray(owner, dtype=np.int64)
    keys = _Keys(crs, group)
    uk, inv = np.unique(keys.key(), return_inverse=True)
    inv = inv.reshape(-1)
    # distinct (voxel node, owner), sorted by node: the owners of node v are own[start[v]:start[v + 1]]
    no = np.unique(np.stack((inv, owner), axis=1), axis=0)
    node, own = no[:, 0], no[:, 1]
    start = np.searchsorted(node, np.arange(len(uk) + 1))
    out = set()
    for d in np.concatenate((np.zeros((1, 3), np.int64), BACK)):
        nk = keys.key(d)
        j = np.minimum(np.searchsorted(uk, nk), len(uk) - 1)
        hit = uk[j] == nk
        # every (entry owner, owner of the neighbouring node) combination
        src_owner, v = owner[hit], j[hit]
        cnt = start[v + 1] - start[v]
        a = np.repeat(src_owner, cnt)
        b = own[np.repeat(start[v], cnt) + (np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt))]
        keep = a != b
        lo, hi = np.minimum(a[keep], b[keep]), np.maximum(a[keep], b[keep])
        out.update(zip(lo.tolist(), hi.tolist()))
    return out


def _pack_grouped(c, r, s, g):
    """The grouped key layout of pe_cluster.cu: 22 bits of group, three 14-bit axes holding index + 2^13 - 1."""
    off = (1 << 13) - 1
    return (np.uint64(g) << np.uint64(42)) | (np.uint64(c + off) << np.uint64(28)) | (np.uint64(r + off) << np.uint64(14)) | \
        np.uint64(s + off)


def _hash_slot(key, n):
    l2 = 6
    while (1 << l2) < 2 * n + 16:
        l2 += 1
    with np.errstate(over="ignore"):
        return (np.asarray(key, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)) >> np.uint64(64 - l2)


# ---------------------------------------------------------------------------------------------------- inputs
def _blob_voxels(shape, frac, seed, origin=(0, 0, 0)):
    """Voxels of smoothed random blobs (the top `frac` of a smoothed noise field), row-major, shifted by `origin`."""
    rng = np.random.default_rng(seed)
    v = ndimage.gaussian_filter(rng.standard_normal(shape).astype(np.float32), 1.5)
    cut = np.quantile(v, 1.0 - frac)
    return np.argwhere(v > cut).astype(np.int64) + np.asarray(origin, np.int64)


def _with_repeats(crs, frac, rng, group=None):
    """Appends `frac` x n repeated entries (same voxel, same group) and shuffles."""
    n = len(crs)
    rep = rng.integers(0, n, int(frac * n))
    idx = rng.permutation(np.concatenate((np.arange(n), rep)))
    return crs[idx], (None if group is None else group[idx])


def _cluster_device(crs, group=None, first=True):
    label, fst, ncl = cutils.clusterCrs(np.ascontiguousarray(crs, dtype=np.int32), None if group is None else
                                        np.ascontiguousarray(group, dtype=np.int32), wantFirst=first)
    return label.cpu().numpy(), ncl, (fst.cpu().numpy() if first else None)


def _check_clusters(crs, group=None):
    label, ncl, first = _cluster_device(crs, group)
    want_label, want_n, want_first = host_clusters(crs, group)
    assert ncl == want_n
    assert np.array_equal(label, want_label)
    assert np.array_equal(first, want_first)
    if group is None:
        plain, n2 = _device.cluster_crs(np.ascontiguousarray(crs, dtype=np.int32))
        assert n2 == want_n and np.array_equal(plain.cpu().numpy(), want_label)
    return want_n


# ---------------------------------------------------------------------------------------------------- clustering
def test_host_helper_equals_the_oracle():
    """The adjacency helper is createCrsLists: checked against orc.cluster_crs (pinned by tests/golden) on small shuffled
    lists of distinct voxels (the oracle, like createCrsLists' callers, takes sets)."""
    rng = np.random.default_rng(1)
    for seed in range(4):
        crs = _blob_voxels((14, 12, 13), 0.25, seed, origin=(-7, 3, -20))
        crs = crs[rng.permutation(len(crs))][:1500]
        want, n = orc.cluster_crs(crs)
        got, m, _ = host_clusters(crs)
        assert m == n and np.array_equal(got, want)


@pytest.mark.parametrize("n", [1, 31, 32, 33, 257, 50000])
def test_cluster_blobs_with_repeats(n):
    rng = np.random.default_rng(n)
    crs = _blob_voxels((60, 64, 56), 0.25, 7 + n, origin=(-30, -5, -41))     # negative un-wrapped indices
    crs, _ = _with_repeats(crs, 0.1 + 0.2 * rng.random(), rng)
    near = np.argsort(np.abs(crs - crs[0]).max(axis=1), kind="stable")[:n]      # a compact piece, in shuffled order
    crs = crs[rng.permutation(near)]
    assert len(crs) == n
    ncl = _check_clusters(crs)
    if n >= 257:
        assert 1 < ncl < n


@pytest.mark.parametrize("layout", ["interleaved", "single", "sparse_ids"])
def test_cluster_grouped(layout):
    rng = np.random.default_rng({"interleaved": 2, "single": 3, "sparse_ids": 4}[layout])
    crs = _blob_voxels((40, 44, 36), 0.2, 21, origin=(-20, -22, 5))
    if layout == "single":
        group = np.full(len(crs), 6, np.int64)
    elif layout == "interleaved":
        group = rng.integers(0, 5, len(crs)) * 2                                 # ids 0, 2, .., 8: odd ids are empty
    else:
        group = rng.choice(np.array([0, 77, 4096, 123457, GMAX]), len(crs))
    # the same voxels once more under another group: they must not join across groups
    crs = np.concatenate((crs, crs[::3]))
    group = np.concatenate((group, (group[::3] + 1) % (GMAX + 1)))
    crs, group = _with_repeats(crs, 0.25, rng, group)
    ncl = _check_clusters(crs, group)
    assert ncl > len(np.unique(group))


def test_cluster_grid_stride():
    """About 700,000 entries: more than the 16 blocks per SM of grid_for, so every kernel runs its grid-stride loop."""
    rng = np.random.default_rng(9)
    crs = _blob_voxels((180, 180, 180), 0.1, 33, origin=(-90, -60, -30))
    crs, _ = _with_repeats(crs, 0.2, rng)
    assert len(crs) > 148 * 16 * 256
    _check_clusters(crs)
    group = (crs[:, 0] // 16 + 3 * (crs[:, 1] // 16)) % 7
    _check_clusters(crs, group)


def test_cluster_key_range_edges():
    """The largest accepted keys give the host result; one step beyond raises the overflow flag."""
    top = (IMAX_G, IMAX_G, IMAX_G)
    base = [top, (IMAX_G - 1, IMAX_G, IMAX_G), (-IMAX_G, -IMAX_G, -IMAX_G), (-IMAX_G, IMAX_G, 0), top, (IMAX_G, 0, -IMAX_G)]
    groups = [GMAX, GMAX, 0, GMAX, GMAX - 1, 3]
    # more entries whose keys start probing at the same table slot as the largest key
    n = len(base) + 3
    rng = np.random.default_rng(5)
    cand = rng.integers(-IMAX_G, IMAX_G + 1, (200000, 3))
    cg = rng.integers(0, GMAX + 1, 200000)
    slots = _hash_slot(_pack_grouped(cand[:, 0], cand[:, 1], cand[:, 2], cg), n)
    want_slot = _hash_slot(_pack_grouped(*top, GMAX), n)
    same = np.flatnonzero(slots == want_slot)[:3]
    assert len(same) == 3
    crs = np.array(base + [tuple(x) for x in cand[same]], dtype=np.int64)
    group = np.array(groups + cg[same].tolist(), dtype=np.int64)
    for order in (np.arange(n), np.arange(n)[::-1], rng.permutation(n)):
        _check_clusters(crs[order], group[order])
        pairs = cutils.overlapPairs(crs[order].astype(np.int32), np.arange(n, dtype=np.int32), group[order].astype(np.int32))
        assert set(map(tuple, pairs.tolist())) == host_pairs(crs[order], np.arange(n), group[order])
    # without groups: the largest / smallest index on every axis
    plain = np.array([(IMAX, IMAX, IMAX), (IMAX, IMAX - 1, IMAX), (-IMAX, -IMAX, -IMAX), (IMAX, -IMAX, 0), (-IMAX, IMAX, IMAX)])
    _check_clusters(plain)
    # one step outside, on each axis, and bad group ids
    for axis in range(3):
        for v in (IMAX_G + 1, -IMAX_G - 1):
            bad = crs.copy()
            bad[2, axis] = v
            with pytest.raises(_lib.PdbEdaLibError):
                cutils.clusterCrs(bad.astype(np.int32), group.astype(np.int32))
            with pytest.raises(_lib.PdbEdaLibError):
                cutils.overlapPairs(bad.astype(np.int32), np.arange(n, dtype=np.int32), group.astype(np.int32))
        for v in (IMAX + 1, -IMAX - 1):
            bad = plain.copy()
            bad[1, axis] = v
            with pytest.raises(_lib.PdbEdaLibError):
                cutils.clusterCrs(bad.astype(np.int32))
            with pytest.raises(_lib.PdbEdaLibError):
                _device.cluster_crs(bad.astype(np.int32))
    for g in (-1, GMAX + 1):
        bad = group.copy()
        bad[4] = g
        with pytest.raises(_lib.PdbEdaLibError):
            cutils.clusterCrs(crs.astype(np.int32), bad.astype(np.int32))


# ---------------------------------------------------------------------------------------------------- overlap pairs
def _pair_set(arr):
    return set(map(tuple, np.asarray(arr).reshape(-1, 2).tolist()))


def test_overlap_pairs_sparse_owners():
    rng = np.random.default_rng(12)
    crs = _blob_voxels((30, 30, 30), 0.15, 41, origin=(-3, -17, 2))
    nblob = 400
    owner_ids = np.sort(rng.choice(2_000_000_000, nblob, replace=False))
    owner = owner_ids[rng.integers(0, nblob, len(crs))]
    crs, owner = _with_repeats(crs, 0.2, rng, owner)
    got = cutils.overlapPairs(crs.astype(np.int32), owner.astype(np.int32))
    want = host_pairs(crs, owner)
    assert len(want) > 500
    assert _pair_set(got) == want and len(got) == len(want)
    group = rng.integers(0, 3, len(crs))
    got = cutils.overlapPairs(crs.astype(np.int32), owner.astype(np.int32), group.astype(np.int32))
    assert _pair_set(got) == host_pairs(crs, owner, group)


def test_overlap_pairs_hand_made():
    # owner 10 and 20 share a voxel; 30 touches 20 only diagonally; 40 is two steps away from everyone; 50 and 60 share
    # one isolated voxel and nothing else
    crs = np.array([(0, 0, 0), (0, 1, 0), (0, 1, 0), (1, 2, 1), (5, 5, 5), (0, 0, 0), (9, 9, 9), (9, 9, 9)])
    owner = np.array([10, 10, 20, 30, 40, 10, 60, 50])
    want = {(10, 20), (10, 30), (20, 30), (50, 60)}
    assert host_pairs(crs, owner) == want
    assert _pair_set(cutils.overlapPairs(crs.astype(np.int32), owner.astype(np.int32))) == want
    # one group: the same answer; the same geometry with every owner in its own group: no pairs at all
    same = np.zeros(len(crs), np.int32)
    assert _pair_set(cutils.overlapPairs(crs.astype(np.int32), owner.astype(np.int32), same)) == want
    split = (owner // 10).astype(np.int32)
    assert len(cutils.overlapPairs(crs.astype(np.int32), owner.astype(np.int32), split)) == 0
    assert host_pairs(crs, owner, split) == set()
    # a whole blob list duplicated under a second group and a second owner range: pairs only inside each copy
    rng = np.random.default_rng(4)
    blob = _blob_voxels((20, 20, 20), 0.2, 8)
    own = rng.integers(0, 60, len(blob))
    crs2 = np.concatenate((blob, blob))
    own2 = np.concatenate((own, own + 1000))
    grp2 = np.concatenate((np.zeros(len(blob)), np.ones(len(blob)))).astype(np.int32)
    got = _pair_set(cutils.overlapPairs(crs2.astype(np.int32), own2.astype(np.int32), grp2))
    inner = host_pairs(blob, own)
    assert got == inner | {(a + 1000, b + 1000) for a, b in inner}


def test_overlap_pairs_capacity():
    """cap_pairs 0, 1 and 64 on a list with thousands of distinct pairs: the reported count exceeds the capacity (the pair set
    overflows).  The output is then incomplete by contract -- insertions and overflow events share one counter, so a slot
    below cap_pairs may be left unwritten -- but every row that is written is a true, distinct pair.  The wrapper's retry
    returns exactly the host set."""
    lib = _lib.load()
    rng = np.random.default_rng(6)
    cube = np.argwhere(np.ones((16, 16, 16), bool)).astype(np.int64) - 8
    owner = rng.permutation(len(cube)).astype(np.int64) * 7 + 3
    want = host_pairs(cube, owner)
    assert len(want) > 4 * 1024
    crs_t = torch.from_numpy(np.ascontiguousarray(cube, dtype=np.int32)).cuda()
    own_t = torch.from_numpy(np.ascontiguousarray(owner, dtype=np.int32)).cuda()
    n = len(cube)
    for cap in (0, 1, 64):
        counts = torch.zeros(2, dtype=torch.int64, device="cuda")
        pairs = torch.full((max(cap, 1), 2), -1, dtype=torch.int32, device="cuda")      # owners are >= 3: -1 marks "not written"
        ws = torch.empty(max(int(lib.pe_overlap_workspace_bytes(n, cap)), 256), dtype=torch.uint8, device="cuda")
        _lib.check(lib.pe_overlap_pairs(n, _ptr(crs_t), _ptr(own_t), None, cap, _ptr(counts), _ptr(pairs if cap else None),
                                        _ptr(ws), _stream()), "pe_overlap_pairs")
        found, bad = counts.tolist()
        assert bad == 0 and found > cap
        rows = pairs.cpu().numpy()[:cap]
        written = rows[(rows != -1).any(axis=1)]
        assert (written != -1).all()
        assert _pair_set(written) <= want and len(_pair_set(written)) == len(written)
    got = cutils.overlapPairs(cube.astype(np.int32), owner.astype(np.int32))
    assert _pair_set(got) == want and len(got) == len(want)


# ---------------------------------------------------------------------------------------------------- per-cluster sums
def _case(name, seed=11, shift=0.0):
    g = cases.GEOMETRIES[name]
    values = cases._noise(g["shape"], seed) + np.float32(shift)
    data = synthetic.ccp4Bytes(values, g["cell"], g["intervals"], crsStart=g["crsStart"], axisOrder=g["axisOrder"])
    return ccp4.parse(io.BytesIO(data), name)


def _host_geom(dm):
    return orc.geom(dm.header, dm.origin, mv=_blas.probe()), np.ascontiguousarray(dm.densityArray, dtype=np.float32)


def _unwrapped_crs(dm, n, rng):
    """Indices spread over +-3 intervals around the stored block (most wrap; uncovered cells where the map is partial)."""
    iv = np.asarray(dm.header.crsInterval, dtype=np.int64)
    return np.stack([rng.integers(-3 * iv[a], 3 * iv[a] + 1, n) for a in range(3)], axis=1)


def _labels(kind, n, ncl, rng):
    if kind == "sorted":          # runs of 1..100 entries: longer than a warp and crossing warp boundaries
        runs = rng.integers(1, 101, n)
        lab = np.repeat(np.arange(n), runs)[:n] % ncl
        return np.sort(lab)
    if kind == "interleaved":
        return np.arange(n) % ncl
    return rng.permutation(np.sort(np.repeat(np.arange(ncl), n // ncl + 1)[:n]))


def _close_sums(got, want, mag, rtol=1e-12):
    """Sums that differ only in their addition order: |got - want| <= rtol x (sum of the magnitudes of the terms)."""
    got, want, mag = (np.asarray(x, dtype=np.float64) for x in (got, want, mag))
    bad = np.abs(got - want) > rtol * mag + 1e-300
    assert not bad.any(), np.argwhere(bad)[:5].tolist()


@pytest.mark.parametrize("name", gc.CASES)
def test_crs_stats(name):
    rng = np.random.default_rng(len(name))
    dm = _case(name)
    g, rho = _host_geom(dm)
    n = 20000
    crs = _unwrapped_crs(dm, n, rng)
    val, valid = orc.point_density(g, rho, crs)
    d = np.where(valid != 0, val, 0.0)
    xyz = orc.crs2xyz(g, crs)
    if name == "perm":
        assert (valid == 0).any() and (valid != 0).any()
    terms = np.concatenate((np.ones((n, 1)), d[:, None], d[:, None] * xyz, xyz), axis=1)
    ncl = 97
    for kind in ("sorted", "interleaved", "shuffled"):
        label = _labels(kind, n, ncl, rng).astype(np.int64)
        label[rng.random(n) < 0.03] = -1                       # ignored
        label[rng.random(n) < 0.03] = ncl + 5                   # >= n_clusters: ignored
        for take in (None, (rng.random(n) < 0.7).astype(np.uint8)):
            sel = (label >= 0) & (label < ncl) & (take is None or take.astype(bool))
            rows = ncl + 4                                      # extra rows stay zero
            want = np.zeros((rows, 8))
            mag = np.zeros((rows, 8))
            for q in range(8):
                want[:, q] = np.bincount(label[sel], weights=terms[sel, q], minlength=rows)
                mag[:, q] = np.bincount(label[sel], weights=np.abs(terms[sel, q]), minlength=rows)
            got = cutils.crsStats(dm, crs.astype(np.int32), label.astype(np.int32), take, rows).cpu().numpy()
            assert np.array_equal(got[:, 0], want[:, 0]), (kind, take is None)
            assert not got[ncl:].any()
            _close_sums(got, want, mag)
    # no label: one cluster
    got = cutils.crsStats(dm, crs.astype(np.int32), None, None, 1).cpu().numpy()[0]
    assert got[0] == n
    _close_sums(got, terms.sum(axis=0), np.abs(terms).sum(axis=0))


# ---------------------------------------------------------------------------------------------------- RSCC / RSR sums
def _host_pair_metrics(fo, df, label, ngroups, take=None):
    fc = fo - df * 2.0
    sel = (label >= 0) & (label < ngroups) & (np.ones(len(fo), bool) if take is None else take.astype(bool))
    lab, fo, fc = label[sel], fo[sel], fc[sel]
    out = np.zeros((ngroups, 8))
    out[:, 0] = np.bincount(lab, minlength=ngroups)
    out[:, 1] = np.bincount(lab, weights=fo, minlength=ngroups)
    out[:, 2] = np.bincount(lab, weights=fc, minlength=ngroups)
    out[:, 3] = np.bincount(lab, weights=np.abs(fo - fc), minlength=ngroups)
    out[:, 4] = np.bincount(lab, weights=np.abs(fo + fc), minlength=ngroups)
    with np.errstate(invalid="ignore", divide="ignore"):
        xm = fo - (out[:, 1] / out[:, 0])[lab]
        ym = fc - (out[:, 2] / out[:, 0])[lab]
    out[:, 5] = np.bincount(lab, weights=xm * xm, minlength=ngroups)
    out[:, 6] = np.bincount(lab, weights=ym * ym, minlength=ngroups)
    out[:, 7] = np.bincount(lab, weights=xm * ym, minlength=ngroups)
    mag = np.zeros((ngroups, 8))
    for q, w in enumerate((np.ones(len(fo)), fo, fc, np.abs(fo - fc), np.abs(fo + fc), xm * xm, ym * ym, xm * ym)):
        mag[:, q] = np.bincount(lab, weights=np.abs(w), minlength=ngroups)
    return out, mag, (lab, fo, fc)


@pytest.mark.parametrize("name,shift", [("ortho", 0.0), ("perm", 0.0), ("hex", 0.0), ("tric", 0.0), ("over", 0.0), ("ortho", 1000.0)])
def test_pair_metrics(name, shift):
    rng = np.random.default_rng(int(shift) + len(name))
    fo_dm = _case(name, 11, shift)
    df_dm = _case(name, 12)
    g, rho_fo = _host_geom(fo_dm)
    _, rho_df = _host_geom(df_dm)
    crs = _unwrapped_crs(fo_dm, 30000, rng)
    v1, ok1 = orc.point_density(g, rho_fo, crs)
    v2, ok2 = orc.point_density(g, rho_df, crs)
    assert np.array_equal(ok1, ok2)
    if shift:       # only covered voxels: every fo is 1,000 +- a few, so one-pass moments would cancel catastrophically
        keep = ok1 != 0
        crs, v1, ok1, v2, ok2 = crs[keep], v1[keep], ok1[keep], v2[keep], ok2[keep]
    n = len(crs)
    fo, df = np.where(ok1 != 0, v1, 0.0), np.where(ok2 != 0, v2, 0.0)
    ngroups = 64
    label = rng.integers(0, 50, n)                               # groups 50..63 stay empty
    label[:5] = 50 + np.arange(5)                                # one-voxel groups 50..54 ...
    label[rng.random(n) < 0.02] = -1
    label[rng.random(n) < 0.02] = 99                             # out of range: ignored
    label[:5] = 50 + np.arange(5)                                # ... kept whatever the random draws did
    for take in (None, (rng.random(n) < 0.8).astype(np.uint8)):
        if take is not None:
            take[:5] = 1
        got = cutils.pairMetrics(fo_dm, df_dm, crs.astype(np.int32), label.astype(np.int32), take, ngroups).cpu().numpy()
        want, mag, (lab, fo_s, fc_s) = _host_pair_metrics(fo, df, label, ngroups, take)
        assert np.array_equal(got[:, 0], want[:, 0])
        assert not got[55:].any() and not want[55:].any()          # empty groups: all-zero rows
        assert not got[50:55, 5:].any()                             # one voxel: no spread
        _close_sums(got, want, mag)
        rscc = got[:50, 7] / np.sqrt(got[:50, 5] * got[:50, 6])
        rsr = got[:50, 3] / got[:50, 4]
        for k in range(50):
            sel = lab == k
            gc.close([rscc[k]], [stats.pearsonr(fo_s[sel], fc_s[sel])[0]], rtol=1e-10)
            gc.close([rsr[k]], [np.abs(fo_s[sel] - fc_s[sel]).sum() / np.abs(fo_s[sel] + fc_s[sel]).sum()], rtol=1e-12)
