"""GPU tier (one CPU check of the references): the slab-decomposed blob labelling (csrc/pe_slab.cu through slab.py) against references that never touch a CUDA
path, on the slabs where a merge goes wrong: non-square planes, permuted / shifted / skewed / over-sampled / partial maps, slabs
of 1, 31, 32 and 33 sections, slabs that straddle the unique volume's end or lie beyond it, unequal slabs, merges that reach
across several cuts, diagonal contacts, blobs on the plane's edges, dense foreground and a giant percolating component.

References: the C oracle's ``full_blobs`` + ``blob_stats`` on the whole map (tests/golden pins it to the reference), and for
crafted and larger maps ``scipy.ndimage.label`` (26-connectivity, no wrap) on the unique volume in [c][r][s] order, renumbered
by first voxel, with the sums from ``orc.blob_stats``.  Voxels, values, labels and blob counts must match bit for bit, the voxel
counts exactly, the other sums within 1e-12 of the sum of their terms' magnitudes (they differ only in addition order).
"""
import numpy as np
import pytest
import torch
from scipy import ndimage

import cases
from oracle import orc
from pdb_eda_b200 import _blas, _lib, ccp4, slab, synthetic


# ---------------------------------------------------------------------------------------------------- maps and references
class _Map:
    """A map given as float32 values [section][row][column] plus its CCP4 geometry; rho on the device, the oracle's geometry."""

    def __init__(self, values, cell, intervals, crsStart=(0, 0, 0), axisOrder=(1, 2, 3)):
        self.values = np.ascontiguousarray(values, dtype=np.float32)
        ns, nr, nc = self.values.shape
        self.header = ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((nc, nr, ns), cell, intervals, crsStart, axisOrder))
        self.U = tuple(int(u) for u in self.header.uniqueNcrs)
        self.ns = ns
        self.g = orc.geom(self.header, None, mv=_blas.probe())

    @property
    def rho(self):
        if not hasattr(self, "_rho"):
            self._rho = torch.from_numpy(self.values.reshape(-1)).cuda()
        return self._rho

    def emulated(self, cp, cn, ranges, **caps):
        return slab.labelSlabsEmulated(self.header, self.rho, None, cp, cn, ranges=ranges, **caps)

    def oracle(self, cp, cn):
        """Per sign (crs, label, stats) of orc.full_blobs + orc.blob_stats; a 0 cutoff gives an empty sign."""
        return [self._sign_ref(orc.full_blobs(self.g, self.values, c)) for c in (cp, cn)]

    def scipy(self, cp, cn):
        U = self.U
        crs_order = self.values[:U[2], :U[1], :U[0]].transpose(2, 1, 0)          # [c][r][s]: C order = canonical order
        out = []
        for c in (cp, cn):
            c32 = np.float32(c)
            if c32 == 0:
                out.append(self._sign_ref(None))
                continue
            mask = crs_order >= c32 if c32 > 0 else crs_order <= c32
            lab, n = ndimage.label(mask, structure=np.ones((3, 3, 3), dtype=bool))
            flat = lab[mask]
            _, first = np.unique(flat, return_index=True)
            remap = np.empty(n + 1, dtype=np.int32)
            remap[1 + np.argsort(first)] = np.arange(n)
            out.append(self._sign_ref((np.argwhere(mask).astype(np.int32), remap[flat], n)))
        return out

    def _sign_ref(self, blobs):
        if blobs is None:
            return np.zeros((0, 3), np.int32), np.zeros(0, np.int32), np.zeros((0, 8))
        crs, label, n = blobs
        return crs, label, orc.blob_stats(self.g, self.values, crs, label, n)

    def magnitudes(self, crs, label, n):
        """Per blob the sums of |term| of the eight columns (the scale of their rounding differences)."""
        h = self.header
        crs = np.asarray(crs, dtype=np.float64)
        m2x = [int(v) for v in h.map2xyz]
        if self.g.orthogonal:
            xyz = np.stack([crs[:, m2x[i]] * h.gridLength[i] + h.origin[i] for i in range(3)], axis=1)
        else:
            frac = np.stack([(crs[:, m2x[i]] + h.crsStart[m2x[i]]) / h.xyzInterval[i] for i in range(3)], axis=1)
            xyz = frac @ np.asarray(h.orthoMat, dtype=np.float64).T
        d = np.abs(self.values[crs[:, 2].astype(np.int64), crs[:, 1].astype(np.int64), crs[:, 0].astype(np.int64)].astype(np.float64))
        terms = np.concatenate((np.ones((len(d), 1)), d[:, None], d[:, None] * np.abs(xyz), np.abs(xyz)), axis=1)
        return np.stack([np.bincount(label, weights=terms[:, q], minlength=n) for q in range(8)], axis=1)


def _noise_map(shape, seed, cell, intervals, crsStart=(0, 0, 0), axisOrder=(1, 2, 3)):
    return _Map(cases._noise(shape, seed), cell, intervals, crsStart, axisOrder)


def _geometry_map(name, seed=11):
    g = cases.GEOMETRIES[name]
    return _noise_map(g["shape"], seed, g["cell"], g["intervals"], g["crsStart"], g["axisOrder"])


def _check(m, parts, ref):
    """The slab result equals the reference: voxels, values, labels and blob counts bit for bit, sums as documented above."""
    for k, (part, (crs, label, stats)) in enumerate(zip(parts, ref)):
        got_crs = part["crs"].cpu().numpy()
        assert np.array_equal(got_crs, crs.astype(np.int64)), ("sign", k, len(got_crs), len(crs))
        assert np.array_equal(part["value"].cpu().numpy(), m.values[crs[:, 2], crs[:, 1], crs[:, 0]]), ("sign", k)
        assert np.array_equal(part["label"].cpu().numpy(), label.astype(np.int64)), ("sign", k)
        assert part["n_blobs"] == len(stats), ("sign", k, part["n_blobs"], len(stats))
        got = part["stats"].cpu().numpy()
        assert got.shape == stats.shape
        assert np.array_equal(got[:, 0], stats[:, 0]), ("sign", k)
        mag = m.magnitudes(crs, label, len(stats))
        bad = np.abs(got - stats) > 1e-12 * mag + 1e-300
        assert not bad.any(), ("sign", k, np.argwhere(bad)[:5].tolist())


def _whole_slab_caps(m, ranges):
    """Capacities that hold every voxel of the largest slab (dense foreground, giant components)."""
    maxCovered = max(slab.coveredSections(s0, s1, m.U[2]) for s0, s1 in ranges)
    return dict(capVoxels=m.U[0] * m.U[1] * max(maxCovered, 1), capPlane=m.U[0] * m.U[1])


def _layouts(ns):
    return {"w2": slab.slabRanges(ns, 2), "w3": slab.slabRanges(ns, 3), "w5": slab.slabRanges(ns, 5),
            "each": [(s, s + 1) for s in range(ns)]}


def test_scipy_reference_equals_the_oracle():
    """The two references agree on the five geometries (partial, over-sampled and skewed maps included), incl. a dense cutoff
    and a sign switched off: the scipy statement may stand in for the oracle on the maps below."""
    for name in cases.GEOMETRIES:
        m = _geometry_map(name, seed=3)
        for cp, cn in ((2.5, -2.5), (0.8, -0.8), (1.5, 0.0)):
            for (c1, l1, s1), (c2, l2, s2) in zip(m.scipy(cp, cn), m.oracle(cp, cn)):
                assert np.array_equal(c1, c2) and np.array_equal(l1, l2) and np.array_equal(s1, s2), (name, cp)


# ---------------------------------------------------------------------------------------------------- 1. the five geometries
@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["w2", "w3", "w5", "each"])
@pytest.mark.parametrize("name", ["ortho", "perm", "over", "hex", "tric"])
def test_geometries_against_the_oracle(name, layout):
    """Non-square planes, permuted axes, non-zero starts, a partial and an over-sampled map (on ``over`` the slabs beyond the
    unique volume's 30 sections and the one that straddles it), skewed cells; +-2.5, +-1.5 and +-0.8 sigma (a percolating
    component), and one sign switched off."""
    m = _geometry_map(name)
    ranges = _layouts(m.ns)[layout]
    covered = [slab.coveredSections(s0, s1, m.U[2]) for s0, s1 in ranges]
    if name == "over":
        assert m.ns == 36 and m.U[2] == 30
        assert covered.count(0) == 6 if layout == "each" else any(s0 < 30 < s1 for s0, s1 in ranges)
    for cut in (2.5, 1.5, 0.8):
        caps = _whole_slab_caps(m, ranges) if cut < 1 else {}
        ref = m.oracle(cut, -cut)
        parts = m.emulated(cut, -cut, ranges, **caps)
        _check(m, parts, ref)
        if cut < 1:                                      # one blob holds most of the foreground and reaches every slab
            for part in parts:
                sizes = part["stats"][:, 0].cpu().numpy()
                assert sizes.max() > 0.5 * sizes.sum() and part["n_pairs"] >= sum(c > 0 for c in covered) - 1
    ref = m.oracle(1.5, -1.5)
    for cp, cn, on in ((1.5, 0.0, 0), (0.0, -1.5, 1)):
        parts = m.emulated(cp, cn, ranges)
        off = parts[1 - on]
        assert off["n_blobs"] == 0 and off["crs"].shape[0] == 0 and off["stats"].shape[0] == 0
        _check(m, [parts[on]], [ref[on]])


# ---------------------------------------------------------------------------------------------------- 2. crafted structures
CRAFT_SHAPE = (67, 120, 160)                                     # (sections, rows, columns) stored
CUSTOM = [(0, 1), (1, 33), (33, 34), (34, 67)]                   # 1 / 32 / 1 / 33 sections: the bit planes' word edges
CRAFT_LAYOUTS = {"w2": slab.slabRanges(67, 2), "w3": slab.slabRanges(67, 3), "w5": slab.slabRanges(67, 5), "custom": CUSTOM}
CUTS = sorted({s0 for layout in CRAFT_LAYOUTS.values() for s0, _ in layout if s0 > 0})


def _craft_map(values):
    # orthogonal, col -> Z, row -> X, section -> Y, shifted start; every axis holds fewer voxels than its interval
    return _Map(values, (64.0, 40.0, 90.0, 90, 90, 90), (128, 80, 180), crsStart=(5, -7, 3), axisOrder=(3, 1, 2))


class _Canvas:
    """Patterns painted into a zero map: value[s][r][c] = +2 (green) or -2 (red); cutoffs +-1.  Each pattern gets its own
    8 x 8 (column, row) cell of a grid that keeps 3 voxels off the plane's edges, so patterns never touch by accident."""

    def __init__(self):
        self.v = np.zeros(CRAFT_SHAPE, np.float32)
        self.ns, self.U1, self.U0 = CRAFT_SHAPE
        self.next = 0

    def cell(self):
        per_row = (self.U0 - 6) // 8
        c, r = 3 + 8 * (self.next % per_row), 3 + 8 * (self.next // per_row)
        assert r + 8 <= self.U1 - 3
        self.next += 1
        return c, r

    def put(self, c, r, s, sign=1):
        assert 0 <= c < self.U0 and 0 <= r < self.U1 and 0 <= s < self.ns
        self.v[s, r, c] = 2.0 * sign

    def snake(self, sign):
        """One voxel thick, through every section; its lowest column (its smallest key) lies in the top sections, i.e. in
        the last slab of every layout.  Returns its first voxel."""
        c0, r0 = self.cell()
        for s in range(self.ns - 1, -1, -1):
            t = self.ns - 1 - s
            self.put(c0 + t // 9, r0 + t // 11, s, sign)
        return c0, r0, self.ns - 1

    def u_shape(self, k, up, depth, sign):
        """Two bars joined only by a bridge in section k: up = bars in the sections below k (the bridge is above a cut at
        k), else bars in the sections above k (the bridge is below a cut at k + 1)."""
        c, r = self.cell()
        for s in (range(k - depth, k) if up else range(k + 1, k + 1 + depth)):
            if 0 <= s < self.ns:
                self.put(c, r, s, sign)
                self.put(c + 4, r, s, sign)
        for q in range(5):
            self.put(c + q, r, k, sign)

    def diagonal(self, k, dc, dr, sign):
        """One voxel in section k - 1 and one in section k, offset by (dc, dr) in the plane."""
        c, r = self.cell()
        c, r = c + 3, r + 3
        self.put(c, r, k - 1, sign)
        self.put(c + dc, r + dr, k, sign)


def _crafted_values():
    """The crafted map and the first voxel of its green and its red snake."""
    cv = _Canvas()
    snakes = [cv.snake(sign) for sign in (1, -1)]
    for k in CUTS:
        for sign in (1, -1):
            cv.u_shape(k, True, 4, sign)                          # two blobs of the lower slab joined through the upper one
            cv.u_shape(k - 1, False, 4, sign)                     # two blobs of the upper slab joined through the lower one
        for dc, dr in ((1, 1), (1, -1), (-1, 1), (-1, -1), (0, 1), (1, 0), (0, 0)):
            cv.diagonal(k, dc, dr, 1)                             # joined across the cut
        for dc, dr in ((2, 0), (0, 2), (-2, 1), (1, -2), (2, 2)):
            cv.diagonal(k, dc, dr, -1)                            # near misses: not joined
    # joined only through the 1-section slab [33, 34) and the one after it; and through two slabs of the 5-way split
    for lo, top in ((28, 34), (20, 41)):
        for sign in (1, -1):
            c, r = cv.cell()
            for s in range(lo, top):
                cv.put(c, r, s, sign)
                cv.put(c + 3, r + 3, s, sign)
            for q in range(4):
                cv.put(c + q, r + q, top, sign)
    # green and red side by side across cuts: the signs never mix
    for k in CUTS:
        c, r = cv.cell()
        for s in range(max(k - 2, 0), k):
            cv.put(c, r, s, 1)
        for s in range(k, k + 2):
            cv.put(c, r, s, -1)
            cv.put(c + 1, r + 1, s, -1)
    # the plane's edges at cuts: columns 0 / U0-1 and rows 0 / U1-1, corners, and pairs that only wrap-around or an r/c
    # mix-up could join ((c, 0) against (c-1, U1-1); (0, r) against (U0-1, r))
    U0, U1 = cv.U0, cv.U1
    for i, k in enumerate(CUTS):
        a = 4 + 12 * i
        for c, r in ((0, a), (U0 - 1, a + 3), (a, 0), (a + 3, U1 - 1)):
            for s in range(max(k - 2, 0), k + 2):
                cv.put(c, r, s, 1)
        cv.put(0, a + 6, k - 1, -1)
        cv.put(U0 - 1, a + 6, k, -1)
        cv.put(a + 6, 0, k - 1, -1)
        cv.put(a + 5, U1 - 1, k, -1)
    cv.put(0, 0, 33, 1)
    cv.put(1, 1, 34, 1)
    cv.put(U0 - 1, U1 - 1, 33, -1)
    cv.put(U0 - 2, U1 - 2, 34, -1)
    return cv.v, snakes


@pytest.mark.gpu
@pytest.mark.parametrize("layout", sorted(CRAFT_LAYOUTS))
def test_crafted_structures_against_scipy(layout):
    """A 160 x 120 x 67 map (non-square plane, permuted axes, shifted start, default capacities above their floors) with the
    patterns placed at every cut of every layout.  The world-2 split (34 / 33 sections) is one where sizing each slab for
    itself gives the two ranks different exchange layouts."""
    values, snakes = _crafted_values()
    m = _craft_map(values)
    assert m.U == (160, 120, 67)
    ranges = CRAFT_LAYOUTS[layout]
    if layout == "w2":
        own = [slab.slabCapacities(m.U[0], m.U[1], s1 - s0) for s0, s1 in ranges]
        assert own[0][1] != own[1][1] and min(c[0] for c in own) > 4096
    ref = m.scipy(1.0, -1.0)
    assert len(ref[0][2]) > 100 and len(ref[1][2]) > 100
    parts = m.emulated(1.0, -1.0, ranges)
    _check(m, parts, ref)
    for part, head in zip(parts, snakes):
        assert part["n_pairs"] > len(ranges)
        crs, label = part["crs"].cpu().numpy(), part["label"].cpu().numpy()
        snake = label == label[(crs == head).all(axis=1)][0]
        assert all((snake & (crs[:, 2] >= s0) & (crs[:, 2] < s1)).any() for s0, s1 in ranges)


@pytest.mark.gpu
@pytest.mark.parametrize("sign", [1, -1])
@pytest.mark.parametrize("layout", sorted(CRAFT_LAYOUTS))
def test_full_planes_across_cuts(layout, sign):
    """Every voxel of the sections on both sides of every cut is foreground (of one sign; the crafted patterns elsewhere): the
    boundary planes hold U0 x U1 voxels and need capPlane = U0 * U1."""
    v, _ = _crafted_values()
    ranges = CRAFT_LAYOUTS[layout]
    for s0, _ in ranges[1:]:
        v[s0 - 1] = 2.0
        v[s0] = 2.0
    m = _craft_map(sign * v)
    ref = m.scipy(1.0, -1.0)
    _check(m, m.emulated(1.0, -1.0, ranges, **_whole_slab_caps(m, ranges)), ref)


# ---------------------------------------------------------------------------------------------------- 3. skewed medium map
@pytest.mark.gpu
def test_skewed_medium_map_in_two_unequal_slabs():
    """Hexagonal, shifted, 128 x 112 x 61 (slabs of 31 / 30 sections, above the capacity floors): the relabel sums use the
    whole map's crs -> xyz at the global section on a skewed cell."""
    m = _noise_map((61, 112, 128), 23, (64.0, 64.0, 40.0, 90, 90, 120), (128, 128, 64), crsStart=(3, -2, 5))
    ranges = slab.slabRanges(61, 2)
    assert ranges == [(0, 31), (31, 61)] and not m.g.orthogonal
    _check(m, m.emulated(2.5, -2.5, ranges), m.oracle(2.5, -2.5))                       # default capacities
    _check(m, m.emulated(1.5, -1.5, ranges, **_whole_slab_caps(m, ranges)), m.oracle(1.5, -1.5))


# ---------------------------------------------------------------------------------------------------- 4. layout invariance
@pytest.mark.gpu
def test_layout_invariance():
    """A ~1e6-voxel permuted, shifted noise map through ten layouts, unequal ones included: every layout gives the reference's
    voxels, labels, counts and sums (and so the same as every other layout)."""
    m = _noise_map((81, 104, 120), 5, (42.0, 62.0, 54.0, 90, 90, 90), (84, 124, 108), crsStart=(-4, 9, 2), axisOrder=(2, 3, 1))
    assert m.U == (120, 104, 81)
    layouts = [slab.slabRanges(81, w) for w in (1, 2, 3, 4, 6, 7)] + [
        [(0, 1), (1, 81)], [(0, 80), (80, 81)], [(0, 31), (31, 32), (32, 64), (64, 65), (65, 81)], [(0, 33), (33, 66), (66, 81)]]
    ref = m.scipy(2.5, -2.5)
    dense = m.scipy(1.2, -1.2)
    for ranges in layouts:
        _check(m, m.emulated(2.5, -2.5, ranges), ref)
        _check(m, m.emulated(1.2, -1.2, ranges, **_whole_slab_caps(m, ranges)), dense)


# ---------------------------------------------------------------------------------------------------- 5. reuse
@pytest.mark.gpu
def test_labeller_reuse_at_new_cutoffs_and_maps():
    """One world-1 SlabLabeller (the calling pattern bench.py times) at cutoff A, then B, then on a second map, then A again:
    each call equals the reference of that call, so no exchange, plane or sums state leaks from the previous one."""
    a = _geometry_map("hex", seed=11)
    b = _geometry_map("hex", seed=12)
    lab = slab.SlabLabeller(a.header, 0, a.ns, 1, 0, a.rho.device)
    for m, cut in ((a, 2.5), (a, 1.5), (b, 2.5), (a, 2.5), (b, 1.5)):
        _check(m, lab.label(m.rho, cut, -cut), m.oracle(cut, -cut))


# ---------------------------------------------------------------------------------------------------- 6. overflow
@pytest.mark.gpu
def test_too_dense_cutoff_raises_and_the_labeller_recovers():
    """Default capacities at +-0.3 sigma: the capacity flag raises instead of returning a result, on one slab and on two
    unequal ones; the same labeller then labels a sane cutoff correctly."""
    m = _noise_map((61, 112, 128), 29, (64.0, 56.0, 30.5, 90, 90, 90), (128, 112, 61))
    for ranges in ([(0, 61)], slab.slabRanges(61, 2)):
        with pytest.raises(RuntimeError, match="capacity was exceeded"):
            m.emulated(0.3, -0.3, ranges)
    lab = slab.SlabLabeller(m.header, 0, m.ns, 1, 0, m.rho.device)
    with pytest.raises(RuntimeError, match="capacity was exceeded"):
        lab.label(m.rho, 0.3, -0.3)
    _check(m, lab.label(m.rho, 2.5, -2.5), m.oracle(2.5, -2.5))


@pytest.mark.gpu
def test_mismatched_capacities_are_flagged():
    """Two ranks whose exchange buffers have the same size but different layouts (capBlobs / capPlane 2,048 / 4,096 against
    5,120 / 3,072): every rank's merge sees the other stamp and raises instead of reading the buffers at the wrong offsets."""
    m = _geometry_map("ortho")
    ranges = slab.slabRanges(m.ns, 2)
    lib = _lib.load()
    assert lib.pe_slab_exchange_bytes(2048, 4096) == lib.pe_slab_exchange_bytes(5120, 3072)
    labs = [slab.SlabLabeller(m.header, s0, s1, 2, r, m.rho.device, None, None, 8192, cb, cp)
            for r, ((s0, s1), (cb, cp)) in enumerate(zip(ranges, ((2048, 4096), (5120, 3072))))]
    vol = m.rho.reshape(m.ns, -1)
    for lab, (s0, s1) in zip(labs, ranges):
        lab._labelLocal(vol[s0:s1].contiguous(), 2.5, -2.5)
        lab._boundary()
    gathered = torch.cat([lab.exchange for lab in labs])
    for lab in labs:
        lab._mergeAndRelabel(gathered)
        with pytest.raises(RuntimeError, match="capacity was exceeded"):
            lab._readCounts()
