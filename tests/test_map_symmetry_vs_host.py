"""The whole-map reductions, the skewed-cell conversions, the symmetry expansion and the nearest-atom search (pe_map.cu,
pe_symmetry.cu, pe_scan.cu, pe_common.cuh) against host references that do not use CUDA, at the shapes and edges where these
kernels go wrong.

- Reductions: exact sums (float32 values split into integer mantissas per exponent, added exactly), at sizes around the grid's
  thread count, at pointers off 16-byte alignment, with a large mean and a small spread, with voxels at the float32-narrowed
  cutoff, and beyond 2^31 values.  Dyadic inputs symmetric about 0 and the closed-form pattern beyond 2^31 compare bit for bit;
  other inputs within 1e-12 of the sum of the magnitudes of their terms.
- Conversions: half-integer ties of fractional coordinate x interval in skewed cells, against the C oracle and the numpy statement.
- Symmetry: images exactly on the box faces and one ulp outside, atoms outside the box, a non-identity operator 0, a small
  capacity, candidates on both sides of 1,024 scan tiles and beyond 2^31; against the C oracle and a numpy restatement.
- Nearest atom: exact ties across lanes, warps and strides, equal roots of different squares, and a structure whose atoms sit
  on 2-fold axes; against scipy's cdist + argmin and the C oracle.
- The C2 workload at full size: expansion, nearest atoms of its Fo-Fc blobs and both maps' statistics."""
import ctypes
import io
import itertools
import math
from fractions import Fraction

import numpy as np
import pytest
from scipy.spatial.distance import cdist

import bench
import cases
from oracle import orc
from pdb_eda_b200 import _blas, ccp4, synthetic

ABS_CUT = 17.0                  # a multiple of 1/64: dyadic voxels land on it exactly
PATTERN = np.array([0.5, 1.0, 0.0, 1.75, -0.75, 3.5, -2.5, 0.5], dtype=np.float32)   # 0.5 + a zero-sum pattern
BIG_N = (1 << 31) + 12_345      # = 8 k + 1: the last value is PATTERN[0]
SCAN_TILE = 2048                # candidates per tile of the exclusive scan (pe_scan.cu)


# ---------------------------------------------------------------------------------------------------- exact host sums
def _parts(v):
    """v (float32 values) as integer mantissas m < 2^24 and exponents e with v = m 2^e."""
    m, e = np.frexp(np.asarray(v, dtype=np.float32).astype(np.float64).reshape(-1))
    return m * 2.0 ** 24, e.astype(np.int64) - 24


def _exact(ints, exps):
    """sum(ints x 2^exps) as a Fraction.  The per-exponent sums stay below 2^53 (|int| < 2^25, n < 2^28), so bincount is exact."""
    if len(ints) == 0:
        return Fraction(0)
    e0 = int(exps.min())
    s = np.bincount(exps - e0, weights=ints)
    return sum((Fraction(int(x)) * Fraction(2) ** (k + e0) for k, x in enumerate(s) if x), Fraction(0))


def exact_sum(v):
    return _exact(*_parts(v))


def exact_sum_sq(v):
    """sum(v^2) exactly: m^2 = a^2 2^24 + 2ab 2^12 + b^2 with m = a 2^12 + b, each term below 2^25."""
    m, e = _parts(v)
    a, b = np.floor(np.abs(m) / 4096.0), np.abs(m) % 4096.0
    return _exact(np.concatenate((a * a, 2 * a * b, b * b)), np.concatenate((2 * e + 24, 2 * e + 12, 2 * e)))


def exact_stats(v, cut):
    """(mean, std, sum of |v| over |v| > float32(cut), sum of |v|): mean and sum correctly rounded, std within an ulp or two."""
    v = np.asarray(v, dtype=np.float32).reshape(-1)
    n = len(v)
    s, s2 = exact_sum(v), exact_sum_sq(v)
    a = np.abs(v)
    return float(s / n), math.sqrt(float(s2 / n - (s / n) ** 2)), float(exact_sum(a[a > np.float32(cut)])), float(exact_sum(a))


def _pattern_closed_form(n, cuts):
    """mean, std and sums above the cuts of PATTERN repeated over n = 8k + 1 values: every partial sum is exact."""
    k = (n - 1) // 8
    dev = PATTERN.astype(np.float64) - 0.5
    ss = k * float(np.sum(dev * dev))
    above = [k * float(np.sum(np.abs(PATTERN)[np.abs(PATTERN) > np.float32(c)])) + (0.5 if 0.5 > c else 0.0) for c in cuts]
    return 0.5, math.sqrt(ss / n), above


def _dyadic_symmetric(n, seed):
    """n float32 multiples of 1/64 in [-64, 64], symmetric about 0: mean exactly 0, and every partial sum of the values, their
    squares and their magnitudes is exact in float64 in any order, so mean, std and sum_abs are correctly rounded on both sides."""
    rng = np.random.default_rng(seed)
    half = rng.integers(-4096, 4097, n // 2) / 64.0
    return rng.permutation(np.concatenate((half, -half, np.zeros(n % 2)))).astype(np.float32)


def _dyadic_ref(v):
    w = v.astype(np.float64)
    a = np.abs(w)
    return 0.0, math.sqrt(float(np.sum(w * w)) / len(w)), float(np.sum(a[a > ABS_CUT]))


def _close(got, want, mag, rtol=1e-12, what=""):
    """|got - want| <= rtol x mag (the sum of the magnitudes of the terms); NaN fails."""
    assert abs(got - want) <= rtol * mag, (what, got, want, mag)


# ---------------------------------------------------------------------------------------------------- device entry points
def _check(rc, what):
    from pdb_eda_b200 import _lib
    _lib.check(rc, what)


def _L():
    from pdb_eda_b200 import _lib
    return _lib.load()


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _dev_mean_std(t):
    """pe_map_mean_std over a float32 CUDA view (any offset)."""
    import torch
    L = _L()
    out = torch.full((2,), float("nan"), dtype=torch.float64, device=t.device)
    ws = torch.empty(L.pe_stats_workspace_bytes(), dtype=torch.uint8, device=t.device)
    _check(L.pe_map_mean_std(t.data_ptr(), t.numel(), out.data_ptr(), ws.data_ptr(), _stream()), "pe_map_mean_std")
    return tuple(out.tolist())


def _dev_sum_abs(t, cut):
    """pe_map_sum_abs (float32 view) or pe_sum_abs_f64 (float64 view) with the cutoff narrowed to float32."""
    import torch
    L = _L()
    out = torch.full((1,), float("nan"), dtype=torch.float64, device=t.device)
    ws = torch.empty(L.pe_stats_workspace_bytes(), dtype=torch.uint8, device=t.device)
    fn = L.pe_map_sum_abs if t.dtype == torch.float32 else L.pe_sum_abs_f64
    _check(fn(t.data_ptr(), t.numel(), ctypes.c_float(float(np.float32(cut))), out.data_ptr(), ws.data_ptr(), _stream()), "sum_abs")
    return out.item()


def _offset_view(values, offset, poison=1.0e30):
    """values on the device at ``offset`` elements into a larger buffer whose other elements are ``poison``."""
    import torch
    v = torch.from_numpy(np.ascontiguousarray(values))
    base = torch.full((len(v) + 4,), poison, dtype=v.dtype, device="cuda")
    base[offset:offset + len(v)] = v.cuda()
    view = base[offset:offset + len(v)]
    assert (view.data_ptr() % 16 == 0) == (offset * v.element_size() % 16 == 0)
    return view


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _reduction_sizes():
    """n below the thread count, n % 4 tails, and both sides of the two-loads-per-thread loop's boundary: T = 256 threads x 8
    blocks per SM, so n / 4 float4 loads meet T and 2 T at n = 4 T and 8 T."""
    t = 2048 * _sm_count()
    return [1, 2, 3, 4, 5, 7] + [m * t + d for m in (4, 8) for d in (-3, -2, -1, 1, 2, 3)]


# ---------------------------------------------------------------------------------------------------- geometries
def _header(ncrs, cell, intervals, crsStart=(0, 0, 0), axisOrder=(1, 2, 3)):
    return ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header(ncrs, cell, intervals, crsStart, axisOrder))


def _host_geom(hdr):
    return orc.geom(hdr, hdr.origin, mv=_blas.probe())


def _probe_exact():
    """True when _blas.probe's order reproduces np.dot on every one of its samples (else it fell back to the closest order)."""
    perm, fused = _blas.probe()
    rng = np.random.default_rng(12345)
    for _ in range(64):
        m = rng.uniform(-100.0, 100.0, (3, 3))
        x = rng.uniform(-100.0, 100.0, 3)
        x32 = x.astype(np.float32)
        for xx, y in ((x, np.dot(m.tolist(), x.tolist())), (x32.astype(np.float64), np.dot(m, x32))):
            if any(_blas._row([float(v) for v in m[i]], [float(v) for v in xx], perm, fused) != float(y[i]) for i in range(3)):
                return False
    return True


NOT_EXACT = "the BLAS probe fell back to its closest order: the host's np.dot is not reproduced on every sample"
SKEWED = ("hex", "tric", "random1", "random2")


def _skewed(name):
    """(header, float32 values) of a golden skewed geometry or of cases.random_geometry(1) (monoclinic) / (2) (triclinic)."""
    data, values = cases.random_geometry(int(name[-1])) if name.startswith("random") else cases.make_case(name)
    dm = cases.parse_with(ccp4, data)
    assert not dm.header.orthogonal
    return dm.header, values


def _frac_product(hdr, xyz, axis):
    """fl(deOrtho[axis] . xyz x interval) in the probed BLAS order (exact fma), i.e. the value xyz2crs rounds."""
    perm, fused = _blas.probe()
    d = np.asarray(hdr.deOrthoMat, dtype=np.float64)
    f = _blas._row([float(v) for v in d[axis]], [float(v) for v in xyz], perm, fused)
    return f * float(hdr.xyzInterval[axis])


def _tie_points(hdr, seed, per_axis=10, reach=8):
    """xyz points whose fractional coordinate x interval on one axis is a half-integer exactly, or 1, 2 or 3 ulp from one.
    Returns (points, offsets): offsets[i] = (axis, ulps from the half-integer)."""
    rng = np.random.default_rng(seed)
    om = np.asarray(hdr.orthoMat, dtype=np.float64)
    d = np.asarray(hdr.deOrthoMat, dtype=np.float64)
    iv = np.asarray(hdr.xyzInterval, dtype=np.float64)
    steps = np.array(list(itertools.product(range(-reach, reach + 1), repeat=3)), dtype=np.float64)
    pts, offs = [], []
    for axis in range(3):
        for _ in range(per_axis):
            k = int(rng.integers(1, int(iv[axis]) * 2)) * int(rng.choice((-1, 1)))
            h = k + 0.5
            t = rng.uniform(-0.5, 1.5, 3)
            t[axis] = h / iv[axis]
            x0 = np.dot(om, t)
            cand = x0 + steps * np.spacing(x0)
            approx = (cand @ d[axis]) * iv[axis]
            near = cand[np.abs(approx - h) <= 16 * np.spacing(h)]
            want = {0: h}
            for u in (1, 2, 3):
                want[u] = np.nextafter(want[u - 1], np.inf)
                want[-u] = np.nextafter(want[-u + 1], -np.inf)
            lookup = {v: u for u, v in want.items()}
            seen = set()
            for x in near:
                u = lookup.get(_frac_product(hdr, x, axis))
                if u is not None and u not in seen:
                    seen.add(u)
                    pts.append(x)
                    offs.append((axis, u))
    return np.array(pts), offs


def _numpy_xyz2crs(hdr, xyz):
    """DensityHeader.xyz2crsCoord: np.dot(deOrthoMat, xyz) x interval, Python round()."""
    return np.array([hdr.xyz2crsCoord(np.asarray(p, dtype=np.float64)) for p in xyz], dtype=np.int64)


def _numpy_crs2xyz(hdr, crs):
    return np.array([np.asarray(hdr.crs2xyzCoord([int(v) for v in c]), dtype=np.float64) for c in crs])


def _random_crs(hdr, n, seed):
    rng = np.random.default_rng(seed)
    return np.stack([rng.integers(-3 * int(hdr.ncrs[a]), 4 * int(hdr.ncrs[a]), n) for a in range(3)], axis=1).astype(np.int32)


# ---------------------------------------------------------------------------------------------------- symmetry
def _sym_geom():
    """Only mv_perm / mv_fma of the geometry matter to the expansion."""
    return _host_geom(_header((8, 8, 8), (40.0, 40.0, 40.0, 90, 90, 90), (8, 8, 8)))


def _box(xs, ys, zs):
    return [xs[0] - 5, ys[0] - 5, zs[0] - 5], [xs[-1] + 5, ys[-1] + 5, zs[-1] + 5]


def _shifts(orthoMat):
    return np.array([np.dot(orthoMat, ijk) for ijk in itertools.product((-1, 0, 1), repeat=3)], dtype=np.float64)


def sym_oracle(xyz, rot, orthoMat, xs, ys, zs):
    lo, hi = _box(xs, ys, zs)
    return orc.symmetry(_sym_geom(), xyz, np.asarray(rot, dtype=np.float64).reshape(-1, 12), _shifts(orthoMat), lo, hi)


def sym_numpy(xyz, rot, orthoMat, xs, ys, zs):
    """createSymmetryAtoms restated in numpy (pdb_eda/cutils.pyx:73-103): itertools.product([-1, 0, 1]^3, ops), np.dot(R, x) +
    t + np.dot(orthoMat, ijk), the inclusive box test, and (0,0,0,0) keeping every atom untouched.  Returns the kept images
    and every candidate's coordinates (n_codes x n_atoms x 3) for the tests below to inspect."""
    lo, hi = _box(xs, ys, zs)
    xyz = np.asarray(xyz, dtype=np.float64).reshape(-1, 3)
    atom, code, out, cand = [], [], [], []
    for c, sym in enumerate(itertools.product((-1, 0, 1), (-1, 0, 1), (-1, 0, 1), range(len(rot)))):
        m = np.asarray(rot[sym[3]], dtype=np.float64)
        ot = np.dot(orthoMat, sym[0:3])
        row = []
        for a, x in enumerate(xyz):
            p = np.dot(m[:, 0:3], x) + m[:, 3] + ot
            row.append(p)
            if sym == (0, 0, 0, 0) or (lo[0] <= p[0] <= hi[0] and lo[1] <= p[1] <= hi[1] and lo[2] <= p[2] <= hi[2]):
                atom.append(a)
                code.append(c)
                out.append(x if sym == (0, 0, 0, 0) else p)
        cand.append(row)
    return (np.array(atom, dtype=np.int32), np.array(code, dtype=np.int32), np.array(out).reshape(-1, 3)), np.array(cand)


def _op(r, t):
    return np.concatenate((np.asarray(r, dtype=np.float64), np.asarray(t, dtype=np.float64)[:, None]), axis=1)


FACE_CELL = 40.0
FACE_ORTHO = np.diag([FACE_CELL] * 3)
FACE_XS, FACE_YS, FACE_ZS = [2.5, 37.5], [1.25, 30.0], [0.0, 35.5]      # box -2.5..42.5, -3.75..35.0, -5..40.5
FACE_OPS = [_op(np.eye(3), (0, 0, 0)),                                    # operator 0
            _op(np.eye(3), (0, 0, 0)),                                    # the identity again, not operator 0
            _op(np.diag([-1.0, -1.0, 1.0]), (20.0, 0.0, 20.0)),           # a 2_1 screw
            _op([[0, 1, 0], [1, 0, 0], [0, 0, -1]], (0, 0, 0))]           # a 2-fold on x = y, z = 0


def face_atoms():
    """Atoms whose images under operators 1-3 and the lattice shifts land exactly on lo / hi of each axis, one ulp inside and
    one ulp outside; atoms far outside the box, and atoms one ulp outside it (kept only as (0,0,0,0))."""
    lo, hi = (np.array(b) for b in _box(FACE_XS, FACE_YS, FACE_ZS))
    mid = (lo + hi) / 2
    pts = []
    for op in FACE_OPS[1:]:
        r, t = op[:, :3], op[:, 3]
        for axis in range(3):
            for face, out in ((lo[axis], -np.inf), (hi[axis], np.inf)):
                for target in (face, np.nextafter(face, out), np.nextafter(face, -out)):
                    for s in (-1, 0, 1):
                        p = mid.copy()
                        p[axis] = target
                        shift = np.zeros(3)
                        shift[axis] = s * FACE_CELL
                        x = r.T @ (p - shift - t)                # r is a signed permutation: r^-1 = r^T, exact
                        pts.append(x)
                        if target == face:                       # neighbours: the closest images past the face a translation allows
                            for k in range(3):
                                for way in (-np.inf, np.inf):
                                    y = x.copy()
                                    y[k] = np.nextafter(x[k], way)
                                    pts.append(y)
    for axis in range(3):
        for face, out in ((lo[axis], -np.inf), (hi[axis], np.inf)):
            p = mid.copy()
            p[axis] = np.nextafter(face, out)
            pts.append(p)
    pts += [(200.0, -150.0, 300.0), (-160.0, 10.0, 10.0), (10.0, 10.0, 195.5)]      # beyond any image of the box
    return np.array(pts)


def composed_ops(space_group, cell, translations):
    """The operators of ``space_group`` each composed with fractional translations (translation-major), rounded like REMARK 290
    prints them: larger operator lists than any space group has, for the scan sizes."""
    omat = synthetic.orthoMatrix(cell)
    out = []
    for tau in translations:
        for m in synthetic.cartesianOperators(space_group, cell):
            m = m.copy()
            m[:, 3] = np.round(m[:, 3] + omat @ np.asarray(tau, dtype=np.float64), 5) + 0.0
            out.append(m)
    return out


def _atoms_in_cell(n, cell, seed):
    rng = np.random.default_rng(seed)
    frac = rng.uniform(0.0, 1.0, (n, 3))
    return np.round(frac @ synthetic.orthoMatrix(cell).T, 3).astype(np.float32).astype(np.float64)


def _corner_box(cell, n):
    """xs / ys / zs of _calculateSymmetryAtoms for a whole-cell map of n^3 voxels."""
    hdr = _header((n, n, n), cell, (n, n, n))
    corners = [hdr.crs2xyzCoord([c, r, s]) for c in (0, n - 1) for r in (0, n - 1) for s in (0, n - 1)]
    return [sorted(float(p[a]) for p in corners) for a in range(3)]


BIG_CELL = (60.0,) * 3 + (90.0,) * 3
BIG_TRANSLATIONS = list(itertools.product((0, 0.5), (0, 1 / 3, 2 / 3), (0, 0.25, 0.5, 0.75)))   # 24 x 8 = 192 operators
BIG_ATOMS = 420_000
BIG_LO, BIG_HI = [60.0, 60.0, 60.0], [66.0, 66.0, 66.0]


def big_symmetry_case():
    """> 2^31 candidates: 192 operators x 420,000 atoms x 27 shifts with a 6 A box one cell over, so that few images are kept
    and some of them come from candidates beyond 2^31 (shift (1,1,1), operators above 121)."""
    xyz = _atoms_in_cell(BIG_ATOMS, BIG_CELL, seed=31)
    rot = np.array(composed_ops("P 43 21 2", BIG_CELL, BIG_TRANSLATIONS)).reshape(-1, 12)
    return xyz, rot, _shifts(synthetic.orthoMatrix(BIG_CELL))


def big_symmetry_oracle(xyz, rot, shift, cap):
    """orc_symmetry over all candidates, storing the first ``cap`` kept images; returns (count, atom, code, xyz)."""
    lib = orc.lib()
    atom, code, out = np.empty(cap, np.int32), np.empty(cap, np.int32), np.empty((cap, 3))
    lo, hi = np.array(BIG_LO), np.array(BIG_HI)
    n = lib.orc_symmetry(ctypes.byref(_sym_geom()), len(xyz), orc._p(xyz), len(rot), orc._p(rot), orc._p(shift), orc._p(lo),
                         orc._p(hi), orc._p(atom), orc._p(code), orc._p(out), cap)
    k = min(n, cap)
    return n, atom[:k], code[:k], out[:k]


def _dev_expand(xyz, rot, shift, lo, hi, cap, ws=None, guard=16):
    """pe_symmetry_expand through ctypes with an explicit capacity; outputs carry ``guard`` sentinel entries past cap."""
    import torch
    from pdb_eda_b200 import _device
    L = _L()
    g = _device.geom_from_header(_header((8, 8, 8), (40.0, 40.0, 40.0, 90, 90, 90), (8, 8, 8)))
    x = torch.from_numpy(np.ascontiguousarray(xyz, dtype=np.float64)).cuda()
    r = torch.from_numpy(np.ascontiguousarray(rot, dtype=np.float64)).cuda()
    s = torch.from_numpy(np.ascontiguousarray(shift, dtype=np.float64)).cuda()
    if ws is None:
        ws = torch.empty(max(L.pe_symmetry_workspace_bytes(len(xyz), len(rot)), 256), dtype=torch.uint8, device="cuda")
    count = torch.full((1,), -5, dtype=torch.int64, device="cuda")
    atom = torch.full((cap + guard,), -7, dtype=torch.int32, device="cuda")
    code = torch.full((cap + guard,), -7, dtype=torch.int32, device="cuda")
    out = torch.full((cap + guard, 3), float("nan"), dtype=torch.float64, device="cuda")
    rc = L.pe_symmetry_expand(ctypes.byref(g), len(xyz), x.data_ptr(), len(rot), r.data_ptr(), s.data_ptr(),
                              (ctypes.c_double * 3)(*lo), (ctypes.c_double * 3)(*hi), cap, count.data_ptr(), atom.data_ptr(),
                              code.data_ptr(), out.data_ptr(), ws.data_ptr(), _stream())
    _check(rc, "pe_symmetry_expand")
    return int(count.item()), atom.cpu().numpy(), code.cpu().numpy(), out.cpu().numpy()


def _assert_same_images(got, want, what=""):
    for k, name in enumerate(("atom", "code", "xyz")):
        assert got[k].shape == want[k].shape and np.array_equal(got[k], want[k]), (what, name, len(got[k]), len(want[k]))


# ---------------------------------------------------------------------------------------------------- nearest atom
def nearest_cdist(cent, coords, chunk=4096):
    """np.argmin / min of cdist rows, in chunks over atoms (an earlier chunk keeps a tie) and over blobs."""
    cent = np.asarray(cent, dtype=np.float64).reshape(-1, 3)
    coords = np.asarray(coords, dtype=np.float64).reshape(-1, 3)
    idx = np.full(len(cent), -1, dtype=np.int64)
    dist = np.full(len(cent), np.inf)
    for b0 in range(0, len(cent), chunk):
        sl = slice(b0, b0 + chunk)
        for a0 in range(0, len(coords), chunk):
            d = cdist(cent[sl], coords[a0:a0 + chunk])
            j = np.argmin(d, axis=1)
            m = d[np.arange(len(j)), j]
            better = m < dist[sl]
            idx[sl] = np.where(better, a0 + j, idx[sl])
            dist[sl] = np.where(better, m, dist[sl])
    return idx, dist


def _sq(u, v):
    """cdist's euclidean arithmetic before the root: (d0 d0 + d1 d1) + d2 d2."""
    d = np.asarray(u, dtype=np.float64) - np.asarray(v, dtype=np.float64)
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def root_pair(u, seed, converse=False, reach=5):
    """Two atoms near u: (a, b) with sq(a) > sq(b) and sqrt(sq(a)) == sqrt(sq(b)); with ``converse``, sqrt(sq(b)) one ulp below
    sqrt(sq(a)).  Found among ulp-perturbations of one random atom."""
    rng = np.random.default_rng(seed)
    v0 = u + rng.uniform(1.0, 2.5, 3) * rng.choice((-1, 1), 3)
    steps = np.array(list(itertools.product(range(-reach, reach + 1), repeat=3)), dtype=np.float64)
    cand = v0 + steps * np.spacing(v0)
    s = _sq(u, cand)
    r = np.sqrt(s)
    order = np.lexsort((s, r))
    s, r, cand = s[order], r[order], cand[order]
    for i in range(len(r) - 1):
        j = i + 1
        if converse:
            if r[j] == np.nextafter(r[i], np.inf):          # b = i (smaller root), a = j
                return cand[j], cand[i]
        elif r[j] == r[i] and s[j] > s[i]:
            return cand[j], cand[i]
    raise AssertionError("no pair found")


TIE_STARTS = (0, 31, 100, 255, 273, 509, 1000, 1535)
TIE_GAPS = (1, 32, 256, 2048)       # other lane, other warp, next stride of the same thread, eight strides on


def planted(gap, kind, n_atoms=4096, seed=0):
    """One blob per start s in TIE_STARTS, 100 A apart; atoms s and s + gap are its nearest pair, every other atom is > 40 A from
    every blob.  kind: 'tie' (one atom twice), 'root' (equal roots, the larger square first) or 'converse' (the smaller root at
    the higher index).  Returns (centroids, coords, the index that must win)."""
    rng = np.random.default_rng(seed + gap)
    cent = np.array([(100.0 * k + 0.123, -7.25, 3.5) for k in range(len(TIE_STARTS))])
    coords = np.stack((rng.uniform(-50, 900, n_atoms), rng.uniform(-50, 50, n_atoms), rng.uniform(60, 90, n_atoms)), axis=1)
    slots = [(s, s + gap) for s in TIE_STARTS]
    assert len({i for p in slots for i in p}) == 2 * len(slots) and max(s + gap for s in TIE_STARTS) < n_atoms
    want = []
    for k, (i, j) in enumerate(slots):
        if kind == "tie":
            a = b = cent[k] + rng.uniform(0.5, 2.0, 3)
            w = i
        else:
            a, b = root_pair(cent[k], seed=1000 * gap + k, converse=kind == "converse")
            w = j if kind == "converse" else i
        coords[i], coords[j] = a, b
        want.append(w)
    return cent, coords, np.array(want)


def axis_structure(cell_len):
    """Poly-ALA residues whose atoms all lie on the 2-fold axis x = y, z = 0 of P 43 21 2's operator (y, x, -z) in a cubic cell.
    The axis passes through the origin, so every symmetry image of such an atom coincides exactly with another image."""
    from pdb_eda_b200 import structure as S
    st = S.Structure("axis")
    st.header["resolution"] = 2.0
    chain = st.add(S.Model(0)).add(S.Chain("A"))
    us = np.arange(1.5, cell_len - 1.5, 0.5)             # multiples of 1/8: the coordinates print and parse exactly
    names = ("N", "CA", "C", "O", "CB")
    for k in range(0, len(us) - 4, 5):
        res = chain.add(S.Residue((" ", k // 5 + 1, " "), "ALA"))
        for name, u in zip(names, us[k:k + 5]):
            res.add(S.Atom(name, np.array((u, u, 0.0), dtype=np.float32), 20.0, 1.0, element=name[0]))
    return st


# ==================================================================================================== 1. host references
def test_host_references_agree():
    """Without a GPU: the exact sums equal math.fsum and Fractions; the closed form of the > 2^31 pattern equals exact sums of a
    short copy; a one-pass variance misses the offset-spread std by far more than the bar; the oracle's xyz2crs / crs2xyz equal
    the numpy statement on the skewed ties, and every axis of every cell has exact ties and 1-3 ulp neighbours; the numpy
    symmetry loop equals orc.symmetry on the face, outside-atom and non-identity-operator-0 cases, and the faces are really hit;
    the oracle's nearest atoms equal chunked cdist on the planted ties, and comparing squares alone would pick another atom."""
    rng = np.random.default_rng(0)
    for v in (rng.standard_normal(10_001).astype(np.float32) * 1e3, (1e4 + 1e-2 * rng.standard_normal(5_000)).astype(np.float32),
              np.array([3e38, -3e38, 1e-45, 1.0], dtype=np.float32)):
        w = v.astype(np.float64)
        assert float(exact_sum(v)) == math.fsum(w) and exact_sum(v) == sum(Fraction(float(x)) for x in w)
        assert exact_sum_sq(v[:500]) == sum(Fraction(float(x)) ** 2 for x in w[:500])
    # the > 2^31 pattern's closed form, on a short copy
    n = 8 * 1001 + 1
    v = np.concatenate((np.tile(PATTERN, 1001), PATTERN[:1]))
    mean, std, above = _pattern_closed_form(n, (1.0, 1.75))
    e = exact_stats(v, 1.0)
    assert (mean, std, above[0]) == e[:3] and above[1] == exact_stats(v, 1.75)[2]
    # offset spread: a one-pass formula loses about 8 digits
    v = (1e4 + 1e-2 * rng.standard_normal(1_000_003)).astype(np.float32)
    w = v.astype(np.float64)
    _, std, _, _ = exact_stats(v, 0.0)
    one_pass = math.sqrt(max(float(np.mean(w * w)) - float(np.mean(w)) ** 2, 0.0))
    assert abs(one_pass - std) > 1e-9 * std and abs(float(np.std(w)) - std) <= 1e-12 * std
    # skewed conversions
    if _probe_exact():
        for name in SKEWED:
            hdr, _ = _skewed(name)
            g = _host_geom(hdr)
            pts, offs = _tie_points(hdr, seed=len(name))
            assert {(a, u) for a, u in offs} >= {(a, u) for a in range(3) for u in range(-3, 4)}, name
            assert np.array_equal(orc.xyz2crs(g, pts), _numpy_xyz2crs(hdr, pts)), name
            crs = _random_crs(hdr, 300, seed=1)
            assert np.array_equal(orc.crs2xyz(g, crs), _numpy_crs2xyz(hdr, crs)), name
    # symmetry
    xyz = face_atoms()
    (atom, code, out), cand = sym_numpy(xyz, FACE_OPS, FACE_ORTHO, FACE_XS, FACE_YS, FACE_ZS)
    for rot in (FACE_OPS, [FACE_OPS[2], FACE_OPS[0], FACE_OPS[3]]):
        (a2, c2, o2), _ = sym_numpy(xyz, rot, FACE_ORTHO, FACE_XS, FACE_YS, FACE_ZS)
        _assert_same_images(sym_oracle(xyz, rot, FACE_ORTHO, FACE_XS, FACE_YS, FACE_ZS), (a2, c2, o2))
    lo, hi = (np.array(b) for b in _box(FACE_XS, FACE_YS, FACE_ZS))
    nops = len(FACE_OPS)
    cand = cand.reshape(27, nops, len(xyz), 3)
    for op in (1, 2, 3):
        p = cand[:, op].reshape(-1, 3)
        for axis in range(3):
            others = [b for b in range(3) if b != axis]
            inside = np.all((p[:, others] >= lo[others]) & (p[:, others] <= hi[others]), axis=1)
            for face, sign in ((lo[axis], -1), (hi[axis], 1)):
                past = sign * (p[:, axis] - face) / abs(np.spacing(face))     # ulps beyond the face
                assert (inside & (past == 0)).sum() >= 3, (op, axis, face)                       # kept, on the face
                reach = 16 if op == 2 else 1    # the screw's translation of 20 A makes the step past -2.5 / 42.5 coarser
                assert (inside & (past > 0) & (past <= reach)).sum() >= 1, (op, axis, face)      # dropped, just outside
    far, just_out = np.arange(len(xyz) - 3, len(xyz)), np.arange(len(xyz) - 9, len(xyz) - 3)
    assert not np.all((xyz[just_out] >= lo) & (xyz[just_out] <= hi), axis=1).any()
    assert np.array_equal(atom[np.isin(atom, far)], far) and (code[np.isin(atom, far)] == 13 * nops).all()
    for a in just_out:                   # kept as (0,0,0,0), dropped as the same identity under operator 1
        assert (13 * nops) in code[atom == a] and (13 * nops + 1) not in code[atom == a]
    # nearest
    for gap in TIE_GAPS:
        for kind in ("tie", "root", "converse"):
            cent, coords, want = planted(gap, kind)
            idx, dist = nearest_cdist(cent, coords, chunk=1024)
            assert np.array_equal(idx, want), (gap, kind)
            oi, od = orc.nearest(cent, coords)
            assert np.array_equal(oi, want) and np.array_equal(od, dist)
            assert np.array_equal(dist, np.sqrt(_sq(cent, coords[want])))
            if kind == "root":
                assert not np.array_equal(np.argmin(_sq(cent[:, None], coords[None]), axis=1), want)      # squares alone differ


# ==================================================================================================== 2. reductions
@pytest.mark.gpu
def test_reduction_sizes_and_alignment():
    """n in {1, 2, 3, 4, 5, 7} and 4 T +- {1, 2, 3}, 8 T +- {1, 2, 3} (T = 2048 x SMs), at 0-3 floats off a 16-byte boundary
    (offsets 1-3 take the scalar path): mean, std and sum_abs bit-identical to the exact values on dyadic inputs symmetric
    about 0.  pe_sum_abs_f64 on the same values as float64, at 0 and 1 doubles off.  The buffer around the view holds 1e30, so
    a read past either end shows."""
    import torch
    for n in _reduction_sizes():
        v = _dyadic_symmetric(n, seed=n)
        mean, std, above = _dyadic_ref(v)
        if n > 100:
            assert above > 0 and (np.abs(v) == ABS_CUT).any()
        for off in (0, 1, 2, 3):
            t = _offset_view(v, off)
            assert _dev_mean_std(t) == (mean, std), (n, off)
            assert _dev_sum_abs(t, ABS_CUT) == above, (n, off)
        for off in (0, 1):
            assert _dev_sum_abs(_offset_view(v.astype(np.float64), off), ABS_CUT) == above, (n, off)
    del t
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_reductions_of_general_values():
    """Random float32 values over nine decades at 4 T + 1 (aligned) and 8 T - 3 (one float off): mean, std and sum_abs within
    1e-12 of the sum of their terms' magnitudes of the exact values; the same call twice gives identical bits."""
    t_threads = 2048 * _sm_count()
    rng = np.random.default_rng(3)
    for n, off in ((4 * t_threads + 1, 0), (8 * t_threads - 3, 1)):
        v = (rng.standard_normal(n) * 10.0 ** rng.uniform(-4, 5, n)).astype(np.float32)
        mean, std, above, mag = exact_stats(v, 2.0)
        t = _offset_view(v, off)
        m, s = _dev_mean_std(t)
        _close(m, mean, mag / n, what="mean")
        _close(s, std, std, what="std")            # every term (v - mean)^2 is positive
        _close(_dev_sum_abs(t, 2.0), above, above, what="sum_abs")
        _close(_dev_sum_abs(_offset_view(v.astype(np.float64), off), 2.0), above, above, what="sum_abs f64")
        assert _dev_mean_std(t) == (m, s) and _dev_sum_abs(t, 2.0) == _dev_sum_abs(t, 2.0)


@pytest.mark.gpu
def test_std_of_a_large_mean_with_a_small_spread():
    """Values near 1e4 with a spread near 1e-2: the two-pass std is within 1e-12 relative of the exact value (a one-pass
    E[v^2] - mean^2 is off by about 1e-4 relative here), aligned and one float off."""
    rng = np.random.default_rng(4)
    v = (1e4 + 1e-2 * rng.standard_normal(1_000_003)).astype(np.float32)
    mean, std, _, mag = exact_stats(v, 0.0)
    for off in (0, 1):
        m, s = _dev_mean_std(_offset_view(v, off))
        _close(m, mean, mag / len(v), what="mean")
        _close(s, std, std, what="std")


@pytest.mark.gpu
def test_sum_abs_at_the_float32_cutoff():
    """Voxels at exactly +-float32(cut) and one float32 ulp either side, with a Python-float cutoff that float32 rounds onto a
    voxel: only |v| > float32(cut) counts (strict), through DeviceMap.sum_abs, cutils.sumOfAbs and the offset entry point.
    float64 values within float32 resolution of the cutoff (double(float32(cut)), the Python float itself, one double ulp
    either side) go through pe_sum_abs_f64 against double(float32(cut)); Python lists and integer arrays too."""
    import torch
    from pdb_eda_b200 import _device, cutils
    cut = 1.3
    c32 = np.float32(cut)
    assert float(c32) != cut
    edge = np.array([c32, np.nextafter(c32, np.float32(np.inf)), np.nextafter(c32, np.float32(0))], dtype=np.float32)
    edge = np.concatenate((edge, -edge))
    rng = np.random.default_rng(5)
    shape = (40, 48, 64)
    v = rng.standard_normal(int(np.prod(shape))).astype(np.float32)
    pos = rng.choice(v.size, 600, replace=False)
    v[pos] = np.resize(edge, 600)
    a = np.abs(v)
    want = float(exact_sum(a[a > c32]))
    assert want != float(exact_sum(a[a >= c32]))
    hdr = _header(shape[::-1], (32.0, 24.0, 20.0, 90, 90, 90), shape[::-1])
    dm = _device.DeviceMap(_device.geom_from_header(hdr), torch.from_numpy(v).cuda())
    got = [dm.sum_abs(cut), cutils.sumOfAbs(v, cut), _dev_sum_abs(_offset_view(v, 3), cut)]
    for g in got:
        _close(g, want, want)
    assert got[0] == got[1]
    # float64 input: the comparison is against double(float32(cut)), not the Python float
    c = float(c32)
    e64 = np.array([c, np.nextafter(c, np.inf), np.nextafter(c, -np.inf), cut, np.nextafter(cut, np.inf), np.nextafter(cut, -np.inf)])
    assert c < cut and (np.abs(e64) > c).sum() == 4 and (np.abs(e64) > cut).sum() == 1
    w = rng.standard_normal(50_001) * 2.0
    w[rng.choice(w.size, 1200, replace=False)] = np.resize(np.concatenate((e64, -e64)), 1200)
    kept = np.abs(w)[np.abs(w) > c]
    want64 = math.fsum(kept)
    assert want64 != math.fsum(np.abs(w)[np.abs(w) > cut])
    for g in (cutils.sumOfAbs(w, cut), cutils.sumOfAbs(w.tolist(), cut), _dev_sum_abs(_offset_view(w, 1), cut)):
        _close(g, want64, want64)
    ints = np.arange(-50, 51, dtype=np.int64)
    assert cutils.sumOfAbs(ints, 7.0) == cutils.sumOfAbs(ints.tolist(), 7.0) == 2 * sum(range(8, 51))
    assert cutils.sumOfAbs(ints.astype(np.int32), 7.5) == 2 * sum(range(8, 51))


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_reductions_beyond_2_31_values():
    """n = 2^31 + 12,345 float32 values of a period-8 pattern, written on the device: mean, std and the sums above 1.0 and 1.75
    (a voxel value, kept out by the strict test) equal their closed forms bit for bit, on a 16-byte aligned view (float4 loads,
    scalar tail past 2^31) and one float off (every load scalar, indices up to 2^31 + 12,345)."""
    import torch
    n = BIG_N
    k = (n - 1) // 8
    mean, std, above = _pattern_closed_form(n, (1.0, 1.75))
    pat = torch.from_numpy(PATTERN).cuda()
    base = torch.empty(n + 1, dtype=torch.float32, device="cuda")
    for off in (0, 1):
        base.fill_(1.0e30)
        t = base[off:off + n]
        t[:8 * k].view(k, 8).copy_(pat.expand(k, 8))
        t[8 * k] = float(PATTERN[0])
        assert _dev_mean_std(t) == (mean, std), off
        assert [_dev_sum_abs(t, c) for c in (1.0, 1.75)] == above, off
    del base, t
    torch.cuda.empty_cache()


# ==================================================================================================== 3. skewed conversions
@pytest.mark.gpu
@pytest.mark.parametrize("name", SKEWED)
def test_skewed_conversion_ties(name):
    """xyz whose fractional coordinate x interval is a half-integer, or 1-3 ulp from one, on each axis: the device's index equals
    the oracle's, and the numpy statement's when the BLAS probe reproduces np.dot.  crs2xyz in the same cell is bit-identical
    to both."""
    import torch
    from pdb_eda_b200 import _device
    hdr, values = _skewed(name)
    g = _host_geom(hdr)
    dm = _device.DeviceMap(_device.geom_from_header(hdr), torch.from_numpy(np.ascontiguousarray(values).reshape(-1)).cuda())
    pts, offs = _tie_points(hdr, seed=len(name))
    assert {(a, u) for a, u in offs} >= {(a, u) for a in range(3) for u in range(-3, 4)}
    got = dm.xyz2crs(pts).cpu().numpy()
    assert np.array_equal(got, orc.xyz2crs(g, pts))
    crs = np.concatenate((_random_crs(hdr, 2000, seed=2), got))
    xyz = dm.crs2xyz(crs).cpu().numpy()
    assert np.array_equal(xyz, orc.crs2xyz(g, crs))
    if not _probe_exact():
        pytest.skip(NOT_EXACT)
    assert np.array_equal(got, _numpy_xyz2crs(hdr, pts))
    assert np.array_equal(xyz, _numpy_crs2xyz(hdr, crs))


# ==================================================================================================== 4. symmetry expansion
@pytest.mark.gpu
def test_symmetry_box_faces_and_outside_atoms():
    """Images exactly on lo / hi of each axis are kept and one ulp outside dropped, for the identity as operator 1, a screw and a
    2-fold, with every lattice shift; atoms outside the box keep only their (0,0,0,0) image, coordinate untouched.  With a
    non-identity operator 0, (0,0,0,0) still keeps the atom where it is: the rule goes by index, not by matrix."""
    from pdb_eda_b200 import cutils
    xyz = face_atoms()
    for rot in (FACE_OPS, [FACE_OPS[2], FACE_OPS[0], FACE_OPS[3]]):
        want, _ = sym_numpy(xyz, rot, FACE_ORTHO, FACE_XS, FACE_YS, FACE_ZS)
        got = cutils.symmetryImages(xyz, rot, FACE_ORTHO, FACE_XS, FACE_YS, FACE_ZS)
        _assert_same_images(got, want)
        _assert_same_images(got, sym_oracle(xyz, rot, FACE_ORTHO, FACE_XS, FACE_YS, FACE_ZS))
        ident = got[1] == 13 * len(rot)
        assert np.array_equal(got[0][ident], np.arange(len(xyz))) and np.array_equal(got[2][ident], xyz)


@pytest.mark.gpu
def test_symmetry_small_capacity():
    """A capacity below the kept count: the count still reports every kept image, the first cap entries are the head of the full
    list, and nothing is written past cap."""
    xyz = face_atoms()
    lo, hi = _box(FACE_XS, FACE_YS, FACE_ZS)
    rot = np.array(FACE_OPS).reshape(-1, 12)
    shift = _shifts(FACE_ORTHO)
    full = sym_oracle(xyz, FACE_OPS, FACE_ORTHO, FACE_XS, FACE_YS, FACE_ZS)
    total = len(full[0])
    for cap in (0, 1, 5, total - 1, total, total + 3):
        n, atom, code, out = _dev_expand(xyz, rot, shift, lo, hi, cap)
        k = min(cap, total)
        assert n == total, cap
        _assert_same_images((atom[:k], code[:k], out[:k]), tuple(x[:k] for x in full), cap)
        assert (atom[k:] == -7).all() and (code[k:] == -7).all() and np.isnan(out[k:]).all(), cap


@pytest.mark.gpu
@pytest.mark.parametrize("group,cell", [("P 1", (48.0, 52.0, 44.0, 90, 90, 90)), ("P 21 21 21", (48.0, 52.0, 44.0, 90, 90, 90)),
                                        ("P 43 21 2", (50.0, 50.0, 44.0, 90, 90, 90)), ("P 65 2 2", (40.0, 40.0, 60.0, 90, 90, 120)),
                                        ("P 43 21 2, F-centred", (50.0, 50.0, 44.0, 90, 90, 90))])
def test_symmetry_scan_tiles(group, cell):
    """1, 4, 8 and 12 operators (the hexagonal cell makes every product count) and 32 (P 43 21 2 with F-centring), with atom
    counts that put the candidates one atom below and one above 1,024 scan tiles (2,097,152), and at about 3,000 tiles: atoms,
    image codes, coordinates and counts equal the oracle's."""
    from pdb_eda_b200 import cutils
    if group == "P 43 21 2, F-centred":
        rot = composed_ops("P 43 21 2", cell, [(0, 0, 0), (0, 0.5, 0.5), (0.5, 0, 0.5), (0.5, 0.5, 0)])
    else:
        rot = synthetic.cartesianOperators(group, cell)
    nops = len(rot)
    orthoMat = synthetic.orthoMatrix(cell)
    xs, ys, zs = _corner_box(cell, 48)
    below = (1024 * SCAN_TILE - 1) // (27 * nops)
    for n in (below, below + 1, 3 * below):
        tiles = -(-27 * nops * n // SCAN_TILE)
        assert (n != below or tiles <= 1024) and (n != below + 1 or tiles > 1024)
        xyz = _atoms_in_cell(n, cell, seed=n)
        got = cutils.symmetryImages(xyz, rot, orthoMat, xs, ys, zs)
        want = sym_oracle(xyz, rot, orthoMat, xs, ys, zs)
        _assert_same_images(got, want, (group, n))
        assert len(want[0]) > n


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_symmetry_beyond_2_31_candidates():
    """192 operators x 420,000 atoms x 27 shifts = 2,177,280,000 candidates with a tight box: count, atoms, codes and
    coordinates equal the oracle's, and some kept images are candidates beyond 2^31."""
    import torch
    xyz, rot, shift = big_symmetry_case()
    L = _L()
    ws = torch.empty(L.pe_symmetry_workspace_bytes(len(xyz), len(rot)), dtype=torch.uint8, device="cuda")
    n_dev = _dev_expand(xyz, rot, shift, BIG_LO, BIG_HI, 0, ws=ws, guard=1)[0]
    n, atom, code, out = big_symmetry_oracle(xyz, rot, shift, n_dev + 16)
    assert n == n_dev
    q = code.astype(np.int64) * len(xyz) + atom
    assert 27 * len(rot) * len(xyz) > 1 << 31 and (q >= 1 << 31).sum() > 100
    got = _dev_expand(xyz, rot, shift, BIG_LO, BIG_HI, n, ws=ws)
    del ws
    torch.cuda.empty_cache()
    assert got[0] == n
    _assert_same_images(tuple(x[:n] for x in got[1:]), (atom, code, out))


@pytest.mark.gpu
def test_symmetry_refuses_2_32_candidates():
    """At 2^32 candidates or more the call returns an argument error before any device work: nothing is launched and the count
    is not written.  (The buffers are full size, so the call would be safe even without the check.)"""
    import torch
    from pdb_eda_b200 import _device, _lib
    L = _L()
    n_atoms, n_ops = 1 << 16, 2428
    assert 27 * n_ops * n_atoms >= 1 << 32 > 27 * (n_ops - 1) * n_atoms
    g = _device.geom_from_header(_header((8, 8, 8), (40.0, 40.0, 40.0, 90, 90, 90), (8, 8, 8)))
    xyz = torch.zeros((n_atoms, 3), dtype=torch.float64, device="cuda")
    rot = torch.zeros((n_ops, 12), dtype=torch.float64, device="cuda")
    shift = torch.zeros((27, 3), dtype=torch.float64, device="cuda")
    ws = torch.empty(L.pe_symmetry_workspace_bytes(n_atoms, n_ops), dtype=torch.uint8, device="cuda")
    count = torch.full((1,), -5, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    launches = _lib.launch_count()
    box = (ctypes.c_double * 3)(0.0, 0.0, 0.0)
    rc = L.pe_symmetry_expand(ctypes.byref(g), n_atoms, xyz.data_ptr(), n_ops, rot.data_ptr(), shift.data_ptr(), box, box, 0,
                              count.data_ptr(), None, None, None, ws.data_ptr(), _stream())
    assert rc == -1 and b"2^32" in L.pe_last_error()
    assert _lib.launch_count() == launches and count.item() == -5
    del ws
    torch.cuda.empty_cache()


# ==================================================================================================== 5. nearest atom
@pytest.mark.gpu
def test_nearest_sizes():
    """n_blobs in {1, 7, 8, 9, 83} x n_atoms in {1, 31, 32, 255, 256, 257}, then 100,003 blobs x 257 atoms and 83 blobs x
    100,003 atoms: indices equal cdist + argmin's, distances bit-identical."""
    from pdb_eda_b200 import _device
    rng = np.random.default_rng(6)
    shapes = [(b, a) for b in (1, 7, 8, 9, 83) for a in (1, 31, 32, 255, 256, 257)] + [(100_003, 257), (83, 100_003)]
    for nb, na in shapes:
        cent = rng.uniform(-20, 60, (nb, 3))
        coords = np.round(rng.uniform(-20, 60, (na, 3)), 3).astype(np.float32).astype(np.float64)
        idx, dist = _device.nearest_atom(cent, coords)
        want_i, want_d = nearest_cdist(cent, coords)
        assert np.array_equal(idx.cpu().numpy(), want_i) and np.array_equal(dist.cpu().numpy(), want_d), (nb, na)
        if nb * na <= 83 * 257:
            oi, od = orc.nearest(cent, coords)
            assert np.array_equal(oi, want_i) and np.array_equal(od, want_d)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["tie", "root", "converse"])
@pytest.mark.parametrize("gap", TIE_GAPS)
def test_nearest_ties_and_equal_roots(gap, kind):
    """Per blob, two nearest candidates at index gaps of 1, 32, 256 and 2,048 (another lane, another warp, a later stride of the
    same thread), starting in lanes 0, 31, 100, 255, ... so that the higher index often sits in a lower thread.  'tie': one atom
    twice, the lower index wins.  'root': the first has the larger square but the same root, and wins (np.argmin over the
    roots).  'converse': the second's root is one ulp smaller, and it wins."""
    from pdb_eda_b200 import _device
    cent, coords, want = planted(gap, kind)
    idx, dist = _device.nearest_atom(cent, coords)
    want_i, want_d = nearest_cdist(cent, coords)
    assert np.array_equal(want_i, want)
    assert np.array_equal(idx.cpu().numpy(), want) and np.array_equal(dist.cpu().numpy(), want_d)


@pytest.mark.gpu
def test_blob_statistics_on_two_fold_axes():
    """A P 43 21 2 structure whose atoms all sit on 2-fold axes, so that every symmetry image coincides with another:
    calculateAtomSpecificBlobStatistics reports, for every green and red blob, the distance, atom and symmetry code of
    cdist([centroid], symmetryAtomCoords) + argmin, with the expansion itself equal to the oracle's."""
    from pdb_eda_b200 import densityAnalysis, structure
    cell_len = 40.0
    cell = (cell_len,) * 3 + (90.0,) * 3
    st = axis_structure(cell_len)
    ops = synthetic.cartesianOperators("P 43 21 2", cell)
    d1, d2 = synthetic.mapPair(st, (48, 48, 48), cell, seed=9)
    text = structure.formatPDB(st, remark290=ops, cell=cell, spaceGroup="P 43 21 2")
    densityAnalysis.setGlobals(synthetic.defaultParams())
    m = densityAnalysis.fromFile(io.StringIO(text), io.BytesIO(synthetic.ccp4Bytes(d1, cell, (48,) * 3)),
                                 io.BytesIO(synthetic.ccp4Bytes(d2, cell, (48,) * 3)))
    assert m != 0
    m._densityElectronRatio = 1.0          # the electron column is not under test; this skips the cloud aggregation
    atoms = list(m.biopdbObj.get_atoms())
    xyz = np.array([a.coord for a in atoms], dtype=np.float64)
    hdr = m.densityObj.header
    corners = [hdr.crs2xyzCoord([c, r, s]) for c in (0, 47) for r in (0, 47) for s in (0, 47)]
    xs, ys, zs = (sorted(float(p[a]) for p in corners) for a in range(3))
    ref_atom, ref_code, ref_xyz = sym_oracle(xyz, m.pdbObj.header.rotationMats, hdr.orthoMat, xs, ys, zs)
    assert np.array_equal(np.asarray(m.symmetryAtomCoords, dtype=np.float64), ref_xyz)
    blobs = m.greenBlobList + m.redBlobList
    assert len(blobs) >= 10
    rows = m.calculateAtomSpecificBlobStatistics(blobs)
    ties = 0
    for blob, row in zip(blobs, rows):
        d = cdist(np.asarray([blob.centroid], dtype=np.float64), ref_xyz)[0]
        k = int(np.argmin(d))
        ties += int((d == d[k]).sum() > 1)
        img, op = divmod(int(ref_code[k]), 8)
        a = atoms[ref_atom[k]]
        assert row[0] == d[k] and row[9] == (img // 9 - 1, (img // 3) % 3 - 1, img % 3 - 1, op)
        assert row[5:9] == [a.parent.parent.id, a.parent.id[1], a.parent.resname, a.name]
    assert ties == len(blobs)


# ==================================================================================================== 6. full size
@pytest.fixture(scope="module")
def c2():
    work = bench.build_workload(bench.FULL, seed=2)
    return work


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["P 21 21 21", "P 43 21 2"])
def test_full_size_expansion_and_nearest(c2, group):
    """The C2 workload (40,000 atoms, 384^3 cubic cell) under P 21 21 21 (4.3 M candidates) and P 43 21 2 (8.6 M) with the map-corner
    box of _calculateSymmetryAtoms: the expansion equals the oracle's; the nearest kept image of every green and red blob
    centroid of the Fo-Fc map (at mean +- 3 std) equals chunked cdist + argmin, distances bit for bit."""
    import torch
    from pdb_eda_b200 import _device, cutils
    n, cell = c2["n"], c2["cell"]
    xyz = c2["xyz"].astype(np.float64)
    rot = synthetic.cartesianOperators(group, cell)
    orthoMat = synthetic.orthoMatrix(cell)
    xs, ys, zs = _corner_box(cell, n)
    got = cutils.symmetryImages(xyz, rot, orthoMat, xs, ys, zs)
    want = sym_oracle(xyz, rot, orthoMat, xs, ys, zs)
    _assert_same_images(got, want)
    hdr = _header((n, n, n), cell, (n, n, n))
    dm = _device.DeviceMap(_device.geom_from_header(hdr), torch.from_numpy(np.ascontiguousarray(c2["fofc"]).reshape(-1)).cuda())
    mean, std = dm.mean_std()
    cent = []
    for part in dm.blob_label(mean + 3 * std, -(mean + 3 * std)):
        s = part["stats"].cpu().numpy()
        cent.append(s[:, 2:5] / s[:, 1:2])
    cent = np.concatenate(cent)
    assert len(cent) > 100
    idx, dist = _device.nearest_atom(cent, want[2])
    want_i, want_d = nearest_cdist(cent, want[2])
    assert np.array_equal(idx.cpu().numpy(), want_i) and np.array_equal(dist.cpu().numpy(), want_d)


@pytest.mark.gpu
def test_full_size_map_statistics(c2):
    """mean_std and sum_abs at the 1.5 / 3 std cutoffs of the C2 2Fo-Fc and Fo-Fc maps (384^3) against exact sums."""
    import torch
    from pdb_eda_b200 import _device
    n, cell = c2["n"], c2["cell"]
    hdr = _header((n, n, n), cell, (n, n, n))
    for name, k in (("fofc2", 1.5), ("fofc", 3.0)):
        v = np.ascontiguousarray(c2[name], dtype=np.float32).reshape(-1)
        dm = _device.DeviceMap(_device.geom_from_header(hdr), torch.from_numpy(v).cuda())
        mean, std = dm.mean_std()
        cut = float(np.float32(mean + k * std))
        e_mean, e_std, e_above, mag = exact_stats(v, cut)
        _close(mean, e_mean, mag / len(v), what=name)
        _close(std, e_std, e_std, what=name)
        _close(dm.sum_abs(cut), e_above, e_above, what=name)
