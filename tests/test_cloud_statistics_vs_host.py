"""The statistics block of the batched aggregateCloud (csrc/pe_cloudstats.cu) and the radix-select medians it shares with
the centroid cutoff (csrc/pe_select.cuh) against exact host references.

GPU tier, ``pe_cloud_statistics`` through ctypes on hand-made per-atom records:
  A  every order-statistic column bit for bit against np.nanmedian, at lengths around the 1,024-thread stride and the
     12,288-key shared-memory stage, on ties across the middle, keys that differ in one byte only, signed zeros,
     subnormals, infinities, NaN and non-contributing rows;
  B  the staged and the unstaged select on the same rows: all 14 output columns bit for bit;
  C  the slope's p-value test at p = 0.05 (1 +- delta) against mpmath's regularised incomplete beta, df from 1 to 1e5;
  D  degenerate fits against scipy.stats.linregress and the reference's calcSlope rule;
  E  ``CloudBatch`` on a poly-ALA structure whose atom-type segments exceed the stage, against the host statement.
CPU tier: the host statement ``cloudBatch.batchAtomTypeStatistics`` on the cases of C and D.

The library is built with -fmad=false, so the per-element arithmetic (der / nv * median, (adj - ratio) / ratio, ...) is
numpy's operation for operation.  Centroid distances are NaN on every contributing row unless a test says otherwise:
that turns the second centroid filter off, so every contributing row is kept.
"""
import warnings

import numpy as np
import pytest
from scipy import stats

STAGE = 12288                 # stats_segment_kernel stages a column in shared memory up to min(max_segment, 12288) rows
CURRENT = 1000.0              # the current slope of atom type t is CURRENT + t: no fit in these tests comes near it
LENGTHS = (1, 2, 3, 4, 31, 32, 33, 1023, 1024, 1025, 1026, STAGE - 1, STAGE, STAGE + 1, 65537, 200003)
DBL_MAX = np.finfo(np.float64).max


def _segment(nv, td, bf, cd=None, flags=None, density=500.0, electrons=1000.0, atomType=0, unitVolume=0.125):
    """One (structure, atom type) segment: per-row num_voxels, total_density (electrons = occupancy = 1, so the
    density/electron ratio is total_density itself), b-factor, centroid distance, flags (1 contributes, 3 also complete);
    the structure's total density and electrons (map_out[:, 1:3])."""
    n = len(nv)
    return {"nv": np.asarray(nv, dtype=np.float64), "td": np.asarray(td, dtype=np.float64), "bf": np.asarray(bf, dtype=np.float64),
            "cd": np.full(n, np.nan) if cd is None else np.asarray(cd, dtype=np.float64),
            "flags": np.ones(n) if flags is None else np.asarray(flags, dtype=np.float64),
            "map": (float(density), float(electrons)), "type": int(atomType), "uvol": float(unitVolume)}


def _run_statistics(segments, nTypes=None, minTotalElectrons=400.0):
    """pe_cloud_statistics with every segment a structure of its own (identity permutation); max_segment is the longest
    segment.  Returns seg_out (n_segments x 14) and map_stats (n_segments x 4)."""
    import ctypes
    import torch
    from pdb_eda_b200 import _lib
    from pdb_eda_b200._device import _ptr, _stream
    lib = _lib.load()
    nS = len(segments)
    sizes = np.array([len(s["nv"]) for s in segments], dtype=np.int64)
    start = np.concatenate(([0], np.cumsum(sizes)))
    nA = int(start[-1])
    recs = np.zeros((nA, 8))                           # clouds, num_voxels, centroid_distance, total_density, cx, cy, cz, flags
    static = np.ones((nA, 3))                          # electrons, occupancy, bfactor
    for k, s in enumerate(segments):
        a = slice(int(start[k]), int(start[k + 1]))
        recs[a, 0], recs[a, 1], recs[a, 2], recs[a, 3], recs[a, 7] = 1.0, s["nv"], s["cd"], s["td"], s["flags"]
        static[a, 2] = s["bf"]
    maps = (_lib.PeBatchMap * nS)()
    for k in range(nS):
        maps[k].atom_begin, maps[k].atom_end = int(start[k]), int(start[k + 1])
    mapOut = np.zeros((nS, 8))
    mapOut[:, 1:3] = [s["map"] for s in segments]
    types = np.array([s["type"] for s in segments], dtype=np.int32)
    nT = int(types.max()) + 1 if nTypes is None else nTypes
    dev = "cuda"
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d = dict(maps=torch.frombuffer(bytearray(bytes(maps)), dtype=torch.uint8).to(dev), recs=up(recs), mapOut=up(mapOut), static=up(static),
             perm=up(np.arange(nA, dtype=np.int32)), sm=up(np.arange(nS, dtype=np.int32)), st=up(types),
             sb=up(start[:-1].astype(np.int32)), se=up(start[1:].astype(np.int32)), uv=up(np.array([s["uvol"] for s in segments])),
             sl=up(CURRENT + np.arange(nT, dtype=np.float64)))
    scratch = torch.empty((9, max(nA, 1)), dtype=torch.float64, device=dev)
    segOut = torch.full((nS, 14), -12345.0, dtype=torch.float64, device=dev)
    mapStats = torch.empty((nS, 4), dtype=torch.float64, device=dev)
    _lib.check(lib.pe_cloud_statistics(nS, _ptr(d["maps"]), nA, _ptr(d["recs"]), _ptr(d["mapOut"]), _ptr(d["static"]), _ptr(d["perm"]),
                                       nS, _ptr(d["sm"]), _ptr(d["st"]), _ptr(d["sb"]), _ptr(d["se"]), int(sizes.max()), _ptr(d["uv"]),
                                       _ptr(d["sl"]), ctypes.c_double(minTotalElectrons), _ptr(scratch), _ptr(segOut), _ptr(mapStats),
                                       _stream()), "pe_cloud_statistics")
    return segOut.cpu().numpy(), mapStats.cpu().numpy()


def _nanmedian(v):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return float(np.nanmedian(v)) if len(v) else np.nan


def _same(a, b):
    """Bit-identical up to the sign of zero; NaN matches NaN."""
    return bool(np.array_equal(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64), equal_nan=True))


def _host_order_statistics(s):
    """Columns 0-6 and 8 of seg_out from the numpy statement, for a segment whose contributing rows all have NaN centroid
    distances (every contributing row kept)."""
    rows = (s["flags"].astype(np.int64) & 1) != 0
    assert np.isnan(s["cd"][rows]).all()
    nv, der, bf = s["nv"][rows], s["td"][rows], s["bf"][rows]
    ratio = s["map"][0] / s["map"][1]
    with np.errstate(all="ignore"):
        medNv = _nanmedian(nv)
        adj = der / nv * medNv
        out = {0: float(rows.sum()), 1: medNv, 2: _nanmedian(der), 3: _nanmedian(s["cd"][rows]), 4: _nanmedian(adj),
               5: _nanmedian(nv * s["uvol"]), 6: _nanmedian(bf[bf > 0]), 8: _nanmedian((adj - ratio) / ratio)}
    return out


# ------------------------------------------------------------------------------------------------------ A: order statistics
def _with_byte(rng, n, j, base=1.2345):
    """Values whose bit patterns are base's except byte j (random): the select decides in the pass of byte j alone.
    Byte 7 holds the sign, so that variant mixes signs; patterns that are not finite fall back to base."""
    bits = np.full(n, np.float64(base).view(np.uint64))
    k = rng.integers(0, 256, n).astype(np.uint64)
    bits = (bits & ~np.uint64(0xff << (8 * j))) | (k << np.uint64(8 * j))
    v = bits.view(np.float64).copy()
    v[~np.isfinite(v)] = base
    return v


def _values(kind, rng, n):
    if kind == "equal":
        return np.full(n, 7.25)
    if kind in ("halves", "majority"):           # exactly n/2 copies of each value, or n/2 + 1 copies of the smaller one
        low = n // 2 + (1 if kind == "majority" else 0)
        return rng.permutation(np.where(np.arange(n) < low, 3.0, 5.5))
    if kind == "last_byte":                       # x (1 + k 2^-52), k in 0..255
        return 2.0 * (1.0 + rng.integers(0, 256, n) * 2.0 ** -52)
    if kind.startswith("byte"):
        return _with_byte(rng, n, int(kind[4:]))
    if kind == "negative":
        return -np.round(np.exp(rng.normal(size=n)), 3)
    if kind == "signed_zeros":
        v = np.round(rng.normal(size=n), 2)
        z = rng.random(n) < 0.4
        v[z] = np.where(rng.random(int(z.sum())) < 0.5, -0.0, 0.0)
        return v
    if kind == "extremes":
        pool = np.array([5e-324, -5e-324, 1e-310, -3e-315, 2.2250738585072014e-308, -2.2250738585072014e-308, np.inf, -np.inf,
                         DBL_MAX, -DBL_MAX, 0.0, -0.0, 1.0])
        return pool[rng.integers(0, len(pool), n)]
    if kind in ("nan10", "nan90"):
        v = np.round(rng.normal(10.0, 3.0, n), 2)
        v[rng.random(n) < (0.1 if kind == "nan10" else 0.9)] = np.nan
        return v
    if kind == "all_nan":
        return np.full(n, np.nan)
    raise ValueError(kind)


KINDS = ("equal", "halves", "majority", "last_byte") + tuple("byte%d" % j for j in range(1, 8)) + \
        ("negative", "signed_zeros", "extremes", "nan10", "nan90", "all_nan", "noncontributing", "bfactors_not_positive")


def _order_case(kind, rng, n):
    if kind == "noncontributing":                 # a third of the rows do not contribute and carry values that would move the median
        flags = np.where(rng.random(n) < 1 / 3, 0.0, rng.choice([1.0, 3.0], n))
        flags[0] = 1.0
        v = [np.round(rng.normal(10.0, 3.0, n), 2) for _ in range(3)]
        for col in v:
            col[flags == 0] = rng.choice([np.inf, DBL_MAX, 1e300, 1e6], int((flags == 0).sum()))
        return _segment(v[0], v[1], v[2], flags=flags)
    if kind == "bfactors_not_positive":           # b-factors <= 0 (and NaN) do not enter the b-factor median
        bf = np.round(rng.uniform(5, 60, n), 1)
        bad = rng.random(n) < 0.3
        bf[bad] = rng.choice([0.0, -0.0, -1.0, -1e300, -np.inf, np.nan], int(bad.sum()))
        return _segment(rng.integers(5, 40, n).astype(np.float64), np.round(rng.uniform(2, 7, n), 3), bf,
                        flags=rng.choice([1.0, 3.0], n))
    return _segment(_values(kind, rng, n), _values(kind, rng, n), _values(kind, rng, n), flags=rng.choice([1.0, 3.0], n),
                    density=float(rng.uniform(400, 600)), electrons=float(rng.uniform(900, 1100)), unitVolume=float(rng.uniform(0.1, 0.2)))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_medians_are_exact_order_statistics(kind):
    """Columns 1-6 and 8 equal np.nanmedian over the contributing rows bit for bit, at every length in LENGTHS (one
    segment each, so 12,287 and 12,288 take the staged select and the longer ones read global memory)."""
    rng = np.random.default_rng(KINDS.index(kind) + 100)
    segments = [_order_case(kind, rng, n) for n in LENGTHS]
    segOut, _ = _run_statistics(segments)
    bad = []
    for s, out, n in zip(segments, segOut, LENGTHS):
        want = _host_order_statistics(s)
        for col, value in want.items():
            if not _same(out[col], value):
                bad.append((n, col, out[col], value))
    assert not bad, bad[:10]


# ------------------------------------------------------------------------------------------- B: staged and unstaged select
def _mixed_rows(rng, n, correlated):
    """Rows with integer voxel counts, b-factors <= 0 and ties, centroid distances with outliers and NaN, some rows that
    do not contribute; with ``correlated`` the domain fraction follows log(b-factor), so the slope is a fit."""
    bf = np.round(rng.uniform(5, 60, n), 1)
    low = rng.random(n) < 0.08
    bf[low] = rng.choice([0.0, -1.0], int(low.sum()))
    nv = rng.integers(5, 40, n).astype(np.float64)
    td = nv * 0.5 * (1.0 + (0.2 * np.log(np.where(bf > 0, bf, 20.0)) if correlated else 0.0) + 0.05 * rng.normal(size=n))
    cd = np.abs(rng.normal(0.1, 0.05, n))
    out = rng.random(n) < 0.02
    cd[out] = np.where(rng.random(int(out.sum())) < 0.7, rng.uniform(1, 2, int(out.sum())), np.nan)
    flags = np.where(rng.random(n) < 0.1, 0.0, rng.choice([1.0, 3.0], n))
    return nv, td, bf, cd, flags


def _padded(rows, total, rng):
    """The same rows followed by non-contributing rows up to ``total`` rows (after the real rows, so every block-wide sum
    adds the same terms in the same order)."""
    nv, td, bf, cd, flags = rows
    m = total - len(nv)
    pad = lambda a, fill: np.concatenate((a, fill))
    return (pad(nv, rng.choice([np.inf, 1e300, 7.0], m)), pad(td, rng.uniform(-1e6, 1e6, m)), pad(bf, rng.uniform(-5, 1e6, m)),
            pad(cd, np.full(m, np.nan)), pad(flags, np.zeros(m)))


@pytest.mark.gpu
def test_staged_and_unstaged_select_agree():
    """Segment pairs in one call (max_segment > 12,288, so stage_cap = 12,288): 12,288 rows against the same rows padded
    with one non-contributing row, and 5,000 contributing rows against the same rows padded past the stage.  All 14 output
    columns are bit-identical."""
    rng = np.random.default_rng(21)
    segments = []
    for k, (n, total) in enumerate([(STAGE, STAGE + 1), (5000, STAGE + 2000), (STAGE, STAGE + 1), (5000, 3 * STAGE)]):
        rows = _mixed_rows(rng, n, correlated=k % 2 == 0)
        if n == 5000:
            rows = rows[:4] + (np.where(rows[4] == 0.0, 1.0, rows[4]),)
        density, electrons = float(rng.uniform(400, 600)), float(rng.uniform(900, 1100))
        for r in (rows, _padded(rows, total, rng)):
            segments.append(_segment(*r[:3], cd=r[3], flags=r[4], density=density, electrons=electrons, atomType=k, unitVolume=0.125))
    segOut, _ = _run_statistics(segments)
    for k in range(0, len(segments), 2):
        staged, unstaged = segOut[k], segOut[k + 1]
        assert len(segments[k]["nv"]) <= STAGE < len(segments[k + 1]["nv"])
        assert staged[0] > 0.8 * (segments[k]["flags"] != 0).sum()
        assert _same(staged, unstaged), (k, staged, unstaged)
        if segments[k]["type"] % 2 == 0:             # the correlated pairs take the fitted slope
            assert staged[7] != CURRENT + segments[k]["type"]


# --------------------------------------------------------------------------------------------- C: the slope's p-value test
DFS = (1, 2, 3, 5, 10, 30, 100, 1000, 10 ** 4, 10 ** 5)
DELTAS = (1e-2, 1e-4, 1e-6, 1e-8)


def _exact_p(x, y):
    """The two-sided p-value of the slope of y on x: I_{1 - r^2}(df / 2, 1 / 2), r from long-double moments of the float64
    arrays, the incomplete beta function by mpmath at 40 digits."""
    import mpmath
    x, y = np.asarray(x, dtype=np.longdouble), np.asarray(y, dtype=np.longdouble)
    dx, dy = x - x.mean(), y - y.mean()
    df = len(x) - 2
    with mpmath.workdps(40):
        mp = lambda v: mpmath.mpf(float(v)) + mpmath.mpf(float(v - np.longdouble(float(v))))   # a long double, exactly
        sxx, syy, sxy = mp((dx * dx).sum()), mp((dy * dy).sum()), mp((dx * dy).sum())
        return float(mpmath.betainc(mpmath.mpf(df) / 2, mpmath.mpf(1) / 2, 0, 1 - sxy * sxy / (sxx * syy), regularized=True))


def _slope_case(df, p, rng, atomType):
    """A segment of n = df + 2 contributing rows whose slope test has p-value ~p: random positive b-factors, the domain
    fraction y = r z(x) + sqrt(1 - r^2) w with x = log(b-factor) standardised to z and w random, orthogonal to x and
    standardised; r = t / sqrt(df + t^2), t = stats.t.isf(p / 2, df).  The total density is solved so that the kernel's
    y = ((der / nv) med_nv - ratio) / ratio has this value (num_voxels constant 16, a power of two).  Returns the segment
    and (x, y) recomputed from its rows exactly as the kernel computes them."""
    n = df + 2
    bf = np.round(rng.uniform(5, 60, n), 3)
    while len(np.unique(bf)) < 2:
        bf = np.round(rng.uniform(5, 60, n), 3)
    x = np.log(bf)
    z = (x - x.mean()) / x.std()
    w = rng.normal(size=n)
    w -= w.mean()
    w -= (w @ z) / (z @ z) * z
    w /= w.std()
    t = stats.t.isf(p / 2, df)
    r = t / np.sqrt(df + t * t)
    density, electrons = float(rng.uniform(400, 600)), float(rng.uniform(900, 1100))
    ratio = density / electrons
    target = 0.1 * (r * z + np.sqrt(1 - r * r) * w)
    nv = np.full(n, 16.0)
    td = ratio * (1.0 + target)
    y = (td / nv * 16.0 - ratio) / ratio
    return _segment(nv, td, bf, density=density, electrons=electrons, atomType=atomType), x, y


def _slope_cases():
    rng = np.random.default_rng(77)
    cases = []
    for df in DFS:
        for delta in DELTAS:
            for sign in (-1, 1):
                p = 0.05 * (1 + sign * delta)
                seg, x, y = _slope_case(df, p, rng, len(cases))
                cases.append({"df": df, "delta": sign * delta, "segment": seg, "x": x, "y": y, "p": _exact_p(x, y),
                              "fit": stats.linregress(x, y)})
    return cases


def _calc_slope(bf, y, current):
    """The reference's calcSlope (pdb_eda/densityAnalysis.py:729-733, :806-810) on the b-factors after the <= 0 ones took
    the median."""
    if len(y) <= 2 or len(np.unique(bf)) == 1:
        return current
    with np.errstate(all="ignore"):
        fit = stats.linregress(np.log(bf), y)
    return current if fit.pvalue > 0.05 else fit.slope


def _host_statement(segments):
    """batchAtomTypeStatistics on the contributing rows of the segments, one structure each."""
    from pdb_eda_b200 import cloudBatch
    rows = [np.flatnonzero(s["flags"].astype(np.int64) & 1) for s in segments]
    cat = lambda key: np.concatenate([s[key][r] for s, r in zip(segments, rows)])
    structure = np.concatenate([np.full(len(r), k) for k, r in enumerate(rows)])
    types = np.concatenate([np.full(len(r), s["type"]) for s, r in zip(segments, rows)])
    nT = max(s["type"] for s in segments) + 1
    return cloudBatch.batchAtomTypeStatistics(structure, types, nT, cat("td"), cat("nv"), cat("cd"), cat("bf"),
                                              [s["map"][0] / s["map"][1] for s in segments], [s["uvol"] for s in segments],
                                              CURRENT + np.arange(nT))


def _check_slope_cases(cases, slopes):
    """Decisions and fitted slopes against mpmath and linregress; returns the cases that disagree."""
    bad = []
    for c, slope in zip(cases, slopes):
        assert abs(c["p"] / 0.05 - 1) >= 1e-12, ("construction failed", c["df"], c["delta"], c["p"])
        current = CURRENT + c["segment"]["type"]
        if c["p"] > 0.05:
            ok = slope == current
        else:
            ok = slope != current and abs(slope - c["fit"].slope) <= 1e-10 * abs(c["fit"].slope)
        if not ok:
            bad.append((c["df"], c["delta"], c["p"], slope, c["fit"].slope))
    return bad


@pytest.fixture(scope="module")
def slope_cases():
    return _slope_cases()


@pytest.mark.gpu
def test_slope_decision_matches_mpmath(slope_cases):
    """Column 7 is the current slope iff the exact p-value exceeds 0.05, for p = 0.05 (1 +- delta), delta down to 1e-8 and
    df up to 1e5 (the two largest segments leave the stage); a kept fit equals scipy's slope to 1e-10, and columns 8-10
    equal the host statement to 1e-10."""
    cases = slope_cases
    segments = [c["segment"] for c in cases]
    segOut, _ = _run_statistics(segments)
    assert not _check_slope_cases(cases, segOut[:, 7])
    _, med, present = _host_statement(segments)
    k = np.arange(len(segments))
    assert present[k, k].all() and np.array_equal(segOut[:, 0], [len(s["nv"]) for s in segments])
    for col, column in ((8, "domain_fraction"), (9, "corrected_fraction"), (10, "corrected_density_electron_ratio")):
        np.testing.assert_allclose(segOut[:, col], med[column][k, k], rtol=1e-10, atol=0, err_msg=column)
    assert np.array_equal(segOut[:, 8], [_nanmedian(c["y"]) for c in cases])


# ----------------------------------------------------------------------------------------------------- D: degenerate fits
def _degenerate_cases():
    """(name, segment) pairs: n = 1, 2, 3; all b-factors equal, also only after the ones <= 0 took the median; y constant
    (r and p NaN: `NaN > 0.05` is false, so the fitted slope 0.0 is kept); y linear in log(b-factor) (r = +-1)."""
    rng = np.random.default_rng(41)
    cases = []
    add = lambda name, bf, td, nv=None: cases.append((name, _segment(np.full(len(bf), 1.0) if nv is None else nv, td, bf,
                                                                          atomType=len(cases))))
    for n in (1, 2, 3):
        add("n=%d" % n, rng.uniform(5, 60, n), rng.uniform(0.3, 0.7, n))
    add("n=3 linear", np.array([10.0, 20.0, 40.0]), 0.5 * (1 + 0.1 * np.log([10.0, 20.0, 40.0])))
    add("equal b-factors", np.full(50, 20.0), rng.uniform(0.3, 0.7, 50))
    add("equal after the median replaces b <= 0", np.array([20.0, 0.0, -3.0, 20.0, 20.0, -0.0, 20.0]), rng.uniform(0.3, 0.7, 7))
    add("distinct after the median replaces b <= 0", np.array([20.0, 30.0, 0.0, -1.0, 30.0, 20.0, 25.0]), 0.5 * (1 + 0.05 * np.arange(7)))
    bf = np.round(rng.uniform(5, 60, 40), 2)
    add("y = 0", bf, np.full(40, 0.5))                        # ratio 0.5 (500 / 1000): y = (0.5 - 0.5) / 0.5
    add("y = 0.25", bf, np.full(40, 0.625))                   # exactly representable: the mean of y is y
    add("y = 0.3 log(b)", bf, 0.5 * (1 + 0.3 * np.log(bf)))
    add("y = -0.3 log(b)", bf, 0.5 * (1 - 0.3 * np.log(bf)))
    return cases


def _replaced_bfactors(bf):
    bf = bf.copy()
    med = _nanmedian(bf[bf > 0])
    bf[bf <= 0] = med
    return bf


@pytest.mark.gpu
def test_degenerate_fits_follow_calc_slope():
    cases = _degenerate_cases()
    segOut, _ = _run_statistics([s for _, s in cases])
    _, med, _ = _host_statement([s for _, s in cases])
    for k, (name, s) in enumerate(cases):
        y = (s["td"] / s["nv"] * _nanmedian(s["nv"]) - 0.5) / 0.5
        want = _calc_slope(_replaced_bfactors(s["bf"]), y, CURRENT + k)
        got = segOut[k, 7]
        if want == CURRENT + k or want == 0.0:
            assert got == want, (name, got, want)
        else:
            assert abs(got - want) <= 1e-10 * abs(want), (name, got, want)
        for col, column in ((7, "slopes"), (8, "domain_fraction"), (9, "corrected_fraction"), (10, "corrected_density_electron_ratio")):
            np.testing.assert_allclose(segOut[k, col], med[column][k, k], rtol=1e-10, atol=0, err_msg="%s %s" % (name, column))


# ---------------------------------------------------------------------------------------------------------------- F: CPU
def test_host_statement_slope_decisions(slope_cases):
    """batchAtomTypeStatistics takes the same decisions as mpmath and the same slopes as linregress on the cases of C, and
    follows calcSlope on the degenerate cases of D."""
    _, med, _ = _host_statement([c["segment"] for c in slope_cases])
    k = np.arange(len(slope_cases))
    assert not _check_slope_cases(slope_cases, med["slopes"][k, k])
    cases = _degenerate_cases()
    _, med, _ = _host_statement([s for _, s in cases])
    for k, (name, s) in enumerate(cases):
        y = (s["td"] / s["nv"] * _nanmedian(s["nv"]) - 0.5) / 0.5
        want = _calc_slope(_replaced_bfactors(s["bf"]), y, CURRENT + k)
        got = med["slopes"][k, k]
        assert got == want or abs(got - want) <= 1e-10 * abs(want), (name, got, want)
    assert [med["slopes"][k, k] for k in range(len(cases))].count(0.0) == 2    # the two constant-y cases keep the fit 0.0


# ------------------------------------------------------------------------------------- E: production flow beyond the stage
@pytest.mark.gpu
def test_cloud_batch_beyond_the_stage():
    """CloudBatch on one poly-ALA structure of 16,000 residues (300^3 map): each ALA atom type is a segment of more than
    12,288 atoms.  The centroid cutoff (cutoff_kernel) against nanmedian + 2.5 nanstd of the device's own atom rows, and
    the per-type medians against batchAtomTypeStatistics on those rows."""
    from pdb_eda_b200 import _device, ccp4, cloudBatch, synthetic
    params = synthetic.defaultParams()
    atomTypes = sorted(params["radii"])
    params["slopes"] = {t: CURRENT + k for k, t in enumerate(atomTypes)}
    n, residues, seed = 300, 16000, 9
    cell = (0.5 * n,) * 3 + (90.0, 90.0, 90.0)
    coords, bf = synthetic.fastPolyAla(residues, cell, seed)
    table = synthetic.polyAlaTable(coords, bf, params)
    assert table.supported
    electronsOf = np.array([synthetic.ALA_ELECTRONS["ALA_" + a] for a, _, _ in synthetic._ALA_ATOMS])
    rho = synthetic.densityMapDevice(coords, np.tile(electronsOf, residues), n, cell, seed + 1)
    hdr = ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((n, n, n), cell, (n, n, n)))
    dmap = _device.DeviceMap(_device.geom_from_header(hdr), rho.reshape(-1))
    m, s = dmap.mean_std()
    batch = cloudBatch.CloudBatch([(cloudBatch.MapRef(dmap, m + 1.5 * s, hdr.unitVolume, "big"), table)], params)
    assert batch.maxSegment > STAGE and batch.nSegments == 5
    batch.launch()
    arr = batch.collectArrays()
    rows = batch.atomRows()
    assert arr["ok"][0]
    # centroid cutoff: median exact (a neighbouring order statistic is ~1e-3 away), standard deviation to 1e-12
    d = rows[(rows[:, 0] > 0) & ~np.isnan(rows[:, 2]), 2]
    assert len(d) > 5 * STAGE
    med, std = float(np.median(d)), float(np.std(d))
    assert abs(arr["centroidCutoff"][0] - (med + 2.5 * std)) <= 2.5 * std * 1e-12 + 4 * np.spacing(med + 2.5 * std)
    # the statistics block on the contributing rows
    acc = (rows[:, 7].astype(np.int64) & 1) != 0
    assert (batch.segEnd - batch.segBegin).min() > STAGE and acc.sum() > 0.5 * len(rows)
    ratio = arr["totalDensity"][0] / arr["totalElectrons"][0]
    keep, host, present = cloudBatch.batchAtomTypeStatistics(
        np.zeros(int(acc.sum()), dtype=np.int64), batch.typeIndex[acc], len(atomTypes), rows[acc, 3] / batch.electrons[acc] / batch.occupancy[acc],
        rows[acc, 1], rows[acc, 2], batch.bfactor[acc], [ratio], batch.unitVolume, [params["slopes"][t] for t in atomTypes])
    assert arr["ratio"][0] == ratio and arr["analysed"][0] == keep.sum()
    assert np.array_equal(arr["present"], present) and present.all()
    for column in cloudBatch.MEDIAN_COLUMNS:
        got, want = arr["medians"][column][0], host[column][0]
        if column in ("slopes", "corrected_fraction", "corrected_density_electron_ratio"):
            np.testing.assert_allclose(got, want, rtol=1e-10, atol=0, err_msg=column)
        else:
            assert np.array_equal(got, want), (column, got, want)
