"""Recorded results for the tests that compare this package with pdb_eda 2.7.1 (the reference).

Where the reference is installed (oracle/_ref, see oracle/build_ref.py) those tests compare with it live.  Everywhere
else they compare with tests/golden/recorded/<test>.npz.  Those files hold this package's results (the CUDA library,
or for the CPU tier the C oracle), not the reference's: the reference is not part of this repository and was not
installed where they were recorded.  They pin what the package computes, so a clean checkout checks every later
change against them; they do not replace the live comparison, which stays the test of correctness.

Inputs: the recorded branch hands the package the inputs of the live branch.  The cutoffs the live branch takes from
the reference (mean + k sigma by np.mean / np.std over the stored voxels in float64, pdb_eda/ccp4.py:350-363) are
computed the same way on the host and stored (``inputs``); the live branch asserts that the reference's own cutoffs
equal the stored ones bit for bit, and the recorded branch uses the stored ones.

A recorded value is a digest of the nested result (lists, tuples, dicts, sets, numpy arrays, scalars, strings):
  exact part  sha256 of every count, index, flag, string and shape, in order -- bit-exact like the live bars;
  float part  every float64 in order, compared within the test's own rtol / atol: all of them when there are at most
              SAMPLE, otherwise a seeded sample of SAMPLE; always their count and NaN pattern, and three sums bounded
              by the same tolerance: the signed sum, the sum of magnitudes and a sum with seeded random signs (which
              errors that cancel in the signed sum do not escape).
Record:  PDB_EDA_RECORD_DIR=<dir> python -m pytest <tests> writes <dir>/<test>.npz instead of checking.
"""
import hashlib
import os
import re

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "recorded")
SAMPLE = 256


def reference():
    """The modules of the installed reference (ccp4, densityAnalysis, cutils, pdbParser), or None without oracle/_ref."""
    from oracle import refload
    return refload.load() if refload.available() else None


def host_mean_std(densityMatrix):
    """np.mean / np.std (population) over the stored voxels in float64, the reference's statistics (pdb_eda/ccp4.py:350-363)."""
    values = np.asarray(densityMatrix.densityArray, dtype=np.float64).ravel()
    return float(np.mean(values)), float(np.std(values))


def inputs(name, values, live=False):
    """The stored inputs ``name`` (cutoffs) of a test.  ``live``: ``values`` come from the reference and must equal the stored
    ones.  Otherwise ``values`` are the host restatement, written when recording and replaced by the stored ones when checking."""
    values = [float(v) for v in values]
    out = os.environ.get("PDB_EDA_RECORD_DIR")
    if out and not live:
        os.makedirs(out, exist_ok=True)
        np.savez_compressed(os.path.join(out, _path(name + "-inputs")), values=np.array(values))
        return values
    stored = np.load(os.path.join(GOLDEN_DIR, _path(name + "-inputs")))["values"].tolist()
    if live:
        assert values == stored, "%s: the reference's inputs %r differ from the stored %r" % (name, values, stored)
    return stored


def _walk(v, tok, flt):
    if v is None:
        tok.append(b"N")
    elif isinstance(v, (bool, np.bool_)):
        tok.append(b"b1" if v else b"b0")
    elif isinstance(v, (int, np.integer)):
        tok.append(b"i%d" % int(v))
    elif isinstance(v, (float, np.floating)):
        tok.append(b"f")
        flt.append(np.array([v], dtype=np.float64))
    elif isinstance(v, str):
        tok.append(b"s" + v.encode())
    elif isinstance(v, np.ndarray):
        tok.append(b"a" + repr(v.shape).encode())
        if v.dtype.names:
            for name in v.dtype.names:
                tok.append(b"F" + name.encode())
                _walk(v[name], tok, flt)
        elif v.dtype.kind == "f":
            flt.append(v.astype(np.float64).ravel())
        elif v.dtype.kind in "iub":
            tok.append(np.ascontiguousarray(v, dtype=np.int64).tobytes())
        elif v.dtype.kind in "US":
            tok.append("\0".join(str(x) for x in v.ravel()).encode())
        else:
            for x in v.ravel():
                _walk(x, tok, flt)
    elif isinstance(v, dict):
        tok.append(b"{%d" % len(v))
        for k in sorted(v, key=repr):
            _walk(k, tok, flt)
            _walk(v[k], tok, flt)
    elif isinstance(v, (set, frozenset)):
        _walk(sorted(v), tok, flt)
    elif isinstance(v, (list, tuple)):
        tok.append(b"[%d" % len(v))
        for x in v:
            _walk(x, tok, flt)
    elif hasattr(v, "__array__"):          # torch tensors and the like
        _walk(np.asarray(v), tok, flt)
    else:
        raise TypeError("no digest for %r" % type(v))


def digest(value):
    tok, flt = [], []
    _walk(value, tok, flt)
    f = np.concatenate(flt) if flt else np.zeros(0)
    h = hashlib.sha256()
    for t in tok:
        h.update(len(t).to_bytes(8, "little"))
        h.update(t)
    idx = np.arange(f.size) if f.size <= SAMPLE else np.sort(np.random.default_rng(f.size).choice(f.size, SAMPLE, replace=False))
    return {"exact": np.array(h.hexdigest()), "n": np.array(f.size), "idx": idx, "sample": f[idx],
            "nan": np.array(hashlib.sha256(np.packbits(np.isnan(f)).tobytes()).hexdigest()),
            "sum": np.array(np.nansum(f)), "abssum": np.array(np.nansum(np.abs(f))), "signsum": np.array(np.nansum(_signs(f.size) * f))}


def _signs(n):
    return np.where(np.random.default_rng(n + 1).random(n) < 0.5, -1.0, 1.0)


def _path(name):
    return re.sub(r"[^A-Za-z0-9_.-]+", "_", name) + ".npz"


def check(name, value, rtol=1e-9, atol=1e-9):
    """Compares ``value`` with the recorded result ``name`` (or records it under $PDB_EDA_RECORD_DIR)."""
    got = digest(value)
    out = os.environ.get("PDB_EDA_RECORD_DIR")
    if out:
        os.makedirs(out, exist_ok=True)
        np.savez_compressed(os.path.join(out, _path(name)), **got)
        return
    z = np.load(os.path.join(GOLDEN_DIR, _path(name)))
    want = {k: z[k] for k in z.files}
    assert str(got["exact"]) == str(want["exact"]), "%s: counts, indices, flags or strings differ from the recorded result" % name
    assert int(got["n"]) == int(want["n"]) and str(got["nan"]) == str(want["nan"]), "%s: float values differ in number or NaN pattern" % name
    a, b = got["sample"], want["sample"]
    scale = np.maximum(np.abs(a), np.abs(b))
    bad = ~((np.abs(a - b) <= rtol * scale + atol) | (np.isnan(a) & np.isnan(b)))
    assert not bad.any(), "%s: float values differ from the recorded result at %s" % (name, want["idx"][bad][:5].tolist())
    slack = (rtol + 2.3e-16 * int(want["n"])) * float(want["abssum"]) + atol * int(want["n"])     # plus the summation's rounding
    for key in ("sum", "abssum", "signsum"):
        assert abs(float(got[key]) - float(want[key])) <= slack, "%s: the %s of the float values differs from the recorded one" % (name, key)
