"""VoxelPass.step on an SM partition (blob pass on its own SMs, sphere kernel on the others) against the shared-SM schedule
(PDB_EDA_B200_BLOB_SMS=0): the same cloud and region rows bit for bit, the same blob keys, labels and counts, blob sums equal or
within 1e-12 relative (float64 atomics that a different grid may group differently); refused counts fall back; partitions can be
destroyed and made again; the sparse kernel's placement flag stays clear on a partition."""
import ctypes
import io
import os
import sys
import warnings

import numpy as np
import pytest

from pdb_eda_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_partition_arguments_without_a_device():
    lib = _lib.load()
    sb, sr, nb, nr = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_int32(), ctypes.c_int32()
    assert lib.pe_sm_partition_create(0, 32, None, ctypes.byref(sr), ctypes.byref(nb), ctypes.byref(nr)) == -1
    assert b"pe_sm_partition_create" in lib.pe_last_error()
    assert lib.pe_sm_partition_create(0, 0, ctypes.byref(sb), ctypes.byref(sr), ctypes.byref(nb), ctypes.byref(nr)) == -1
    assert lib.pe_sm_partition_destroy(None, None) == -1
    import torch
    if not torch.cuda.is_available():
        assert lib.pe_sm_partition_create(0, 32, ctypes.byref(sb), ctypes.byref(sr), ctypes.byref(nb), ctypes.byref(nr)) == -4


def _small_pass():
    from pdb_eda_b200 import ccp4, synthetic
    from pdb_eda_b200.pipeline import VoxelPass
    cell, n = (32.0, 32.0, 32.0, 90, 90, 90), (64, 64, 64)
    st = synthetic.polyAlaStructure(60, (0, 0, 0), cell[:3], seed=8)
    a, b = synthetic.mapPair(st, n, cell, seed=9)
    dens = ccp4.parse(io.BytesIO(synthetic.ccp4Bytes(a, cell, n)), "d")
    diff = ccp4.parse(io.BytesIO(synthetic.ccp4Bytes(b, cell, n)), "f")
    xyz = np.array([at.coord for at in st.get_atoms()], dtype=np.float64)
    radii = np.tile(np.array([0.78, 0.72, 0.66, 0.81, 0.84], dtype=np.float32), 60)
    start = np.arange(0, 301, 5, dtype=np.int32)
    return VoxelPass(dens.deviceMap, diff.deviceMap, xyz, radii, start, 3.5)


def _c2_pass():
    """The 384^3 workload bench.py times (seed 2)."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from pdb_eda_b200 import _device, ccp4, synthetic
    from pdb_eda_b200.pipeline import VoxelPass
    work = bench.build_workload(bench.FULL, seed=2)
    n, cell = work["n"], work["cell"]
    geom = _device.geom_from_header(ccp4.DensityHeader.fromFileHeader(synthetic.ccp4Header((n, n, n), cell, (n, n, n))))
    dens = _device.DeviceMap(geom, torch.from_numpy(work["fofc2"].reshape(-1)).cuda())
    diff = _device.DeviceMap(geom, torch.from_numpy(work["fofc"].reshape(-1)).cuda())
    return VoxelPass(dens, diff, work["xyz"].astype(np.float64), work["radii"], work["res_start"], bench.REGION_RADIUS)


def _step(vp, blob_sms, monkeypatch):
    """One step with PDB_EDA_B200_BLOB_SMS = blob_sms into outputs filled with garbage first; its results (deep copies)."""
    monkeypatch.setenv("PDB_EDA_B200_BLOB_SMS", str(blob_sms))
    for t in (vp.cloud_out, vp.region_out, vp.blob_stats):
        t.fill_(float("nan"))
    vp.blob_key.fill_(-7)
    vp.blob_label.fill_(-7)
    vp.step()
    res = vp.results()
    return {"cloud": res["cloud"].copy(), "region": res["region"].copy(), "blob_counts": res["blob_counts"].copy(),
            **{tag: {k: v.copy() for k, v in res[tag].items()} for tag in ("green", "red")}}


def _assert_same(a, b):
    assert np.array_equal(a["cloud"], b["cloud"]) and np.array_equal(a["region"], b["region"])
    assert np.array_equal(a["blob_counts"], b["blob_counts"]) and a["blob_counts"][4] == 0
    for tag in ("green", "red"):
        assert np.array_equal(a[tag]["key"], b[tag]["key"]) and np.array_equal(a[tag]["label"], b[tag]["label"])
        sa, sb = a[tag]["stats"], b[tag]["stats"]
        if not np.array_equal(sa, sb):
            np.testing.assert_allclose(sa, sb, rtol=1e-12, atol=0)


def _sms():
    return _lib.require_device()[0]


@pytest.mark.gpu
def test_partitioned_step_matches_shared_sms_small(monkeypatch):
    vp = _small_pass()
    want = _step(vp, 0, monkeypatch)
    assert len(want["green"]["key"]) > 0 and len(want["red"]["key"]) > 0
    for k in (16, 32, 56):
        _assert_same(_step(vp, k, monkeypatch), want)


@pytest.mark.gpu
def test_partitioned_step_matches_shared_sms_c2(monkeypatch):
    from pdb_eda_b200 import pipeline
    vp = _c2_pass()
    want = _step(vp, 0, monkeypatch)
    for k in sorted({16, pipeline.BLOB_SMS, 48}):
        got = _step(vp, k, monkeypatch)
        assert pipeline.smPartition(vp.device, k) is not None
        _assert_same(got, want)
        assert int(vp.blob_counts[4].item()) == 0           # placement flag of the sparse kernel: 3 blocks on every SM


@pytest.mark.gpu
def test_refused_counts_fall_back_to_shared_sms(monkeypatch):
    from pdb_eda_b200 import pipeline
    vp = _small_pass()
    want = _step(vp, 0, monkeypatch)
    for k in (20, _sms(), _sms() + 8, -8, "many"):
        with pytest.warns(RuntimeWarning, match="no partition"):
            got = _step(vp, k, monkeypatch)
        _assert_same(got, want)
        with warnings.catch_warnings():
            warnings.simplefilter("error")                  # said once per count
            _step(vp, k, monkeypatch)
    assert all(pipeline._partitions[(vp.device.index or 0, k)] is None for k in (20, _sms(), -8))


@pytest.mark.gpu
def test_partition_create_destroy_create(monkeypatch):
    from pdb_eda_b200 import pipeline
    lib = _lib.load()
    sms = _sms()
    for _ in range(2):
        sb, sr, nb, nr = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_int32(), ctypes.c_int32()
        assert lib.pe_sm_partition_create(0, 24, ctypes.byref(sb), ctypes.byref(sr), ctypes.byref(nb), ctypes.byref(nr)) == 0
        assert (nb.value, nr.value) == (24, sms - 24) and sb.value and sr.value
        assert lib.pe_sm_partition_destroy(sb, sr) == 0
        assert lib.pe_sm_partition_destroy(sb, sr) == -1     # already gone
    vp = _small_pass()
    want = _step(vp, 0, monkeypatch)
    first = _step(vp, 32, monkeypatch)
    pipeline.releasePartitions()
    assert not pipeline._partitions
    again = _step(vp, 32, monkeypatch)
    _assert_same(first, want)
    _assert_same(again, want)
    assert pipeline.smPartition(vp.device, 32) is not None
