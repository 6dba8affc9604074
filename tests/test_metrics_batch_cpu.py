"""CPU tier of the batched RSCC / RSR path (pdb_eda_b200/metricsBatch.py, pe_pair_union_metrics): argument errors without a
device, the ``--single-mode`` surface of ``multiple``, the numpy row builder against a per-residue loop, and the all-reduced
summary over two gloo ranks."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch.multiprocessing as mp


def test_argument_errors_without_a_device():
    from pdb_eda_b200 import _lib
    lib = _lib.load()
    assert lib.pe_pair_union_workspace_bytes(-1) == -1
    assert lib.pe_pair_union_workspace_bytes(10) >= 10 * 32
    assert lib.pe_pair_union_metrics(-1, None, 1, None, None, None, None, None, None, None) == -1
    assert b"negative size" in lib.pe_last_error()
    assert lib.pe_pair_union_metrics(1, None, -3, None, None, None, None, None, None, None) == -1
    assert lib.pe_pair_union_metrics(1, None, 2, None, None, None, None, None, None, None) == -1
    assert b"null pointer" in lib.pe_last_error()
    assert lib.pe_pair_union_metrics(0, None, 2, None, None, None, None, None, None, None) == -1
    assert lib.pe_pair_union_metrics(0, None, 0, None, None, None, None, None, None, None) == 0   # nothing to do


def test_single_mode_parsing():
    from pdb_eda_b200 import multipleStructures
    a = multipleStructures.parseSingleMode("statistics --residue --out-format csv --include-pdbid")
    assert a.submode == "statistics" and a.residue and not a.atom and a.out_format == "csv" and a.include_pdbid
    a = multipleStructures.parseSingleMode("density --residue --radius 2.5")
    assert a.submode == "density" and a.radius == 2.5
    for bad in ("nosuchmode", "statistics --pdb-file x.pdb"):
        with pytest.raises(SystemExit):
            multipleStructures.parseSingleMode(bad)
    e = multipleStructures._entryArgs(multipleStructures.parseSingleMode("statistics --atom"), "1abc", "/out", "/data")
    assert e.pdbid == "1abc" and e.out_file == os.path.join("/out", "1abc.result")
    assert e.density_file == os.path.join("/data", "1abc.ccp4") and e.diff_file == os.path.join("/data", "1abc_diff.ccp4")


def test_metrics_radius_and_rscc_rsr():
    from pdb_eda_b200 import metricsBatch
    assert metricsBatch.metricsRadius(0.5) == 0.7 and metricsBatch.metricsRadius(3.3) == 3.3 * 0.5
    assert metricsBatch.metricsRadius(2.0) == (2.0 - 0.6) / 3 + 0.7
    with pytest.raises(TypeError):
        metricsBatch.metricsRadius(None)
    sums = np.array([[0, 0, 0, 0, 0, 0, 0, 0], [3, 1, 1, 2.0, 4.0, 1.0, 4.0, 2.5]], dtype=np.float64)
    rscc, rsr = metricsBatch.rsccRsr(sums)
    assert np.isnan(rscc[0]) and np.isnan(rsr[0]) and rscc[1] == 1.0 and rsr[1] == 0.5


class _Map:
    def __init__(self, n):
        import torch
        self.rho = torch.zeros(n)


class _Analyzer:
    def __init__(self, st, n=8, nd=8):
        self.biopdbObj = st
        self.densityObj = type("D", (), {"deviceMap": _Map(n)})()
        self.diffDensityObj = type("D", (), {"deviceMap": _Map(nd)})()


def _structure(seed):
    from pdb_eda_b200 import synthetic
    st = synthetic.polyAlaStructure(23, (0, 0, 0), (30.0, 30.0, 30.0), seed=seed, residuesPerChain=10, hetero=4)
    rng = np.random.default_rng(seed)
    for atom in st.get_atoms():
        atom.occupancy = float(rng.choice([0.0, 0.25, 0.5, 1.0], p=[0.1, 0.2, 0.2, 0.5]))
    for residue in st.get_residues():            # every residue keeps one occupied atom
        residue.child_list[0].occupancy = 0.75
    return st


def test_residue_rows_against_a_per_residue_loop():
    from pdb_eda_b200 import metricsBatch
    st = _structure(5)
    entry = metricsBatch.residueEntry(_Analyzer(st))
    residues = list(st.get_residues())
    assert entry.nGroups == len(residues) and entry.radius == metricsBatch.metricsRadius(2.0)
    assert entry.groupStart.tolist() == np.cumsum([0] + [len(r.child_list) for r in residues]).tolist()
    np.testing.assert_array_equal(entry.coords32, np.asarray([a.coord for r in residues for a in r.child_list], dtype=np.float32))
    rng = np.random.default_rng(3)
    rscc, rsr = rng.uniform(-1, 1, len(residues)), rng.uniform(0, 1, len(residues))
    rscc[2] = np.nan
    got = entry.finish(rscc, rsr)
    for k, residue in enumerate(residues):          # residueMetrics()'s loop (pdb_eda_b200/densityAnalysis.py)
        bfactorWeightedSum = occupancySum = 0.0
        for atom in residue.child_list:
            bfactorWeightedSum += atom.get_bfactor() * atom.get_occupancy()
            occupancySum += atom.get_occupancy()
        want = [residue.parent.id, residue.id[1], residue.resname, rscc[k], rsr[k], occupancySum / len(residue.child_list),
                bfactorWeightedSum / occupancySum]
        assert got[k][:3] == want[:3] and got[k][5:] == want[5:]          # bit-identical
        np.testing.assert_array_equal(got[k][3:5], want[3:5])


def test_entries_that_fail_like_the_single_call():
    from pdb_eda_b200 import metricsBatch
    st = _structure(6)
    for atom in list(st.get_residues())[4].child_list:
        atom.occupancy = 0.0
    with pytest.raises(ZeroDivisionError):
        metricsBatch.residueEntry(_Analyzer(st))
    st = _structure(7)
    with pytest.raises(ValueError):
        metricsBatch.residueEntry(_Analyzer(st, 8, 9))       # maps on different grids
    st.header["resolution"] = None
    with pytest.raises(TypeError):
        metricsBatch.residueEntry(_Analyzer(st))
    # failed and missing entries yield None without a device
    out = metricsBatch.analyzeMetrics([0, _Analyzer(st)], "residue")
    assert out == [None, None]


def _worker(rank, world, port, out):
    import torch.distributed as dist
    from pdb_eda_b200 import multi
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    loads = []
    run = multi.runMultipleMetrics(list(range(7)), lambda i: loads.append(i) or 0, "residue", costs=[3, 1, 4, 1, 5, 9, 2],
                                   device="cpu")
    summary = multi.summarizeMetrics(rank + 1, 2 * rank, 10 * rank + 5, "cpu")
    out[rank] = (run, summary, loads)
    dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


@pytest.mark.timeout(120)
def test_two_rank_summary_over_gloo():
    manager = mp.Manager()
    out = manager.dict()
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    for rank in range(2):
        run, summary, _ = out[rank]
        assert run == {"ok": 0, "failed": 7, "rows": 0}
        assert summary == {"ok": 3, "failed": 2, "rows": 20}
    assert sorted(out[0][2] + out[1][2]) == list(range(7))      # every entry loaded once, by its owner
    from pdb_eda_b200 import multi
    shards = multi.shardStructures([3, 1, 4, 1, 5, 9, 2], 2)
    assert out[0][2] == shards[0] and out[1][2] == shards[1] and shards[0][0] == 5   # longest first
