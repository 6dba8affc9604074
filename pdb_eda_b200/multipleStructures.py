"""``multiple`` mode command line: many PDB entries, sharded over the GPUs of the node (pdb_eda/multipleStructures.py:61-194).

Usage:
    python -m pdb_eda_b200 multiple <pdbid-file> <out-result-file> [--out-format json|csv] [--params FILE] [--data-dir DIR] [--workers W]
    python -m pdb_eda_b200 multiple <pdbid-file> <out-dir> --single-mode "<single options>" [--data-dir DIR]
    torchrun --nproc-per-node N -m pdb_eda_b200 multiple ...        (one rank per GPU; rank 0 writes the result)

<pdbid-file>: JSON list or whitespace-separated text of PDB ids.  --data-dir: analyse DIR/<id>.ccp4, DIR/<id>_diff.ccp4,
DIR/pdb<id>.ent(.gz) instead of downloading.  Result: per-entry ``stats`` and ``diffs`` as in ``analyzePDBID``
(pdb_eda/multipleStructures.py:320-356), plus the all-reduced cumulative statistics.

--single-mode runs a ``single`` submode on every entry (the reference's ``multiple --single-mode``): "<single options>" are
the options of ``single`` after <pdbid> <out-file>, e.g. "statistics --residue --out-format csv --include-pdbid", and every
entry's result goes to <out-dir>/<pdbid>.result in the schema ``single`` writes.  ``statistics --residue`` / ``--atom`` runs
batched on the device (``multi.runMultipleMetrics``; with --print-validation, entry by entry); every other submode runs
``single`` entry by entry on the rank that owns the entry.  Entries are sharded over the ranks and every rank writes the
files of its own entries; the summary line (entries ok / failed, rows) is printed by rank 0.
"""
import argparse
import csv
import functools
import json
import copy
import os
import shlex
import sys

import torch
import torch.distributed as dist

from . import densityAnalysis, multi, singleStructure

statsHeaders = ['density_electron_ratio', 'voxel_volume', 'num_voxels_aggregated', 'total_aggregated_electrons', 'num_atoms_analyzed',
                'num_residue_clouds_analyzed', 'num_domain_clouds_analyzed', 'atom_overlap_completeness']


def readIds(path):
    text = open(path).read()
    try:
        ids = json.loads(text)
    except ValueError:
        ids = text.split()
    return [str(i).lower() for i in ids]


def loadEntry(dataDir, pdbid):
    """DensityAnalysis of one entry: downloaded (``dataDir`` empty) or read from DIR/<id>.ccp4, DIR/<id>_diff.ccp4, DIR/pdb<id>.ent(.gz)."""
    if not dataDir:
        return densityAnalysis.fromPDBid(pdbid)
    pdb = os.path.join(dataDir, "pdb" + pdbid + ".ent.gz")
    if not os.path.isfile(pdb):
        pdb = os.path.join(dataDir, "pdb" + pdbid + ".ent")
    an = densityAnalysis.fromFile(pdb, os.path.join(dataDir, pdbid + ".ccp4"), os.path.join(dataDir, pdbid + "_diff.ccp4"))
    if an:
        an.pdbid = pdbid
    return an


def makeLoader(dataDir):
    return functools.partial(loadEntry, dataDir)     # picklable: usable by the host worker pool


def main(argv=None):
    p = argparse.ArgumentParser(prog="pdb_eda_b200 multiple")
    p.add_argument("pdbid_file")
    p.add_argument("out_result_file")
    p.add_argument("--out-format", default="json", choices=["json", "csv"])
    p.add_argument("--params", default="")
    p.add_argument("--data-dir", default="")
    p.add_argument("--workers", type=int, default=1, help="host worker processes per rank (all drive the rank's GPU)")
    p.add_argument("--single-mode", default=None, help="options of a single-structure submode, run on every entry")
    args = p.parse_args(argv)
    single = parseSingleMode(args.single_mode) if args.single_mode is not None else None
    if args.params:
        densityAnalysis.setGlobals(json.load(open(args.params)))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 and not dist.is_initialized():
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")
    rank = dist.get_rank() if dist.is_initialized() else 0
    ids = readIds(args.pdbid_file)
    if single is not None:
        summary = runSingleMode(ids, args.out_result_file, single, args.data_dir)
        if rank == 0:
            print(json.dumps(summary, sort_keys=True))
        if dist.is_initialized():
            dist.barrier()
        return
    types = sorted(densityAnalysis.paramsGlobal["radii"])
    summary = multi.runMultipleStructures(ids, makeLoader(args.data_dir), None, types, workers=args.workers)
    if rank == 0:
        cols = summary["columns"]
        full = {}
        for row in summary["rows"]:
            rec = dict(zip(cols, row.tolist()))
            pdbid = ids[int(rec["index"])]
            full[pdbid] = {"pdbid": pdbid, "stats": {h: rec[h] for h in statsHeaders},
                           "diffs": {t: rec["diff:" + t] for t in types}, "execution_time": rec["execution_time"]}
        with open(args.out_result_file, "w", newline="") if args.out_result_file != "-" else sys.stdout as out:
            if args.out_format == "csv":
                writer = csv.writer(out)
                writer.writerow(["pdbid"] + statsHeaders + types)
                for rec in full.values():
                    writer.writerow([rec["pdbid"]] + [rec["stats"][h] for h in statsHeaders] + [rec["diffs"][t] for t in types])
            else:
                print(json.dumps({"entries": full, "cumulative": summary["cumulative"]}, indent=2, sort_keys=True), file=out)
    if dist.is_initialized():
        dist.barrier()


def parseSingleMode(text):
    """The options of ``--single-mode`` as the ``single`` parser reads them (<pdbid> and <out-file> are set per entry)."""
    args = singleStructure.buildParser().parse_args(["-", "-"] + shlex.split(text))
    if args.pdb_file or args.density_file or args.diff_file:
        raise SystemExit("--single-mode: entries come from --data-dir or the PDB, not from --pdb-file / --density-file / --diff-file")
    return args


def _entryArgs(single, pdbid, outDir, dataDir):
    a = copy.copy(single)
    a.pdbid, a.out_file = pdbid, os.path.join(outDir, pdbid + ".result")
    if dataDir:
        pdb = os.path.join(dataDir, "pdb" + pdbid + ".ent.gz")
        a.pdb_file = pdb if os.path.isfile(pdb) else os.path.join(dataDir, "pdb" + pdbid + ".ent")
        a.density_file, a.diff_file = os.path.join(dataDir, pdbid + ".ccp4"), os.path.join(dataDir, pdbid + "_diff.ccp4")
    return a


def runSingleMode(ids, outDir, single, dataDir="", group=None):
    """``single`` with the options ``single`` (``parseSingleMode``) on every entry of ``ids``; this rank writes the result files
    of its own entries.  Returns the all-reduced counts of ``multi.summarizeMetrics`` (entries ok / failed, rows)."""
    os.makedirs(outDir, exist_ok=True)
    sizeOf = lambda path: os.path.getsize(path) if os.path.isfile(path) else 0
    costs = [sizeOf(os.path.join(dataDir, i + ".ccp4")) + 1 for i in ids] if dataDir else None     # longest first
    if single.submode == "statistics" and not single.print_validation:
        level = "residue" if single.residue else "atom"

        def write(idx, rows):
            header = (densityAnalysis.DensityAnalysis.residueMetricsHeaderList if level == "residue"
                      else densityAnalysis.DensityAnalysis.atomMetricsHeaderList)
            a = _entryArgs(single, ids[idx], outDir, dataDir)
            singleStructure.writeResult(a, *singleStructure.statisticsResult(a, header, rows, ids[idx]))

        return multi.runMultipleMetrics(ids, makeLoader(dataDir), level, costs=costs, write=write, group=group)
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    ok = failed = nrows = 0
    for idx in multi.shardStructures(costs or [1.0] * len(ids), world)[rank]:
        a = _entryArgs(single, ids[idx], outDir, dataDir)
        try:
            header, rows = singleStructure.analyze(a)
        except Exception:
            failed += 1
            continue
        singleStructure.writeResult(a, header, rows)
        ok += 1
        nrows += len(rows)
    device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
    return multi.summarizeMetrics(ok, failed, nrows, device, group)


if __name__ == "__main__":
    main()
