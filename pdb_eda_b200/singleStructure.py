"""``single`` mode command line: one PDB entry analysed on the GPU (argument surface and output schemas of
pdb_eda/singleStructure.py:1-178; docopt is not required).

Usage:
    python -m pdb_eda_b200 single <pdbid> <out-file> map (--density | --diff-density)
    python -m pdb_eda_b200 single <pdbid> <out-file> cloud (--atom | --residue | --domain) [options]
    python -m pdb_eda_b200 single <pdbid> <out-file> density (--atom | --residue | --symmetry-atom) [options]
    python -m pdb_eda_b200 single <pdbid> <out-file> difference (--atom | --residue | --symmetry-atom) [options]
    python -m pdb_eda_b200 single <pdbid> <out-file> blob [--green] [--red] [--blue] [options]
    python -m pdb_eda_b200 single <pdbid> <out-file> statistics (--atom | --residue) [--print-validation] [options]

Options (as in the reference): --type, --radius (3.5), --num-sd (3.0 for green / red / difference, else 1.5),
--out-format json|csv, --params, --include-pdbid, --atom-mask, --optimized-radii.
Extra: --pdb-file / --density-file / --diff-file analyse local files instead of downloading <pdbid>.
"""
import argparse
import json
import sys

import numpy

from . import densityAnalysis

SUBMODES = ("map", "cloud", "density", "difference", "blob", "statistics")


def buildParser():
    p = argparse.ArgumentParser(prog="pdb_eda_b200 single", description="single structure analysis mode")
    p.add_argument("pdbid")
    p.add_argument("out_file")
    p.add_argument("submode", choices=SUBMODES)
    for flag in ("density", "diff-density", "atom", "residue", "symmetry-atom", "domain", "green", "red", "blue", "include-pdbid",
                 "optimized-radii", "print-validation"):
        p.add_argument("--" + flag, action="store_true")
    p.add_argument("--type", default=None)
    p.add_argument("--radius", type=float, default=3.5)
    p.add_argument("--num-sd", type=float, default=None)
    p.add_argument("--out-format", default="json", choices=["json", "csv"])
    p.add_argument("--params", default="")
    p.add_argument("--atom-mask", default=None)
    p.add_argument("--pdb-file", default=None)
    p.add_argument("--density-file", default=None)
    p.add_argument("--diff-file", default=None)
    return p


def numpyConverter(obj):
    """numpy scalars / arrays -> plain Python (pdb_eda/singleStructure.py:180-196)."""
    if isinstance(obj, numpy.integer):
        return int(obj)
    if isinstance(obj, numpy.floating):
        return float(obj)
    if isinstance(obj, numpy.ndarray):
        return [numpyConverter(item) for item in obj]
    return obj


def _loadJson(path, what):
    try:
        with open(path, "r") as handle:
            return json.load(handle)
    except Exception:
        raise RuntimeError("Error: %s file \"%s\" does not exist or is not parsable." % (what, path))


def analyze(args):
    """Returns (headerList, rows) of the requested submode."""
    numSD = args.num_sd
    if numSD is None:
        numSD = 3.0 if (args.green or args.red or args.submode == "difference") else 1.5
    if args.params:
        densityAnalysis.setGlobals(_loadJson(args.params, "params"))
    atomMask = _loadJson(args.atom_mask, "atom mask") if args.atom_mask else None
    if args.pdb_file:
        analyzer = densityAnalysis.fromFile(args.pdb_file, args.density_file, args.diff_file)
        if analyzer:
            analyzer.pdbid = args.pdbid.lower()
    else:
        analyzer = densityAnalysis.fromPDBid(args.pdbid)
    if not analyzer:
        raise RuntimeError("Error: Unable to parse or download PDB entry or associated ccp4 file.")
    DA = densityAnalysis.DensityAnalysis
    sub = args.submode
    if sub == "map":
        dm = analyzer.densityObj if args.density or not args.diff_density else analyzer.diffDensityObj
        hdr = dm.header
        return None, {"pdbid": dm.pdbid, "ncrs": list(hdr.ncrs), "crsStart": list(hdr.crsStart), "xyzInterval": list(hdr.xyzInterval),
                      "cell": [hdr.xlength, hdr.ylength, hdr.zlength, hdr.alpha, hdr.beta, hdr.gamma], "origin": [float(v) for v in hdr.origin],
                      "meanDensity": dm.meanDensity, "stdDensity": dm.stdDensity, "density": numpy.asarray(dm.densityArray, dtype=float).tolist()}
    if sub == "cloud":
        analyzer.aggregateCloud()
        ratio = analyzer.densityElectronRatio
        if args.atom:
            header = list(map(str, list(analyzer.atomCloudDescriptions.dtype.names) + ['density_electron_ratio']))
            rows = [[numpyConverter(e) for e in item] + [ratio] for item in analyzer.atomCloudDescriptions]
        elif args.residue:
            header, rows = DA.residueCloudHeader + ['density_electron_ratio'], [list(i) + [ratio] for i in analyzer.residueCloudDescriptions]
        else:
            header, rows = DA.domainCloudHeader + ['density_electron_ratio'], [list(i) + [ratio] for i in analyzer.domainCloudDescriptions]
    elif sub in ("density", "difference"):
        symmetry = args.symmetry_atom
        if sub == "density":
            if args.atom:
                header, rows = DA.atomRegionDensityHeader, analyzer.calculateAtomRegionDensity(args.radius, numSD, args.type, args.optimized_radii)
            elif args.residue:
                header, rows = DA.residueRegionDensityHeader, analyzer.calculateResidueRegionDensity(args.radius, numSD, args.type, atomMask, args.optimized_radii)
            else:
                header, rows = DA.symmetryAtomRegionDensityHeader, analyzer.calculateSymmetryAtomRegionDensity(args.radius, numSD, args.type, args.optimized_radii)
        else:
            if args.atom:
                header, rows = DA.atomRegionDiscrepancyHeader, analyzer.calculateAtomRegionDiscrepancies(args.radius, numSD, args.type)
            elif args.residue:
                header, rows = DA.residueRegionDiscrepancyHeader, analyzer.calculateResidueRegionDiscrepancies(args.radius, numSD, args.type, atomMask)
            else:
                header, rows = DA.symmetryAtomRegionDiscrepancyHeader, analyzer.calculateSymmetryAtomRegionDiscrepancies(args.radius, numSD, args.type)
        if symmetry:
            for info in rows:
                info[5] = [val for val in info[5]]
                info[6] = [float(val) for val in info[6]]
    elif sub == "blob":
        header, rows = DA.blobStatisticsHeader, []
        diff, dens = analyzer.diffDensityObj, analyzer.densityObj
        if args.green or args.red:
            cut = diff.meanDensity + numSD * diff.stdDensity
            green, red = diff.createFullBlobLists(cut if args.green else 0.0, -cut if args.red else 0.0)   # one pass for both
            for blobs in (green, red):
                if blobs:
                    rows.extend(analyzer.calculateAtomSpecificBlobStatistics(blobs))
        else:
            rows.extend(analyzer.calculateAtomSpecificBlobStatistics(dens.createFullBlobList(dens.meanDensity + numSD * dens.stdDensity)))
        for info in rows:
            info[0] = float(info[0])
            info[9] = [val for val in info[9]]
            info[10] = [float(val) for val in info[10]]
            info[11] = [float(val) for val in info[11]]
    else:  # statistics
        if args.print_validation:
            fo, fc = analyzer.medianAbsFoFc()
            print("Median abs Fo(<1sd):", fo, "Median abs Fc(<1sd):", fc, "Relative Difference:", (fo - fc) / max(fo, fc))
        if args.residue:
            header, rows = analyzer.residueMetricsHeaderList, analyzer.residueMetrics()
        else:
            header, rows = analyzer.atomMetricsHeaderList, analyzer.atomMetrics()
        return statisticsResult(args, header, rows, analyzer.pdbid)
    if args.include_pdbid:
        header = ["pdbid"] + header
        rows = [[analyzer.pdbid] + row for row in rows]
    return header, rows


def statisticsResult(args, header, rows, pdbid):
    """(header, rows) of ``statistics`` from the rows of residueMetrics() / atomMetrics(), as written to the result file."""
    if not args.residue:
        for info in rows:
            info[4] = [x for x in info[4]]
            info[5] = [float(x) for x in info[5]]
    rows = [[numpyConverter(e) for e in row] for row in rows]
    if args.include_pdbid:
        header = ["pdbid"] + header
        rows = [[pdbid] + row for row in rows]
    return header, rows


def main(argv=None):
    args = buildParser().parse_args(argv)
    header, rows = analyze(args)
    writeResult(args, header, rows)


def writeResult(args, header, rows):
    """Writes (header, rows) to ``args.out_file`` ("-": stdout) in ``args.out_format``."""
    with open(args.out_file, "w") if args.out_file != "-" else sys.stdout as out:
        if header is None:
            out.write(json.dumps(rows))
        elif args.out_format == "csv":
            print(*[",".join(map(str, row)) for row in [header] + rows], sep="\n", file=out)
        else:
            print(json.dumps([dict(zip(header, row)) for row in rows], indent=2, sort_keys=True, default=numpyConverter), file=out)


if __name__ == "__main__":
    main()
