"""compare_models command line: model 1 (Hill fixed) against model 2 (Hill free) by PSIS-LOO, from the `_loo.txt` files
PyHillFit --loo writes beside the temperature-1 chain files.  Host only, mirroring assemble_BFs: for every pair of the data
file that has both models' files it writes one line to LOO/loo_compare.txt,
    drug channel n elpd1 se1 elpd2 se2 diff se_diff max_khat1 max_khat2
(diff = elpd1 - elpd2 with the paired standard error of loo.compare), and prints how many pairs prefer each model by
more than 2 se_diff.  A file written with --loo-refit has two more columns, elpd_refit_i se_refit_i: a point uses its
exact refit value where that is finite and its PSIS value otherwise.  When any file has them, each line (and the header)
ends with n_refit1 n_refit2, the points of each model that used a refit (kind-3 points, whose exact value is a
constant, are not counted).

    python -m pyhillfit_b200.compare_models --data-file data/crumb_data.csv
"""
import argparse
import itertools as it
import os
import sys

import numpy as np

HEADER = "# drug channel n elpd1 se1 elpd2 se2 diff se_diff max_khat1 max_khat2\n"
HEADER_REFIT = "# drug channel n elpd1 se1 elpd2 se2 diff se_diff max_khat1 max_khat2 n_refit1 n_refit2\n"


def read_loo(f):
    """[N, 7] rows of a _loo.txt file: index dose response elpd_loo_i lppd_i p_waic_i khat_i; [N, 9] with
    elpd_refit_i se_refit_i."""
    return np.loadtxt(f, ndmin=2)


def elpd_points(rows):
    """(pointwise elpd, points that used a refit) of one file's rows: elpd_refit_i where it is finite, elpd_loo_i
    otherwise.  A point of kind 3 (response in no mask) carries its exact constant, not a refit, and is not counted."""
    from .packing import masks, point_kinds
    if rows.shape[1] < 9:
        return rows[:, 3], 0
    done = np.isfinite(rows[:, 7])
    return np.where(done, rows[:, 7], rows[:, 3]), int(np.count_nonzero(done & (point_kinds(*masks(rows[:, 2])) != 3)))


def compare_rows(rows1, rows2):
    """(n, elpd1, se1, elpd2, se2, diff, se_diff, max_khat1, max_khat2, n_refit1, n_refit2) of one pair from the two
    models' file rows."""
    from . import loo
    if len(rows1) != len(rows2) or not np.array_equal(rows1[:, :3], rows2[:, :3]):
        raise ValueError("the two models' files do not list the same points")
    (e1, n1), (e2, n2) = elpd_points(rows1), elpd_points(rows2)
    n = len(e1)
    diff, se_diff = loo.compare(e1, e2)
    return (n, e1.sum(), np.sqrt(n * np.var(e1)), e2.sum(), np.sqrt(n * np.var(e2)), diff, se_diff,
            rows1[:, 6].max(), rows2[:, 6].max(), n1, n2)


def build_parser():
    parser = argparse.ArgumentParser()
    requiredNamed = parser.add_argument_group('required arguments')
    requiredNamed.add_argument("--data-file", type=str, required=True,
                               help="csv file from which to read in data, in same format as provided crumb_data.csv")
    return parser


def main(argv=None):
    parser = build_parser()
    argv = sys.argv[1:] if argv is None else argv
    if len(argv) == 0:
        parser.print_help()
        return 1
    args = parser.parse_args(argv)
    from . import chainio
    from . import doseresponse as dr
    dr.setup(args.data_file)
    results, prefer = [], [0, 0, 0]   # model 1, model 2, neither (|diff| <= 2 se_diff)
    refit_columns = False
    for top_drug, top_channel in it.product(dr.drugs, dr.channels):
        files = []
        for m in (1, 2):
            drug, channel, chain_file, _ = dr.nonhierarchical_chain_file_and_figs_dir(m, top_drug, top_channel, 1)
            files.append(chainio.loo_name(chain_file))
        if not all(os.path.exists(f) for f in files):
            continue
        rows1, rows2 = read_loo(files[0]), read_loo(files[1])
        refit_columns |= rows1.shape[1] >= 9 or rows2.shape[1] >= 9
        r = compare_rows(rows1, rows2)
        results.append((drug, channel, r))
        diff, se_diff = r[5], r[6]
        prefer[0 if diff > 2 * se_diff else (1 if -diff > 2 * se_diff else 2)] += 1
    lines = []
    for drug, channel, r in results:
        tail = " {:d} {:d}".format(r[9], r[10]) if refit_columns else ""
        lines.append("{} {} {:d} ".format(drug, channel, r[0]) + " ".join("{:.18e}".format(v) for v in r[1:9]) + tail
                     + "\n")
    if not os.path.exists("LOO"):
        os.makedirs("LOO")
    with open("LOO/loo_compare.txt", "w") as out:
        out.write(HEADER_REFIT if refit_columns else HEADER)
        out.writelines(lines)
    summary = "{} pairs: model 1 preferred by more than 2 se_diff in {}, model 2 in {}, neither in {}".format(
        len(lines), *prefer)
    if refit_columns:
        summary += "; exact refits used at {} points of model 1 and {} of model 2".format(
            sum(r[9] for _, _, r in results), sum(r[10] for _, _, r in results))
    print(summary)
    return 0


if __name__ == "__main__":
    sys.exit(main())
