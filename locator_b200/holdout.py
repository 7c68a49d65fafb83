"""K-fold holdout predictions for every sample of known location.

    python -m locator_b200.holdout --vcf data.vcf.gz --sample_data samples.txt --out out/run [--folds 10]

The located samples are split into k folds; for each fold a model is trained on the other folds (with an inner
validation split drawn as the reference's split_train_test draws it) and predicts the held-out fold.  Every located
sample thus gets a prediction from a model that never saw it, and the error of each sample can be read off.
The folds are independent models on one SNP matrix: they run as work items of the replicate queue
(locator_b200.replicates), side by side on each GPU (``--replicates_per_gpu``) and over ``--gpus``; their
training sets differ by up to one sample when k does not divide the number of located samples.

Takes every ``locator`` flag plus ``--folds``; refuses --windows, --bootstrap, --jacknife and --load_weights.
Every numpy draw is taken serially in this process, so the outputs do not depend on --gpus or
--replicates_per_gpu.  Outputs:
  {out}_holdout_predlocs.txt     x,y,sampleID,fold -- one row per located sample, ascending sample index
  {out}_holdout{f}_history.txt   per fold
  {out}_holdout{f}.weights.npz   per fold, with --keep_weights
  {out}_holdout{f}.sites.tsv     per fold, with --keep_weights --keep_sites (python -m locator_b200.predict)
  {out}_params.json              as a plain locator run writes it
"""
from __future__ import annotations

import sys

import numpy as np

from . import locator as L
from . import replicates


def build_parser():
    parser = L.command_parser()
    parser.prog = "python -m locator_b200.holdout"
    parser.add_argument("--folds", default=10, type=int,
                        help="number of folds k: every located sample is predicted by the model trained on the other "
                        "k - 1 folds. default: 10")
    return parser


def check_args(ns):
    """The flags this command cannot honour, refused before any data is read."""
    problems = [f"--{name}: not available with k-fold holdout" for name in ("windows", "bootstrap", "jacknife")
                if getattr(ns, name)]
    if ns.load_weights:
        problems.append("--load_weights: k-fold holdout trains its own models")
    if int(ns.folds) < 2:
        problems.append(f"--folds {ns.folds}: must be >= 2")
    if problems:
        raise SystemExit("holdout: " + "\n         ".join(problems))


def draw_folds(locs, k, train_split):
    """Fold partition and inner splits, from numpy's global stream: a permutation of the located samples split
    into k folds (np.array_split), then for f = 0..k-1 the inner validation set of fold f drawn from its training
    candidates (located samples outside fold f, ascending) by the rule of split_train_test (locator.py:296-302).
    Returns [(held, train, val)] index arrays per fold."""
    known = np.array([x[0] for x in np.argwhere(~np.isnan(locs[:, 0]))], dtype=np.int64)
    if k > len(known):
        raise SystemExit(f"holdout: --folds {k}: more folds than the {len(known)} samples of known location")
    perm = np.random.choice(known, len(known), replace=False)
    folds = np.array_split(perm, k)
    out = []
    for f, held in enumerate(folds):
        out_f = set(held.tolist())
        cands = np.array([x for x in known if x not in out_f], dtype=np.int64)
        val = np.random.choice(cands, round((1 - train_split) * len(cands)), replace=False)
        vs = set(val.tolist())
        train = np.array([x for x in cands if x not in vs], dtype=np.int64)
        if len(train) == 0:
            raise SystemExit(f"holdout: fold {f} leaves no training sample (--train_split {train_split})")
        out.append((np.sort(held), train, val))
    return out


def predict_fold(model, history, rep):
    """Called for each trained fold model (replicates._run_items): writes the fold's history and returns
    (fold, held-out sample indices, predictions de-normalised as in predict_locs)."""
    import pandas as pd

    meanlong, sdlong, meanlat, sdlat = rep["norm"]
    p = model.predict(rep["predgen"])
    xy = np.array([[x[0] * sdlong + meanlong, x[1] * sdlat + meanlat] for x in p])
    pd.DataFrame(history.history).to_csv(rep["out"] + "_history.txt", sep="\t", index=False)
    return rep["fold"], np.asarray(rep["pred"]), xy


def run(ac, locs, norm, samples, folds):
    """Train and predict every fold through the replicate queue; returns the fold results in fold order."""
    args = L.args
    base = {"genotypes": ac.packed, "locs": locs, "norm": norm, "samples": samples, "sites": ac.sites}
    items = [{"kind": "fold", "fold": f, "held": held, "train": train, "val": val, "fold_out": f"{args.out}_holdout{f}"}
             for f, (held, train, val) in enumerate(folds)]
    return replicates.run_work(L, items, base)


def write_predictions(results, locs, norm, samples):
    """{out}_holdout_predlocs.txt and the summary over all located samples (R2 and errors in the reference's
    print format, predict_locs :440-447)."""
    import pandas as pd
    from scipy import spatial

    meanlong, sdlong, meanlat, sdlat = norm
    pred = np.full((len(locs), 2), np.nan)
    fold = np.full(len(locs), -1, dtype=np.int64)
    for f, held, xy in results:
        pred[held] = xy
        fold[held] = f
    known = np.array([x[0] for x in np.argwhere(~np.isnan(locs[:, 0]))], dtype=np.int64)
    assert (fold[known] >= 0).all() and len(known) == sum(len(r[1]) for r in results)
    samples = np.array([s.decode() if isinstance(s, bytes) else s for s in np.asarray(samples)])
    out = pd.DataFrame(pred[known], columns=["x", "y"])
    out["sampleID"] = samples[known]
    out["fold"] = fold[known]
    out.to_csv(L.args.out + "_holdout_predlocs.txt", index=False)

    true = np.array([[x[0] * sdlong + meanlong, x[1] * sdlat + meanlat] for x in locs[known]])
    p = pred[known]
    r2_long = np.corrcoef(p[:, 0], true[:, 0])[0][1] ** 2
    r2_lat = np.corrcoef(p[:, 1], true[:, 1])[0][1] ** 2
    dists = [spatial.distance.euclidean(p[x, :], true[x, :]) for x in range(len(p))]
    print("R2(x)=" + str(r2_long) + "\nR2(y)=" + str(r2_lat) + "\n" + "mean holdout error " + str(np.mean(dists))
          + "\n" + "median holdout error " + str(np.median(dists)) + "\n")


def main(argv=None):
    ns = build_parser().parse_args(argv)
    check_args(ns)
    args = L.start_run(ns, extensions=("gpus", "replicates_per_gpu", "load_weights", "folds", "bed", "keep_sites"))
    check_args(args)  # a --load_params file may ask for one of them
    L.validate_args(args)
    L._write_params()
    replicates.start_pool_early(args)  # several GPUs: the workers boot while this process reads and draws
    try:
        genotypes, samples = L.load_genotypes()
        sample_data, locs = L.sort_samples(samples, genotypes)
        meanlong, sdlong, meanlat, sdlat, locs = L.normalize_locs(locs)
        norm = (meanlong, sdlong, meanlat, sdlat)
        ac = L.filter_snps(genotypes)
        folds = draw_folds(locs, int(args.folds), float(args.train_split))
        results = run(ac, locs, norm, samples, folds)
    finally:
        replicates.abort_early_pool()  # only still there if the run failed before handing it over
    write_predictions(results, locs, norm, samples)
    return 0


if __name__ == "__main__":
    sys.exit(main())
