"""python -m locator_b200.holdout: k-fold holdout predictions for every sample of known location.

On the reference's fixture (450 of 500 samples located): the fold partition and the inner validation splits equal a
numpy restatement of the rule, every located sample is predicted exactly once, the outputs do not depend on
--replicates_per_gpu or --gpus, and a fold's predictions equal those of the same model trained alone on the fold's
matrices.  With --folds 8 the training sets differ in size (ragged replicate groups).
"""
import glob
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
VCF = os.path.join(HERE, "golden", "data", "test_genotypes.vcf.gz")
SAMPLES = os.path.join(HERE, "golden", "data", "test_sample_data.txt")
SEED, FOLDS, EPOCHS = 12345, 8, 3


def _argv(out, *extra):
    return ["--vcf", VCF, "--sample_data", SAMPLES, "--out", str(out), "--seed", str(SEED), "--max_epochs", str(EPOCHS),
            "--keras_verbose", "0", "--folds", str(FOLDS), *extra]


@pytest.mark.parametrize("extra,match", [
    (["--windows"], "--windows"),
    (["--bootstrap"], "--bootstrap"),
    (["--jacknife"], "--jacknife"),
    (["--load_weights", "w.weights.npz"], "--load_weights"),
    (["--folds", "1"], "--folds 1"),
], ids=["windows", "bootstrap", "jacknife", "load_weights", "one-fold"])
def test_refused_flags(tmp_path, extra, match):
    """Refused before any data is read (CPU only: the input files are never opened)."""
    from locator_b200 import holdout

    argv = ["--vcf", str(tmp_path / "missing.vcf.gz"), "--sample_data", str(tmp_path / "missing.txt"),
            "--out", str(tmp_path / "r")] + extra
    with pytest.raises(SystemExit, match=match):
        holdout.main(argv)
    assert not os.listdir(tmp_path)


def test_folds_restated():
    """draw_folds against the rule written out with numpy (CPU only)."""
    from locator_b200 import holdout

    locs = np.random.default_rng(0).normal(size=(60, 2))
    locs[::7] = np.nan
    np.random.seed(3)
    got = holdout.draw_folds(locs, 4, 0.8)
    np.random.seed(3)
    known = np.flatnonzero(~np.isnan(locs[:, 0]))
    perm = np.random.choice(known, len(known), replace=False)
    parts = np.array_split(perm, 4)
    for f, (held, train, val) in enumerate(got):
        assert np.array_equal(held, np.sort(parts[f]))
        cands = np.setdiff1d(known, parts[f])
        want_val = np.random.choice(cands, round(0.2 * len(cands)), replace=False)
        assert np.array_equal(val, want_val)
        assert np.array_equal(train, np.setdiff1d(cands, want_val))
    with pytest.raises(SystemExit, match="more folds"):
        holdout.draw_folds(locs, len(known) + 1, 0.8)


@pytest.fixture(scope="module")
def cuda():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _run(tmp_path, tag, *extra):
    from locator_b200 import holdout

    d = tmp_path / tag
    d.mkdir()
    assert holdout.main(_argv(d / "r", *extra)) == 0
    return d, {os.path.basename(f): open(f, "rb").read() for f in sorted(glob.glob(str(d / "*")))}


def _ingest(tmp_path):
    """The run's located samples, normalised targets, filtered matrix and folds, as the command draws them."""
    from locator_b200 import holdout
    from locator_b200 import locator as L

    args = L.start_run(holdout.build_parser().parse_args(_argv(tmp_path / "ingest")),
                       extensions=("gpus", "replicates_per_gpu", "load_weights", "folds"))
    genotypes, samples = L.load_genotypes()
    _, locs = L.sort_samples(samples, genotypes)
    meanlong, sdlong, meanlat, sdlat, locs = L.normalize_locs(locs)
    ac = L.filter_snps(genotypes)
    return args, locs, (meanlong, sdlong, meanlat, sdlat), ac, holdout.draw_folds(locs, FOLDS, args.train_split)


@pytest.mark.gpu
def test_holdout_outputs(cuda, tmp_path, capsys):
    import pandas as pd

    from locator_b200.model import LocatorModel, spare_cluster_l1_ctas
    from locator_b200 import locator as L

    d1, f1 = _run(tmp_path, "g1", "--replicates_per_gpu", "1", "--keep_weights")
    d4, f4 = _run(tmp_path, "g4", "--replicates_per_gpu", "4", "--keep_weights")
    text = capsys.readouterr().out
    assert "replicates side by side" in text and "mean holdout error" in text and "R2(x)=" in text
    want = (["r_holdout_predlocs.txt", "r_params.json"] + [f"r_holdout{f}_history.txt" for f in range(FOLDS)]
            + [f"r_holdout{f}.weights.npz" for f in range(FOLDS)])
    assert sorted(f1) == sorted(want)
    for name in want:
        if name.endswith(".npz"):  # the arrays (a zip member carries its write time)
            a, b = np.load(d1 / name), np.load(d4 / name)
            assert a.files == b.files and all(np.array_equal(a[k], b[k]) for k in a.files), name
        elif name != "r_params.json":  # holds --out
            assert f1[name] == f4[name], name

    out = pd.read_csv(d1 / "r_holdout_predlocs.txt", float_precision="round_trip")
    assert list(out.columns) == ["x", "y", "sampleID", "fold"]
    args, locs, (meanlong, sdlong, meanlat, sdlat), ac, folds = _ingest(tmp_path)
    known = np.flatnonzero(~np.isnan(locs[:, 0]))
    assert len(known) == 450 and len(out) == len(known)
    samples = pd.read_csv(SAMPLES, sep="\t")
    assert out["sampleID"].is_unique and set(out["sampleID"]) == set(samples["sampleID"][samples["x"].notna()])

    # fold partition and inner splits: numpy's global stream after the plain run's draws (none before the split
    # with the fixture's flags), restated
    np.random.seed(SEED)
    perm = np.random.choice(known, len(known), replace=False)
    parts = np.array_split(perm, FOLDS)
    sizes = set()
    for f, (held, train, val) in enumerate(folds):
        assert np.array_equal(held, np.sort(parts[f]))
        cands = np.setdiff1d(known, parts[f])
        want_val = np.random.choice(cands, round((1 - args.train_split) * len(cands)), replace=False)
        assert np.array_equal(val, want_val) and np.array_equal(train, np.setdiff1d(cands, want_val))
        assert np.array_equal(out["fold"].to_numpy()[np.searchsorted(known, held)], np.full(len(held), f))
        sizes.add(len(train))
    assert sizes == {354, 355}  # folds of 57 and 56 samples: ragged training sets

    # folds 0 and 7 (different training-set sizes): the same model trained alone on the fold's matrices
    g = ac.packed
    for f in (0, FOLDS - 1):
        held, train, val = folds[f]
        K = g.K
        m = LocatorModel(K, width=args.width, nlayers=args.nlayers, dropout_prop=args.dropout_prop,
                         batch_size=args.batch_size, max_epochs=EPOCHS, seed=(SEED * 1000003 + f + 1) & (2**64 - 1),
                         l1_ctas=spare_cluster_l1_ctas() if K >= L.RING_MIN_SNPS else None)
        m.fit(g.take_rows(train), locs[train], epochs=EPOCHS, batch_size=args.batch_size,
              validation_data=(g.take_rows(val), locs[val]), patience=args.patience)
        m.restore_best()
        p = m.predict(g.take_rows(held))
        xy = np.array([[x[0] * sdlong + meanlong, x[1] * sdlat + meanlat] for x in p])
        rows = out.iloc[np.searchsorted(known, held)]
        assert np.array_equal(rows[["x", "y"]].to_numpy(), xy), f


@pytest.mark.gpu
def test_holdout_two_gpus(cuda, tmp_path):
    if cuda.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _, f1 = _run(tmp_path, "g1", "--replicates_per_gpu", "4")
    _, f2 = _run(tmp_path, "n2", "--replicates_per_gpu", "4", "--gpus", "2")
    f1.pop("r_params.json"), f2.pop("r_params.json")  # holds --out
    assert f1 == f2
