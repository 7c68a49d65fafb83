#!/usr/bin/env python3
"""`locator` command of the B200-native build: same flags, same output files, same function
surface as /root/reference/locator/locator.py, with the work done by the CUDA library.

    locator --vcf data.vcf.gz --sample_data samples.txt --out out/run [--bootstrap ...]

Mirrored functions (reference file:line):
  load_genotypes :187-228   sort_samples :231-247   replace_md :250-262   filter_snps :265-281
  normalize_locs :284-292   split_train_test :295-308   load_network :311-327
  load_callbacks :330-362   train_network :365-394   predict_locs :397-470
  plot_history :473-484     main :487-749 (single / --windows / --bootstrap / --jacknife drivers)

Differences that are deliberate and documented in DESIGN.md:
  * arguments are parsed in main() (the reference parses at import); the module-level ``args`` is
    set by main() or by ``set_args`` for programmatic use;
  * genotype matrices handed between the functions are 2-bit packed device matrices
    (``AlleleCounts`` / ``PackedGenotypes``; ``.to_numpy()`` gives the reference's uint8 arrays);
  * every draw the reference takes from numpy's legacy global stream is taken here with the same
    call in the same order, so split / subsample / bootstrap / jacknife indices are bit-identical
    for a given ``--seed``; weight init, batch order and dropout (unseeded TensorFlow in the
    reference) come from Philox streams keyed by ``--seed``;
  * weights files are ``.weights.npz`` (no HDF5 on this image) and only exist with --keep_weights
    (the best-epoch checkpoint lives in device memory, not on disk);
  * ``--bed PREFIX`` (extension, not written to params.json): PLINK 1 .bed input, filtered and packed on the
    device straight from its 2-bit records (locator_b200.io.BedRows, loc_bed_* kernels);
  * ``--keep_sites`` (extension, not written to params.json): next to every weights file, X.sites.tsv with the
    model's sites and location normalisation (locator_b200.sites), which python -m locator_b200.predict reads;
  * ``--gpus N`` and ``--replicates_per_gpu G`` (extensions, not written to params.json): --bootstrap
    replicates (the FULL model included), --windows replicates and the folds of a k-fold holdout run
    (locator_b200.holdout) are work items of one queue at every GPU count, spread over N GPUs of the box,
    G models trained side by side on each GPU (locator_b200.replicates); results do not depend on either.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

args = None  # set by main() / set_args(); the functions below read it like the reference does

_REFERENCE_KEYS = [
    "vcf", "zarr", "matrix", "sample_data", "train_split", "windows", "window_start", "window_stop", "window_size",
    "bootstrap", "jacknife", "jacknife_prop", "nboots", "batch_size", "max_epochs", "patience", "min_mac", "max_SNPs",
    "impute_missing", "dropout_prop", "nlayers", "width", "out", "seed", "gpu_number", "plot_history", "keep_weights",
    "load_params", "keras_verbose",
]


def build_parser():
    """The reference's argparse surface, flag for flag (locator.py:12-166), plus --gpus."""
    parser = argparse.ArgumentParser(prog="locator")
    parser.add_argument("--vcf", help="VCF with SNPs for all samples.")
    parser.add_argument("--zarr", help="zarr file of SNPs for all samples.")
    parser.add_argument("--matrix", help="tab-delimited matrix of minor allele counts with first column named 'sampleID'.")
    parser.add_argument("--sample_data", help="tab-delimited text file with columns 'sampleID \\t x \\t y'. SampleIDs must "
                        "exactly match those in the VCF. X and Y values for samples without known locations should be NA.")
    parser.add_argument("--train_split", default=0.9, type=float, help="0-1, proportion of samples to use for training. default: 0.9")
    parser.add_argument("--windows", default=False, action="store_true",
                        help="Run windowed analysis over a single chromosome (requires zarr or --bed input).")
    parser.add_argument("--window_start", default=0, help="default: 0")
    parser.add_argument("--window_stop", default=None, help="default: max snp position")
    parser.add_argument("--window_size", default=5e5, help="default: 500000")
    parser.add_argument("--bootstrap", default=False, action="store_true",
                        help="Run bootstrap replicates by retraining on bootstrapped data.")
    parser.add_argument("--jacknife", default=False, action="store_true",
                        help="Run jacknife uncertainty estimate on a trained network.")
    parser.add_argument("--jacknife_prop", default=0.05, type=float,
                        help="proportion of SNPs to remove for jacknife resampling. default: 0.05")
    parser.add_argument("--nboots", default=50, type=int, help="number of bootstrap replicates to run. default: 50")
    parser.add_argument("--batch_size", default=32, type=int,
                        help="default: 32 (locator_b200: 1..256; above 32 rows a step runs as 32-row chunks with batch statistics over the "
                        "whole step)")
    parser.add_argument("--max_epochs", default=5000, type=int, help="default: 5000")
    parser.add_argument("--patience", type=int, default=100,
                        help="n epochs to run the optimizer after last improvement in validation loss. default: 100")
    parser.add_argument("--min_mac", default=2, type=int, help="minimum minor allele count. default: 2.")
    parser.add_argument("--max_SNPs", default=None, type=int,
                        help="randomly select max_SNPs variants to use in the analysis default: None.")
    parser.add_argument("--impute_missing", default=False, action="store_true",
                        help="default: True (if False, all alleles at missing sites are ancestral)")
    parser.add_argument("--dropout_prop", default=0.25, type=float,
                        help="proportion of weights to zero at the dropout layer. default: 0.25")
    parser.add_argument("--nlayers", default=10, type=int, help="number of layers in the network. default: 10")
    parser.add_argument("--width", default=256, type=int,
                        help="number of units per layer in the network default:256 (locator_b200: a multiple of 32 in [32, 1024]; "
                        "256 runs on the tensor cores, other widths on fp32 CUDA-core kernels)")
    parser.add_argument("--out", help="file name stem for output")
    parser.add_argument("--seed", default=None, type=int, help="random seed for train/test splits and SNP subsetting.")
    parser.add_argument("--gpu_number", default=None, type=str)
    parser.add_argument("--plot_history", default=True, type=bool, help="plot training history? default: True")
    parser.add_argument("--keep_weights", default=False, action="store_true",
                        help="keep model weights after training? default: False.")
    parser.add_argument("--load_params", default=None, type=str,
                        help="Path to a _params.json file to load parameters from a previous run. Parameters from the "
                        "json file will supersede all parameters provided via command line.")
    parser.add_argument("--keras_verbose", default=1, type=int,
                        help="verbose argument passed to keras in model training. 0 = silent. default: 1.")
    # extension of this build (kept out of params.json)
    parser.add_argument("--gpus", default=1, type=int,
                        help="(locator_b200) GPUs of this box to spread --bootstrap / --windows replicates over. default: 1")
    parser.add_argument("--load_weights", default=None,
                        help="(locator_b200) predict from a weights file written by --keep_weights (.weights.npz, Keras "
                        "weight order; see python -m locator_b200.keras_weights for .weights.h5) instead of training: "
                        "with --jacknife a prediction-only sweep on the stored model; not with --bootstrap or --windows, "
                        "which train every model they predict from. default: None")
    parser.add_argument("--replicates_per_gpu", default=4, type=int,
                        help="(locator_b200) bootstrap / window models trained side by side on each GPU (1-8; neither "
                        "the indices nor the predictions depend on it; width 256 with more than 14 layers trains one "
                        "model at a time). default: 4")
    return parser


def command_parser():
    """The parser of the `locator` command: build_parser() plus the genotype input formats of this build (--bed), which
    the reference's function surface does not have."""
    parser = build_parser()
    parser.add_argument("--bed", default=None, metavar="PREFIX",
                        help="(locator_b200) PLINK 1 binary fileset PREFIX.bed / .bim / .fam (SNP-major) instead of --vcf / "
                        "--zarr / --matrix: A1 (.bim column 5) is the counted allele, the role ALT plays in a VCF; sample "
                        "IDs are the .fam IIDs, positions .bim column 4 (--windows: one chromosome). default: None")
    parser.add_argument("--keep_sites", default=False, action="store_true",
                        help="(locator_b200) with --keep_weights: next to every X.weights.npz write X.sites.tsv -- the "
                        "model's sites (CHROM POS REF ALT, one row per first-layer weight row) and the location mean / sd "
                        "-- so that python -m locator_b200.predict can locate samples of another file. default: False")
    return parser


def set_args(namespace):
    """Install the module-level ``args`` (programmatic use / tests)."""
    global args
    args = namespace
    return args


def validate_args(ns):
    """Limits of this build, checked before any data is read (the reference accepts any value and fails -- or
    not -- inside Keras).  Documented in INTEGRATION.md as deliberate deviations of the boundary."""
    from ._cabi import lib  # fails loudly here when the CUDA library is missing

    problems = []
    if getattr(ns, "bed", None) is not None:
        other = [f"--{k}" for k in ("vcf", "zarr", "matrix") if getattr(ns, k) is not None]
        if other:
            problems.append(f"--bed with {' / '.join(other)}: give one genotype input")
    if getattr(ns, "keep_sites", False):
        if not ns.keep_weights:
            problems.append("--keep_sites without --keep_weights: the sites file describes a weights file")
        if ns.matrix is not None:
            problems.append("--keep_sites with --matrix: a matrix has no site identity (CHROM / POS / REF / ALT)")
    if not 1 <= int(ns.batch_size) <= 256:
        problems.append(f"--batch_size {ns.batch_size}: must be in [1, 256] (up to 32, the reference's default, a step runs "
                        "on the fused tensor-core kernels; 33..256 rows go through the stack in 32-row chunks)")
    width, nlayers = int(ns.width), int(ns.nlayers)
    # every model needs the CUDA-core hidden stack's shared-memory layout to hold at least one weight slice
    deepest = int(lib.loc_hidden_max_nlayers(width))
    if width < 32 or width > 1024 or width % 32:
        problems.append(f"--width {ns.width}: must be a multiple of 32 in [32, 1024] (256, the default, runs on the "
                        "tensor cores; other widths on the CUDA-core kernels)")
    elif deepest == 0:
        ok = ", ".join(str(w) for w in range(32, 1025, 32) if lib.loc_hidden_max_nlayers(w) > 0)
        problems.append(f"--width {ns.width}: this build cannot hold a hidden layer of that width in shared memory at any "
                        f"--nlayers (widths that build: {ok})")
    if not 2 <= nlayers <= 64:
        problems.append(f"--nlayers {ns.nlayers}: must be in [2, 64]")
    elif 0 < deepest < nlayers:
        problems.append(f"--nlayers {ns.nlayers}: at --width {width} this build holds at most {deepest} hidden layers "
                        "(the CUDA-core hidden stack keeps one layer's weight slice in shared memory)")
    if not 0.0 <= float(ns.dropout_prop) < 1.0:
        problems.append(f"--dropout_prop {ns.dropout_prop}: must be in [0, 1)")
    if int(ns.max_epochs) < 1:
        problems.append(f"--max_epochs {ns.max_epochs}: must be >= 1")
    if int(ns.patience) < 0:
        problems.append(f"--patience {ns.patience}: must be >= 0")
    if not 1 <= int(getattr(ns, "replicates_per_gpu", 4) or 1) <= 8:
        problems.append(f"--replicates_per_gpu {ns.replicates_per_gpu}: must be in [1, 8]")
    if getattr(ns, "load_weights", None) and (ns.bootstrap or ns.windows):
        problems.append(f"--load_weights with --{'bootstrap' if ns.bootstrap else 'windows'}: replicate runs train every "
                        "model they predict from")
    if ns.windows:
        # the reference takes int(args.window_start / _stop / _size) inside its loop (locator.py:524-531): a value
        # such as "2e5" only fails there, after the genome has been read; here it fails now
        for name in ("window_start", "window_stop", "window_size"):
            v = getattr(ns, name)
            if v is None:
                continue
            try:
                iv = int(v)
            except (TypeError, ValueError):
                problems.append(f"--{name} {v!r}: not an integer (the reference calls int() on it)")
                continue
            if name == "window_size" and iv <= 0:
                problems.append(f"--window_size {v!r}: must be positive")
    if problems:
        raise SystemExit("locator: " + "\n         ".join(problems))


def _params_dict(ns):
    return {k: getattr(ns, k) for k in _REFERENCE_KEYS}


def _write_params():
    with open(args.out + "_params.json", "w") as f:
        json.dump(_params_dict(args), f, indent=2)


# ---------------------------------------------------------------------------------------------
# genotype containers handed between the mirrored functions
# ---------------------------------------------------------------------------------------------
class AlleleCounts:
    """``ac``: derived-allele counts [K sites, N samples] (reference orientation), stored packed
    sample-major on the device."""

    def __init__(self, packed, sites=None):
        self.packed = packed  # PackedGenotypes [N, K]
        self.sites = sites  # --keep_sites: site table of the K columns (locator_b200.sites)

    @property
    def shape(self):
        return (self.packed.K, self.packed.n)

    def __len__(self):
        return self.packed.K

    def to_numpy(self):
        return self.packed.to_counts().cpu().numpy().T.copy()

    def take_samples(self, idx):
        """np.transpose(ac[:, idx]) -> PackedGenotypes [len(idx), K] (locator.py:303-307)."""
        return self.packed.take_rows(np.asarray(idx, dtype=np.int64))

    def site_sums(self):
        """int64 [K]: sum over ALL samples of the allele counts (jacknife af, locator.py:714-717)."""
        return self.packed.site_sums().cpu().numpy()


def _matrix_shape(g):
    return (g.n, g.K)


# ---------------------------------------------------------------------------------------------
# ingest
# ---------------------------------------------------------------------------------------------
def load_genotypes():
    from . import io

    keep_sites = bool(getattr(args, "keep_sites", False))
    if args.zarr is not None:
        print("reading zarr")
        # calldata/GT is decoded on first use (row ranges for --windows)
        callset = io.read_zarr(args.zarr, lazy=True, sites=keep_sites)
        genotypes = io.Genotypes(callset["calldata/GT"], callset["samples"], callset["variants/POS"],
                                 io.variant_ids(callset))
        samples = callset["samples"]
    elif args.vcf is not None:
        print("reading VCF")
        vcf = io.read_vcf(args.vcf, sites=keep_sites)
        genotypes = io.Genotypes(vcf["calldata/GT"], vcf["samples"], vcf["variants/POS"], io.variant_ids(vcf))
        samples = vcf["samples"]
    elif args.matrix is not None:
        genotypes = io.read_matrix(args.matrix)
        samples = genotypes.samples
    elif getattr(args, "bed", None) is not None:
        print("reading PLINK .bed")
        try:
            # .bim / .fam parsed, .bed header and size checked; no genotype byte read
            callset = io.read_bed(args.bed, sites=keep_sites)
        except ValueError as e:
            raise SystemExit(f"locator: {e}")
        chroms = np.unique(callset["variants/CHROM"])
        if args.windows and len(chroms) > 1:
            raise SystemExit(f"locator: --windows on {args.bed}.bim, which lists {len(chroms)} chromosomes "
                             f"({', '.join(chroms[:5])}{', ...' if len(chroms) > 5 else ''}): windows are positional and "
                             "run over a single chromosome")
        genotypes = io.Genotypes(callset["calldata/GT"], callset["samples"], callset["variants/POS"],
                                 io.variant_ids(callset))
        samples = callset["samples"]
    else:
        raise SystemExit("one of --vcf, --zarr, --matrix or --bed is required")
    if keep_sites and genotypes.ids is None:
        raise SystemExit(f"locator: --keep_sites: {args.zarr} has no variants/CHROM, variants/REF and variants/ALT "
                         "arrays, so the sites of a model cannot be named")
    return genotypes, samples


def sort_samples(samples, genotypes):
    import pandas as pd

    sample_data = pd.read_csv(args.sample_data, sep="\t")
    sample_data["sampleID2"] = sample_data["sampleID"]
    sample_data.set_index("sampleID", inplace=True)
    samples = np.asarray(samples)
    samples = np.array([s.decode() if isinstance(s, bytes) else s for s in samples]).astype("str")
    sample_data = sample_data.reindex(np.array(samples))
    if not all([sample_data["sampleID2"].iloc[x] == samples[x] for x in range(len(samples))]):
        print("sample ordering failed! Check that sample IDs match the VCF.")
        sys.exit()
    locs = np.array(sample_data[["x", "y"]])
    print("loaded " + str(np.shape(genotypes)) + " genotypes\n\n")
    return sample_data, locs


def replace_md(genotypes, stats=None):
    """Impute missing calls with binomial(2, site allele frequency) -- locator.py:250-262.

    The scalar draws are taken from numpy's global stream in the reference's row-major (site, sample) order
    (by the library's restatement of numpy's sampler, nprandom.legacy_binomial); everything around them stays
    on the device: the per-site counts are the ones the site filter already produced (loc_site_stats), the
    list of missing calls comes from loc_missing_calls, the draws are patched into the packed matrix.
    ``stats`` = (device GT cube or .bed records, alt_count, n_missing, kept-site indices, packed matrix) from
    filter_snps;
    called on its own (as the reference's function can be) it imputes every site of ``genotypes``.
    """
    import torch
    from . import genotypes as G

    print("imputing missing data")
    if stats is None:
        g, na, alt, miss, keep = G.site_stats(genotypes.gt, min_mac=1)
        idx = torch.arange(g.shape[0], dtype=torch.int64, device=g.device)
        packed = G.pack_sites(g, idx)
    else:
        g, alt, miss, idx, packed = stats
    N = g.shape[1]
    dc = alt[idx].cpu().numpy().astype(np.int64)          # count_alleles()[:, 1]
    ninds = N - miss[idx].cpu().numpy().astype(np.int64)  # samples with a called genotype
    with np.errstate(divide="ignore", invalid="ignore"):
        af = dc / (2 * ninds)
    if isinstance(g, G.BedRecords):
        ks, samps = G.bed_missing_calls(g, idx, miss)  # row-major (site, sample) order
    else:
        ks, samps = G.missing_calls(g, idx, miss)
    if ks.numel():
        from .nprandom import legacy_binomial

        vals = legacy_binomial(2, af[ks.cpu().numpy()], 1)[:, 0]  # the reference's scalar draws, in its order
        packed.patch(ks, samps, vals)
    return AlleleCounts(packed)


def filter_snps(genotypes):
    from . import genotypes as G
    from . import sites
    from .io import BedRows

    print("filtering SNPs")
    on_disk = getattr(genotypes, "rows_on_disk", None)
    if isinstance(on_disk, BedRows):
        # .bed records -> pinned staging -> device as they are on disk (2 bits a call); no cube anywhere
        g = G.BedRecords.upload(on_disk)
        n_alleles, alt_count, n_missing, keep = G.bed_site_stats(g, min_mac=int(args.min_mac))
        keep_idx = G.compact_sites(keep)
        packed = G.bed_pack_sites(g, keep_idx)
    else:
        if on_disk is not None and on_disk.dtype == np.int8:
            gt = G.upload_rows(on_disk)  # zarr chunks -> pinned staging -> device; the host never holds the cube
        else:
            gt = genotypes.gt
        g, n_alleles, alt_count, n_missing, keep = G.site_stats(gt, min_mac=int(args.min_mac))
        keep_idx = G.compact_sites(keep)  # device-side prefix sum: the mask never visits the host
        packed = G.pack_sites(g, keep_idx)
    if args.impute_missing:
        ac = replace_md(genotypes, (g, alt_count, n_missing, keep_idx, packed))
    else:
        ac = AlleleCounts(packed)
    if getattr(args, "keep_sites", False):
        ac.sites = sites.table(genotypes.ids, genotypes.positions, keep_idx.cpu().numpy())
    if not args.max_SNPs == None:  # noqa: E711  (as in the reference)
        sel = np.random.choice(range(ac.shape[0]), args.max_SNPs, replace=False)
        ac = AlleleCounts(ac.packed.take_cols(sel), None if ac.sites is None else sites.take(ac.sites, sel))
    print("running on " + str(len(ac)) + " genotypes after filtering\n\n\n")
    return ac


def windows_are_data_independent():
    """True when no draw from numpy's global stream depends on the genotypes (no imputation, no SNP
    subsampling): a window's random indices can then be drawn before anybody has read its genotypes."""
    return not args.impute_missing and args.max_SNPs is None


def normalize_locs(locs):
    meanlong = np.nanmean(locs[:, 0])
    sdlong = np.nanstd(locs[:, 0])
    meanlat = np.nanmean(locs[:, 1])
    sdlat = np.nanstd(locs[:, 1])
    locs = np.array([[(x[0] - meanlong) / sdlong, (x[1] - meanlat) / sdlat] for x in locs])
    return meanlong, sdlong, meanlat, sdlat, locs


def draw_split(locs):
    """The index draws of split_train_test (locator.py:296-302) without touching the genotypes: the
    validation samples come from numpy's global stream, everything else is deterministic."""
    train = np.argwhere(~np.isnan(locs[:, 0]))
    train = np.array([x[0] for x in train])
    tr = set(train.tolist())
    pred = np.array([x for x in range(len(locs)) if x not in tr], dtype=np.int64)
    test = np.random.choice(train, round((1 - args.train_split) * len(train)), replace=False)
    te = set(test.tolist())
    train = np.array([x for x in train if x not in te])
    return train, test, pred


def split_train_test(ac, locs, drawn=None):
    train, test, pred = draw_split(locs) if drawn is None else drawn
    traingen = ac.take_samples(train)
    trainlocs = locs[train]
    testgen = ac.take_samples(test)
    testlocs = locs[test]
    predgen = ac.take_samples(pred)
    return train, test, traingen, testgen, trainlocs, testlocs, pred, predgen


# ---------------------------------------------------------------------------------------------
# model / training / prediction
# ---------------------------------------------------------------------------------------------
_seed_tag = [0]  # replicate index (0 = the single / FULL model): model seeds do not depend on scheduling


def _model_seed():
    """Weight-init / shuffle / dropout seed: derived from --seed and the replicate index when --seed
    is given (reproducible runs), fresh entropy otherwise (the reference never seeds TensorFlow)."""
    if args.seed is not None:
        return (int(args.seed) * 1000003 + _seed_tag[0]) & 0xFFFFFFFFFFFFFFFF
    return int.from_bytes(os.urandom(8), "little")


RING_MIN_SNPS = 32768


def load_network(traingen, dropout_prop):
    from .model import LocatorModel, spare_cluster_l1_ctas

    K = traingen.shape[1] if hasattr(traingen, "shape") else traingen.K
    # Replicate runs (--bootstrap / --windows) train several models per GPU side by side and keep one cluster's
    # worth of SMs free of the first-layer kernels, so that one model's hidden stack overlaps another's weight
    # stream (ring schedule of loc_group_train_epochs).  The CTA count fixes the fp32 summation order of the
    # layer, hence the same setting for EVERY model of such a run whatever --replicates_per_gpu / --gpus say:
    # the outputs of a replicate run never depend on how it was scheduled.
    # (Only where the weight stream outlasts the hidden stack: RING_MIN_SNPS mirrors kRingMinK of the library.)
    # The folds of a k-fold holdout run (locator_b200.holdout) are such replicates too.
    grouped = (args.bootstrap or args.windows or getattr(args, "folds", None)) and K >= RING_MIN_SNPS
    return LocatorModel(K, width=args.width, nlayers=args.nlayers, dropout_prop=args.dropout_prop,
                        batch_size=args.batch_size, max_epochs=args.max_epochs, seed=_model_seed(),
                        l1_ctas=spare_cluster_l1_ctas() if grouped else None)


class _Callback:
    def __init__(self, kind, **kw):
        self.kind = kind
        self.__dict__.update(kw)


def load_callbacks(boot):
    """(checkpointer, earlystop, reducelr) descriptors with the reference's settings (:330-362)."""
    if args.bootstrap or args.jacknife:
        path = args.out + "_boot" + str(boot) + ".weights.npz"
    else:
        path = args.out + ".weights.npz"
    checkpointer = _Callback("ModelCheckpoint", filepath=path, save_best_only=True, save_weights_only=True,
                             monitor="val_loss")
    earlystop = _Callback("EarlyStopping", monitor="val_loss", min_delta=0, patience=args.patience)
    reducelr = _Callback("ReduceLROnPlateau", monitor="val_loss", factor=0.5, patience=int(args.patience / 6),
                         min_delta=0, cooldown=0, min_lr=0)
    return checkpointer, earlystop, reducelr


def train_network(model, traingen, testgen, trainlocs, testlocs, callbacks, boot=0):
    start = time.time()
    checkpointer, earlystop, reducelr = callbacks
    history = model.fit(traingen, trainlocs, epochs=args.max_epochs, batch_size=args.batch_size, shuffle=True,
                        verbose=1 if args.keras_verbose == 2 else 0, validation_data=(testgen, testlocs),
                        callbacks=callbacks, patience=earlystop.patience)
    # load_weights(best checkpoint): the checkpoint lives in device memory
    model.restore_best()
    if args.keep_weights:
        model.save_weights(checkpointer.filepath)
    elapsed = time.time() - start
    print("run time " + str(elapsed / 60) + " minutes")
    return history, model


def save_sites(weights_path, site_table, norm):
    """--keep_sites: the sidecar of a weights file just written (locator_b200.sites)."""
    if args.keep_weights and getattr(args, "keep_sites", False):
        from . import sites

        sites.write(sites.sidecar_path(weights_path), site_table, args.width, args.nlayers, norm)


def predict_locs(model, predgen, sdlong, meanlong, sdlat, meanlat, testlocs, pred, samples, testgen, history, boot=0,
                 verbose=True):
    import pandas as pd
    from scipy import spatial

    if verbose == True:  # noqa: E712
        print("predicting locations...")
    prediction = model.predict(predgen)
    prediction = np.array([[x[0] * sdlong + meanlong, x[1] * sdlat + meanlat] for x in prediction])
    predout = pd.DataFrame(prediction.reshape(-1, 2))
    predout.columns = ["x", "y"]
    samples = np.array([s.decode() if isinstance(s, bytes) else s for s in np.asarray(samples)])
    predout["sampleID"] = samples[pred]
    if args.bootstrap or args.jacknife:
        outfile = args.out + "_boot" + str(boot) + "_predlocs.txt"
    elif args.windows:
        window_start = int(args.window_start)
        window_size = int(args.window_size)
        outfile = f"{args.out}_{window_start}-{window_start + window_size - 1}_predlocs.txt"
    else:
        outfile = args.out + "_predlocs.txt"
    predout.to_csv(outfile, index=False)

    testlocs2 = np.array([[x[0] * sdlong + meanlong, x[1] * sdlat + meanlat] for x in testlocs])
    p2 = model.predict(testgen)
    p2 = np.array([[x[0] * sdlong + meanlong, x[1] * sdlat + meanlat] for x in p2])
    r2_long = np.corrcoef(p2[:, 0], testlocs2[:, 0])[0][1] ** 2
    r2_lat = np.corrcoef(p2[:, 1], testlocs2[:, 1])[0][1] ** 2
    dists = [spatial.distance.euclidean(p2[x, :], testlocs2[x, :]) for x in range(len(p2))]
    mean_dist = np.mean(dists)
    median_dist = np.median(dists)
    if verbose == True:  # noqa: E712
        print("R2(x)=" + str(r2_long) + "\nR2(y)=" + str(r2_lat) + "\n" + "mean validation error " + str(mean_dist)
              + "\n" + "median validation error " + str(median_dist) + "\n")
    hist = pd.DataFrame(history.history)
    hist.to_csv(args.out + "_history.txt", sep="\t", index=False)
    return dists


def plot_history(history, dists):
    if args.plot_history:
        try:
            import matplotlib

            matplotlib.use("agg")
            from matplotlib import pyplot as plt
        except ImportError:
            return  # matplotlib is not part of this image; the fit plot is cosmetic
        fig = plt.figure(figsize=(4, 1.5), dpi=200)
        plt.rcParams.update({"font.size": 7})
        ax1 = fig.add_axes([0, 0, 0.4, 1])
        ax1.plot(history.history["val_loss"][3:], "-", color="black", lw=0.5)
        ax1.set_xlabel("Validation Loss")
        ax2 = fig.add_axes([0.55, 0, 0.4, 1])
        ax2.plot(history.history["loss"][3:], "-", color="black", lw=0.5)
        ax2.set_xlabel("Training Loss")
        fig.savefig(args.out + "_fitplot.pdf", bbox_inches="tight")


# ---------------------------------------------------------------------------------------------
# drivers
# ---------------------------------------------------------------------------------------------
def _run_one(traingen, testgen, trainlocs, testlocs, predgen, norm, pred, samples, boot, cb_boot, sites=None):
    meanlong, sdlong, meanlat, sdlat = norm
    model = load_network(traingen, args.dropout_prop)
    callbacks = load_callbacks(cb_boot)
    if getattr(args, "load_weights", None):
        # prediction from stored weights (the reference only ever reloads the checkpoint of the run itself,
        # locator.py:380,386): no training, an empty history
        from .model import History

        model.load_weights(args.load_weights)
        print("loaded weights from " + str(args.load_weights))
        history = History()
    else:
        history, model = train_network(model, traingen, testgen, trainlocs, testlocs, callbacks, boot)
        save_sites(callbacks[0].filepath, sites, norm)
    dists = predict_locs(model, predgen, sdlong, meanlong, sdlat, meanlat, testlocs, pred, samples, testgen, history,
                         boot)
    if args.plot_history and history.history["loss"]:
        plot_history(history, dists)
    return model, history, dists


def _jacknife_draws(af, K, n_pred):
    """(sites_to_remove, vals uint8 [nsites, n_pred]) per replicate, from numpy's global stream in the
    reference's order (locator.py:722-727): choice without replacement, then per chosen site, in the
    returned order, binomial(2, af[site], n_pred).  The binomials are taken by the library's restatement of
    numpy's generator (nprandom.legacy_binomial: same stream, a few ns per draw instead of ~50, GIL
    released), and the draws of replicate r+1 run in a helper thread while replicate r is predicted and
    written.  Nothing else touches the stream during the sweep."""
    import queue
    import threading

    from .nprandom import legacy_binomial, legacy_choice_without_replacement

    nsites = int(K * args.jacknife_prop)
    q = queue.Queue(maxsize=2)

    def produce():
        try:
            for _ in range(args.nboots):
                sites = legacy_choice_without_replacement(K, nsites)
                vals = legacy_binomial(2, af[sites], n_pred)
                q.put((sites, vals))
            q.put(None)
        except BaseException as e:  # surfaces in the consumer
            q.put(e)

    t = threading.Thread(target=produce, daemon=True)
    t.start()
    while True:
        item = q.get()
        if item is None:
            break
        if isinstance(item, BaseException):
            raise item
        yield item
    t.join()


def start_run(ns, extensions=("gpus", "replicates_per_gpu", "load_weights", "bed", "keep_sites")):
    """Install ``ns`` as ``args`` and set the run up as the reference does: seed and gpu (locator.py:170-173),
    load stored parameters (:177-184), seed again in main() (:491-494) -- with --load_params it is the stored
    seed that decides the run's draws.  ``extensions``: flags of this build, kept from the command line (a
    params file does not hold them)."""
    set_args(ns)
    if args.seed is not None:
        np.random.seed(args.seed)
    if args.gpu_number is not None:
        os.environ["CUDA_VISIBLE_DEVICES"] = args.gpu_number
    if args.load_params is not None:
        kept = {k: getattr(args, k) for k in extensions if hasattr(args, k)}
        with open(args.load_params, "r") as f:
            args.__dict__ = json.load(f)
        args.__dict__.update(kept)
    if args.seed is not None:
        np.random.seed(args.seed)
    if args.gpu_number is not None:
        os.environ["CUDA_VISIBLE_DEVICES"] = args.gpu_number
    if args.out is None:
        raise SystemExit("--out is required")
    return args


def main(argv=None):
    parser = command_parser()
    start_run(parser.parse_args(argv))
    validate_args(args)
    _write_params()
    from . import replicates

    replicates.start_pool_early(args)  # several GPUs: the workers boot while this process reads and draws
    try:
        return _main_body()
    finally:
        replicates.abort_early_pool()  # only still there if the run failed before handing it over


def _main_body():
    genotypes, samples = load_genotypes()
    sample_data, locs = sort_samples(samples, genotypes)
    meanlong, sdlong, meanlat, sdlat, locs = normalize_locs(locs)
    norm = (meanlong, sdlong, meanlat, sdlat)
    if args.windows and (args.zarr is not None or getattr(args, "bed", None) is not None) and windows_are_data_independent():
        # The reference filters and splits the whole genome before its window loop (main :500-517) and then
        # never uses the result; only the split's draws matter for what follows.  Take the draws, leave the
        # genome on disk: every window decodes just its own chunks (possibly inside a worker process).
        print("filtering SNPs\n(windows run: the genome-wide matrix is not materialised; every window is filtered on its own)")
        draw_split(locs)
        ac = traingen = testgen = predgen = None
    else:
        ac = filter_snps(genotypes)
        train, test, traingen, testgen, trainlocs, testlocs, pred, predgen = split_train_test(ac, locs)

    if args.windows:
        from . import replicates

        if args.zarr is None and getattr(args, "bed", None) is None:
            raise SystemExit("--windows requires --zarr or --bed input")
        replicates.run_windows(sys.modules[__name__], genotypes, samples)
    elif not args.bootstrap and not args.jacknife:
        _run_one(traingen, testgen, trainlocs, testlocs, predgen, norm, pred, samples, 0, None, ac.sites)
    elif args.bootstrap:
        from . import replicates

        replicates.run_bootstrap(sys.modules[__name__], traingen, testgen, trainlocs, testlocs, predgen, norm, pred,
                                 samples, ac.sites)
    elif args.jacknife:
        boot = "FULL"
        start = time.time()
        model, history, dists = _run_one(traingen, testgen, trainlocs, testlocs, predgen, norm, pred, samples, boot,
                                         boot, ac.sites)
        print("run time " + str((time.time() - start) / 60) + " minutes")
        print("starting jacknife resampling")
        af = ac.site_sums() / (ac.shape[1] * 2)  # wide integer sums (numpy >= 2 would wrap uint8 in the reference)
        n_pred = _matrix_shape(predgen)[0]
        for boot, (sites_to_remove, vals) in enumerate(_jacknife_draws(af, _matrix_shape(predgen)[1], n_pred)):
            pg = predgen.clone()
            if len(sites_to_remove):
                pg.replace_cols(sites_to_remove, vals)
            predict_locs(model, pg, sdlong, meanlong, sdlat, meanlat, testlocs, pred, samples, testgen, history, boot,
                         verbose=False)
    return 0


if __name__ == "__main__":
    sys.exit(main())
