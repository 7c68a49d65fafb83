"""Locate the samples of a new genotype file with stored models.

    python -m locator_b200.predict --weights A.weights.npz [B.weights.npz ...] (--vcf F | --zarr D | --bed PREFIX)
                                   --out STEM

Every model needs the sites file a run writes with ``--keep_weights --keep_sites`` (A.sites.tsv next to
A.weights.npz: the model's sites in W1 order and the location normalisation, locator_b200.sites).  The query is read
and uploaded once; per model its records are joined to the model's sites on the host (sites.join: equal CHROM and
POS, {REF, ALT} equal as a set, swapped alleles flipped), then packed in the model's site order on the GPU
(loc_pack_sites_mapped / loc_bed_pack_sites_mapped).  A missing call, a call with an allele index >= 2 and every call
of a site the query lacks are entered as code 3, which the first layer reads as x = the model's moving mean (xhat =
beta: mean imputation in BatchNorm's space).  Every query sample is predicted; no sample data is needed.

Output per model: {out}_{A}_predlocs.txt (x,y,sampleID; A = the weights file name without .weights.npz), so that the
folder can be summarised with python -m locator_b200.summarize.
"""
from __future__ import annotations

import argparse
import os
import sys
import zipfile

import numpy as np

from . import sites


def build_parser():
    parser = argparse.ArgumentParser(prog="python -m locator_b200.predict")
    parser.add_argument("--weights", nargs="+", required=True,
                        help="weights files written with --keep_weights --keep_sites (X.weights.npz; X.sites.tsv must "
                        "be next to each)")
    parser.add_argument("--vcf", help="query VCF (.vcf / .vcf.gz)")
    parser.add_argument("--zarr", help="query zarr store with variants/CHROM, variants/REF and variants/ALT")
    parser.add_argument("--bed", metavar="PREFIX", help="query PLINK 1 fileset PREFIX.bed / .bim / .fam (SNP-major; "
                        "REF = A2, ALT = A1)")
    parser.add_argument("--out", required=True, help="file name stem for output")
    return parser


def _npz_shapes(path):
    """{array name: shape} of an .npz, from the array headers only."""
    out = {}
    with zipfile.ZipFile(path) as z:
        for name in z.namelist():
            with z.open(name) as fh:
                version = np.lib.format.read_magic(fh)
                shape = (np.lib.format.read_array_header_1_0(fh) if version == (1, 0)
                         else np.lib.format.read_array_header_2_0(fh))[0]
            out[name[:-4] if name.endswith(".npy") else name] = shape
    return out


def model_name(weights_path):
    base = os.path.basename(weights_path)
    return base[: -len(".weights.npz")] if base.endswith(".weights.npz") else os.path.splitext(base)[0]


def check_models(paths):
    """[(weights path, site table, {"width", "nlayers"}, norm)] -- refuses a weights file without its sites file, or
    whose sites file disagrees with it, before any genotype is read."""
    models, problems = [], []
    for p in paths:
        sp = sites.sidecar_path(p)
        if not os.path.exists(p):
            problems.append(f"{p}: no such weights file")
            continue
        if not os.path.exists(sp):
            problems.append(f"{p}: no sites file {sp} (train with --keep_weights --keep_sites)")
            continue
        try:
            table, shape, norm = sites.read(sp)
            ws = _npz_shapes(p)
        except (ValueError, OSError, zipfile.BadZipFile) as e:
            problems.append(f"{p}: {e}")
            continue
        names = sorted(ws)
        K, width, nlayers = len(table["pos"]), shape["width"], shape["nlayers"]
        if len(names) != 4 + 2 * (nlayers + 2) or len(names) < 6:
            problems.append(f"{p}: {len(names)} weight arrays, but {sp} says nlayers {nlayers} "
                            f"({4 + 2 * (nlayers + 2)} arrays)")
        elif ws[names[4]] != (K, width):
            problems.append(f"{p}: first-layer weights of shape {ws[names[4]]}, but {sp} lists {K} sites at width {width}")
        else:
            models.append((p, table, shape, norm))
    if problems:
        raise SystemExit("predict: " + "\n         ".join(problems))
    return models


def read_query(ns):
    """(callset of the query file, site table of its records, sample IDs); no genotype is decoded yet for a zarr
    store or a .bed file."""
    from . import io

    if ns.bed is not None:
        cs = io.read_bed(ns.bed, sites=True)
    elif ns.zarr is not None:
        cs = io.read_zarr(ns.zarr, lazy=True, sites=True)
    else:
        cs = io.read_vcf(ns.vcf, sites=True)
    ids = io.variant_ids(cs)
    if ids is None:
        raise SystemExit(f"predict: {ns.zarr} has no variants/CHROM, variants/REF and variants/ALT arrays: its records "
                         "cannot be matched to a model's sites")
    query = sites.table(ids, cs["variants/POS"], np.arange(len(cs["variants/POS"])))
    samples = np.array([s.decode() if isinstance(s, bytes) else s for s in np.asarray(cs["samples"])]).astype(str)
    return cs, query, samples


def upload_query(cs):
    """The query's genotypes on the device, once for all models: .bed records as they are on disk
    (genotypes.BedRecords), else the GT int8 cube (zarr chunks decoded into pinned staging on the way)."""
    import torch

    from . import genotypes as G
    from . import io

    gt = cs["calldata/GT"]
    if isinstance(gt, io.BedRows):
        return G.BedRecords.upload(gt)
    if isinstance(gt, io.ZarrRows):
        return G.upload_rows(gt)
    return torch.as_tensor(gt).to(G._dev())


def code3_fraction(packed):
    """Share of code-3 entries (missing or absent) among the n x K entries of a packed matrix (pad bits are 0)."""
    w = packed.words
    m = w & (w >> 1) & 0x55555555  # bit 2j set where field j holds 3 (bit 31 of the shift is masked off)
    n3 = sum(int(((m >> (2 * j)) & 1).sum()) for j in range(16))
    return n3 / max(1, packed.n * packed.K)


def predict_model(dev, src, flip, weights_path, shape, norm):
    """Mapped pack of the query + one model's prediction, de-normalised as predict_locs does (locator.py:470).
    Returns (xy float64 [N, 2], packed matrix)."""
    from . import genotypes as G
    from .model import LocatorModel

    packed = G.pack_sites_mapped(dev, src, flip)
    model = LocatorModel(len(src), width=shape["width"], nlayers=shape["nlayers"], seed=0)
    model.load_weights(weights_path)
    prediction = model.predict(packed)
    meanlong, sdlong, meanlat, sdlat = (np.float64(v) for v in norm)  # float64 products, as in predict_locs
    xy = np.array([[x[0] * sdlong + meanlong, x[1] * sdlat + meanlat] for x in prediction])
    return xy, packed


def write_predlocs(path, xy, samples):
    import pandas as pd

    out = pd.DataFrame(xy.reshape(-1, 2))
    out.columns = ["x", "y"]
    out["sampleID"] = samples
    out.to_csv(path, index=False)


def main(argv=None):
    ns = build_parser().parse_args(argv)
    given = [f"--{k}" for k in ("vcf", "zarr", "bed") if getattr(ns, k) is not None]
    if len(given) != 1:
        raise SystemExit("predict: give exactly one genotype input (--vcf, --zarr or --bed)"
                         + (f", not {' and '.join(given)}" if given else ""))
    models = check_models(ns.weights)
    cs, query, samples = read_query(ns)
    joins = []
    for p, table, _, _ in models:
        src, flip = sites.join(table, query)
        if not (src >= 0).any():
            raise SystemExit(f"predict: {p}: none of its {len(src)} sites is in the query")
        joins.append((src, flip))
    dev = upload_query(cs)
    for (p, table, shape, norm), (src, flip) in zip(models, joins):
        xy, packed = predict_model(dev, src, flip, p, shape, norm)
        out = f"{ns.out}_{model_name(p)}_predlocs.txt"
        write_predlocs(out, xy, samples)
        matched = int((src >= 0).sum())
        print(f"{p}: {len(src)} sites, {matched} matched ({int(flip.sum())} flipped), {len(src) - matched} absent; "
              f"code-3 calls {code3_fraction(packed):.6f}; {len(samples)} samples -> {out}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
