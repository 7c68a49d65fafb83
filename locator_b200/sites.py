"""The sites of a stored model, and where a query file has them.

A model trained with ``--keep_weights --keep_sites`` gets, next to every ``X.weights.npz``, a sidecar
``X.sites.tsv``: the model's shape, the location normalisation its outputs are de-normalised with, and one
``CHROM POS REF ALT`` row per W1 row, in W1 order (REF = allele index 0, ALT = allele index 1: the packed value of a
site is its count of ALT).  ``python -m locator_b200.predict`` reads it to put a query's genotypes in the model's
site order (``join``).

Sidecar layout (tab-separated)::

    #width	256
    #nlayers	10
    #meanlong	<repr float>     (also sdlong, meanlat, sdlat: repr, so that de-normalisation is exact)
    #CHROM	POS	REF	ALT
    1	12345	A	T           (one row per W1 row)
"""
from __future__ import annotations

import numpy as np

NORM_KEYS = ("meanlong", "sdlong", "meanlat", "sdlat")


def sidecar_path(weights_path):
    """X.weights.npz -> X.sites.tsv"""
    stem = weights_path[: -len(".weights.npz")] if weights_path.endswith(".weights.npz") else weights_path
    return stem + ".sites.tsv"


def table(ids, positions, idx):
    """Site table {"chrom", "pos", "ref", "alt"} of rows ``idx`` (int array, duplicates allowed) of a genotype
    input's identity arrays (io.Genotypes.ids / .positions)."""
    idx = np.asarray(idx, dtype=np.int64)
    return {"chrom": np.asarray(ids["chrom"])[idx], "pos": np.asarray(positions, dtype=np.int64)[idx],
            "ref": np.asarray(ids["ref"])[idx], "alt": np.asarray(ids["alt"])[idx]}


def take(t, idx):
    """Rows ``idx`` of a site table (bootstrap site orders, --max_SNPs)."""
    idx = np.asarray(idx, dtype=np.int64)
    return {k: v[idx] for k, v in t.items()}


def write(path, t, width, nlayers, norm):
    """The sidecar of one model; ``norm`` = (meanlong, sdlong, meanlat, sdlat)."""
    head = [f"#width\t{int(width)}", f"#nlayers\t{int(nlayers)}"]
    head += [f"#{k}\t{float(v)!r}" for k, v in zip(NORM_KEYS, norm)]
    head.append("#CHROM\tPOS\tREF\tALT")
    rows = [f"{c}\t{p}\t{r}\t{a}" for c, p, r, a in zip(t["chrom"], t["pos"].tolist(), t["ref"], t["alt"])]
    with open(path, "w") as fh:
        fh.write("\n".join(head + rows) + "\n")


def read(path):
    """-> (site table, {"width", "nlayers"}, norm tuple).  Raises ValueError on a malformed file."""
    import pandas as pd

    meta = {}
    with open(path) as fh:
        for _ in range(len(NORM_KEYS) + 3):
            line = fh.readline().rstrip("\n")
            if not line.startswith("#"):
                raise ValueError(f"{path}: header line expected, found {line[:40]!r}")
            key, _, val = line[1:].partition("\t")
            meta[key] = val
    want = ["width", "nlayers", *NORM_KEYS, "CHROM"]
    if list(meta) != want or meta["CHROM"] != "POS\tREF\tALT":
        raise ValueError(f"{path}: not a sites file (header keys {list(meta)}, expected {want})")
    t = pd.read_csv(path, sep="\t", header=None, skiprows=len(want), dtype=str, keep_default_na=False,
                    names=["chrom", "pos", "ref", "alt"])
    sites = {"chrom": t["chrom"].to_numpy(dtype=str), "pos": t["pos"].to_numpy(dtype=np.int64),
             "ref": t["ref"].to_numpy(dtype=str), "alt": t["alt"].to_numpy(dtype=str)}
    shape = {"width": int(meta["width"]), "nlayers": int(meta["nlayers"])}
    return sites, shape, tuple(float(meta[k]) for k in NORM_KEYS)


def join(model, query):
    """Where a query has each model site: (src int64 [K], flip uint8 [K]).

    Model site k matches query record r when CHROM and POS are equal and {REF, ALT} are equal as sets; swapped
    alleles set flip[k] (the query's count of allele 0 is the model's count of ALT).  No strand complement is
    applied: A/T and C/G sites match as written.  Of several matching records the first in file order is taken;
    src[k] = -1 when none matches."""
    K = len(model["pos"])
    src = np.full(K, -1, dtype=np.int64)
    flip = np.zeros(K, dtype=np.uint8)
    if K == 0 or len(query["pos"]) == 0:
        return src, flip
    # (CHROM, POS) -> one int64 key; chromosome names numbered over both tables
    names, inv = np.unique(np.concatenate([np.asarray(model["chrom"], dtype=str), np.asarray(query["chrom"], dtype=str)]),
                           return_inverse=True)
    span = int(max(model["pos"].max(), query["pos"].max())) + 1
    mkey = inv[:K].astype(np.int64) * span + model["pos"]
    qkey = inv[K:].astype(np.int64) * span + query["pos"]
    order = np.argsort(qkey, kind="stable")  # equal keys stay in file order
    qs = qkey[order]
    lo = np.searchsorted(qs, mkey, "left")
    hi = np.searchsorted(qs, mkey, "right")
    mref, malt = np.asarray(model["ref"]), np.asarray(model["alt"])
    qref, qalt = np.asarray(query["ref"]), np.asarray(query["alt"])

    def match(k, r):
        if qref[r] == mref[k] and qalt[r] == malt[k]:
            return 0
        if qref[r] == malt[k] and qalt[r] == mref[k]:
            return 1
        return -1

    one = np.nonzero(hi - lo == 1)[0]
    r1 = order[lo[one]]
    same = (qref[r1] == mref[one]) & (qalt[r1] == malt[one])
    swap = ~same & (qref[r1] == malt[one]) & (qalt[r1] == mref[one])
    src[one[same | swap]] = r1[same | swap]
    flip[one[swap]] = 1
    for k in np.nonzero(hi - lo > 1)[0]:  # several records at one position: the first that matches
        for r in np.sort(order[lo[k]:hi[k]]):
            m = match(k, r)
            if m >= 0:
                src[k], flip[k] = r, m
                break
    return src, flip
