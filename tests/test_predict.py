"""CPU: the sites file of --keep_sites, the join of a query to a model's sites, the site identity the readers give,
and every refusal of --keep_sites and of python -m locator_b200.predict (all before any GPU work)."""
import gzip
import json
import os

import numpy as np
import pytest

from locator_b200 import io, sites


def _table(rows):
    c, p, r, a = zip(*rows) if rows else ((), (), (), ())
    return {"chrom": np.array(c, dtype=str), "pos": np.array(p, dtype=np.int64), "ref": np.array(r, dtype=str),
            "alt": np.array(a, dtype=str)}


def test_sites_file_round_trip(tmp_path):
    t = _table([("1", 100, "A", "T"), ("chr2", 5, "AC", "A"), ("1", 100, "A", "T"), ("X", 2**40, "G", "C")])
    norm = (np.float64(1) / 3, np.float64(2.000000000000001), -7.123456789012345e-300, 1e300)
    path = str(tmp_path / "m.sites.tsv")
    sites.write(path, t, 128, 6, norm)
    back, shape, norm2 = sites.read(path)
    assert shape == {"width": 128, "nlayers": 6}
    assert norm2 == tuple(float(x) for x in norm)  # repr: exact
    for k in t:
        assert np.array_equal(back[k], t[k]) and back[k].dtype.kind == t[k].dtype.kind, k
    assert sites.sidecar_path(str(tmp_path / "run_boot3.weights.npz")) == str(tmp_path / "run_boot3.sites.tsv")
    with open(path) as fh:
        head = [next(fh) for _ in range(7)]
    assert head[0] == "#width\t128\n" and head[-1] == "#CHROM\tPOS\tREF\tALT\n"
    with open(tmp_path / "bad.sites.tsv", "w") as fh:
        fh.write("CHROM\tPOS\tREF\tALT\n1\t2\tA\tT\n")
    with pytest.raises(ValueError):
        sites.read(str(tmp_path / "bad.sites.tsv"))


def test_join_rules():
    model = _table([
        ("1", 10, "A", "T"),   # 0: same alleles
        ("1", 20, "A", "G"),   # 1: swapped in the query -> flip
        ("1", 30, "C", "T"),   # 2: absent
        ("1", 40, "A", "C"),   # 3: query has {A, G}: allele mismatch -> absent
        ("1", 50, "G", "T"),   # 4: three query records at 50: the first that matches, in file order
        ("2", 10, "A", "T"),   # 5: same POS as site 0, other chromosome
        ("1", 60, "A", "T"),   # 6: A/T site: no strand complement (query T/A is a swap, not a complement)
        ("1", 10, "A", "T"),   # 7: a duplicate of site 0 (bootstrap models)
        ("1", 70, "C", "G"),   # 8: query lists the complement G/C at 70 -> a swap as written; TA/AT no match
    ])
    query = _table([
        ("1", 50, "G", "A"),   # 0
        ("1", 20, "G", "A"),   # 1
        ("1", 10, "A", "T"),   # 2
        ("1", 40, "A", "G"),   # 3
        ("1", 50, "T", "G"),   # 4 (swap) -- first match in file order
        ("1", 50, "G", "T"),   # 5 (same) -- later
        ("2", 10, "T", "A"),   # 6
        ("1", 60, "T", "A"),   # 7
        ("1", 70, "G", "C"),   # 8
        ("3", 30, "C", "T"),   # 9: other chromosome, POS of the absent site
    ])
    src, flip = sites.join(model, query)
    assert src.tolist() == [2, 1, -1, -1, 4, 6, 7, 2, 8]
    assert flip.tolist() == [0, 1, 0, 0, 1, 1, 1, 0, 1]
    src, flip = sites.join(model, _table([]))
    assert (src == -1).all() and not flip.any()


def _vcf_text(lines, samples=("a", "b", "c")):
    head = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(samples) + "\n"
    return head + "".join("\t".join(map(str, ln)) + "\n" for ln in lines)


def test_readers_give_site_identity(tmp_path):
    lines = [("chr1", 5, ".", "A", "T", ".", ".", ".", "GT", "0/1", "1/1", "./."),
             ("chr1", 9, "rs1", "AC", "A,G", ".", ".", ".", "GT", "0/2", "0/0", "1|0"),
             ("chr2", 9, ".", "G", "C", ".", ".", ".", "GT", "0/0", "0/1", "1/1")]
    p = tmp_path / "q.vcf.gz"
    with gzip.open(p, "wt") as fh:
        fh.write(_vcf_text(lines))
    v = io.read_vcf(str(p), sites=True)
    assert v["variants/CHROM"].tolist() == ["chr1", "chr1", "chr2"]
    assert v["variants/REF"].tolist() == ["A", "AC", "G"] and v["variants/ALT"].tolist() == ["T", "A", "C"]
    assert "variants/REF" not in io.read_vcf(str(p))  # opt-in: a plain run reads what it always read
    z = str(tmp_path / "q.zarr")
    io.write_zarr(z, v["calldata/GT"], v["samples"], v["variants/POS"], chrom=v["variants/CHROM"],
                  ref=v["variants/REF"], alt=v["variants/ALT"])
    back = io.read_zarr(z, lazy=True, sites=True)
    ids = io.variant_ids(back)
    assert {k: x.tolist() for k, x in ids.items()} == {"chrom": ["chr1", "chr1", "chr2"], "ref": ["A", "AC", "G"],
                                                        "alt": ["T", "A", "C"]}
    io.write_zarr(str(tmp_path / "bare.zarr"), v["calldata/GT"], v["samples"], v["variants/POS"])
    assert io.variant_ids(io.read_zarr(str(tmp_path / "bare.zarr"), lazy=True, sites=True)) is None
    gt = np.zeros((2, 3, 2), np.int8)
    io.write_bed(str(tmp_path / "b"), gt, ["a", "b", "c"], [7, 8])
    cs = io.read_bed(str(tmp_path / "b"), sites=True)
    assert cs["variants/REF"].tolist() == ["A", "A"] and cs["variants/ALT"].tolist() == ["T", "T"]  # REF = A2, ALT = A1
    g = io.Genotypes(cs["calldata/GT"], cs["samples"], cs["variants/POS"], io.variant_ids(cs))
    assert g[1:2].ids["alt"].tolist() == ["T"] and g[1:2].positions.tolist() == [8]


def test_keep_sites_refusals_and_params(tmp_path):
    from locator_b200 import locator as L

    base = ["--vcf", "x.vcf", "--sample_data", "s.txt", "--out", str(tmp_path / "r")]
    with pytest.raises(SystemExit, match="--keep_sites without --keep_weights"):
        L.validate_args(L.command_parser().parse_args(base + ["--keep_sites"]))
    with pytest.raises(SystemExit, match="--keep_sites with --matrix"):
        L.validate_args(L.command_parser().parse_args(["--matrix", "m.txt", "--out", "o", "--keep_weights", "--keep_sites"]))
    L.validate_args(L.command_parser().parse_args(base + ["--keep_weights", "--keep_sites"]))
    # not a reference key: params.json does not hold it, and a --load_params run keeps it from the command line
    ns = L.start_run(L.command_parser().parse_args(base + ["--keep_weights", "--keep_sites"]))
    L._write_params()
    params = json.load(open(str(tmp_path / "r") + "_params.json"))
    assert "keep_sites" not in params
    ns = L.start_run(L.command_parser().parse_args(["--load_params", str(tmp_path / "r") + "_params.json",
                                                    "--keep_sites"]))
    assert ns.keep_sites is True and ns.keep_weights is True
    from locator_b200 import holdout

    hs = holdout.build_parser().parse_args(base + ["--keep_weights", "--keep_sites"])
    assert hs.keep_sites


def test_keep_sites_refuses_a_zarr_store_without_alleles(tmp_path):
    from locator_b200 import locator as L

    z = str(tmp_path / "bare.zarr")
    io.write_zarr(z, np.zeros((3, 2, 2), np.int8), ["a", "b"], [1, 2, 3])
    L.set_args(L.command_parser().parse_args(["--zarr", z, "--out", "o", "--keep_weights", "--keep_sites"]))
    with pytest.raises(SystemExit, match="variants/CHROM"):
        L.load_genotypes()


def _model_files(tmp_path, name="m", K=5, width=64, nlayers=2, rows=None, sidecar=True):
    ws = [np.zeros(K, np.float32)] * 4 + [np.zeros((K, width), np.float32), np.zeros(width, np.float32)]
    for _ in range(nlayers - 1):
        ws += [np.zeros((width, width), np.float32), np.zeros(width, np.float32)]
    ws += [np.zeros((width, 2), np.float32), np.zeros(2, np.float32), np.zeros((2, 2), np.float32), np.zeros(2, np.float32)]
    w = str(tmp_path / f"{name}.weights.npz")
    np.savez(w, **{f"w{i:03d}": x for i, x in enumerate(ws)})
    if sidecar:
        t = _table(rows or [("1", 10 * (k + 1), "A", "T") for k in range(K)])
        sites.write(sites.sidecar_path(w), t, width, nlayers, (0.0, 1.0, 0.0, 1.0))
    return w


def test_predict_refusals_before_reading_genotypes(tmp_path, monkeypatch):
    from locator_b200 import predict

    good = _model_files(tmp_path)
    # a genotype read would fail loudly: every refusal below comes first
    monkeypatch.setattr(io, "read_vcf", lambda *a, **k: (_ for _ in ()).throw(AssertionError("genotypes read")))
    q = ["--vcf", "q.vcf", "--out", str(tmp_path / "p")]
    with pytest.raises(SystemExit, match="exactly one genotype input"):
        predict.main(["--weights", good, "--out", "o"])
    with pytest.raises(SystemExit, match="--vcf and --bed"):
        predict.main(["--weights", good, "--vcf", "a", "--bed", "b", "--out", "o"])
    nosc = _model_files(tmp_path, "nosc", sidecar=False)
    with pytest.raises(SystemExit, match="no sites file"):
        predict.main(["--weights", good, nosc] + q)
    rows = _model_files(tmp_path, "rows", K=5)
    sites.write(sites.sidecar_path(rows), _table([("1", 1, "A", "T")] * 4), 64, 2, (0.0, 1.0, 0.0, 1.0))
    with pytest.raises(SystemExit, match="lists 4 sites"):
        predict.main(["--weights", rows] + q)
    wid = _model_files(tmp_path, "wid")
    sites.write(sites.sidecar_path(wid), _table([("1", 1, "A", "T")] * 5), 128, 2, (0.0, 1.0, 0.0, 1.0))
    with pytest.raises(SystemExit, match="at width 128"):
        predict.main(["--weights", wid] + q)
    deep = _model_files(tmp_path, "deep")
    sites.write(sites.sidecar_path(deep), _table([("1", 1, "A", "T")] * 5), 64, 3, (0.0, 1.0, 0.0, 1.0))
    with pytest.raises(SystemExit, match="nlayers 3"):
        predict.main(["--weights", deep] + q)
    assert predict.model_name(good) == "m" and len(predict.check_models([good])) == 1


def test_predict_refuses_a_model_with_no_site_in_the_query(tmp_path, monkeypatch):
    from locator_b200 import predict

    w = _model_files(tmp_path, rows=[("9", 10 * (k + 1), "A", "T") for k in range(5)])
    p = tmp_path / "q.vcf"
    p.write_text(_vcf_text([("1", 10, ".", "A", "T", ".", ".", ".", "GT", "0/1", "1/1", "./.")]))
    monkeypatch.setattr(predict, "upload_query", lambda cs: (_ for _ in ()).throw(AssertionError("uploaded")))
    with pytest.raises(SystemExit, match="none of its 5 sites"):
        predict.main(["--weights", w, "--vcf", str(p), "--out", str(tmp_path / "o")])
