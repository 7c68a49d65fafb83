"""CPU: PLINK 1 .bed input (--bed) -- the format against a hand-computed record, write_bed round trips through the
oracle's decoder, .bim / .fam parsing, and every refusal."""
import builtins
import json
import os

import numpy as np
import pytest

from oracle import bed_ref, ingest_ref


def _cube(rng, nvar, N, miss=0.1):
    """Biallelic GT cube as a .bed holds it: hets written as (0, 1), missing calls missing in both alleles."""
    gt = (rng.uniform(size=(nvar, N, 2)) < rng.uniform(0, 1, size=(nvar, 1, 1))).astype(np.int8)
    gt.sort(axis=2)
    gt[rng.uniform(size=(nvar, N)) < miss] = -1
    return gt


def test_known_record_decodes_by_hand():
    """Five samples [hom A1, missing, het, hom A2, het] = bytes 0xE4 0x02; the second byte's three pad fields are 0."""
    rec = np.array([[0xE4, 0x02]], dtype=np.uint8)
    gt = bed_ref.bed_to_gt(rec, 5)
    assert gt[0].tolist() == [[1, 1], [-1, -1], [0, 1], [0, 0], [0, 1]]
    assert ingest_ref.alt_allele_counts(gt)[0].tolist() == [2, 0, 1, 0, 1]  # the missing call counts 0 before imputation
    cnt = ingest_ref.count_alleles(gt)
    assert cnt[0, 1] == 4  # copies of A1
    assert int(ingest_ref.is_missing(gt)[0].sum()) == 1 and int((cnt[0] > 0).sum()) == 2
    assert ingest_ref.filter_snps(gt, min_mac=1).tolist() == [[2, 0, 1, 0, 1]]  # packed values
    # the pad fields read as genotypes would be three more homozygous-A1 calls: alt count 10
    assert ingest_ref.count_alleles(bed_ref.bed_to_gt(rec, 8))[0, 1] == 10
    from locator_b200 import io

    assert np.array_equal(io.decode_bed(rec, 5), gt)


@pytest.mark.parametrize("N", [1, 3, 4, 5, 17, 64, 65])
def test_write_bed_round_trips_through_the_oracle(tmp_path, N):
    from locator_b200 import io

    rng = np.random.default_rng(N)
    nvar = 37
    gt = _cube(rng, nvar, N)
    gt[0] = -1        # all missing
    gt[1] = 1         # monomorphic A1
    gt[2] = 0         # monomorphic A2
    samples = [f"ind{i}" for i in range(N)]
    pos = np.arange(nvar) * 1000 + 7
    prefix = str(tmp_path / "x")
    io.write_bed(prefix, gt, samples, pos)
    assert os.path.getsize(prefix + ".bed") == 3 + nvar * ((N + 3) // 4)
    records = bed_ref.read_bed_file(prefix + ".bed", nvar, N)
    assert np.array_equal(bed_ref.bed_to_gt(records, N), gt)
    # the reference's ingest on the decoded cube is that of the cube
    for mm in (1, 2, 3):
        assert np.array_equal(ingest_ref.filter_snps(bed_ref.bed_to_gt(records, N), min_mac=mm),
                              ingest_ref.filter_snps(gt, min_mac=mm))
    cs = io.read_bed(prefix)
    assert cs["samples"].tolist() == samples and cs["variants/POS"].tolist() == pos.tolist()
    assert set(cs["variants/CHROM"].tolist()) == {"1"}
    rows = cs["calldata/GT"]
    assert rows.shape == (nvar, N, 2) and rows.stored_shape == (nvar, (N + 3) // 4)
    assert np.array_equal(rows.read(), records)
    out = np.empty(((30 - 5), (N + 3) // 4), dtype=np.uint8)
    rows.rows(5, 30).read(out=out)  # positioned read of a record range into a given buffer
    assert np.array_equal(out, records[5:30])
    g = io.Genotypes(rows, cs["samples"], cs["variants/POS"])
    assert g.lazy == (prefix, 0, nvar) and g[5:30].lazy == (prefix, 5, 30)
    assert np.array_equal(g[5:30].gt, gt[5:30]) and g[5:30].positions.tolist() == pos[5:30].tolist()
    assert np.array_equal(g.gt, gt) and g.rows_on_disk is None


def test_write_bed_refuses_what_a_bed_cannot_hold(tmp_path):
    from locator_b200 import io

    gt = np.zeros((2, 3, 2), np.int8)
    bad = gt.copy()
    bad[1, 2, 1] = 2
    with pytest.raises(ValueError, match="allele indices >= 2"):
        io.write_bed(str(tmp_path / "a"), bad, ["a", "b", "c"], [1, 2])
    bad = gt.copy()
    bad[0, 1, 0] = -1
    with pytest.raises(ValueError, match="half-missing"):
        io.write_bed(str(tmp_path / "b"), bad, ["a", "b", "c"], [1, 2])


def test_bim_and_fam_parsing(tmp_path):
    from locator_b200 import io

    (tmp_path / "p.fam").write_text("famA s1 0 0 1 -9\nfamA  s2\t0 0 2 1\n\nfamB s3 s1 s2 0 -9\n")
    (tmp_path / "p.bim").write_text("1\trs1\t0\t1500\tA\tG\n1 rs2 0.5 2500 C T\n2\trs3\t0\t100\tG\tA\n")
    assert io.read_fam(str(tmp_path / "p.fam")).tolist() == ["s1", "s2", "s3"]  # IID, not FID
    chrom, pos = io.read_bim(str(tmp_path / "p.bim"))
    assert chrom.tolist() == ["1", "1", "2"] and pos.tolist() == [1500, 2500, 100] and pos.dtype == np.int64
    (tmp_path / "p.bed").write_bytes(b"\x6c\x1b\x01" + bytes([0xE4, 0x1B, 0x00]))
    cs = io.read_bed(str(tmp_path / "p"))
    assert cs["calldata/GT"].shape == (3, 3, 2)
    assert io.decode_bed(cs["calldata/GT"].read(), 3).tolist() == [
        [[1, 1], [-1, -1], [0, 1]], [[0, 0], [0, 1], [-1, -1]], [[1, 1], [1, 1], [1, 1]]]


def _fileset(tmp_path, nvar=6, N=5, chrom="1", name="g"):
    from locator_b200 import io

    prefix = str(tmp_path / name)
    io.write_bed(prefix, _cube(np.random.default_rng(0), nvar, N), [f"s{i}" for i in range(N)], np.arange(nvar) + 1,
                 chrom=chrom)
    return prefix


@pytest.mark.parametrize("damage,word", [(lambda b: b"\x6c\x1c" + b[2:], "magic bytes"),
                                         (lambda b: b[:2] + b"\x00" + b[3:], "sample-major"),
                                         (lambda b: b[:-1], "bytes"), (lambda b: b + b"\x00", "bytes")])
def test_bed_refusals_before_any_genotype_byte(tmp_path, damage, word):
    from locator_b200 import io, locator as L

    prefix = _fileset(tmp_path)
    data = open(prefix + ".bed", "rb").read()
    open(prefix + ".bed", "wb").write(damage(data))
    with pytest.raises(ValueError, match=word):
        io.read_bed(prefix)
    L.set_args(L.command_parser().parse_args(["--bed", prefix, "--out", str(tmp_path / "o")]))
    with pytest.raises(SystemExit, match=word):
        L.load_genotypes()


def test_windows_refused_on_several_chromosomes(tmp_path, monkeypatch):
    from locator_b200 import io, locator as L

    prefix = _fileset(tmp_path, chrom=np.array(["1", "1", "1", "2", "2", "X"]))
    monkeypatch.setattr(io.BedRows, "read", lambda *a, **k: pytest.fail("genotype bytes read"))
    L.set_args(L.command_parser().parse_args(["--bed", prefix, "--out", str(tmp_path / "o"), "--windows"]))
    with pytest.raises(SystemExit, match="3 chromosomes"):
        L.load_genotypes()
    L.set_args(L.command_parser().parse_args(["--bed", prefix, "--out", str(tmp_path / "o")]))
    genotypes, samples = L.load_genotypes()  # without --windows the chromosomes do not matter
    assert genotypes.shape == (6, 5, 2) and samples.tolist() == [f"s{i}" for i in range(5)]
    one = _fileset(tmp_path, chrom="22", name="one")
    L.set_args(L.command_parser().parse_args(["--bed", one, "--out", str(tmp_path / "o"), "--windows"]))
    assert L.load_genotypes()[0].lazy == (one, 0, 6)


def test_bed_with_another_input_refused_before_any_file_is_opened(tmp_path, monkeypatch):
    from locator_b200 import locator as L

    def ns(*extra):
        return L.command_parser().parse_args(["--sample_data", "s.txt", "--out", "o"] + list(extra))

    def no_open(*a, **k):
        raise AssertionError(f"opened {a[:1]}")

    L.validate_args(ns("--bed", "missing/prefix"))
    for other in (["--vcf", "x.vcf"], ["--zarr", "x.zarr"], ["--matrix", "m.txt"]):
        monkeypatch.setattr(builtins, "open", no_open)
        monkeypatch.setattr(os, "open", no_open)
        try:
            with pytest.raises(SystemExit, match="--bed with " + other[0]):
                L.validate_args(ns("--bed", "missing/prefix", *other))
        finally:
            monkeypatch.undo()
    with pytest.raises(SystemExit, match="--bed with --vcf"):
        L.main(["--bed", str(tmp_path / "none"), "--vcf", str(tmp_path / "none.vcf"), "--out", str(tmp_path / "o")])
    assert not os.path.exists(str(tmp_path / "o") + "_params.json")


def test_bed_is_an_extension_flag(tmp_path):
    """Not in params.json (the reference's keys), and kept over --load_params like --gpus."""
    from locator_b200 import locator as L

    ns = L.command_parser().parse_args(["--bed", "p", "--sample_data", "s.txt", "--out", str(tmp_path / "o")])
    assert "bed" not in L._params_dict(ns)
    L.set_args(ns)
    L._write_params()
    params = json.load(open(str(tmp_path / "o") + "_params.json"))
    assert "bed" not in params and params["vcf"] is None
    args = L.start_run(L.command_parser().parse_args(["--bed", "q", "--load_params", str(tmp_path / "o") + "_params.json",
                                                    "--out", str(tmp_path / "o2")]))
    assert args.bed == "q" and args.out == str(tmp_path / "o")
    from locator_b200 import holdout

    args = L.start_run(holdout.build_parser().parse_args(["--bed", "r", "--load_params",
                                                          str(tmp_path / "o") + "_params.json"]),
                       extensions=("gpus", "replicates_per_gpu", "load_weights", "folds", "bed"))
    assert args.bed == "r"


def test_bed_loads_like_a_vcf(tmp_path, fixture_gt, golden_dir, capsys):
    """The fixture's cube (third-allele calls set missing) from a .bed: same samples, positions and the same
    'loaded (nvar, N, 2) genotypes' line as the VCF run; the GT cube the records stand for is the cube."""
    from locator_b200 import io, locator as L

    gt = fixture_gt["calldata/GT"].copy()
    gt[(gt >= 2).any(axis=2)] = -1
    gt[(gt < 0).any(axis=2)] = -1
    gt.sort(axis=2)
    prefix = str(tmp_path / "fx")
    io.write_bed(prefix, gt, fixture_gt["samples"], fixture_gt["variants/POS"])
    sd = os.path.join(golden_dir, "data", "test_sample_data.txt")
    L.set_args(L.command_parser().parse_args(["--bed", prefix, "--sample_data", sd, "--out", str(tmp_path / "o")]))
    genotypes, samples = L.load_genotypes()
    L.sort_samples(samples, genotypes)
    text = capsys.readouterr().out
    assert f"loaded ({gt.shape[0]}, {gt.shape[1]}, 2) genotypes" in text
    assert np.array_equal(samples, fixture_gt["samples"]) and np.array_equal(genotypes.positions, fixture_gt["variants/POS"])
    assert genotypes.rows_on_disk is not None  # nothing decoded on the host
    assert np.array_equal(genotypes[100:900].gt, gt[100:900])
