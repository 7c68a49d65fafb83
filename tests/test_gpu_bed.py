"""GPU: --bed input.  The .bed kernels (loc_bed_site_stats / _pack_sites / _missing_calls) equal the int8 kernels on
the cube the records stand for, bit for bit; filter_snps and every driver give byte-identical outputs from a .bed
and from a VCF / zarr store of the same cube."""
import glob
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

HERE = os.path.dirname(os.path.abspath(__file__))
VCF = os.path.join(HERE, "golden", "data", "test_genotypes.vcf.gz")
SAMPLES = os.path.join(HERE, "golden", "data", "test_sample_data.txt")


@pytest.fixture(scope="module")
def G():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from locator_b200 import genotypes

    return genotypes


def _cube(rng, nvar, N, miss=0.05):
    """Biallelic cube with missing calls, an all-missing, a monomorphic-A1 and a monomorphic-A2 site."""
    gt = (rng.uniform(size=(nvar, N, 2)) < rng.uniform(0, 1, size=(nvar, 1, 1)) ** 2).astype(np.int8)
    gt.sort(axis=2)
    gt[rng.uniform(size=(nvar, N)) < miss] = -1
    gt[0] = -1
    gt[1] = 1
    gt[2] = 0
    if nvar > 4:
        gt[3, :, 0] = 0
        gt[3, :, 1] = 1
        gt[3, : N // 2] = -1
    return gt


def _both(G, tmp_path, gt, name="b"):
    """(device cube, device .bed records) of one cube, the records written and read back through the files."""
    from locator_b200 import io

    prefix = str(tmp_path / name)
    io.write_bed(prefix, gt, [f"s{i}" for i in range(gt.shape[1])], np.arange(gt.shape[0]))
    bed = G.BedRecords.upload(io.read_bed(prefix)["calldata/GT"])
    return torch.as_tensor(gt).cuda(), bed


def _check_equal(G, g, bed, min_mac):
    na, alt, miss, keep = G.bed_site_stats(bed, min_mac=min_mac)
    _, na0, alt0, miss0, keep0 = G.site_stats(g, min_mac=min_mac)
    for a, b in ((na, na0), (alt, alt0), (miss, miss0), (keep, keep0)):
        assert torch.equal(a, b)
    idx = G.compact_sites(keep)
    p = G.bed_pack_sites(bed, idx)
    p0 = G.pack_sites(g, idx)
    assert p.row_words == p0.row_words and torch.equal(p.words, p0.words)  # pad bits included
    ks, ss = G.bed_missing_calls(bed, idx, miss)
    ks0, ss0 = G.missing_calls(g, idx, miss0)
    assert torch.equal(ks, ks0) and torch.equal(ss, ss0)
    return int(idx.numel())


@pytest.mark.parametrize("min_mac", [1, 2, 3])
@pytest.mark.parametrize("N", [1, 3, 4, 5, 15, 16, 17, 63, 64, 65, 500, 2500])
def test_bed_kernels_equal_int8_kernels(G, tmp_path, N, min_mac):
    rng = np.random.default_rng(N * 10 + min_mac)
    nvar = 300 if N < 500 else 120
    gt = _cube(rng, nvar, N)
    g, bed = _both(G, tmp_path, gt)
    K = _check_equal(G, g, bed, min_mac)
    assert K > 0 or N == 1  # one sample: a kept site is one het call, alt count 1 < min_mac 2 / 3
    # no site kept
    g, bed = _both(G, tmp_path, np.ones((20, N, 2), np.int8), "mono")
    assert _check_equal(G, g, bed, min_mac) == 0


@pytest.mark.parametrize("offset", [1, 2, 3])
def test_bed_kernels_at_any_pointer_offset(G, offset):
    """The C ABI takes any record-area address (records are byte-aligned anyway when ceil(N/4) is odd)."""
    from locator_b200 import io
    from locator_b200._cabi import lib, check

    rng = np.random.default_rng(offset)
    nvar, N = 301, 37
    gt = _cube(rng, nvar, N)
    rb = (N + 3) // 4
    q = np.zeros((nvar, rb * 4), np.uint8)
    q[:, :N] = np.select([gt[:, :, 0] < 0, gt.sum(2) == 2, gt.sum(2) == 1], [1, 0, 2], 3)
    q = q.reshape(nvar, rb, 4)
    rec = (q[:, :, 0] | q[:, :, 1] << 2 | q[:, :, 2] << 4 | q[:, :, 3] << 6).astype(np.uint8)
    assert np.array_equal(io.decode_bed(rec, N), gt)
    buf = torch.full((rec.size + 64,), 0x55, dtype=torch.uint8, device="cuda")  # neighbours: "missing" fields
    buf[offset:offset + rec.size] = torch.as_tensor(rec.reshape(-1)).cuda()
    ptr = buf.data_ptr() + offset
    st = torch.cuda.current_stream().cuda_stream
    na = torch.empty(nvar, dtype=torch.int32, device="cuda")
    alt, miss = torch.empty_like(na), torch.empty_like(na)
    keep = torch.empty(nvar, dtype=torch.uint8, device="cuda")
    check(lib.loc_bed_site_stats(ptr, nvar, N, 2, na.data_ptr(), alt.data_ptr(), miss.data_ptr(), keep.data_ptr(), st))
    g = torch.as_tensor(gt).cuda()
    _, na0, alt0, miss0, keep0 = G.site_stats(g, min_mac=2)
    assert torch.equal(na, na0) and torch.equal(alt, alt0) and torch.equal(miss, miss0) and torch.equal(keep, keep0)
    idx = G.compact_sites(keep)
    out = G.PackedGenotypes.empty(N, int(idx.numel()))
    check(lib.loc_bed_pack_sites(ptr, nvar, N, idx.data_ptr(), int(idx.numel()), out.ptr, out.row_words, st))
    assert torch.equal(out.words, G.pack_sites(g, idx).words)


def test_bed_pack_beyond_65535_word_groups(G, tmp_path):
    """loc_bed_pack_sites takes any K in one launch (the grid's rows loop over the word groups)."""
    rng = np.random.default_rng(7)
    nvar, N = 1_100_000, 5
    gt = (rng.uniform(size=(nvar, N, 2)) < 0.5).astype(np.int8)
    gt.sort(axis=2)
    g, bed = _both(G, tmp_path, gt)
    idx = torch.arange(nvar, device="cuda")
    assert torch.equal(G.bed_pack_sites(bed, idx).words, G.pack_sites(g, idx).words)


def _fixture_cube():
    """The fixture's cube with its third-allele (and half-missing) calls set to missing: what a .bed can hold."""
    from locator_b200 import io

    v = io.read_vcf(VCF)
    gt = v["calldata/GT"].copy()
    gt[((gt >= 2) | (gt < 0)).any(axis=2)] = -1
    gt.sort(axis=2)
    return gt, v["samples"], v["variants/POS"]


def _write_vcf(path, gt, samples, pos):
    txt = {(-1, -1): "./.", (0, 0): "0/0", (0, 1): "0/1", (1, 1): "1/1"}
    with open(path, "w") as fh:
        fh.write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(samples) + "\n")
        for row, p in zip(gt, pos):
            fh.write(f"1\t{p}\t.\tA\tT\t.\t.\t.\tGT\t" + "\t".join(txt[(int(a), int(b))] for a, b in row) + "\n")


@pytest.fixture(scope="module")
def inputs(tmp_path_factory):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from locator_b200 import io

    d = tmp_path_factory.mktemp("bed_inputs")
    gt, samples, pos = _fixture_cube()
    _write_vcf(str(d / "fx.vcf"), gt, samples, pos)
    io.write_bed(str(d / "fx"), gt, samples, pos)
    io.write_zarr(str(d / "fx.zarr"), gt, samples, pos, chunk_variants=1500)
    return {"vcf": str(d / "fx.vcf"), "bed": str(d / "fx"), "zarr": str(d / "fx.zarr"), "gt": gt}


def test_filter_snps_impute_and_subsample_match_the_vcf_path(G, inputs, tmp_path):
    """Same packed matrix and numpy's stream left at the same position (imputation draws, --max_SNPs)."""
    from locator_b200 import io, locator as L

    got = {}
    for src in ("vcf", "bed"):
        L.set_args(L.command_parser().parse_args([f"--{src}", inputs[src], "--out", str(tmp_path / "r"),
                                                "--impute_missing", "--max_SNPs", "3000", "--min_mac", "2"]))
        genotypes, _ = L.load_genotypes()
        assert (genotypes.rows_on_disk is not None) == (src == "bed")
        np.random.seed(99)
        ac = L.filter_snps(genotypes)
        got[src] = (ac.packed.words.cpu().numpy(), ac.shape, np.random.random())
    assert np.array_equal(got["vcf"][0], got["bed"][0]) and got["vcf"][1:] == got["bed"][1:]
    # and the oracle's ingest of the cube
    from oracle import ingest_ref

    np.random.seed(99)
    ref = ingest_ref.filter_snps(inputs["gt"], min_mac=2, impute_missing=True, max_SNPs=3000)
    assert np.array_equal(G.PackedGenotypes(torch.as_tensor(got["bed"][0]).cuda(), *got["bed"][1][::-1]).to_numpy(), ref.T)


def _outputs(stem):
    """{file suffix: contents} of a run: text files as bytes, weights as arrays."""
    out = {}
    for f in sorted(glob.glob(stem + "*")):
        key = f[len(stem):]
        if key.endswith(("_params.json", ".pdf")):  # the fit plot carries its creation date
            continue
        if f.endswith(".npz"):
            with np.load(f) as z:
                out[key] = [z[k] for k in sorted(z.files)]
        else:
            out[key] = open(f, "rb").read()
    return out


def _same(a, b):
    assert sorted(a) == sorted(b) and a
    for k in a:
        if isinstance(a[k], list):
            assert len(a[k]) == len(b[k]) and all(np.array_equal(x, y) for x, y in zip(a[k], b[k])), k
        else:
            assert a[k] == b[k], k


@pytest.mark.parametrize("mode", ["plain", "bootstrap", "jacknife", "holdout"])
def test_runs_from_bed_equal_runs_from_vcf(G, inputs, tmp_path, mode):
    from locator_b200 import holdout, locator as L

    extra = {"plain": [], "bootstrap": ["--bootstrap", "--nboots", "2"], "jacknife": ["--jacknife", "--nboots", "2"],
             "holdout": ["--folds", "3"]}[mode]
    outs = {}
    for src in ("vcf", "bed"):
        stem = str(tmp_path / src / "r")
        os.makedirs(os.path.dirname(stem), exist_ok=True)
        argv = [f"--{src}", inputs[src], "--sample_data", SAMPLES, "--out", stem, "--seed", "4242", "--max_epochs", "3",
                "--keras_verbose", "0", "--keep_weights"] + extra
        assert (holdout.main(argv) if mode == "holdout" else L.main(argv)) == 0
        outs[src] = _outputs(stem)
    _same(outs["vcf"], outs["bed"])


@pytest.mark.parametrize("gpus,parent_ingest,impute", [(1, False, False), (1, True, False), (2, False, False),
                                                       (2, True, False), (1, False, True), (2, False, True)])
def test_windows_from_bed_equal_windows_from_zarr(G, inputs, tmp_path, monkeypatch, gpus, parent_ingest, impute):
    from locator_b200 import locator as L

    if parent_ingest:
        monkeypatch.setenv("LOC_WINDOWS_PARENT_INGEST", "1")
    else:
        monkeypatch.delenv("LOC_WINDOWS_PARENT_INGEST", raising=False)
    outs = {}
    for src in ("zarr", "bed"):
        stem = str(tmp_path / src / "w")
        os.makedirs(os.path.dirname(stem), exist_ok=True)
        argv = [f"--{src}", inputs[src], "--sample_data", SAMPLES, "--out", stem, "--seed", "777", "--max_epochs", "3",
                "--keras_verbose", "0", "--windows", "--window_size", "1250000", "--gpus", str(gpus),
                "--replicates_per_gpu", "2", "--keep_weights"] + (["--impute_missing"] if impute else [])
        assert L.main(argv) == 0
        outs[src] = _outputs(stem)
    assert sum(k.endswith("_predlocs.txt") for k in outs["bed"]) == 2
    _same(outs["zarr"], outs["bed"])
