"""GPU: prediction of a new genotype file with stored models (python -m locator_b200.predict).

The mapped packs (loc_pack_sites_mapped / loc_bed_pack_sites_mapped) against the plain-loop oracle
(oracle/predict_ref.py); code 3 in every inference forward against the oracle fed the moving mean there; and the
command end to end: on the file a model was trained on (no missing call, so no code 3) it reproduces the run's own
predictions byte for byte, for every kind of run that keeps weights."""
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


# ---- mapped packs --------------------------------------------------------------------------------------------
def _query_cube(rng, nvar, N):
    """Calls of every kind: 0/0, 0/1, 1/0, 1/1, missing, half-missing, allele index 2."""
    gt = (rng.uniform(size=(nvar, N, 2)) < rng.uniform(0.1, 0.9, size=(nvar, 1, 1))).astype(np.int8)
    u = rng.uniform(size=(nvar, N))
    gt[u < 0.05] = -1
    gt[(u >= 0.05) & (u < 0.08), 0] = -1
    gt[(u >= 0.08) & (u < 0.10), 1] = 2
    return gt


def _mapping(rng, nvar, K):
    src = rng.integers(0, nvar, K)
    src[rng.uniform(size=K) < 0.1] = -1  # absent sites
    src[K // 2:K // 2 + 5] = src[0]      # duplicates
    flip = (rng.uniform(size=K) < 0.3).astype(np.uint8)
    return src, flip


def _bed_cube(gt):
    """What a .bed can hold: half-missing -> missing, allele 2 -> 1, alleles sorted."""
    g = gt.copy()
    g[(g < 0).any(axis=2)] = -1
    g[g >= 2] = 1
    g.sort(axis=2)
    return g


@pytest.mark.parametrize("N", [1, 3, 4, 5, 15, 16, 17, 63, 64, 65, 500])
def test_mapped_packs_equal_oracle(G, tmp_path, N):
    from locator_b200 import io
    from oracle import predict_ref

    rng = np.random.default_rng(N)
    nvar, K = 90, 300
    gt = _query_cube(rng, nvar, N)
    src, flip = _mapping(rng, nvar, K)
    ref = predict_ref.mapped_counts(gt, src, flip)
    got = G.pack_sites_mapped(torch.as_tensor(gt).cuda(), src, flip)
    assert torch.equal(got.words, G.PackedGenotypes.from_counts(ref).words)  # pad bits included
    gb = _bed_cube(gt)
    prefix = str(tmp_path / "q")
    io.write_bed(prefix, gb, [f"s{i}" for i in range(N)], np.arange(nvar))
    bed = G.BedRecords.upload(io.read_bed(prefix)["calldata/GT"])
    got = G.pack_sites_mapped(bed, src, flip)
    assert torch.equal(got.words, G.PackedGenotypes.from_counts(predict_ref.mapped_counts(gb, src, flip)).words)


@pytest.mark.parametrize("offset", [1, 2, 3])
def test_bed_mapped_pack_at_any_pointer_offset(G, offset):
    from locator_b200._cabi import lib, check
    from oracle import bed_ref, predict_ref

    rng = np.random.default_rng(offset)
    nvar, N, K = 301, 37, 500
    rec = rng.integers(0, 256, size=(nvar, (N + 3) // 4), dtype=np.uint8)
    buf = torch.full((rec.size + 64,), 0x55, dtype=torch.uint8, device="cuda")
    buf[offset:offset + rec.size] = torch.as_tensor(rec.reshape(-1)).cuda()
    src, flip = _mapping(rng, nvar, K)
    out = G.PackedGenotypes.empty(N, K)
    s, f = torch.as_tensor(src).cuda(), torch.as_tensor(flip).cuda()
    check(lib.loc_bed_pack_sites_mapped(buf.data_ptr() + offset, nvar, N, s.data_ptr(), f.data_ptr(), K, out.ptr,
                                        out.row_words, torch.cuda.current_stream().cuda_stream))
    ref = predict_ref.mapped_counts(bed_ref.bed_to_gt(rec, N), src, flip)
    assert torch.equal(out.words, G.PackedGenotypes.from_counts(ref).words)


def test_mapped_packs_over_many_word_groups(G, tmp_path):
    """K = 1.1 M model sites (4,297 word groups of 256) from 400 records: both kernels agree with each other and, on
    a sample of columns, with the oracle."""
    from locator_b200 import io
    from oracle import predict_ref

    rng = np.random.default_rng(11)
    nvar, N, K = 400, 5, 1_100_000
    gt = _bed_cube(_query_cube(rng, nvar, N))
    src, flip = _mapping(rng, nvar, K)
    io.write_bed(str(tmp_path / "q"), gt, [f"s{i}" for i in range(N)], np.arange(nvar))
    bed = G.BedRecords.upload(io.read_bed(str(tmp_path / "q"))["calldata/GT"])
    a = G.pack_sites_mapped(bed, src, flip)
    b = G.pack_sites_mapped(torch.as_tensor(gt).cuda(), src, flip)
    assert torch.equal(a.words, b.words)
    cols = np.concatenate([np.arange(300), rng.integers(0, K, 300), np.arange(K - 300, K)])
    assert np.array_equal(a.to_numpy()[:, cols], predict_ref.mapped_counts(gt, src[cols], flip[cols]))


# ---- code 3 in the inference forwards -------------------------------------------------------------------------
# family -> oracle numerics and tolerance |dy| <= tol * (1 + |y|) (those of tests/test_gpu_model.py)
FAMILIES = {"tcgen05": ("tf32", 2e-3), "simt": ("fp32", 2e-4)}


@pytest.mark.parametrize("path,width,n", [("wide", 256, 100), ("narrow", 256, 100), ("narrow", 256, 20),
                                          ("simt", 128, 100)])
def test_code3_is_the_moving_mean(G, monkeypatch, path, width, n):
    """Prediction with code-3 entries (whole absent columns and scattered missing calls) equals the oracle fed x =
    the moving mean there: tcgen05 wide forward, the narrow one (LOC_NO_WIDE=1, and <= 32 rows), CUDA-core."""
    from locator_b200 import model as M
    from oracle import model_ref, predict_ref

    rng = np.random.default_rng(n + width)
    K = 3000
    counts = rng.binomial(2, rng.uniform(0.05, 0.95, K), size=(n, K)).astype(np.uint8)
    counts[:, rng.uniform(size=K) < 0.1] = 3
    counts[rng.uniform(size=(n, K)) < 0.05] = 3
    m = M.LocatorModel(K, width=width, nlayers=4, seed=5)
    assert m.impl == ("simt" if path == "simt" else "tcgen05")
    ws = m.get_weights()
    ws[0] = rng.uniform(0.5, 1.5, K).astype(np.float32)
    ws[1] = rng.normal(0, 0.5, K).astype(np.float32)  # beta: what code 3 enters as
    ws[2] = rng.uniform(0, 1.5, K).astype(np.float32)
    ws[3] = rng.uniform(0.1, 0.8, K).astype(np.float32)
    for i in range(5, len(ws), 2):
        ws[i] = rng.normal(0, 0.05, ws[i].shape).astype(np.float32)
    m.set_weights(ws)
    if path == "narrow":
        monkeypatch.setenv("LOC_NO_WIDE", "1")
    else:
        monkeypatch.delenv("LOC_NO_WIDE", raising=False)
    yp = m.predict(G.PackedGenotypes.from_counts(counts))
    numerics, tol = FAMILIES[m.impl]
    ref = model_ref.RefLocator(K, width, 4, weights=ws, numerics=numerics)
    yr = ref.predict(predict_ref.first_layer_input(counts, ws[2]))
    np.testing.assert_allclose(yp, yr, rtol=tol, atol=tol)
    # and code 3 is not read as a count: the same matrix with 3 -> 0 predicts something else
    assert not np.allclose(yp, m.predict(G.PackedGenotypes.from_counts(np.where(counts == 3, 0, counts))), atol=1e-3)


# ---- the command end to end -----------------------------------------------------------------------------------
def _write_vcf(path, gt, samples, pos, ref="A", alt="T"):
    txt = {(-1, -1): "./.", (0, 0): "0/0", (0, 1): "0/1", (1, 0): "1/0", (1, 1): "1/1", (0, -1): "0/.", (1, -1): "1/."}
    ref = np.broadcast_to(np.asarray(ref, dtype=str), len(pos))
    alt = np.broadcast_to(np.asarray(alt, dtype=str), len(pos))
    with open(path, "w") as fh:
        fh.write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(samples) + "\n")
        for row, p, r, a in zip(gt, pos, ref, alt):
            fh.write(f"1\t{p}\t.\t{r}\t{a}\t.\t.\t.\tGT\t" + "\t".join(txt[(int(x), int(y))] for x, y in row) + "\n")


@pytest.fixture(scope="module")
def inputs(tmp_path_factory):
    """The fixture's cube without missing calls (third alleles -> 1) as VCF (REF A, ALT T), .bed and zarr."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from locator_b200 import io

    d = tmp_path_factory.mktemp("predict_inputs")
    v = io.read_vcf(VCF)
    gt, samples, pos = v["calldata/GT"].copy(), v["samples"], v["variants/POS"]
    assert (gt >= 0).all()
    gt[gt >= 2] = 1
    gt.sort(axis=2)
    _write_vcf(str(d / "fx.vcf"), gt, samples, pos)
    io.write_bed(str(d / "fx"), gt, samples, pos)
    io.write_zarr(str(d / "fx.zarr"), gt, samples, pos, chunk_variants=1500, chrom="1", ref="A", alt="T")
    return {"vcf": str(d / "fx.vcf"), "bed": str(d / "fx"), "zarr": str(d / "fx.zarr"), "gt": gt, "samples": samples,
            "pos": pos, "dir": d}


def _rows(path, ncols=3):
    """{sampleID: the row's first ncols fields, as written}"""
    with open(path) as fh:
        lines = fh.read().splitlines()[1:]
    return {ln.split(",")[2]: ",".join(ln.split(",")[:ncols]) for ln in lines}


def _predict(weights, src, path, out):
    from locator_b200 import predict

    assert predict.main(["--weights", *weights, f"--{src}", path, "--out", out]) == 0


def _check_reproduced(run_predlocs, pred_out):
    run, got = _rows(run_predlocs), _rows(pred_out)
    assert run and set(run) <= set(got)
    for sid, row in run.items():
        assert got[sid] == row, sid


def _train(argv, holdout=False):
    from locator_b200 import holdout as H, locator as L

    assert (H.main(argv) if holdout else L.main(argv)) == 0


def _common(src, path, stem):
    return [f"--{src}", path, "--sample_data", SAMPLES, "--out", stem, "--seed", "31", "--max_epochs", "3",
            "--keras_verbose", "0", "--keep_weights", "--keep_sites"]


def test_predict_reproduces_plain_run_and_bed_equals_vcf(G, inputs, tmp_path, capsys):
    from locator_b200 import sites

    stem = str(tmp_path / "plain")
    _train(_common("vcf", inputs["vcf"], stem))
    t, shape, norm = sites.read(stem + ".sites.tsv")
    assert shape == {"width": 256, "nlayers": 10} and len(t["pos"]) == np.load(stem + ".weights.npz")["w004"].shape[0]
    assert (t["ref"] == "A").all() and (t["alt"] == "T").all()
    outs = {}
    for src in ("vcf", "bed", "zarr"):
        _predict([stem + ".weights.npz"], src, inputs[src], str(tmp_path / f"q_{src}"))
        outs[src] = open(str(tmp_path / f"q_{src}_plain_predlocs.txt"), "rb").read()
    assert outs["vcf"] == outs["bed"] == outs["zarr"]
    assert "code-3 calls 0.000000" in capsys.readouterr().out
    _check_reproduced(stem + "_predlocs.txt", str(tmp_path / "q_vcf_plain_predlocs.txt"))
    assert len(_rows(str(tmp_path / "q_vcf_plain_predlocs.txt"))) == len(inputs["samples"])


def test_predict_reproduces_bootstrap_models(G, inputs, tmp_path):
    from locator_b200 import sites

    stem = str(tmp_path / "b")
    _train(_common("vcf", inputs["vcf"], stem) + ["--bootstrap", "--nboots", "2"])
    models = [f"{stem}_boot{b}.weights.npz" for b in ("FULL", 0, 1)]
    t = sites.read(f"{stem}_boot0.sites.tsv")[0]
    assert len(np.unique(t["pos"])) < len(t["pos"])  # a replicate's resampled sites, duplicates included
    _predict(models, "vcf", inputs["vcf"], str(tmp_path / "q"))
    for b in ("FULL", 0, 1):
        _check_reproduced(f"{stem}_boot{b}_predlocs.txt", str(tmp_path / f"q_b_boot{b}_predlocs.txt"))


@pytest.mark.parametrize("src,parent_ingest", [("zarr", False), ("zarr", True), ("bed", False)])
def test_predict_reproduces_window_models(G, inputs, tmp_path, monkeypatch, src, parent_ingest):
    if parent_ingest:
        monkeypatch.setenv("LOC_WINDOWS_PARENT_INGEST", "1")
    else:
        monkeypatch.delenv("LOC_WINDOWS_PARENT_INGEST", raising=False)
    stem = str(tmp_path / "w")
    _train(_common(src, inputs[src], stem) + ["--windows", "--window_size", "1250000", "--replicates_per_gpu", "2"])
    models = sorted(glob.glob(stem + "_*.weights.npz"))
    assert len(models) == 2
    _predict(models, "vcf", inputs["vcf"], str(tmp_path / "q"))
    for wpath in models:
        name = os.path.basename(wpath)[: -len(".weights.npz")]
        (run,) = glob.glob(str(tmp_path / name) + "_*_predlocs.txt")  # the window's stem + the reference's suffix
        _check_reproduced(run, str(tmp_path / f"q_{name}_predlocs.txt"))


def test_predict_reproduces_a_holdout_fold(G, inputs, tmp_path):
    stem = str(tmp_path / "h")
    _train(_common("bed", inputs["bed"], stem) + ["--folds", "3"], holdout=True)
    _predict([stem + "_holdout1.weights.npz"], "bed", inputs["bed"], str(tmp_path / "q"))
    with open(stem + "_holdout_predlocs.txt") as fh:
        fold1 = {ln.split(",")[2]: ",".join(ln.split(",")[:3]) for ln in fh.read().splitlines()[1:]
                 if ln.split(",")[3] == "1"}
    got = _rows(str(tmp_path / "q_h_holdout1_predlocs.txt"))
    assert fold1 and all(got[sid] == row for sid, row in fold1.items())


@pytest.fixture(scope="module")
def trained(inputs, tmp_path_factory):
    """One plain model of the no-missing cube, with its sites file."""
    d = tmp_path_factory.mktemp("predict_model")
    stem = str(d / "m")
    _train(_common("vcf", inputs["vcf"], stem))
    return stem + ".weights.npz"


def test_swapped_alleles_predict_the_same(G, inputs, trained, tmp_path):
    """REF/ALT swapped at a subset of sites and GT 0 <-> 1 rewritten there: the same predictions, byte for byte."""
    rng = np.random.default_rng(3)
    gt = inputs["gt"].copy()
    swap = rng.uniform(size=len(gt)) < 0.3
    gt[swap] = 1 - gt[swap]
    path = str(tmp_path / "swapped.vcf")
    _write_vcf(path, gt, inputs["samples"], inputs["pos"], np.where(swap, "T", "A"), np.where(swap, "A", "T"))
    _predict([trained], "vcf", inputs["vcf"], str(tmp_path / "a"))
    _predict([trained], "vcf", path, str(tmp_path / "b"))
    assert open(str(tmp_path / "a_m_predlocs.txt"), "rb").read() == open(str(tmp_path / "b_m_predlocs.txt"), "rb").read()


def test_absent_sites_and_missing_calls_match_oracle(G, inputs, trained, tmp_path):
    """A query without 10 % of the model's sites and with some calls blanked (missing, half-missing) against the
    oracle: the model's weights, x = the moving mean at every code-3 entry."""
    from locator_b200 import io, predict, sites
    from locator_b200.model import LocatorModel
    from oracle import model_ref, predict_ref

    rng = np.random.default_rng(4)
    table, shape, norm = sites.read(sites.sidecar_path(trained))
    model_pos = set(table["pos"].tolist())
    drop = np.array([p in model_pos and rng.uniform() < 0.1 for p in inputs["pos"]])
    gt = inputs["gt"][~drop].copy()
    u = rng.uniform(size=gt.shape[:2])
    gt[u < 0.03] = -1
    gt[(u >= 0.03) & (u < 0.05), 1] = -1
    path = str(tmp_path / "holes.vcf")
    _write_vcf(path, gt, inputs["samples"], inputs["pos"][~drop])
    ns = predict.build_parser().parse_args(["--weights", trained, "--vcf", path, "--out", str(tmp_path / "o")])
    cs, query, samples = predict.read_query(ns)
    src, flip = sites.join(table, query)
    assert 0.05 < (src < 0).mean() < 0.15
    xy, packed = predict.predict_model(predict.upload_query(cs), src, flip, trained, shape, norm)
    counts = predict_ref.mapped_counts(cs["calldata/GT"], src, flip)
    assert np.array_equal(packed.to_numpy(), counts)
    assert abs(predict.code3_fraction(packed) - (counts == 3).mean()) < 1e-12
    m = LocatorModel(len(src), seed=0)
    m.load_weights(trained)
    ws = m.get_weights()
    numerics, tol = FAMILIES[m.impl]
    yr = model_ref.RefLocator(len(src), 256, 10, weights=ws, numerics=numerics).predict(
        predict_ref.first_layer_input(counts, ws[2]))
    meanlong, sdlong, meanlat, sdlat = norm
    y = np.stack([(xy[:, 0] - meanlong) / sdlong, (xy[:, 1] - meanlat) / sdlat], axis=1)
    np.testing.assert_allclose(y, yr, rtol=tol, atol=tol)
