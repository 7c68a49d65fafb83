"""Replicate groups of large-batch models (--batch_size 33..256, loc_group_train_epochs).

A group step runs the batch statistics of all models in one launch, their 32-row chunks packed whole models per
hidden-stack launch, one step end for all models, the first-layer backwards back to back and the small-layer updates
on side streams (csrc/model.cu: train_step_big).  Every model must end bit-identical to the same model trained
alone with model.fit: histories, weights, Adam moments, predictions and optimizer counters.
"""
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
def M():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from locator_b200 import model

    return model


def _data(rng, n, K):
    p = rng.uniform(0.02, 0.98, size=K)
    x = rng.binomial(2, p, size=(n, K)).astype(np.uint8)
    x[:, ::97] = 0
    w = rng.normal(size=(K, 2)) / np.sqrt(K)
    y = ((x - 2 * p) @ w + 0.3 * rng.normal(size=(n, 2))).astype(np.float32)  # some signal: validation loss moves
    return x, y


def _datasets(rng, Ks, ntr, nva):
    from locator_b200.genotypes import PackedGenotypes

    out = []
    for K in Ks:
        x, y = _data(rng, ntr + nva, K)
        out.append((PackedGenotypes.from_counts(x[:ntr]), y[:ntr], PackedGenotypes.from_counts(x[ntr:]), y[ntr:]))
    return out


def _snapshot(m, h, xv):
    st = m.state()
    return {"history": h.history, "weights": m.get_weights(), "adam4": m.get_adam(4), "adam0": m.get_adam(0),
            "pred": m.predict(xv), "t": st.t, "last_loss": st.last_loss, "epoch": st.epoch}


def _assert_same(a, b):
    assert a["history"] == b["history"]
    assert a["t"] == b["t"] and a["last_loss"] == b["last_loss"] and a["epoch"] == b["epoch"]
    assert len(a["weights"]) == len(b["weights"])
    for i, (u, v) in enumerate(zip(a["weights"], b["weights"])):
        assert np.array_equal(u, v), f"weight {i}"
    for key in ("adam4", "adam0"):
        for u, v in zip(a[key], b[key]):
            assert np.array_equal(u, v), key
    assert np.array_equal(a["pred"], b["pred"])


def _solo_and_group(M, Ks, B, ntr, nva, epochs, seed0, l1_ctas=None, patience=100, epochs_per_call=16):
    rng = np.random.default_rng(seed0)
    datas = _datasets(rng, Ks, ntr, nva)
    solo = []
    for g, (x, y, xv, yv) in enumerate(datas):
        m = M.LocatorModel(Ks[g], batch_size=B, seed=seed0 + g, max_epochs=epochs, l1_ctas=l1_ctas)
        if m.impl != "tcgen05":
            pytest.skip("replicate groups need the tcgen05 kernels")
        h = m.fit(x, y, epochs=epochs, batch_size=B, validation_data=(xv, yv), patience=patience,
                  epochs_per_call=epochs_per_call)
        solo.append(_snapshot(m, h, xv))
        del m
    ms = [M.LocatorModel(Ks[g], batch_size=B, seed=seed0 + g, max_epochs=epochs, l1_ctas=l1_ctas) for g in range(len(Ks))]
    hs = M.fit_group(ms, [d[0] for d in datas], [d[1] for d in datas], [(d[2], d[3]) for d in datas], epochs=epochs,
                     patience=patience, epochs_per_call=epochs_per_call)
    group = [_snapshot(m, h, d[2]) for m, h, d in zip(ms, hs, datas)]
    return solo, group


@pytest.mark.parametrize("Ks,B,ntr,serial,ctas", [
    ([3001] * 4, 64, 300, False, False),          # 4 models x 2 chunks: 8 clusters in one hidden launch
    ([5000] * 3, 100, 250, False, False),         # ragged chunk, ragged last step, third model on a second launch
    ([4096] * 2, 256, 300, False, False),         # one model per launch
    ([20000] * 5, 33, 90, False, True),           # one-row chunk, odd group, several tiles per CTA, 24-row last step
    ([2500, 3001, 3500], 64, 300, False, False),  # models of different K, as windows produce
    ([3001] * 3, 96, 300, True, False),           # LOC_BB_SERIAL=1: one hidden launch per chunk
], ids=["K3001-B64-G4", "K5000-B100-G3", "K4096-B256-G2", "K20000-B33-G5", "mixedK-B64-G3", "serial-B96-G3"])
def test_group_equals_solo_bit_for_bit(M, monkeypatch, Ks, B, ntr, serial, ctas):
    if serial:
        monkeypatch.setenv("LOC_BB_SERIAL", "1")
    else:
        monkeypatch.delenv("LOC_BB_SERIAL", raising=False)
    solo, group = _solo_and_group(M, Ks, B, ntr, 40, 3, 100 + B, l1_ctas=M.spare_cluster_l1_ctas() if ctas else None)
    for s, g in zip(solo, group):
        assert s["t"] == 3 * -(-ntr // B)
        _assert_same(s, g)


def test_early_stopping_inside_a_group(M):
    """Patience 1: the models stop at different epochs; a stopped model's launches are no-ops while the others go on
    (and it leaves the group at the next call).  Each model still equals its solo run."""
    solo, group = _solo_and_group(M, [3001] * 4, 64, 200, 40, 16, 7, patience=1, epochs_per_call=4)
    stops = [s["epoch"] for s in solo]
    assert len(set(stops)) > 1 and max(stops) < 16, stops
    for s, g in zip(solo, group):
        _assert_same(s, g)


def test_grouped_launch_count(M):
    """One epoch of 4 models at 64 rows: the launches the grouped schedule implies, and fewer than four solo epochs."""
    from locator_b200 import _cabi

    G, K, B, ntr, nva = 4, 3001, 64, 300, 40
    rng = np.random.default_rng(3)
    datas = _datasets(rng, [K] * G, ntr, nva)
    m = M.LocatorModel(K, batch_size=B, seed=1, max_epochs=1)
    if m.impl != "tcgen05":
        pytest.skip("replicate groups need the tcgen05 kernels")
    torch.cuda.synchronize()
    l0 = _cabi.launch_count()
    m.fit(datas[0][0], datas[0][1], epochs=1, batch_size=B, validation_data=(datas[0][2], datas[0][3]))
    solo = _cabi.launch_count() - l0
    ms = [M.LocatorModel(K, batch_size=B, seed=1 + g, max_epochs=1) for g in range(G)]
    torch.cuda.synchronize()
    l0 = _cabi.launch_count()
    M.fit_group(ms, [d[0] for d in datas], [d[1] for d in datas], [(d[2], d[3]) for d in datas], epochs=1)
    group = _cabi.launch_count() - l0
    steps = -(-ntr // B)  # 64, 64, 64, 64, 44 rows: two 32-row chunks each
    chunks = 2
    per_step = (1                          # batch statistics of all models
                + G                        # wide first-layer forward per model
                + -(-G // (8 // chunks))   # hidden-stack launches, whole models of floor(8 / chunks)
                + 1                        # step end of all models
                + 2 * G                    # first-layer backward + gamma / beta per model
                + G)                       # small-layer update per model
    per_model = (1                         # set_schedule
                 + 1                       # begin of the call
                 + 3                       # validation: one wide pass of 40 rows (forward, hidden group, sums)
                 + 2)                      # epoch end + checkpoint
    assert group == steps * per_step + G * per_model, (group, solo)
    assert solo == steps * 7 + per_model
    assert group < G * solo


def test_group_of_mixed_batch_sizes_is_refused(M):
    from locator_b200._cabi import LocatorCudaError

    rng = np.random.default_rng(4)
    datas = _datasets(rng, [3001, 3001], 100, 20)
    ms = [M.LocatorModel(3001, batch_size=b, seed=5, max_epochs=1) for b in (32, 64)]
    if ms[0].impl != "tcgen05":
        pytest.skip("replicate groups need the tcgen05 kernels")
    with pytest.raises(LocatorCudaError):
        M.fit_group(ms, [d[0] for d in datas], [d[1] for d in datas], [(d[2], d[3]) for d in datas], epochs=1)


def _cli(tmp_path, tag, argv, G, capsys):
    from locator_b200 import locator as L

    d = tmp_path / f"{tag}{G}"
    d.mkdir()
    assert L.main(argv + ["--out", str(d / "r"), "--seed", "12345", "--max_epochs", "3", "--keras_verbose", "0",
                          "--replicates_per_gpu", str(G)]) == 0
    text = capsys.readouterr().out
    files = sorted(glob.glob(str(d / "*_predlocs.txt")) + glob.glob(str(d / "*_history.txt")))
    return text, {os.path.basename(f): open(f, "rb").read() for f in files}


def test_cli_bootstrap_large_batch_groups(M, tmp_path, capsys):
    argv = ["--vcf", VCF, "--sample_data", SAMPLES, "--bootstrap", "--nboots", "3", "--batch_size", "64"]
    t1, f1 = _cli(tmp_path, "b", argv, 1, capsys)
    t4, f4 = _cli(tmp_path, "b", argv, 4, capsys)
    assert "replicates side by side" in t4 and "replicates side by side" not in t1
    # one history file: every replicate writes <out>_history.txt in turn (locator.py), the last one stays
    assert sorted(f1) == sorted([f"r_boot{b}_predlocs.txt" for b in ("FULL", "0", "1", "2")] + ["r_history.txt"])
    assert f1 == f4


def test_cli_windows_large_batch_groups(M, tmp_path, capsys):
    from locator_b200 import io

    v = io.read_vcf(VCF)
    z = str(tmp_path / "fix.zarr")
    io.write_zarr(z, v["calldata/GT"], v["samples"], v["variants/POS"], chunk_variants=2000)
    argv = ["--zarr", z, "--sample_data", SAMPLES, "--windows", "--window_size", "1000000", "--batch_size", "96"]
    t1, f1 = _cli(tmp_path, "w", argv, 1, capsys)
    t4, f4 = _cli(tmp_path, "w", argv, 4, capsys)
    assert "replicates side by side" in t4
    assert len([f for f in f1 if f.endswith("_predlocs.txt")]) == 3  # three windows of different K
    assert f1 == f4
