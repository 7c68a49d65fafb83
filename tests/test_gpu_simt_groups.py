"""Replicate groups of CUDA-core models (widths other than 256, loc_group_train_epochs).

Up to 32 rows a step the group runs every model's first-layer forward, ONE k_hidden launch holding every model's hidden
stack (one cluster per model), the small-layer updates on side streams and the first-layer backwards back to back.
Above 32 rows (train_step_big) the chunks go one after another: every model's forward of chunk c, then chunk c of every
model in one k_hidden launch.  Every kernel of a model gets the arguments it gets alone, so each model must end
bit-identical to the same model trained alone with model.fit: histories, optimizer state, weights, Adam moments and
predictions.  Width 256 with 15..21 layers (tcgen05 first layer, CUDA-core hidden stack) is not grouped.
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


def cdiv(a, b):
    return -(-a // b)


def _datasets(rng, Ks, ntr, nva):
    from locator_b200.genotypes import PackedGenotypes

    out = []
    for K in Ks:
        p = rng.uniform(0.02, 0.98, size=K)
        x = rng.binomial(2, p, size=(ntr + nva, K)).astype(np.uint8)
        w = rng.normal(size=(K, 2)) / np.sqrt(K)
        y = ((x - 2 * p) @ w + 0.3 * rng.normal(size=(ntr + nva, 2))).astype(np.float32)  # some signal
        out.append((PackedGenotypes.from_counts(x[:ntr]), y[:ntr], PackedGenotypes.from_counts(x[ntr:]), y[ntr:]))
    return out


def _snapshot(m, h, xv):
    st = m.state()
    return {"history": h.history, "state": (st.t, st.epoch, st.stopped, st.best_epoch, st.es_wait, st.rlr_wait, st.lr,
                                            st.ckpt_best, st.last_loss, st.last_val_loss),
            "weights": m.get_weights(), "adam": [m.get_adam(i) for i in (0, 1, 4, 6)], "pred": m.predict(xv)}


def _assert_same(a, b):
    assert a["history"] == b["history"]
    assert a["state"] == b["state"]
    assert len(a["weights"]) == len(b["weights"])
    for i, (u, v) in enumerate(zip(a["weights"], b["weights"])):
        assert np.array_equal(u, v), f"weight {i}"
    for (mu, vu), (mv, vv) in zip(a["adam"], b["adam"]):
        assert np.array_equal(mu, mv) and np.array_equal(vu, vv)
    assert np.array_equal(a["pred"], b["pred"])


def _simt(m):
    assert (m.impl, m.hidden_impl) == ("simt", "simt"), (m.width, m.nlayers)


def _solo_and_group(M, Ks, H, L, B, ntr, nva, epochs, seed0, patience):
    rng = np.random.default_rng(seed0)
    datas = _datasets(rng, Ks, ntr, nva)
    solo = []
    for g, (x, y, xv, yv) in enumerate(datas):
        m = M.LocatorModel(Ks[g], width=H, nlayers=L, batch_size=B, seed=seed0 + g, max_epochs=epochs)
        _simt(m)
        h = m.fit(x, y, epochs=epochs, batch_size=B, validation_data=(xv, yv), patience=patience, epochs_per_call=4)
        solo.append(_snapshot(m, h, xv))
        del m
    ms = [M.LocatorModel(Ks[g], width=H, nlayers=L, batch_size=B, seed=seed0 + g, max_epochs=epochs)
          for g in range(len(Ks))]
    hs = M.fit_group(ms, [d[0] for d in datas], [d[1] for d in datas], [(d[2], d[3]) for d in datas], epochs=epochs,
                     patience=patience, epochs_per_call=4)
    return solo, [_snapshot(m, h, d[2]) for m, h, d in zip(ms, hs, datas)]


@pytest.mark.parametrize("H,L", [(128, 4), (224, 10)], ids=["w128-L4", "w224-L10"])
def test_lockstep_group_equals_solo(M, H, L):
    """G = 3 at 32 rows a step, models of different K (as windows produce).  Width 128 runs 16-CTA clusters; width 224
    x 10 runs 8-CTA clusters with fewer weight slots than uses (the slice ring wraps).  Patience 1: the models stop at
    different epochs, and a stopped model's launches are no-ops while the others go on (it leaves the group at the next
    call of four epochs)."""
    epochs = 12
    solo, group = _solo_and_group(M, [3001, 2500, 3500], H, L, 32, 150, 40, epochs, 300 + H, patience=1)
    stops = [s["state"][1] for s in solo]
    assert len(set(stops)) > 1 and min(stops) < epochs, stops
    for s, g in zip(solo, group):
        _assert_same(s, g)


def test_lockstep_group_full_run_equals_solo(M):
    """The same without early stopping: every epoch of every model runs inside the group."""
    solo, group = _solo_and_group(M, [4000] * 3, 128, 4, 32, 150, 40, 4, 77, patience=100)
    for s, g in zip(solo, group):
        assert s["state"][1] == 4 and s["state"][0] == 4 * cdiv(150, 32)
        _assert_same(s, g)


@pytest.mark.parametrize("serial", [False, True], ids=["lockstep", "serial"])
@pytest.mark.parametrize("B,ntr", [(64, 270), (100, 250)], ids=["B64", "B100"])
def test_large_batch_group_equals_solo(M, monkeypatch, B, ntr, serial):
    """Width 64 x 4 above 32 rows a step: 64 rows (two chunks, a one-chunk last step of 14 rows) and 100 rows (a
    4-row last chunk, a 50-row last step); chunk by chunk in one launch per chunk (lockstep) or one launch per chunk
    and model (LOC_BB_SERIAL=1)."""
    if serial:
        monkeypatch.setenv("LOC_BB_SERIAL", "1")
    else:
        monkeypatch.delenv("LOC_BB_SERIAL", raising=False)
    solo, group = _solo_and_group(M, [3001, 3001, 2600], 64, 4, B, ntr, 40, 3, 500 + B, patience=100)
    for s, g in zip(solo, group):
        assert s["state"][0] == 3 * cdiv(ntr, B)
        _assert_same(s, g)


# launch counts (the `loc` launch counter, as in tests/test_gpu_schedules.py)
K, NVA, E = 3001, 40, 2
VAL_NARROW = 2 * cdiv(NVA, 32)  # per 32 validation rows: forward, hidden stack
EPOCH_END = 2                   # epoch end + checkpoint copy


def _launches(fn):
    from locator_b200 import _cabi

    torch.cuda.synchronize()
    l0 = _cabi.launch_count()
    fn()
    torch.cuda.synchronize()
    return _cabi.launch_count() - l0


def _fit(m, d, B):
    return _launches(lambda: m.fit(d[0], d[1], epochs=E, batch_size=B, validation_data=(d[2], d[3])))


def _fit_group(M, ms, ds):
    return _launches(lambda: M.fit_group(ms, [d[0] for d in ds], [d[1] for d in ds], [(d[2], d[3]) for d in ds], epochs=E))


def test_lockstep_launch_count(M):
    """G = 3 at 32 rows: per step every model's forward, ONE hidden-stack launch, an update and a backward per model."""
    G, ntr = 3, 200
    steps = cdiv(ntr, 32)
    ds = _datasets(np.random.default_rng(40), [K] * G, ntr, NVA)
    m = M.LocatorModel(K, width=128, nlayers=4, seed=1, max_epochs=E)
    _simt(m)
    assert _fit(m, ds[0], 32) == 2 + E * (4 * steps + VAL_NARROW + EPOCH_END)  # set_schedule, begin of the call
    ms = [M.LocatorModel(K, width=128, nlayers=4, seed=1 + g, max_epochs=E) for g in range(G)]
    per_step = G + 1 + 2 * G
    assert _fit_group(M, ms, ds) == 2 * G + E * (steps * per_step + G * (VAL_NARROW + EPOCH_END))


@pytest.mark.parametrize("serial", [False, True], ids=["lockstep", "serial"])
def test_large_batch_launch_count(M, monkeypatch, serial):
    """G = 2 at 64 rows: one hidden-stack launch per chunk for the whole group (LOC_BB_SERIAL=1: per chunk and model)."""
    G, B, ntr = 2, 64, 270
    chunks = [cdiv(min(B, ntr - off), 32) for off in range(0, ntr, B)]  # 2, 2, 2, 2, 1
    if serial:
        monkeypatch.setenv("LOC_BB_SERIAL", "1")
    else:
        monkeypatch.delenv("LOC_BB_SERIAL", raising=False)
    ds = _datasets(np.random.default_rng(41), [K] * G, ntr, NVA)

    def step(nc, n):
        hidden = n * nc if (serial or n == 1) else nc
        return (1             # batch statistics of all models
                + n * nc      # first-layer forward per chunk and model
                + hidden
                + 2 * n       # first-layer backward + gamma / beta per model
                + n)          # small-layer update per model

    m = M.LocatorModel(K, width=64, nlayers=4, batch_size=B, seed=1, max_epochs=E)
    _simt(m)
    assert _fit(m, ds[0], B) == 2 + E * (sum(step(nc, 1) for nc in chunks) + VAL_NARROW + EPOCH_END)
    ms = [M.LocatorModel(K, width=64, nlayers=4, batch_size=B, seed=1 + g, max_epochs=E) for g in range(G)]
    assert _fit_group(M, ms, ds) == 2 * G + E * (sum(step(nc, G) for nc in chunks) + G * (VAL_NARROW + EPOCH_END))


def _cli(tmp_path, tag, argv, G, capsys):
    from locator_b200 import locator as L

    d = tmp_path / f"{tag}{G}"
    d.mkdir()
    assert L.main(argv + ["--out", str(d / "r"), "--seed", "12345", "--max_epochs", "3", "--keras_verbose", "0",
                          "--width", "128", "--nlayers", "4", "--replicates_per_gpu", str(G)]) == 0
    text = capsys.readouterr().out
    files = sorted(glob.glob(str(d / "*_predlocs.txt")) + glob.glob(str(d / "*_history.txt")))
    return text, {os.path.basename(f): open(f, "rb").read() for f in files}


def test_cli_bootstrap_width_128_groups(M, tmp_path, capsys):
    argv = ["--vcf", VCF, "--sample_data", SAMPLES, "--bootstrap", "--nboots", "3"]
    t1, f1 = _cli(tmp_path, "b", argv, 1, capsys)
    t4, f4 = _cli(tmp_path, "b", argv, 4, capsys)
    assert "replicates side by side" in t4 and "replicates side by side" not in t1
    assert sorted(f1) == sorted([f"r_boot{b}_predlocs.txt" for b in ("FULL", "0", "1", "2")] + ["r_history.txt"])
    assert f1 == f4


def test_cli_windows_width_128_groups(M, tmp_path, capsys):
    from locator_b200 import io

    v = io.read_vcf(VCF)
    z = str(tmp_path / "fix.zarr")
    io.write_zarr(z, v["calldata/GT"], v["samples"], v["variants/POS"], chunk_variants=2000)
    argv = ["--zarr", z, "--sample_data", SAMPLES, "--windows", "--window_size", "1000000"]
    t1, f1 = _cli(tmp_path, "w", argv, 1, capsys)
    t4, f4 = _cli(tmp_path, "w", argv, 4, capsys)
    assert "replicates side by side" in t4 and "replicates side by side" not in t1
    assert len([f for f in f1 if f.endswith("_predlocs.txt")]) == 3  # three windows of different K
    assert f1 == f4


@pytest.mark.parametrize("shapes,match", [
    ([(128, 4), (64, 4)], "share width"),
    ([(256, 16), (256, 16)], "different kernel families"),
    ([(128, 16), (256, 16)], "different kernel families"),
    ([(256, 4), (128, 4)], "all run the tcgen05 kernels"),
], ids=["two-widths", "mixed-family", "cuda-core-and-mixed", "tcgen05-and-cuda-core"])
def test_refused_groups(M, shapes, match):
    from locator_b200._cabi import LocatorCudaError

    datas = _datasets(np.random.default_rng(6), [3001] * len(shapes), 64, 20)
    ms = [M.LocatorModel(3001, width=h, nlayers=nl, seed=5 + g, max_epochs=1) for g, (h, nl) in enumerate(shapes)]
    with pytest.raises(LocatorCudaError, match=match) as e:
        M.fit_group(ms, [d[0] for d in datas], [d[1] for d in datas], [(d[2], d[3]) for d in datas], epochs=1)
    assert "loc_group_train_epochs" in str(e.value)
