"""Deep and wide models: the shapes that run off the default 256 x 10.

Every model needs the CUDA-core hidden stack's shared-memory layout to hold at least one weight slice
(csrc/hidden.cu: hidden_slots); loc_hidden_max_nlayers(width) states the deepest nlayers that does, and validate_args
refuses deeper ones before any data is read.  Width-256 models deeper than the tcgen05 hidden stack holds (14 layers)
run the tcgen05 first layer with the CUDA-core hidden stack behind it -- the mixed family, compared here with the
oracle's "tf32_l1" mode -- and train one replicate after the other instead of in replicate groups.
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


def test_envelope_of_buildable_shapes(M):
    """For every width the CLI accepts, the deepest nlayers the host query names builds on the device, one layer
    deeper does not; a width the query rules out does not build at all."""
    from locator_b200._cabi import LocatorCudaError, lib

    deepest = {w: int(lib.loc_hidden_max_nlayers(w)) for w in range(32, 1025, 32)}
    assert deepest[256] == 21 and deepest[32] == deepest[64] == deepest[128] == 64
    for w, d in deepest.items():
        if d > 0:
            m = M.LocatorModel(100, width=w, nlayers=d, seed=1)
            assert m.hidden_impl == "simt", (w, d)
            del m
        if d < 64:
            with pytest.raises(LocatorCudaError, match="cluster"):
                M.LocatorModel(100, width=w, nlayers=max(d + 1, 2), seed=1)
    m14 = M.LocatorModel(100, width=256, nlayers=14, seed=1)
    m15 = M.LocatorModel(100, width=256, nlayers=15, seed=1)
    assert (m14.impl, m14.hidden_impl) == ("tcgen05", "tcgen05")
    assert (m15.impl, m15.hidden_impl) == ("tcgen05", "simt")


def _data(rng, n, K):
    p = rng.uniform(0.02, 0.98, size=K)
    x = rng.binomial(2, p, size=(n, K)).astype(np.uint8)
    w = rng.normal(size=(K, 2)) / np.sqrt(K)
    y = ((x - 2 * p) @ w + 0.3 * rng.normal(size=(n, 2))).astype(np.float32)  # some signal: validation loss falls
    return x, y


def test_mixed_family_fit_and_restore_best(M):
    """fit at 256 x 16 (tcgen05 first layer, whose backward also runs the next step's forward, feeding the CUDA-core
    stack at cluster 16) against the oracle's "tf32_l1" mode; then restore_best (hidden_reslice of the best weights)
    against the same weights uploaded through set_weights."""
    from oracle import model_ref

    rng = np.random.default_rng(16)
    K, H, L, p = 3000, 256, 16, 0.25
    ntr, nva, epochs = 75, 20, 3
    x, y = _data(rng, ntr + nva, K)
    x, y, xv, yv = x[:ntr], y[:ntr], x[ntr:], y[ntr:]
    m = M.LocatorModel(K, width=H, nlayers=L, dropout_prop=p, seed=8, max_epochs=epochs)
    assert (m.impl, m.hidden_impl) == ("tcgen05", "simt")
    w0 = m.get_weights()
    spe = -(-ntr // 32)
    masks = (rng.uniform(size=(epochs * spe, 32, H)) >= p).astype(np.uint8)
    m.set_dropout_masks(masks)
    perms = np.stack([rng.permutation(ntr) for _ in range(epochs)])
    h = m.fit(x, y, epochs=epochs, validation_data=(xv, yv), patience=100, perms=perms)
    # the oracle family: the same products with the first layer's sum over SNPs cut into 1, 8 and 47 (the device's
    # CTA count at K = 3000: one 64-SNP tile each) parts -- trajectories may separate by that much after epoch 1
    fam, refs = [], []
    for parts in (47, 8, 1):
        refs.append(model_ref.RefLocator(K, H, L, dropout=p, weights=[w.copy() for w in w0], numerics="tf32_l1",
                                         l1_parts=parts))
        fam.append(model_ref.fit(refs[-1], x, y, xv, yv, epochs, batch_size=32, patience=100, perms=perms,
                                 masks=lambda step, nb: masks[step][:nb]))
    hr = fam[0]
    assert len(h.history["loss"]) == epochs
    # epoch 1 at the per-step loss tolerance of the family (tests/test_gpu_model.py)
    np.testing.assert_allclose(h.history["loss"][0], hr["loss"][0], rtol=1e-4)
    np.testing.assert_allclose(h.history["val_loss"][0], hr["val_loss"][0], rtol=1e-4)
    for key in ("loss", "val_loss"):
        f = np.array([r[key] for r in fam])
        lo, hi = f.min(axis=0), f.max(axis=0)
        spread = hi - lo
        for e in range(1, epochs):
            v = h.history[key][e]
            assert lo[e] - 1.5 * spread[e] - 0.03 * lo[e] <= v <= hi[e] + 1.5 * spread[e] + 0.03 * hi[e], (key, e, h.history, f)
    assert h.history["learning_rate"] == pytest.approx(hr["learning_rate"])
    m.restore_best()
    st = m.state()
    assert st.best_epoch == int(np.argmin(hr["val_loss"]))
    yp = m.predict(xv)
    np.testing.assert_allclose(yp, refs[0].predict(xv), rtol=0.02, atol=0.02)  # the oracle's restored best weights
    fresh = M.LocatorModel(K, width=H, nlayers=L, dropout_prop=p, seed=9, max_epochs=epochs)
    fresh.set_weights(m.get_weights())
    assert np.array_equal(fresh.predict(xv), yp)
    assert np.array_equal(fresh.predict(x), m.predict(x))


def _cli(tmp_path, argv, G, capsys):
    from locator_b200 import locator as L

    d = tmp_path / f"r{G}"
    d.mkdir()
    assert L.main(argv + ["--out", str(d / "r"), "--seed", "12345", "--keras_verbose", "0",
                          "--replicates_per_gpu", str(G)]) == 0
    text = capsys.readouterr().out
    files = sorted(glob.glob(str(d / "*_predlocs.txt")) + glob.glob(str(d / "*_history.txt")))
    return text, {os.path.basename(f): open(f, "rb").read() for f in files}


def test_cli_bootstrap_deep_width_256(M, tmp_path, capsys):
    """--nlayers 16 at the default width: the replicates run the CUDA-core hidden stack, so they train one after the
    other whatever --replicates_per_gpu says (replicate groups need the tcgen05 hidden stack) -- same bytes."""
    argv = ["--vcf", VCF, "--sample_data", SAMPLES, "--bootstrap", "--nboots", "2", "--nlayers", "16", "--max_epochs", "2"]
    t1, f1 = _cli(tmp_path, argv, 1, capsys)
    t4, f4 = _cli(tmp_path, argv, 4, capsys)
    assert "replicates side by side" not in t1 + t4
    assert sorted(f1) == sorted([f"r_boot{b}_predlocs.txt" for b in ("FULL", "0", "1")] + ["r_history.txt"])
    assert f1 == f4
