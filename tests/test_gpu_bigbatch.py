"""GPU parity for --batch_size > 32 (locator/locator.py:69,371: any batch size goes to model.fit).

Steps of 33..256 rows run as batch statistics over the whole step -> first-layer forward with those statistics ->
32-row chunks through the hidden stack -> one first-layer backward + Adam over all rows -> one small-layer update
(csrc/bigbatch.cu).  Compared with the CPU oracle (oracle/model_ref.py handles any batch size) on the same rows,
weights and dropout masks.

Tolerances: as tests/test_gpu_model.py -- tf32 products in the forward and the hidden stack on the tcgen05 path
(loss 2e-3 relative), plain fp32 on the CUDA-core path (1e-4), and the fp32 bounds against the oracle's "tf32_l1" mode
for the tcgen05 first layer behind a CUDA-core hidden stack; the first-layer gradient of a large step is fp32 on all
of them; moving statistics derive from integer counts (1e-5).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def M():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from locator_b200 import model

    return model


def _data(rng, n, K):
    p = rng.uniform(0.02, 0.98, size=K)
    x = rng.binomial(2, p, size=(n, K)).astype(np.uint8)
    x[:, ::97] = 0  # SNPs that are constant in every batch: dgamma must be exactly 0 there
    y = rng.normal(size=(n, 2)).astype(np.float32)
    return x, y


def _numerics(m):
    """The oracle mode of the model's kernel families (first layer, hidden stack)."""
    if m.impl != "tcgen05":
        return "fp32"
    return "tf32" if m.hidden_impl == "tcgen05" else "tf32_l1"


def _compare_updates(m, ref, w0, tc):
    w1 = m.get_weights()
    r1 = ref.get_weights()
    names = ["gamma", "beta", "mmean", "mvar"] + [f"dense{i // 2}.{'b' if i % 2 else 'W'}" for i in range(len(w1) - 4)]
    for name, a0, a, b in zip(names, w0, w1, r1):
        da, db = a - a0, b - a0
        scale = max(np.abs(db).max(), 1e-6)
        err = np.abs(da - db)
        frac_bad = float((err > 0.05 * scale + 1e-7).mean())
        assert frac_bad < (0.02 if tc else 0.005), (name, frac_bad, float(err.max()), float(scale))
    np.testing.assert_allclose(w1[2], r1[2], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(w1[3], r1[3], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("K,H,L,p,B,sizes", [
    (1000, 64, 4, 0.25, 64, [64, 64, 40]),       # CUDA-core kernels, two chunks, ragged last step
    (3001, 256, 10, 0.25, 96, [96, 96, 70, 33]),  # tcgen05 forward / hidden stack, three chunks
    (777, 128, 3, 0.0, 256, [256, 200]),         # eight chunks
    (4096, 256, 10, 0.25, 250, [250, 250, 17]),  # ragged chunk inside a step; a last step of fewer than 32 rows
    (200, 32, 2, 0.5, 33, [33, 33]),             # one row in the second chunk
    # tcgen05 first layer + CUDA-core hidden stack: no wide forward, every chunk's first-layer forward reads the
    # step's batch statistics
    (3001, 256, 15, 0.25, 96, [96, 70, 33]),
    (1200, 224, 10, 0.5, 64, [64, 40]),          # CUDA-core stack with one weight slice in shared memory
])
def test_large_batch_steps_match_oracle(M, K, H, L, p, B, sizes):
    from oracle import model_ref

    rng = np.random.default_rng(K * 7 + B)
    n = 300
    x, y = _data(rng, n, K)
    m = M.LocatorModel(K, width=H, nlayers=L, dropout_prop=p, batch_size=B, seed=11)
    tc = _numerics(m) == "tf32"  # tf32 products in the hidden stack; the mixed family is held to the fp32 bounds
    w0 = m.get_weights()
    w0[1] = rng.normal(0, 0.05, K).astype(np.float32)  # beta != 0: the beta * c0 term of dW1 is exercised
    m.set_weights(w0)
    # tcgen05 path: the oracle's tf32 operand model (DESIGN.md section 2) -- against plain fp32 the third step of the
    # (4096, 250) case is already 0.8 % off (two sign-like Adam steps amplify the tf32 rounding of the forward);
    # "tf32_l1" behind a CUDA-core hidden stack
    ref = model_ref.RefLocator(K, H, L, dropout=p, weights=w0, numerics=_numerics(m))
    masks = (rng.uniform(size=(len(sizes), B, H)) >= p).astype(np.uint8)
    m.set_dropout_masks(masks)
    m.bind_train(x, y)
    m.set_schedule(patience=100)
    rtol = 2e-3 if tc else 1e-4
    for s, nb in enumerate(sizes):
        rows = rng.permutation(n)[:nb]
        m.train_step(rows)
        st = m.state()
        loss_ref = ref.train_step(x[rows], y[rows], masks[s][:nb])
        assert st.t == s + 1
        np.testing.assert_allclose(st.last_loss, loss_ref, rtol=rtol, err_msg=f"step {s} ({nb} rows)")
        if s == 0:
            # first step: Adam's m = 0.1 * gradient -- the gradient itself, before Adam's sign-like normalisation
            mW, vW = m.get_adam(4)
            gm = ref.m[2].numpy()
            np.testing.assert_allclose(mW, gm, rtol=0.02, atol=(6e-3 if tc else 2e-4) * float(np.abs(gm).max()))
            mg, _ = m.get_adam(0)
            gg = ref.m[0].numpy()
            np.testing.assert_allclose(mg, gg, rtol=0.02, atol=(6e-3 if tc else 2e-4) * float(np.abs(gg).max()))
            assert np.all(mg[::97] == 0.0)  # constant SNPs: exactly zero, as in Keras
            mb, _ = m.get_adam(1)
            gb = ref.m[1].numpy()
            np.testing.assert_allclose(mb, gb, rtol=0.02, atol=(6e-3 if tc else 2e-4) * float(np.abs(gb).max()))
    _compare_updates(m, ref, w0, tc)
    # predictions after training (inference path is the same for every batch size)
    yp, yr = m.predict(x[:50]), ref.predict(x[:50])
    np.testing.assert_allclose(yp, yr, atol=6e-2 if tc else 2e-3)


def test_large_batch_philox_dropout_matches_oracle(M):
    """No injected masks: the device's Philox stream is indexed by the row's position in the whole step."""
    from oracle import model_ref, philox_ref

    K, H, L, p, B = 900, 64, 4, 0.25, 80
    rng = np.random.default_rng(5)
    x, y = _data(rng, 200, K)
    m = M.LocatorModel(K, width=H, nlayers=L, dropout_prop=p, batch_size=B, seed=99)
    w0 = m.get_weights()
    ref = model_ref.RefLocator(K, H, L, dropout=p, weights=w0)
    m.bind_train(x, y)
    m.set_schedule(patience=100)
    for s in range(3):
        rows = rng.permutation(200)[:B]
        m.train_step(rows)
        mk = philox_ref.dropout_keep(B, H, p, 99, s)
        loss_ref = ref.train_step(x[rows], y[rows], mk)
        np.testing.assert_allclose(m.state().last_loss, loss_ref, rtol=1e-4)


def test_chunks_side_by_side_equal_chunks_in_sequence(M, monkeypatch):
    """tcgen05 path: the chunks of a step share one grouped hidden-stack launch; LOC_BB_SERIAL=1 launches them one
    after the other.  Same bits in every weight, loss and counter."""
    K, H, L, B = 5000, 256, 10, 200
    rng = np.random.default_rng(8)
    x, y = _data(rng, 400, K)
    perms = np.stack([rng.permutation(400) for _ in range(2)]).astype(np.int32)
    outs = []
    for serial in (False, True):
        if serial:
            monkeypatch.setenv("LOC_BB_SERIAL", "1")
        else:
            monkeypatch.delenv("LOC_BB_SERIAL", raising=False)
        m = M.LocatorModel(K, width=H, nlayers=L, dropout_prop=0.25, batch_size=B, max_epochs=2, seed=21)
        if m.impl != "tcgen05":
            pytest.skip("needs the tcgen05 kernels")
        h = m.fit(x[:360], y[:360], epochs=2, batch_size=B, validation_data=(x[360:], y[360:]), perms=perms)
        st = m.state()
        outs.append((m.get_weights(), h.history, st.t, st.last_loss))
    (w_a, h_a, t_a, l_a), (w_b, h_b, t_b, l_b) = outs
    assert t_a == t_b == 4 and l_a == l_b and h_a == h_b
    for a, b in zip(w_a, w_b):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("K,H,L,B", [(1500, 64, 4, 64), (5830, 256, 10, 128)])
def test_large_batch_fit_matches_oracle(M, K, H, L, B):
    """model.fit at a large batch size: epoch losses, validation losses, callbacks and the restored best weights."""
    from oracle import model_ref

    rng = np.random.default_rng(K + B)
    n, nv, epochs = 300, 45, 3
    x, y = _data(rng, n, K)
    xv, yv = _data(rng, nv, K)
    m = M.LocatorModel(K, width=H, nlayers=L, dropout_prop=0.25, batch_size=B, max_epochs=epochs, seed=3)
    tc = _numerics(m) == "tf32"
    w0 = m.get_weights()
    ref = model_ref.RefLocator(K, H, L, dropout=0.25, weights=w0, numerics=_numerics(m))
    spe = -(-n // B)
    masks = (rng.uniform(size=(epochs * spe, B, H)) >= 0.25).astype(np.uint8)
    m.set_dropout_masks(masks)
    perms = np.stack([rng.permutation(n) for _ in range(epochs)]).astype(np.int32)
    h = m.fit(x, y, epochs=epochs, batch_size=B, validation_data=(xv, yv), patience=10, perms=perms)
    hr = model_ref.fit(ref, x, y, xv, yv, epochs, batch_size=B, patience=10, perms=perms,
                       masks=lambda step, nb: masks[step][:nb])
    # epoch 1 before trajectories separate (Adam amplifies tf32 rounding, see DESIGN.md section 2)
    np.testing.assert_allclose(h.history["loss"][0], hr["loss"][0], rtol=3e-3 if tc else 2e-4)
    np.testing.assert_allclose(h.history["val_loss"][0], hr["val_loss"][0], rtol=3e-2 if tc else 1e-3)
    np.testing.assert_allclose(h.history["loss"], hr["loss"], rtol=5e-2 if tc else 2e-3)
    np.testing.assert_allclose(h.history["val_loss"], hr["val_loss"], rtol=8e-2 if tc else 5e-3)
    assert h.history["learning_rate"] == pytest.approx(hr["learning_rate"])
    assert m.state().t == epochs * spe


def test_large_batch_cli_runs(M, tmp_path, capsys):
    """The command line with --batch_size 64 on the reference's fixture (locator.py:69,371), plain run and a bootstrap
    run (replicates of a large-batch run train one after the other, not in groups)."""
    import os

    from locator_b200 import locator as L

    here = os.path.dirname(os.path.abspath(__file__))
    vcf = os.path.join(here, "golden", "data", "test_genotypes.vcf.gz")
    sd = os.path.join(here, "golden", "data", "test_sample_data.txt")
    out = str(tmp_path / "bb")
    assert L.main(["--vcf", vcf, "--sample_data", sd, "--out", out, "--batch_size", "64", "--max_epochs", "60",
                   "--patience", "20", "--seed", "12345", "--keras_verbose", "0"]) == 0
    text = capsys.readouterr().out
    lines = open(out + "_predlocs.txt").read().strip().split("\n")
    assert lines[0] == "x,y,sampleID" and len(lines) == 51
    xy = np.array([[float(v) for v in ln.split(",")[:2]] for ln in lines[1:]])
    assert np.all(np.isfinite(xy)) and xy.min() > -20 and xy.max() < 70
    hist = open(out + "_history.txt").read().strip().split("\n")
    h = np.array([[float(v) for v in ln.split("\t")] for ln in hist[1:]])
    assert np.all(np.isfinite(h)) and h[-1, 1] < h[0, 1] * 0.6  # validation loss fell
    med = float(text.split("median validation error ")[1].split()[0])
    assert med < 8.0, med  # 60 epochs at batch 64 on the 50 x 50 landscape (the default run reaches ~3)
    out2 = str(tmp_path / "bs")
    assert L.main(["--vcf", vcf, "--sample_data", sd, "--out", out2, "--batch_size", "100", "--max_epochs", "3",
                   "--seed", "12345", "--keras_verbose", "0", "--bootstrap", "--nboots", "2"]) == 0
    for b in ("FULL", "0", "1"):
        assert len(open(f"{out2}_boot{b}_predlocs.txt").read().strip().split("\n")) == 51
