"""GPU parity: the CUDA training / prediction path (through the C ABI) vs the CPU oracle.

Tolerances, by the model's kernel families (m.impl = first layer, m.hidden_impl = hidden stack; _family):
  CUDA cores throughout (widths other than 256): plain fp32, differences = summation order only -- against the
      fp32 oracle: forward / predict |dy| <= 3e-5 + 2e-4 |y|, per-step loss rel 1e-4, updates 0.5 % off;
  tcgen05 first layer + tcgen05 hidden stack (width 256, nlayers <= 14): TF32 products (10-bit mantissa, as
      TensorFlow does by default on Ampere+ GPUs), fp32 accumulate -- against the oracle's "tf32" mode:
      |dy| <= 2e-3 (1 + |y|), loss rel 2e-3, updates 2 % off;
  tcgen05 first layer + CUDA-core hidden stack (width 256, nlayers 15..21): against the oracle's "tf32_l1" mode
      (first layer rounded as on the device, hidden and output products fp32) the same bounds as plain fp32 --
      what is left is the summation order of the first layer.  Measured on a B200 (1000 W power limit) at 256 x 15
      and 256 x 21: |dy| 5.0e-6, evaluate 2.6e-7 relative, per-step loss 2.5e-6 relative, no disagreeing updates,
      Adam moments of W1 within 1.2e-5 of their largest value.
Weights after N steps are compared through the *update* (w - w0), whose scale is lr = 1e-3.
"""
import os

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


# (m.impl, m.hidden_impl) -> oracle numerics, forward atol / rtol, loss rtol, largest fraction of disagreeing updates,
# Adam-moment atol (relative to the largest moment)
FAMILIES = {
    ("simt", "simt"): dict(numerics="fp32", atol=3e-5, rtol=2e-4, loss=1e-4, frac=0.005, moments=2e-3),
    ("tcgen05", "tcgen05"): dict(numerics="tf32", atol=2e-3, rtol=2e-3, loss=2e-3, frac=0.02, moments=6e-3),
    ("tcgen05", "simt"): dict(numerics="tf32_l1", atol=3e-5, rtol=2e-4, loss=1e-4, frac=0.005, moments=2e-3),
}


def _family(m):
    return FAMILIES[(m.impl, m.hidden_impl)]


def _data(rng, n, K):
    p = rng.uniform(0.02, 0.98, size=K)
    x = rng.binomial(2, p, size=(n, K)).astype(np.uint8)
    y = rng.normal(size=(n, 2)).astype(np.float32)
    return x, y


def _masks(rng, nsteps, H, p):
    return (rng.uniform(size=(nsteps, 32, H)) >= p).astype(np.uint8)


def test_init_matches_oracle_philox(M):
    from oracle import model_ref

    K, H, L = 1000, 64, 4
    m = M.LocatorModel(K, width=H, nlayers=L, seed=1234)
    ws = m.get_weights()
    ref = model_ref.init_weights(K, H, L, seed=1234)
    assert len(ws) == len(ref) == 4 + 2 * (L + 2)
    for a, b in zip(ws, ref):
        assert a.shape == b.shape
        assert np.array_equal(a, b)  # same Philox stream, same fp32 arithmetic


@pytest.mark.parametrize("K,H,L,n", [
    (1000, 64, 4, 70), (5830, 256, 10, 45), (777, 128, 3, 33), (40, 32, 2, 5),
    (2003, 256, 13, 33), (1500, 256, 14, 70),   # tcgen05 stack: odd depth, deepest that fits its shared memory
    (3001, 256, 15, 64), (999, 256, 21, 41),    # tcgen05 first layer + CUDA-core stack: shallowest, deepest
    # CUDA-core stacks with one weight slice in shared memory (the slice ring streams every use), deepest per width
    (1200, 224, 10, 57), (800, 320, 13, 38), (640, 288, 2, 66), (500, 96, 54, 35), (450, 384, 2, 47),
])
def test_predict_and_evaluate_match_oracle(M, K, H, L, n):
    from oracle import model_ref

    rng = np.random.default_rng(K + H)
    x, y = _data(rng, n, K)
    m = M.LocatorModel(K, width=H, nlayers=L, seed=7)
    ws = m.get_weights()
    # non-trivial BN state and biases
    ws[0] = rng.uniform(0.5, 1.5, K).astype(np.float32)
    ws[1] = rng.normal(0, 0.1, K).astype(np.float32)
    ws[2] = rng.uniform(0, 1.5, K).astype(np.float32)
    ws[3] = rng.uniform(0.1, 0.8, K).astype(np.float32)
    for i in range(5, len(ws), 2):
        ws[i] = rng.normal(0, 0.05, ws[i].shape).astype(np.float32)
    m.set_weights(ws)
    got = m.get_weights()
    for a, b in zip(got, ws):
        assert np.array_equal(a, b)
    fam = _family(m)
    ref = model_ref.RefLocator(K, H, L, weights=ws, numerics=fam["numerics"])
    atol, rtol = fam["atol"], fam["rtol"]
    yp = m.predict(x)
    yr = ref.predict(x)
    assert yp.shape == (n, 2)
    np.testing.assert_allclose(yp, yr, rtol=rtol, atol=atol)
    ev = m.evaluate(x, y)
    np.testing.assert_allclose(ev, ref.evaluate(x, y), rtol=rtol)


@pytest.mark.parametrize("K,H,L,p,nsteps", [
    (1000, 64, 4, 0.25, 6), (3001, 256, 10, 0.25, 4), (500, 128, 5, 0.0, 5), (200, 32, 2, 0.5, 3),
    (2003, 256, 13, 0.5, 4), (1500, 256, 14, 0.25, 4), (3001, 256, 15, 0.5, 4), (999, 256, 21, 0.25, 3),
    (1200, 224, 10, 0.5, 4), (800, 320, 13, 0.25, 3), (640, 288, 2, 0.5, 4), (500, 96, 54, 0.25, 3),
    (450, 384, 2, 0.5, 3),
])
def test_train_steps_match_oracle(M, K, H, L, p, nsteps):
    from oracle import model_ref

    rng = np.random.default_rng(K * 3 + L)
    n = 100
    x, y = _data(rng, n, K)
    m = M.LocatorModel(K, width=H, nlayers=L, dropout_prop=p, seed=11)
    fam = _family(m)
    w0 = m.get_weights()
    ref = model_ref.RefLocator(K, H, L, dropout=p, weights=w0, numerics=fam["numerics"])
    masks = _masks(rng, nsteps, H, p)
    m.set_dropout_masks(masks)
    m.bind_train(x, y)
    m.set_schedule(patience=100)
    sizes = [32] * nsteps
    sizes[-1] = 21  # a partial last batch uses its own statistics
    for s in range(nsteps):
        rows = rng.permutation(n)[: sizes[s]]
        m.train_step(rows)
        st = m.state()
        loss_ref = ref.train_step(x[rows], y[rows], masks[s][: sizes[s]])
        assert st.t == s + 1
        np.testing.assert_allclose(st.last_loss, loss_ref, rtol=fam["loss"])
    w1 = m.get_weights()
    r1 = ref.get_weights()
    names = ["gamma", "beta", "mmean", "mvar"] + [f"dense{i // 2}.{'b' if i % 2 else 'W'}" for i in range(len(w1) - 4)]
    for name, a0, a, b in zip(names, w0, w1, r1):
        da, db = a - a0, b - a0
        scale = max(np.abs(db).max(), 1e-6)
        # Adam steps are ~lr in size whatever the gradient scale; sign flips of tiny gradients aside,
        # the bulk of the update must agree
        err = np.abs(da - db)
        frac_bad = float((err > 0.05 * scale + 1e-7).mean())
        assert frac_bad < fam["frac"], (name, frac_bad, float(err.max()), float(scale))
    # Adam moments of the first layer against the oracle
    mW, vW = m.get_adam(4)
    idx = 2  # trainable(): gamma, beta, W1, ...
    am = fam["moments"]
    np.testing.assert_allclose(mW, ref.m[idx].numpy(), rtol=0.02, atol=am * float(np.abs(ref.m[idx].numpy()).max()))
    np.testing.assert_allclose(vW, ref.v[idx].numpy(), rtol=0.05, atol=am * float(np.abs(ref.v[idx].numpy()).max()))
    # moving statistics are exact integer-derived quantities
    np.testing.assert_allclose(w1[2], r1[2], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(w1[3], r1[3], rtol=1e-5, atol=1e-6)


def test_fit_history_matches_oracle(M):
    """Whole fit loop: shuffled batches, validation pass, callbacks, reload of the best epoch."""
    from oracle import model_ref

    rng = np.random.default_rng(99)
    K, H, L, p = 600, 64, 4, 0.25
    ntr, nva, epochs = 75, 20, 6
    x, y = _data(rng, ntr, K)
    xv, yv = _data(rng, nva, K)
    m = M.LocatorModel(K, width=H, nlayers=L, dropout_prop=p, seed=5, max_epochs=epochs)
    w0 = m.get_weights()
    perms = np.stack([rng.permutation(ntr) for _ in range(epochs)])
    h = m.fit(x, y, epochs=epochs, validation_data=(xv, yv), patience=100, perms=perms)
    ref = model_ref.RefLocator(K, H, L, dropout=p, weights=w0)
    hr = model_ref.fit(ref, x, y, xv, yv, epochs, batch_size=32, patience=100, perms=perms, seed=5)
    rtol = _family(m)["rtol"]
    assert len(h.history["loss"]) == epochs
    np.testing.assert_allclose(h.history["loss"], hr["loss"], rtol=max(5 * rtol, 2e-3))
    np.testing.assert_allclose(h.history["val_loss"], hr["val_loss"], rtol=max(5 * rtol, 2e-3))
    np.testing.assert_allclose(h.history["learning_rate"], hr["learning_rate"], rtol=1e-6)
    # reload of the best checkpoint == oracle's best weights (prediction-level check)
    m.restore_best()
    yp = m.predict(xv)
    np.testing.assert_allclose(yp, ref.predict(xv), rtol=0.02, atol=0.02)
    st = m.state()
    assert st.best_epoch == int(np.argmin(hr["val_loss"]))


def test_callbacks_reduce_lr_and_early_stop(M):
    """Small patience: ReduceLROnPlateau (patience//6) and EarlyStopping fire as in the oracle."""
    from oracle import model_ref

    rng = np.random.default_rng(3)
    K, H, L = 300, 32, 2
    ntr, nva, epochs, patience = 64, 16, 60, 12
    x, y = _data(rng, ntr, K)
    xv, yv = _data(rng, nva, K)  # targets are noise -> validation loss stalls quickly
    m = M.LocatorModel(K, width=H, nlayers=L, dropout_prop=0.0, seed=2, max_epochs=epochs)
    w0 = m.get_weights()
    perms = np.stack([rng.permutation(ntr) for _ in range(epochs)])
    h = m.fit(x, y, epochs=epochs, validation_data=(xv, yv), patience=patience, perms=perms, epochs_per_call=7)
    ref = model_ref.RefLocator(K, H, L, dropout=0.0, weights=w0)
    hr = model_ref.fit(ref, x, y, xv, yv, epochs, batch_size=32, patience=patience, perms=perms, seed=2)
    assert len(h.history["loss"]) == len(hr["loss"]) < epochs  # stopped early at the same epoch
    np.testing.assert_allclose(h.history["learning_rate"], hr["learning_rate"], rtol=1e-6)
    assert min(h.history["learning_rate"]) < 1e-3
    assert m.stop_training


def test_step_invariants_full_width(M):
    """BASELINE config-2 shape (K = 100k, batch 32, 10 x 256): properties that need no oracle run."""
    rng = np.random.default_rng(1)
    K, n = 100_000, 64
    x, y = _data(rng, n, K)
    m = M.LocatorModel(K, seed=3)
    m.bind_train(x, y)
    m.set_schedule(patience=100)
    w0 = m.get_weights()
    y0 = m.predict(x)
    assert np.all(np.isfinite(y0))
    # predict is row-wise: any row subset / order gives the same rows
    sub = rng.permutation(n)[:37]
    np.testing.assert_allclose(m.predict(x[sub]), y0[sub], rtol=1e-5, atol=1e-6)
    losses = []
    for s in range(3):
        m.train_step(rng.permutation(n)[:32])
        losses.append(m.state().last_loss)
    assert np.all(np.isfinite(losses))
    w1 = m.get_weights()
    # every Adam step moves a parameter by at most ~lr (|m/sqrt(v)| <= 1/sqrt(1-b2) bound aside)
    dW = np.abs(w1[4] - w0[4])
    assert dW.max() < 3.2e-3 + 1e-6 and dW.max() > 1e-4
    # SNPs that are constant inside every batch have zero-variance columns: finite, bounded update
    assert np.all(np.isfinite(w1[0])) and np.all(np.isfinite(w1[1]))


@pytest.mark.parametrize("schedule", ["all_sms", "fewer_ctas", "ring"])
def test_group_training_matches_individual_training(M, schedule, monkeypatch):
    """Replicate group (loc_group_train_epochs): each model of a group ends bit-identical to the same model
    trained alone -- grouping only changes scheduling.  "all_sms": lockstep schedule (grouped hidden-stack
    launch).  "fewer_ctas": the same with K large enough for several tiles per CTA and the first-layer kernels on
    SMs - 16 (loc_model_set_l1_ctas; same setting for the solo runs, it fixes the summation order) -- the case that
    exposed a shared-memory reuse race between the backward kernel's builder and forward warps.  "ring": the
    schedule large models get (one model's hidden stack concurrent with the previous model's first-layer
    backward + Adam through programmatic dependent launch), forced here at K = 20,000 on a ring of three."""
    rng = np.random.default_rng(12)
    K, ntr, nva, epochs = 3000 if schedule == "all_sms" else 20000, 75, 20, 5
    ctas = None if schedule == "all_sms" else M.spare_cluster_l1_ctas()
    monkeypatch.setenv("LOC_GROUP_SCHEDULE", "ring" if schedule == "ring" else "lockstep")
    pick = slice(None) if schedule == "ring" else slice(None, None, 2)
    datas = []
    for g in range(3):
        x, y = _data(rng, ntr, K)
        xv, yv = _data(rng, nva, K)
        datas.append((x, y, xv, yv))
    solo = []
    for g, (x, y, xv, yv) in enumerate(datas):
        m = M.LocatorModel(K, seed=40 + g, max_epochs=epochs, l1_ctas=ctas)
        h = m.fit(x, y, epochs=epochs, validation_data=(xv, yv), patience=2 if (g == 1 and schedule != "ring") else 100,
                  epochs_per_call=2)
        solo.append((h, m.predict(xv), m.get_weights()[4]))
    ms = [M.LocatorModel(K, seed=40 + g, max_epochs=epochs, l1_ctas=ctas) for g in range(3)]
    if ms[0].impl != "tcgen05":
        pytest.skip("replicate groups need the tcgen05 kernels")
    # one patience for the whole group: compare the models with patience 100 semantics only where equal
    hs = M.fit_group(ms[pick], [d[0] for d in datas[pick]], [d[1] for d in datas[pick]],
                     [(d[2], d[3]) for d in datas[pick]], epochs=epochs, patience=100, epochs_per_call=2)
    assert len(hs) == (3 if schedule == "ring" else 2)
    for (h, yp, w), m, hg, d in zip(solo[pick], ms[pick], hs, datas[pick]):
        assert hg.history["loss"] == h.history["loss"] and hg.history["val_loss"] == h.history["val_loss"]
        assert np.array_equal(m.predict(d[2]), yp)
        assert np.array_equal(m.get_weights()[4], w)


@pytest.mark.parametrize("K,ntr", [(20_000, 75), (100_000, 330), (5830, 405)])
def test_chained_step_matches_unchained_step(M, K, ntr, monkeypatch):
    """train_step's chain (hidden stack -> first-layer backward -> small-layer update as programmatic dependent
    launches that hand over through DevState::hid_seq / bwd_cnt instead of kernel boundaries) only changes WHEN
    kernels start: histories, weights and predictions equal those of the unchained schedule (LOC_NO_CHAIN: update
    on a side stream, plain launches) bit for bit, over several epochs with ragged last batches, validation
    passes and checkpoints in between."""
    rng = np.random.default_rng(K)
    x, y = _data(rng, ntr, K)
    xv, yv = _data(rng, 40, K)
    epochs = 4
    perms = np.stack([rng.permutation(ntr) for _ in range(epochs)])
    out = []
    for chained in (True, False, True):
        if chained:
            monkeypatch.delenv("LOC_NO_CHAIN", raising=False)
        else:
            monkeypatch.setenv("LOC_NO_CHAIN", "1")
        m = M.LocatorModel(K, seed=77, max_epochs=epochs)
        if m.impl != "tcgen05":
            pytest.skip("tcgen05 kernels only")
        h = m.fit(x, y, epochs=epochs, validation_data=(xv, yv), patience=100, perms=perms, epochs_per_call=3)
        st = m.state()
        assert st.nonfinite == 0 and st.t == epochs * int(np.ceil(ntr / 32))
        out.append((h.history, m.get_weights(), m.predict(xv)))
        del m
    monkeypatch.delenv("LOC_NO_CHAIN", raising=False)
    for other in out[1:]:
        assert other[0] == out[0][0]
        for a, b in zip(other[1], out[0][1]):
            assert np.array_equal(a, b)
        assert np.array_equal(other[2], out[0][2])


def test_backward_kernels_survive_many_launches(M):
    """Regression for an mbarrier phase-aliasing race in the tcgen05 backward (the two epilogue groups shared
    one barrier per pipeline stage and could pass a wait one phase early): at K = 100k the unfused kernel
    faulted about once in 500 launches.  600 unfused + 300 fused launches, then the weights must be finite."""
    rng = np.random.default_rng(5)
    K, n = 100_000, 64
    x, y = _data(rng, n, K)
    m = M.LocatorModel(K, seed=9)
    if m.impl != "tcgen05":
        pytest.skip("tcgen05 kernels only")
    m.bind_train(x, y)
    m.set_schedule(patience=100)
    rows = rng.permutation(n)[:32]
    m.debug_stage(0, rows)
    m.debug_stage(1, rows)
    for stage, reps in ((2, 600), (4, 300)):
        for _ in range(reps):
            m.debug_stage(stage, rows)
        torch.cuda.synchronize()
    w = m.get_weights()
    assert all(np.all(np.isfinite(a)) for a in w[:6])


def test_fused_epochs_match_step_by_step_training(M):
    """loc_train_epochs (backward kernel also runs the next step's forward, tiles walked in alternating
    order) vs the same batches issued one loc_train_step at a time (separate forward launches): the two
    schedules differ only in fp32 summation order of the first-layer split-K partials."""
    rng = np.random.default_rng(21)
    K, ntr, nva = 20_000, 96, 32
    x, y = _data(rng, ntr, K)
    xv, yv = _data(rng, nva, K)
    perms = np.stack([rng.permutation(ntr) for _ in range(2)]).astype(np.int32)
    a = M.LocatorModel(K, seed=77, dropout_prop=0.0)
    b = M.LocatorModel(K, seed=77, dropout_prop=0.0)
    for m in (a, b):
        m.bind_train(x, y)
        m.bind_val(xv, yv)
        m.set_schedule(patience=100)
    a.train_epochs(perms)
    for e in range(2):
        for s in range(ntr // 32):
            b.train_step(perms[e, 32 * s:32 * (s + 1)])
    torch.cuda.synchronize()
    wa, wb = a.get_weights(), b.get_weights()
    w0 = M.LocatorModel(K, seed=77, dropout_prop=0.0).get_weights()
    # elementwise comparison is meaningless for Adam (a gradient that rounds to the other side of zero moves
    # a weight by 2 * lr): compare the updates in norm, and the function the two models compute
    for i in (4, 6, 8):  # W1 and the first hidden kernels
        upd = np.linalg.norm(wb[i] - w0[i])
        assert np.linalg.norm(wa[i] - wb[i]) <= 0.05 * upd, f"weight {i}"
    np.testing.assert_allclose(a.predict(xv), b.predict(xv), rtol=5e-3, atol=5e-3)


@pytest.mark.parametrize("K,n", [(200_000, 250), (5830, 33), (20_000, 257), (3000, 300), (100_000, 90)])
def test_wide_inference_matches_oracle_and_narrow_path(M, K, n, monkeypatch):
    """Validation / prediction / jacknife sweeps stream W1 once per 256 rows (k_l1_fwd_wide: MMA N = 32..256,
    the 32-row chunks of a pass through the hidden stack side by side) instead of once per 32 rows.  Against
    RefLocator.predict / evaluate (locator.py:374,414,441) at BASELINE config 5's shape (250 x 200,000) and at
    ragged sizes around the pass / chunk boundaries, and against the chunk-by-chunk path (LOC_NO_WIDE)."""
    from oracle import model_ref

    rng = np.random.default_rng(K + n)
    x, y = _data(rng, n, K)
    m = M.LocatorModel(K, seed=17)
    if m.impl != "tcgen05":
        pytest.skip("tcgen05 kernels only")
    ws = m.get_weights()
    ws[0] = rng.uniform(0.5, 1.5, K).astype(np.float32)
    ws[1] = rng.normal(0, 0.1, K).astype(np.float32)
    ws[2] = rng.uniform(0, 1.5, K).astype(np.float32)
    ws[3] = rng.uniform(0.1, 0.8, K).astype(np.float32)
    for i in range(5, len(ws), 2):
        ws[i] = rng.normal(0, 0.05, ws[i].shape).astype(np.float32)
    m.set_weights(ws)
    yp = m.predict(x)
    ev = m.evaluate(x, y)
    monkeypatch.setenv("LOC_NO_WIDE", "1")
    yp_narrow = m.predict(x)
    ev_narrow = m.evaluate(x, y)
    monkeypatch.delenv("LOC_NO_WIDE")
    assert yp.shape == (n, 2) and np.all(np.isfinite(yp))
    # same products, same split over SNPs, same order of the chunk sums
    np.testing.assert_allclose(yp, yp_narrow, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(ev, ev_narrow, rtol=1e-6)
    # stated tolerance |dy| <= tol * (1 + |y|): 2e-3 against the oracle with the device's operand rounding (what is
    # left is summation order over up to 200,000 SNPs), 5e-3 against the fp32 oracle -- this test's BN scales
    # (gamma up to 1.5, moving variance down to 0.1) put the first layer's inputs at several times the magnitude a
    # trained model sees, and the tf32 rounding error grows with them (measured maxima: 1.0e-3 and 2.5e-3)
    for numerics, tol in (("tf32", 2e-3), ("fp32", 5e-3)):
        ref = model_ref.RefLocator(K, 256, 10, weights=ws, numerics=numerics)
        np.testing.assert_allclose(yp, ref.predict(x), rtol=tol, atol=tol, err_msg=numerics)
        np.testing.assert_allclose(ev, ref.evaluate(x, y), rtol=tol, err_msg=numerics)
