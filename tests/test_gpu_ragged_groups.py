"""Replicate groups whose training-set sizes differ (the folds of a k-fold holdout, loc_group_train_epochs).

The step at row offset off of an epoch holds the models with off < n_train, each over its own min(B, n_train - off)
rows with its own fused-next-forward decision, and a model's epoch ends after its own last step.  Every kernel of a
model gets the arguments it gets alone, so each model must end bit-identical to the same model trained alone with
model.fit: histories, optimizer state, weights, Adam moments and predictions.  Sizes cover a difference inside the
last partial step (405 / 404) and differences of one step or more (405 / 370 / 404 / 341).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

NVA = 40


def cdiv(a, b):
    return -(-a // b)


@pytest.fixture(scope="module")
def M():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from locator_b200 import model

    return model


def _datasets(seed, K, ntrs, nva=NVA):
    from locator_b200.genotypes import PackedGenotypes

    rng = np.random.default_rng(seed)
    out = []
    for ntr in ntrs:
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


def _solo_and_group(M, K, ntrs, width, B, epochs, seed0, ctas=False, patience=100, family="tcgen05"):
    datas = _datasets(seed0, K, ntrs)
    l1_ctas = M.spare_cluster_l1_ctas() if ctas else None
    make = [lambda g=g: M.LocatorModel(K, width=width, nlayers=4, batch_size=B, seed=seed0 + g, max_epochs=epochs,
                                       l1_ctas=l1_ctas) for g in range(len(ntrs))]
    solo = []
    for g, (x, y, xv, yv) in enumerate(datas):
        m = make[g]()
        if (m.impl, m.hidden_impl) != (family, family):
            pytest.skip(f"needs the {family} kernels")
        h = m.fit(x, y, epochs=epochs, batch_size=B, validation_data=(xv, yv), patience=patience, epochs_per_call=4)
        solo.append(_snapshot(m, h, xv))
        del m
    ms = [f() for f in make]
    hs = M.fit_group(ms, [d[0] for d in datas], [d[1] for d in datas], [(d[2], d[3]) for d in datas], epochs=epochs,
                     patience=patience, epochs_per_call=4)
    return solo, [_snapshot(m, h, d[2]) for m, h, d in zip(ms, hs, datas)]


SIZES = {"405-404": [405, 404], "405-370-404": [405, 370, 404], "405-370-404-341": [405, 370, 404, 341]}


@pytest.mark.parametrize("sizes", list(SIZES))
@pytest.mark.parametrize("width,family", [(256, "tcgen05"), (128, "simt")], ids=["tcgen05", "cuda-core-w128"])
def test_lockstep(M, monkeypatch, width, family, sizes):
    """32 rows a step: the grouped hidden launch holds the models with a step at the offset, each with its own rows."""
    monkeypatch.setenv("LOC_GROUP_SCHEDULE", "lockstep")
    epochs = 3
    solo, group = _solo_and_group(M, 3001, SIZES[sizes], width, 32, epochs, 11, family=family)
    for s, g, n in zip(solo, group, SIZES[sizes]):
        assert s["state"][0] == epochs * cdiv(n, 32)
        _assert_same(s, g)


@pytest.mark.parametrize("chain", [True, False], ids=["chained", "LOC_NO_CHAIN"])
@pytest.mark.parametrize("sizes", list(SIZES))
def test_ring(M, monkeypatch, sizes, chain):
    """Ring schedule (forced at K = 20,000, first-layer kernels on SMs - 16): a model without a step left skips its
    slot; in a ring of two the remaining model's steps hand over through its own backward and update."""
    monkeypatch.setenv("LOC_GROUP_SCHEDULE", "ring")
    if chain:
        monkeypatch.delenv("LOC_NO_CHAIN", raising=False)
    else:
        monkeypatch.setenv("LOC_NO_CHAIN", "1")
    epochs = 3
    solo, group = _solo_and_group(M, 20000, SIZES[sizes], 256, 32, epochs, 21, ctas=True)
    for s, g in zip(solo, group):
        _assert_same(s, g)


@pytest.mark.parametrize("serial", [False, True], ids=["grouped", "LOC_BB_SERIAL"])
@pytest.mark.parametrize("B", [64, 100])
@pytest.mark.parametrize("width,family", [(256, "tcgen05"), (128, "simt")], ids=["tcgen05", "cuda-core-w128"])
def test_large_batch(M, monkeypatch, width, family, B, serial):
    """Above 32 rows: at 64 rows the last steps are 21 / 50 / 20 / 21 rows (one and two chunks side by side), at 100
    rows 5 / 70 / 4 / 41 (one, three and two chunks) -- models are packed by their own chunk counts."""
    if serial:
        monkeypatch.setenv("LOC_BB_SERIAL", "1")
    else:
        monkeypatch.delenv("LOC_BB_SERIAL", raising=False)
    epochs = 3
    sizes = SIZES["405-370-404-341"]
    solo, group = _solo_and_group(M, 3001, sizes, width, B, epochs, 31 + B, family=family)
    for s, g, n in zip(solo, group, sizes):
        assert s["state"][0] == epochs * cdiv(n, B)
        _assert_same(s, g)


@pytest.mark.parametrize("B", [32, 64])
def test_early_stopping_at_different_epochs(M, monkeypatch, B):
    """Patience 1: the models stop at different epochs (a stopped model leaves the group at the next call)."""
    monkeypatch.delenv("LOC_GROUP_SCHEDULE", raising=False)
    solo, group = _solo_and_group(M, 3001, SIZES["405-370-404-341"], 256, B, 12, 41 + B, patience=1)
    stops = [s["state"][1] for s in solo]
    assert len(set(stops)) > 1 and min(stops) < 12, stops
    for s, g in zip(solo, group):
        _assert_same(s, g)


# launch counts (the `loc` launch counter, as in tests/test_gpu_schedules.py)
K, E = 3001, 2
VAL_WIDE = 3     # one pass of 40 rows: wide forward, grouped hidden stacks, validation sums in order
EPOCH_END = 2    # epoch end + checkpoint copy


def _launches(fn):
    from locator_b200 import _cabi

    torch.cuda.synchronize()
    l0 = _cabi.launch_count()
    fn()
    torch.cuda.synchronize()
    return _cabi.launch_count() - l0


def _big_step(ncs, serial):
    """Launches of one large-batch step of the models with chunk counts ncs (train_step_big): models of more than one
    chunk packed whole, in order, up to 8 chunks a grouped hidden launch, and one step end for them; a one-chunk model
    (or every chunk with LOC_BB_SERIAL) gets a hidden launch of its own."""
    hidden, packed, side = 0, 0, 0
    for nc in ncs:
        if serial or nc == 1:
            hidden += nc
            hidden += packed > 0
            packed = 0
            continue
        side += 1
        if packed + nc > 8:
            hidden += 1
            packed = 0
        packed += nc
    hidden += packed > 0
    G = len(ncs)
    return 1 + G + hidden + (side > 0) + 2 * G + G  # statistics, wide forwards, hidden, step end, backwards, updates


@pytest.mark.parametrize("B,sizes", [(32, [200, 170, 199]), (64, [300, 270, 199]), (100, [300, 270, 199])])
def test_ragged_group_launch_count(M, monkeypatch, B, sizes):
    monkeypatch.setenv("LOC_GROUP_SCHEDULE", "lockstep")
    monkeypatch.delenv("LOC_BB_SERIAL", raising=False)
    G = len(sizes)
    ds = _datasets(50, K, sizes)
    ms = [M.LocatorModel(K, nlayers=4, batch_size=B, seed=1 + g, max_epochs=E) for g in range(G)]
    if (ms[0].impl, ms[0].hidden_impl) != ("tcgen05", "tcgen05"):
        pytest.skip("needs the tcgen05 kernels")
    offs = range(0, max(sizes), B)
    if B == 32:  # forwards of the first step; per offset one grouped hidden launch, an update and a backward per model
        per_epoch = G + sum(1 + 2 * sum(off < n for n in sizes) for off in offs)
    else:
        per_epoch = sum(_big_step([cdiv(min(B, n - off), 32) for n in sizes if off < n], False) for off in offs)
    n = _launches(lambda: M.fit_group(ms, [d[0] for d in ds], [d[1] for d in ds], [(d[2], d[3]) for d in ds], epochs=E))
    # set_schedule and begin of the call per model; validation and epoch end per model
    assert n == 2 * G + E * (per_epoch + G * (VAL_WIDE + EPOCH_END))
