"""CPU: the oracle against the golden facts frozen from the reference's own fixture, and the
restated Keras math against torch autograd."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from oracle import ingest_ref, model_ref, philox_ref

HERE = os.path.dirname(os.path.abspath(__file__))


def _facts(name):
    return json.load(open(os.path.join(HERE, "golden", name)))


def test_ingest_oracle_matches_fixture_facts(fixture_gt):
    facts = _facts("fixture_facts.json")
    gt = fixture_gt["calldata/GT"]
    assert gt.shape == (facts["nvar"], facts["nsamples"], 2)
    assert fixture_gt["samples"][0] == facts["first_sample"] and fixture_gt["samples"][-1] == facts["last_sample"]
    assert int(fixture_gt["variants/POS"][0]) == facts["pos_first"]
    assert int(fixture_gt["variants/POS"][-1]) == facts["pos_last"]
    cnt = ingest_ref.count_alleles(gt)
    allelism = (cnt > 0).sum(1)
    assert {str(k): int((allelism == k).sum()) for k in (1, 2, 3)} == facts["allelism_hist"]
    assert int(ingest_ref.is_biallelic(cnt).sum()) == facts["n_biallelic"]
    ac, idx = ingest_ref.filter_snps(gt, min_mac=2, return_index=True)
    assert ac.shape == (facts["n_kept_min_mac_2"], facts["nsamples"]) and ac.dtype == np.uint8
    assert hashlib.sha256(idx.astype(np.int64).tobytes()).hexdigest() == facts["kept_index_sha256"]
    assert hashlib.sha256(np.ascontiguousarray(ac).tobytes()).hexdigest() == facts["ac_sha256"]
    assert {str(v): int((ac == v).sum()) for v in (0, 1, 2)} == facts["kept_value_hist"]


def test_sample_data_and_rng_oracle_match_golden(fixture_gt, golden_dir):
    facts, rng = _facts("fixture_facts.json"), _facts("rng_facts.json")
    ids, x, y = ingest_ref.read_sample_data(os.path.join(golden_dir, "data", "test_sample_data.txt"))
    locs = ingest_ref.sort_samples(ids, x, y, fixture_gt["samples"])
    assert int(np.isnan(locs[:, 0]).sum()) == facts["n_na"]
    ml, sl, mt, st, nl = ingest_ref.normalize_locs(locs)
    np.testing.assert_allclose([ml, mt], facts["nanmean"], rtol=1e-12)
    np.testing.assert_allclose([sl, st], facts["nanstd"], rtol=1e-12)
    ac = ingest_ref.filter_snps(fixture_gt["calldata/GT"], min_mac=2)
    np.random.seed(rng["seed"])
    train, test, traingen, testgen, trainlocs, testlocs, pred, predgen = ingest_ref.split_train_test(ac, nl, 0.9)
    assert test.tolist() == rng["test_idx"] and len(train) == 405 and pred.tolist() == list(range(50))
    assert traingen.shape == (405, 5830) and testgen.shape == (45, 5830) and predgen.shape == (50, 5830)
    order = ingest_ref.bootstrap_site_order(ac.shape[0])
    assert order[:16].tolist() == rng["bootstrap_site_order_prefix"]
    assert hashlib.sha256(order.astype(np.int64).tobytes()).hexdigest() == rng["bootstrap_site_order_sha256"]
    # jacknife draws right after the split
    np.random.seed(rng["seed"])
    ingest_ref.split_train_test(ac, nl, 0.9)
    af = ingest_ref.jacknife_af(ac)
    pg, sites = ingest_ref.jacknife_replace(predgen, af, 0.05)
    assert sites[:16].tolist() == rng["jacknife_sites_prefix"] and len(sites) == rng["jacknife_nsites"]
    assert pg[:, sites[0]].tolist() == rng["jacknife_first_col"]


def test_round_is_bankers_rounding_of_float_product():
    # (1 - 0.9) * 450 = 44.99999999999999 -> 45 (SURVEY appendix B)
    assert round((1 - 0.9) * 450) == 45 and round((1 - 0.9) * 900) == 90 and round((1 - 0.9) * 2250) == 225


def test_missing_and_multiallelic_semantics():
    gt = np.array([
        [[0, 1], [1, 1], [-1, -1], [0, 0]],   # biallelic, alt count 3, one missing call
        [[0, 0], [0, 0], [0, 0], [0, 0]],     # monomorphic
        [[1, 2], [2, 1], [1, 1], [2, 2]],     # alleles {1, 2}: passes is_biallelic
        [[0, 1], [2, 0], [1, 1], [0, 0]],     # three alleles
        [[0, -1], [1, 1], [0, 0], [0, 1]],    # half-missing call counts as missing for is_missing
    ], dtype=np.int8)
    cnt = ingest_ref.count_alleles(gt)
    assert cnt[0].tolist() == [3, 3, 0] and cnt[2].tolist() == [0, 4, 4]
    assert ingest_ref.is_biallelic(cnt).tolist() == [True, False, True, False, True]
    assert ingest_ref.is_missing(gt)[4].tolist() == [True, False, False, False]
    ac, idx = ingest_ref.filter_snps(gt, min_mac=2, return_index=True)
    assert idx.tolist() == [0, 2, 4]
    assert ac.tolist() == [[1, 2, 0, 0], [1, 1, 2, 0], [0, 2, 0, 1]]
    assert ingest_ref.filter_snps(gt, min_mac=4).shape[0] == 1  # only the {1,2} site has 4 copies of allele 1
    assert ingest_ref.filter_snps(gt, min_mac=1).shape[0] == 3  # min_mac == 1 skips the count filter


def test_filter_with_no_surviving_or_no_sites():
    """Edge cases: every site fails the biallelic test (all triallelic / monomorphic), and an empty cube."""
    gt = np.array([[[0, 1], [2, 0]], [[0, 0], [0, 0]]], dtype=np.int8)
    ac, idx = ingest_ref.filter_snps(gt, min_mac=2, return_index=True)
    assert ac.shape == (0, 2) and idx.size == 0
    ac, idx = ingest_ref.filter_snps(np.zeros((0, 7, 2), np.int8), min_mac=2, return_index=True)
    assert ac.shape == (0, 7) and idx.size == 0
    assert ingest_ref.count_alleles(np.zeros((0, 7, 2), np.int8)).shape == (0, 1)


def test_philox_known_answer():
    # Philox4x32-10 known-answer test of Random123 (counter = key = 0 and the all-ones vector)
    r = philox_ref.philox4x32_10([0], [0], [0], [0], 0, 0)
    assert [int(v[0]) for v in r] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    r = philox_ref.philox4x32_10([0xFFFFFFFF], [0xFFFFFFFF], [0xFFFFFFFF], [0xFFFFFFFF], 0xFFFFFFFF, 0xFFFFFFFF)
    assert [int(v[0]) for v in r] == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    u = philox_ref.uniform01(1000, 5, 3)
    assert u.dtype == np.float32 and u.min() >= 0 and u.max() < 1 and abs(u.mean() - 0.5) < 0.05


@pytest.mark.parametrize("K,H,L,p,B", [(50, 16, 4, 0.25, 8), (31, 8, 3, 0.0, 5), (20, 8, 2, 0.5, 32),
                                       (40, 16, 4, 0.25, 80), (24, 8, 3, 0.25, 250)])  # batches above 32: --batch_size 33..256
def test_oracle_gradients_match_autograd(K, H, L, p, B):
    rng = np.random.default_rng(K)
    x = rng.integers(0, 3, size=(B, K)).astype(np.uint8)
    x[:, 0] = 1  # a column that is constant within the batch
    y = rng.normal(size=(B, 2)).astype(np.float32)
    ref = model_ref.RefLocator(K, H, L, dropout=p, seed=3)
    ws = ref.get_weights()
    ws[0] = rng.uniform(0.5, 1.5, K).astype(np.float32)
    ws[1] = rng.normal(0, 0.1, K).astype(np.float32)
    ref.set_weights(ws)
    mask = rng.uniform(size=(B, H)) >= p
    loss, grads, _ = ref.gradients(x, y, mask)
    # same network with autograd
    t = [torch.tensor(w, requires_grad=True) for w in ws]
    gamma, beta = t[0], t[1]
    xt = torch.tensor(x, dtype=torch.float32)
    mean = xt.mean(0)
    var = ((xt - mean) ** 2).mean(0)
    a = (xt - mean) * torch.rsqrt(var + 1e-3) * gamma + beta
    nb4 = int(np.floor(L / 2))
    for i in range(L):
        a = torch.nn.functional.elu(a @ t[4 + 2 * i] + t[5 + 2 * i])
        if i == nb4 - 1 and p > 0:
            a = a * torch.tensor(mask, dtype=torch.float32) / (1 - p)
    y1 = a @ t[4 + 2 * L] + t[5 + 2 * L]
    y2 = y1 @ t[6 + 2 * L] + t[7 + 2 * L]
    l = torch.sqrt(((y2 - torch.tensor(y)) ** 2).sum(-1)).mean()
    l.backward()
    assert abs(l.item() - loss) < 1e-5 * max(1.0, abs(loss))
    auto = [t[0].grad, t[1].grad] + [t[i].grad for i in range(4, len(t))]
    for g, ga in zip(grads, auto):
        np.testing.assert_allclose(g.numpy(), ga.numpy(), rtol=2e-4, atol=2e-6)
    assert float(grads[0][0]) == 0.0  # d gamma of the constant column is exactly zero


def test_oracle_tf32_l1_rounds_the_first_layer_only():
    """numerics="tf32_l1" (tcgen05 first layer + CUDA-core hidden stack, width-256 models deeper than 14 layers):
    the first layer's pre-activation equals the "tf32" mode's bit for bit; from that layer's output on, the hidden and
    output layers are the "fp32" mode's arithmetic; the first-layer gradient is the device's formula (as in "tf32")."""
    K, H, L, p, B = 70, 24, 5, 0.25, 12
    rng = np.random.default_rng(4)
    x = rng.integers(0, 3, size=(B, K)).astype(np.uint8)
    y = rng.normal(size=(B, 2)).astype(np.float32)
    ws = model_ref.init_weights(K, H, L, seed=6)
    ws[0] = rng.uniform(0.5, 1.5, K).astype(np.float32)
    ws[1] = rng.normal(0, 0.1, K).astype(np.float32)
    for i in range(5, len(ws), 2):
        ws[i] = rng.normal(0, 0.05, ws[i].shape).astype(np.float32)
    mask = rng.uniform(size=(B, H)) >= p
    out = {}
    for mode in ("fp32", "tf32", "tf32_l1"):
        ref = model_ref.RefLocator(K, H, L, dropout=p, weights=ws, numerics=mode)
        out[mode] = (ref,) + ref.gradients(x, y, mask)
    ref, loss, grads, c = out["tf32_l1"]
    assert torch.equal(c["zs"][0], out["tf32"][3]["zs"][0])
    assert not torch.equal(c["zs"][0], out["fp32"][3]["zs"][0])  # the rounding is visible at these scales
    # the hidden and output layers in plain fp32, fed the first layer's output
    a = c["acts"][1]
    for i in range(1, L):
        z = a @ ref.W[i] + ref.b[i]
        assert torch.equal(z, c["zs"][i]), i
        a = c["acts"][i + 1]
    y2 = (a @ ref.W[L] + ref.b[L]) @ ref.W[L + 1] + ref.b[L + 1]
    assert loss == float(model_ref.RefLocator.loss_per_sample(y2, torch.as_tensor(y)).mean())
    assert loss != out["tf32"][1]
    # hidden-layer backward in fp32: d loss / d z of layer 0 from fp32 products, then the device's first-layer formula
    dz1, W1 = c["dzs"][1], ref.W[1]
    dz0 = torch.where(c["zs"][0] > 0, dz1 @ W1.T, (dz1 @ W1.T) * torch.exp(c["zs"][0]))  # Dropout sits after layer 1
    assert torch.equal(c["dzs"][0], dz0)
    S = model_ref.tf32_rna(c["x"] - c["mean"]).T @ dz0
    assert torch.equal(grads[2], (c["rs"] * ref.gamma)[:, None] * S + ref.beta[:, None] * dz0.sum(0)[None, :])
    # and the whole gradient stays close to the fp32 mode's
    for g, g32 in zip(grads, out["fp32"][2]):
        np.testing.assert_allclose(g.numpy(), g32.numpy(), rtol=2e-2, atol=2e-3 * float(g32.abs().max()))


def test_oracle_adam_and_callbacks_semantics():
    # Keras Adam, one step from zero state: update = -lr * sign(g) * |g| / (|g| + eps*...) ~ -lr * sign(g)
    ref = model_ref.RefLocator(10, 8, 2, dropout=0.0, seed=1)
    w0 = [w.copy() for w in ref.get_weights()]
    rng = np.random.default_rng(0)
    x = rng.integers(0, 3, size=(32, 10)).astype(np.uint8)
    y = rng.normal(size=(32, 2)).astype(np.float32)
    ref.train_step(x, y, np.ones((32, 8), bool))
    w1 = ref.get_weights()
    d = np.abs(w1[4] - w0[4])
    assert d.max() <= 1.0001e-3 and d[d > 0].min() > 0.5e-3
    # moving statistics: 0.99 * old + 0.01 * batch
    np.testing.assert_allclose(w1[2], 0.01 * x.astype(np.float32).mean(0), rtol=1e-5)
    # callbacks: checkpoint on strict improvement, LR halves after patience//6 stale epochs, stop at patience
    cb = model_ref.CallbackState(patience=12, lr=1e-3)
    vals = [1.0, 0.9, 0.95, 0.95, 0.93, 0.92, 0.91, 0.9, 0.9, 0.9, 0.9, 0.9, 0.9, 0.9, 0.9]
    saves, lrs = [], []
    for e, v in enumerate(vals):
        s, lr = cb.on_epoch_end(e, v)
        saves.append(s)
        lrs.append(lr)
        if cb.stop:
            break
    assert saves[:3] == [True, True, False] and sum(saves) == 2
    assert lrs[3] == pytest.approx(1e-3) and lrs[4] == pytest.approx(5e-4) and lrs[6] == pytest.approx(2.5e-4)
    assert cb.stop and e == 13  # 12 epochs without improvement after epoch 1


def _sha(a):
    import hashlib

    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_oracle_matches_vectors_produced_by_the_reference_code(fixture_gt, golden_dir):
    """tests/golden/reference_vectors.* were produced by the REFERENCE'S OWN functions (sort_samples,
    normalize_locs, filter_snps, replace_md, split_train_test and the bootstrap / jacknife loops of main(), compiled
    from /root/reference/locator/locator.py by tests/golden/make_reference_vectors.py).  The oracle must reproduce
    every one of them, bit for bit, from the same inputs and seeds."""
    import json

    vec = json.load(open(os.path.join(golden_dir, "reference_vectors.json")))
    arr = np.load(os.path.join(golden_dir, "reference_vectors.npz"))
    fx = vec["fixture"]
    gt = fixture_gt["calldata/GT"]
    ids, x, y = ingest_ref.read_sample_data(os.path.join(golden_dir, "data", "test_sample_data.txt"))
    np.random.seed(vec["seed"])
    locs = ingest_ref.sort_samples(ids, x, y, fixture_gt["samples"])
    assert _sha(locs.astype(np.float64)) == fx["locs_sha256"]
    meanlong, sdlong, meanlat, sdlat, nlocs = ingest_ref.normalize_locs(locs)
    assert [float(meanlong), float(sdlong), float(meanlat), float(sdlat)] == fx["norm"]
    assert _sha(nlocs.astype(np.float64)) == fx["normalized_locs_sha256"]
    ac = ingest_ref.filter_snps(gt, min_mac=2)
    assert list(ac.shape) == fx["ac_shape"] and str(ac.dtype) == fx["ac_dtype"] and _sha(ac) == fx["ac_sha256"]
    train, test, traingen, testgen, trainlocs, testlocs, pred, predgen = ingest_ref.split_train_test(ac, nlocs, 0.9)
    assert train.tolist() == fx["train"] and test.tolist() == fx["test"] and pred.tolist() == fx["pred"]
    assert _sha(traingen) == fx["traingen_sha256"] and _sha(testgen) == fx["testgen_sha256"]
    assert _sha(predgen) == fx["predgen_sha256"]
    assert _sha(trainlocs) == fx["trainlocs_sha256"] and _sha(testlocs) == fx["testlocs_sha256"]
    after_split = np.random.get_state()
    # bootstrap loop, continuing the run's stream
    for want in vec["bootstrap"]:
        order = ingest_ref.bootstrap_site_order(traingen.shape[1])
        assert order[:16].tolist() == want["site_order_prefix"] and _sha(order.astype(np.int64)) == want["site_order_sha256"]
    # jacknife loop from the same point of the stream
    np.random.set_state(after_split)
    af = ingest_ref.jacknife_af(ac)
    assert _sha(af.astype(np.float64)) == vec["jacknife"]["af_sha256"]
    for want in vec["jacknife"]["replicates"]:
        pg, sites = ingest_ref.jacknife_replace(predgen, af, 0.05)
        assert len(sites) == want["nsites"] and _sha(sites.astype(np.int64)) == want["sites_sha256"]
        assert _sha(pg.astype(np.uint8)) == want["pg_sha256"]
    assert np.random.random() == vec["jacknife"]["next_uniform"]
    # imputation (scalar draws in (site, sample) order) + SNP subsample, and the min_mac == 1 rule
    imp = vec["impute_subsample"]
    np.random.seed(imp["seed"])
    got = ingest_ref.filter_snps(arr["small_gt"], min_mac=imp["min_mac"], impute_missing=True, max_SNPs=imp["max_SNPs"])
    assert np.array_equal(got, arr["small_ac"]) and np.random.random() == imp["next_uniform"]
    assert np.array_equal(ingest_ref.filter_snps(arr["small_gt"], min_mac=1), arr["small_ac_min_mac_1"])


def test_oracle_windows_flow_matches_the_reference_loop(fixture_gt, golden_dir):
    """The --windows loop of the reference's main() (run by make_reference_vectors.py around recording stubs):
    window bounds (SNP b itself excluded), per-window sort / normalise / filter / split continuing one numpy
    stream after the genome-wide split, and the per-window output stem."""
    import json

    w = json.load(open(os.path.join(golden_dir, "reference_vectors.json")))["windows"]
    gt, positions = fixture_gt["calldata/GT"], fixture_gt["variants/POS"]
    ids, x, y = ingest_ref.read_sample_data(os.path.join(golden_dir, "data", "test_sample_data.txt"))
    locs = ingest_ref.sort_samples(ids, x, y, fixture_gt["samples"])
    np.random.seed(w["seed"])
    ingest_ref.split_train_test(ingest_ref.filter_snps(gt, min_mac=2), ingest_ref.normalize_locs(locs)[4], 0.9)
    bounds = list(ingest_ref.window_bounds(positions, 0, w["stop"], w["window_size"]))
    assert [(i, a, b) for i, a, b in bounds] == [(r["i"], r["a"], r["b"]) for r in w["records"]]
    for (i, a, b), r in zip(bounds, w["records"]):
        meanlong, sdlong, meanlat, sdlat, nlocs = ingest_ref.normalize_locs(locs)
        ac = ingest_ref.filter_snps(gt[a:b], min_mac=2)
        train, test, traingen, testgen, trainlocs, testlocs, pred, predgen = ingest_ref.split_train_test(ac, nlocs, 0.9)
        assert ac.shape[0] == r["K"] and _sha(ac) == r["ac_sha256"] and test.tolist() == r["test"]
        assert _sha(train.astype(np.int64)) == r["train_sha256"] and _sha(traingen) == r["traingen_sha256"]
        assert _sha(predgen) == r["predgen_sha256"]
        assert [float(meanlong), float(sdlong), float(meanlat), float(sdlat)] == r["norm"]
        assert r["out"] == f"win_{i}-{i + w['window_size'] - 1}"
    assert np.random.random() == w["next_uniform"]


def test_oracle_builds_what_the_reference_asks_keras_for(golden_dir):
    """load_network of the reference, run around recording stand-ins for Keras (make_reference_vectors.py): the
    layer sequence per nlayers / width / dropout, the optimizer name and the loss expression (numpy as the
    backend).  The oracle's layer plan, weight shapes and per-sample loss must be those."""
    import json

    req = json.load(open(os.path.join(golden_dir, "reference_vectors.json")))["keras_requests"]
    arr = np.load(os.path.join(golden_dir, "reference_vectors.npz"))
    for net in req["networks"]:
        kinds = [l["kind"] for l in net["layers"]]
        L, H, K = net["nlayers"], net["width"], net["layers"][0]["input_shape"][0]
        n_before, n_after = model_ref.layer_plan(L)
        assert kinds == ["BatchNormalization"] + ["Dense"] * n_before + ["Dropout"] + ["Dense"] * n_after + ["Dense", "Dense"]
        dense = [l for l in net["layers"] if l["kind"] == "Dense"]
        assert [d["args"][0] for d in dense] == [H] * L + [2, 2]
        assert [d.get("activation") for d in dense] == ["elu"] * L + [None, None]
        assert [l for l in net["layers"] if l["kind"] == "Dropout"][0]["args"] == [net["dropout_prop"]]
        assert net["compile"] == {"optimizer": "Adam"}
        ref = model_ref.RefLocator(K, H, L, dropout=net["dropout_prop"])
        shapes = [tuple(w.shape) for w in ref.get_weights()]
        dims = [K] + [H] * L + [2, 2]
        want = [(K,)] * 4
        for i in range(L + 2):
            want += [(dims[i], dims[i + 1]), (dims[i + 1],)]
        assert shapes == want and (ref.n_before, ref.n_after) == (n_before, n_after)
        import torch

        got = model_ref.RefLocator.loss_per_sample(torch.as_tensor(arr["loss_y_pred"]), torch.as_tensor(arr["loss_y_true"]))
        assert [float(v) for v in got] == net["loss_of_fixed_arrays"]
    # callback settings the oracle's state machine is built from (patience, patience / 6, factor 0.5 ...)
    for cb in req["callbacks"]:
        ck, es, rl = cb["callbacks"]
        P = es["patience"]
        cbs = model_ref.CallbackState(P)
        assert cbs.P == P and cbs.rlr_patience == rl["patience"] == int(P / 6)
        assert rl["factor"] == 0.5 and rl["min_delta"] == 0 and rl["cooldown"] == 0 and rl["min_lr"] == 0
        assert es["min_delta"] == 0 and es["monitor"] == rl["monitor"] == ck["monitor"] == "val_loss"
        assert ck["save_best_only"] is True and ck["save_weights_only"] is True


@pytest.mark.parametrize("B", [12, 96])
def test_oracle_training_matches_torch_nn_and_torch_optim(B):
    """An independent implementation of the same mathematics: torch.nn.BatchNorm1d (eps 1e-3, momentum 0.01 = Keras
    0.99) / Linear / ELU trained with torch.optim.Adam.  Keras puts epsilon outside the bias-corrected root
    (theta -= lr sqrt(1-b2^t)/(1-b1^t) m / (sqrt(v) + eps)); torch divides v by (1-b2^t) first, which is the same
    update with eps / sqrt(1-b2^t) -- set per step below.  Several optimizer steps from the same weights must give
    the same weights, losses and moving means (moving variances differ by design: torch tracks the unbiased one)."""
    import math

    K, H, L, steps = 37, 16, 4, 6
    rng = np.random.default_rng(17)
    ref = model_ref.RefLocator(K, H, L, dropout=0.0, seed=5)
    ws = ref.get_weights()
    ws[0] = rng.uniform(0.5, 1.5, K).astype(np.float32)
    ws[1] = rng.normal(0, 0.1, K).astype(np.float32)
    ref.set_weights(ws)
    bn = torch.nn.BatchNorm1d(K, eps=1e-3, momentum=0.01)
    dims = [K] + [H] * L + [2, 2]
    lins = [torch.nn.Linear(dims[i], dims[i + 1]) for i in range(L + 2)]
    with torch.no_grad():
        bn.weight.copy_(torch.tensor(ws[0]))
        bn.bias.copy_(torch.tensor(ws[1]))
        for i, lin in enumerate(lins):
            lin.weight.copy_(torch.tensor(ws[4 + 2 * i]).T)
            lin.bias.copy_(torch.tensor(ws[5 + 2 * i]))
    params = [bn.weight, bn.bias] + [p for lin in lins for p in (lin.weight, lin.bias)]
    opt = torch.optim.Adam(params, lr=1e-3, betas=(0.9, 0.999), eps=1e-7)
    bn.train()
    for t in range(1, steps + 1):
        x = rng.integers(0, 3, size=(B, K)).astype(np.uint8)
        y = rng.normal(size=(B, 2)).astype(np.float32)
        for g in opt.param_groups:
            g["eps"] = 1e-7 / math.sqrt(1.0 - 0.999 ** t)
        opt.zero_grad()
        a = bn(torch.tensor(x, dtype=torch.float32))
        for lin in lins[:L]:
            a = torch.nn.functional.elu(lin(a))
        out = lins[L + 1](lins[L](a))
        loss = torch.sqrt(((out - torch.tensor(y)) ** 2).sum(-1)).mean()
        loss.backward()
        opt.step()
        loss_ref = ref.train_step(x, y, np.ones((B, H), bool))
        assert abs(loss.item() - loss_ref) <= 2e-5 * max(1.0, abs(loss_ref)), t
    got = ref.get_weights()
    np.testing.assert_allclose(got[0], bn.weight.detach().numpy(), rtol=2e-4, atol=2e-6)
    np.testing.assert_allclose(got[1], bn.bias.detach().numpy(), rtol=2e-4, atol=2e-6)
    np.testing.assert_allclose(got[2], bn.running_mean.numpy(), rtol=1e-5, atol=1e-7)
    for i, lin in enumerate(lins):
        np.testing.assert_allclose(got[4 + 2 * i], lin.weight.detach().numpy().T, rtol=2e-4, atol=3e-6)
        np.testing.assert_allclose(got[5 + 2 * i], lin.bias.detach().numpy(), rtol=2e-4, atol=3e-6)
    # the weights really moved (6 Adam steps of ~lr each)
    assert np.abs(got[4] - ws[4]).max() > 2e-3
