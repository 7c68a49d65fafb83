"""Launch counts of every host-side schedule in csrc/model.cu.

Each schedule (train_step chained and unchained, the ring and lockstep replicate groups, train_step_big solo and
grouped, infer_rows wide and narrow, the CUDA-core kernels, loc_debug_stage) issues a fixed number of kernel launches
for a given shape.  The counts below are written out from the launches each schedule makes, so a schedule that loses
or gains a launch fails here even when its results stay bit-identical.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

K, NTR, NVA, E = 3001, 200, 40, 2  # 7 steps of 32 rows (the last of 8), one 40-row validation pass, 2 epochs


def cdiv(a, b):
    return -(-a // b)


@pytest.fixture(scope="module")
def M():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from locator_b200 import model

    return model


def _data(seed, ntr=NTR, nva=NVA, k=K):
    from locator_b200.genotypes import PackedGenotypes

    rng = np.random.default_rng(seed)
    x = rng.binomial(2, rng.uniform(0.05, 0.95, k), size=(ntr + nva, k)).astype(np.uint8)
    y = rng.normal(size=(ntr + nva, 2)).astype(np.float32)
    return PackedGenotypes.from_counts(x[:ntr]), y[:ntr], PackedGenotypes.from_counts(x[ntr:]), y[ntr:]


def _launches(fn):
    from locator_b200 import _cabi

    torch.cuda.synchronize()
    l0 = _cabi.launch_count()
    fn()
    torch.cuda.synchronize()
    return _cabi.launch_count() - l0


def _fit(m, d):
    return _launches(lambda: m.fit(d[0], d[1], epochs=E, validation_data=(d[2], d[3])))


def _fit_group(M, ms, ds):
    return _launches(lambda: M.fit_group(ms, [d[0] for d in ds], [d[1] for d in ds], [(d[2], d[3]) for d in ds], epochs=E))


def _tcgen05(m):
    if (m.impl, m.hidden_impl) != ("tcgen05", "tcgen05"):
        pytest.skip("needs the tcgen05 kernels")


STEPS = cdiv(NTR, 32)
VAL_WIDE = 3                  # one pass of 40 rows: wide forward, grouped hidden stacks, validation sums in order
VAL_NARROW = 2 * cdiv(NVA, 32)  # per 32 rows: forward, hidden stack
EPOCH_END = 2                 # epoch end + checkpoint copy


def test_solo_schedules(M, monkeypatch):
    d = _data(0)
    m = M.LocatorModel(K, nlayers=4, seed=1, max_epochs=2 * E)
    _tcgen05(m)
    # set_schedule, begin of the call; per epoch: forward of the first step (later ones are fused into the previous
    # step's backward), hidden stack + small-layer update + first-layer backward per step, validation, epoch end
    per_fit = 2 + E * (1 + 3 * STEPS + VAL_WIDE + EPOCH_END)
    monkeypatch.delenv("LOC_NO_CHAIN", raising=False)
    assert _fit(m, d) == per_fit
    monkeypatch.setenv("LOC_NO_CHAIN", "1")  # the update on the side stream instead of the chain: the same launches
    assert _fit(m, d) == per_fit
    monkeypatch.delenv("LOC_NO_CHAIN")
    rows = np.arange(32)
    # loc_train_step: forward, hidden stack, update, backward (no fused forward across calls)
    assert _launches(lambda: [m.train_step(rows) for _ in range(3)]) == 3 * 4
    for stage in range(5):  # forward | hidden stack | backward | update | backward with the fused forward
        assert _launches(lambda: m.debug_stage(stage, rows)) == 1, stage


@pytest.mark.parametrize("schedule,G", [("ring", 2), ("ring", 3), ("lockstep", 2), ("lockstep", 3)])
def test_group_schedules(M, monkeypatch, schedule, G):
    ds = [_data(10 + g) for g in range(G)]
    ms = [M.LocatorModel(K, nlayers=4, seed=1 + g, max_epochs=E) for g in range(G)]
    _tcgen05(ms[0])
    monkeypatch.setenv("LOC_GROUP_SCHEDULE", schedule)
    if schedule == "ring":  # per model: first forward, then hidden stack, backward, update per step
        per_epoch = G * (1 + 3 * STEPS)
    else:  # forwards of the first step; per step one grouped hidden launch, then an update and a backward per model
        per_epoch = G + STEPS * (1 + 2 * G)
    # set_schedule and begin of the call per model; validation and epoch end per model
    assert _fit_group(M, ms, ds) == 2 * G + E * (per_epoch + G * (VAL_WIDE + EPOCH_END))


def _big_step(nc, G, serial):
    """Launches of one large-batch step of G models with nc 32-row chunks (train_step_big)."""
    if not serial and nc > 1:  # chunks side by side: whole models per grouped hidden launch, one step end
        hidden = cdiv(G, 8 // nc) + 1
    else:  # one hidden-stack launch per chunk
        hidden = G * nc
    return (1          # batch statistics of all models
            + G        # wide first-layer forward per model
            + hidden
            + 2 * G    # first-layer backward + gamma / beta per model
            + G)       # small-layer update per model


@pytest.mark.parametrize("serial", [False, True])
@pytest.mark.parametrize("B,ntr", [(64, 300), (256, 600)])
def test_large_batch_schedules(M, monkeypatch, B, ntr, serial):
    G = 2
    ds = [_data(20 + g, ntr=ntr) for g in range(G)]
    chunks = [cdiv(min(B, ntr - off), 32) for off in range(0, ntr, B)]
    if serial:
        monkeypatch.setenv("LOC_BB_SERIAL", "1")
    else:
        monkeypatch.delenv("LOC_BB_SERIAL", raising=False)
    solo = M.LocatorModel(K, nlayers=4, batch_size=B, seed=1, max_epochs=E)
    _tcgen05(solo)
    assert _fit(solo, ds[0]) == 2 + E * (sum(_big_step(nc, 1, serial) for nc in chunks) + VAL_WIDE + EPOCH_END)
    ms = [M.LocatorModel(K, nlayers=4, batch_size=B, seed=1 + g, max_epochs=E) for g in range(G)]
    assert _fit_group(M, ms, ds) == 2 * G + E * (sum(_big_step(nc, G, serial) for nc in chunks)
                                                + G * (VAL_WIDE + EPOCH_END))


def test_predict_schedules(M, monkeypatch):
    from locator_b200.genotypes import PackedGenotypes

    n = 300
    x = np.random.default_rng(5).binomial(2, 0.3, size=(n, K)).astype(np.uint8)
    xs = [PackedGenotypes.from_counts(x) for _ in range(2)]  # two matrices: predict memoizes per matrix
    m = M.LocatorModel(K, nlayers=4, seed=1)
    _tcgen05(m)
    monkeypatch.delenv("LOC_NO_WIDE", raising=False)
    assert _launches(lambda: m.predict(xs[0])) == 2 * cdiv(n, 256)  # per 256 rows: wide forward, grouped hidden
    monkeypatch.setenv("LOC_NO_WIDE", "1")
    assert _launches(lambda: m.predict(xs[1])) == 2 * cdiv(n, 32)  # per 32 rows: forward, hidden stack


def test_cuda_core_schedules(M):
    d = _data(30)
    m = M.LocatorModel(K, width=128, nlayers=4, seed=1, max_epochs=E)
    assert (m.impl, m.hidden_impl) == ("simt", "simt")
    # no fused forward: forward, hidden stack, update, backward per step; narrow validation
    assert _fit(m, d) == 2 + E * (4 * STEPS + VAL_NARROW + EPOCH_END)
    assert _launches(lambda: m.predict(d[2])) == VAL_NARROW
