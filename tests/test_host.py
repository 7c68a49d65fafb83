"""CPU: host logic -- C-ABI surface, CLI parser / params.json, readers, replicate work queue
(2 worker processes), multi-rank timing reduction over gloo (world_size 2)."""
import argparse
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_exports_every_declared_symbol():
    """The shared library loads without a GPU and exports exactly what include/locator_b200.h declares."""
    lib_path = os.path.join(ROOT, "locator_b200", "lib", "liblocator_b200.so")
    if not os.path.exists(lib_path):
        subprocess.run(["make", "-C", os.path.join(ROOT, "locator_b200", "csrc"), "-j8"], check=True,
                       capture_output=True)
    header = open(os.path.join(ROOT, "include", "locator_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(loc_[a-z0-9_]+)\s*\(", header))
    from locator_b200 import _cabi

    assert declared == set(_cabi.SIGNATURES), (declared ^ set(_cabi.SIGNATURES))
    for name in declared:
        assert hasattr(_cabi.lib, name)
    assert _cabi.lib.loc_abi_version() == 1
    assert _cabi.lib.loc_l1_impl() in (b"tcgen05", b"simt")
    # loading the library launches nothing; counted in a fresh process, since the counter is per process and GPU
    # tests that ran before this one in the same session have launched kernels
    r = subprocess.run([sys.executable, "-c", "from locator_b200 import _cabi; print(_cabi.lib.loc_launch_count())"],
                       cwd=ROOT, capture_output=True, text=True, check=True)
    assert int(r.stdout) == 0


def test_product_package_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "locator_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f


def test_parser_matches_reference_flags_and_params_json(tmp_path):
    from locator_b200 import locator as L

    ns = L.build_parser().parse_args(["--vcf", "a.vcf", "--sample_data", "s.txt", "--out", str(tmp_path / "o")])
    d = L._params_dict(ns)
    assert list(d.keys()) == [
        "vcf", "zarr", "matrix", "sample_data", "train_split", "windows", "window_start", "window_stop", "window_size",
        "bootstrap", "jacknife", "jacknife_prop", "nboots", "batch_size", "max_epochs", "patience", "min_mac",
        "max_SNPs", "impute_missing", "dropout_prop", "nlayers", "width", "out", "seed", "gpu_number", "plot_history",
        "keep_weights", "load_params", "keras_verbose"]
    assert d["train_split"] == 0.9 and d["window_size"] == 5e5 and d["window_start"] == 0 and d["nboots"] == 50
    assert d["batch_size"] == 32 and d["max_epochs"] == 5000 and d["patience"] == 100 and d["min_mac"] == 2
    assert d["impute_missing"] is False and d["dropout_prop"] == 0.25 and d["nlayers"] == 10 and d["width"] == 256
    assert d["plot_history"] is True and d["keras_verbose"] == 1 and d["seed"] is None
    # the reference's quirks: window_* arrive as strings from the CLI; --plot_history uses type=bool
    ns = L.build_parser().parse_args(["--window_size", "250000", "--plot_history", "False", "--out", "x"])
    assert ns.window_size == "250000" and ns.plot_history is True
    L.set_args(ns)
    ns.out = str(tmp_path / "p")
    L._write_params()
    text = open(str(tmp_path / "p") + "_params.json").read()
    assert text.startswith('{\n  "vcf": null,') and json.loads(text)["window_size"] == "250000"


def test_callback_descriptors_follow_reference_settings(tmp_path):
    from locator_b200 import locator as L

    L.set_args(L.build_parser().parse_args(["--out", str(tmp_path / "o"), "--patience", "100", "--bootstrap"]))
    ck, es, rl = L.load_callbacks(3)
    assert ck.filepath.endswith("_boot3.weights.npz") and es.patience == 100 and rl.patience == 16 and rl.factor == 0.5
    L.set_args(L.build_parser().parse_args(["--out", str(tmp_path / "o"), "--patience", "20"]))
    ck, es, rl = L.load_callbacks(None)
    assert ck.filepath.endswith("o.weights.npz") and rl.patience == 3


def test_normalize_locs_and_window_bounds():
    from locator_b200 import locator as L, replicates

    locs = np.array([[1.0, 2.0], [np.nan, np.nan], [3.0, 6.0]])
    ml, sl, mt, st, out = L.normalize_locs(locs)
    assert (ml, mt) == (2.0, 4.0) and (sl, st) == (1.0, 2.0)
    assert out[0].tolist() == [-1.0, -1.0] and np.isnan(out[1]).all()
    pos = np.array([5, 10, 20, 100, 110, 205])
    assert list(replicates.window_bounds(pos, 0, 205, 100)) == [(0, 0, 2), (100, 3, 4), (200, 5, 5)]


def test_vcf_reader_matches_oracle_reader_and_zarr_round_trip(tmp_path, fixture_gt, golden_dir):
    from locator_b200 import io

    v = io.read_vcf(os.path.join(golden_dir, "data", "test_genotypes.vcf.gz"))
    assert np.array_equal(v["calldata/GT"], fixture_gt["calldata/GT"])
    assert np.array_equal(v["variants/POS"], fixture_gt["variants/POS"]) and (v["samples"] == fixture_gt["samples"]).all()
    # generic path: extra FORMAT keys, missing and multi-digit alleles, unphased, haploid
    txt = ("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\ts1\ts2\ts3\n"
           "1\t10\t.\tA\tC\t.\t.\t.\tGT:DP\t0/1:3\t./.:0\t1|1:9\n"
           "1\t20\t.\tA\tC,G\t.\t.\t.\tDP:GT\t3:0|2\t1:10|1\t2:1\n")
    p = tmp_path / "t.vcf"
    p.write_text(txt)
    g = io.read_vcf(str(p))
    assert g["calldata/GT"].tolist() == [[[0, 1], [-1, -1], [1, 1]], [[0, 2], [10, 1], [1, -1]]]
    assert g["samples"].tolist() == ["s1", "s2", "s3"] and g["variants/POS"].tolist() == [10, 20]
    z = str(tmp_path / "z.zarr")
    io.write_zarr(z, v["calldata/GT"][:1000], v["samples"], v["variants/POS"][:1000], chunk_variants=300)
    back = io.read_zarr(z)
    assert np.array_equal(back["calldata/GT"], v["calldata/GT"][:1000])
    assert [s.decode() for s in back["samples"]] == v["samples"].tolist()
    gen = io.Genotypes(back["calldata/GT"], back["samples"], back["variants/POS"])
    assert gen[10:20].shape == (10, 500, 2) and gen[10:20, :, :].positions.tolist() == v["variants/POS"][10:20].tolist()
    # --matrix: counts -> haplotype pairs (c>=1, c>=2)
    m = tmp_path / "m.txt"
    m.write_text("sampleID\ts1\ts2\ts3\nA\t0\t1\t2\nB\t2\t0\t1\n")
    gm = io.read_matrix(str(m))
    assert gm.gt.tolist() == [[[0, 0], [1, 1]], [[1, 0], [0, 0]], [[1, 1], [1, 0]]] and gm.samples.tolist() == ["A", "B"]


def test_replicate_pool_two_workers(tmp_path):
    """The N > 1 replicate path without GPUs: two worker processes drain the shared queue, every item
    runs exactly once, its result comes back in submission order although items of uneven cost finish out of
    order, a failing item surfaces as an error in the parent."""
    from locator_b200 import replicates

    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    np.random.seed(5)
    orders = replicates.draw_bootstrap_orders(1000, 7)
    np.random.seed(5)
    again = replicates.draw_bootstrap_orders(1000, 7)
    assert all(np.array_equal(a, b) for a, b in zip(orders, again))
    args = argparse.Namespace(out=str(tmp_path))
    pool = replicates.ReplicatePool(2, args, runner="_pool_runner:run")
    for b, o in enumerate(orders):
        pool.submit({"kind": "boot", "boot": b, "site_order": o, "cost": 100 if b == 0 else 1})
    assert pool.close() == list(range(7))
    finished = sorted(range(7), key=lambda b: os.path.getmtime(tmp_path / f"item_{b}.txt"))
    assert finished[-1] == 0  # item 0 (100x the cost) finished last, its result still comes first
    ranks = set()
    for b, o in enumerate(orders):
        rank, s = open(tmp_path / f"item_{b}.txt").read().split()
        assert int(s) == int(o.sum())
        ranks.add(rank)
    assert ranks <= {"0", "1"}
    pool = replicates.ReplicatePool(2, args, runner="_pool_runner:run")
    pool.submit({"kind": "boot", "boot": 0, "site_order": orders[0], "fail": True})
    with pytest.raises(RuntimeError, match="boom"):
        pool.close()


_GLOO_SNIPPET = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
import bench
dist.init_process_group("gloo")
r = dist.get_rank()
t = bench.max_over_ranks(10.0 + r, "cpu")
v = bench.aggregate_value(world=dist.get_world_size(), steps=100, batch=32, ms=t)
if r == 0:
    print("RESULT", t, round(v, 3))
dist.destroy_process_group()
"""


def test_bench_multi_rank_reduction_gloo_world2(tmp_path):
    script = tmp_path / "g.py"
    script.write_text(_GLOO_SNIPPET % ROOT)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("RESULT")][0].split()
    assert float(line[1]) == 11.0                      # max over ranks of the per-rank time
    assert float(line[2]) == round(2 * 100 * 32 / 0.011, 3)  # whole-job samples/s over both ranks


_RANKQUEUE_SNIPPET = r"""
import json, os, sys, time, torch.distributed as dist
sys.path.insert(0, %r)
from locator_b200 import replicates
dist.init_process_group("gloo")
r, w = dist.get_rank(), dist.get_world_size()
store = dist.distributed_c10d._get_default_store()
items = [{"kind": "boot", "boot": b} for b in range(23)]     # every rank derives the same list (seeded draws)
q = replicates.RankQueue(items, w, store, key="t_queue", group=4)
mine = []
while True:
    deep = q.queue_is_deep()
    g = q.take_group()
    if g is None:
        break
    mine.append(([it["boot"] for it in g], deep))
    time.sleep(0.02 * len(g) * (1 + r))                       # ranks of different speed
out = [None] * w
dist.all_gather_object(out, mine)
if r == 0:
    print("RESULT", json.dumps(out))
dist.destroy_process_group()
"""


def test_rank_queue_hands_out_every_item_once_gloo_world2(tmp_path):
    """replicates.RankQueue (the work queue of a torchrun job: bench.py's cfg4 leg, `locator` under torchrun): the
    ranks share nothing but one atomic counter in the job's store.  Two gloo ranks of different speed: every work
    item is taken exactly once, in order inside a group, groups hold at most `group` items and shrink towards the
    end of the queue (guided self-scheduling), and prefetching is only allowed while the queue is deep."""
    script = tmp_path / "q.py"
    script.write_text(_RANKQUEUE_SNIPPET % ROOT)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29534", str(script)],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    import json

    per_rank = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("RESULT")][0][7:])
    taken = [b for groups in per_rank for g, _ in groups for b in g]
    assert sorted(taken) == list(range(23))
    for groups in per_rank:
        assert groups, "both ranks must get work"
        for g, deep in groups:
            assert 1 <= len(g) <= 4 and g == sorted(g)
    sizes_by_first = sorted((g[0], len(g), deep) for groups in per_rank for g, deep in groups)
    assert sizes_by_first[0][1] == 4                      # full groups while the queue is long
    assert sizes_by_first[-1][1] < 4                      # ... smaller ones at its end
    assert any(d for _, _, d in sizes_by_first) and not sizes_by_first[-1][2]
    # a single process (world 1, no store) walks the same queue with a local counter
    from locator_b200 import replicates

    q = replicates.RankQueue([{"boot": b} for b in range(6)], 1, None, group=4)
    assert [len(g) for g in iter(q.take_group, None)] == [4, 2]


def test_summarize_centroids_and_kernel_peaks(tmp_path):
    """Post-hoc summariser (reference locator_py/plot_locator.py:26-134): centroid = mean of the replicate
    predictions; kernel peak = the prediction with the highest Gaussian density (bandwidth 0.2)."""
    import pandas as pd
    from locator_b200 import summarize

    rng = np.random.default_rng(3)
    truth = {"a": (1.0, 2.0), "b": (-3.0, 0.5), "c": (10.0, 10.0)}
    d = tmp_path / "boots"
    d.mkdir()
    for r in range(12):
        rows = []
        for sid, (x, y) in truth.items():
            if sid == "c" and r >= 9:   # three far outliers: pull the centroid, not the density peak
                rows.append((x + 5.0 + r, y - 4.0, sid))
            else:
                rows.append((x + 0.05 * rng.normal(), y + 0.05 * rng.normal(), sid))
        pd.DataFrame(rows, columns=["x", "y", "sampleID"]).to_csv(d / f"run_boot{r}_predlocs.txt", index=False)
    (d / "run_history.txt").write_text("ignored")
    sd = tmp_path / "samples.txt"
    pd.DataFrame([(s, x, y) for s, (x, y) in truth.items()], columns=["sampleID", "x", "y"]).to_csv(sd, sep="\t", index=False)
    assert summarize.main(["--infile", str(d), "--sample_data", str(sd), "--out", str(tmp_path / "s"), "--error", "--silence"]) == 0
    t = pd.read_csv(str(tmp_path / "s_centroids.txt"), sep="\t").set_index("sampleID")
    assert list(t.columns) == ["x", "y", "kd_x", "kd_y", "gc_x", "gc_y"]
    allp = summarize.load_predictions(str(d))
    for sid, (x, y) in truth.items():
        g = allp[allp.sampleID == sid]
        assert t.loc[sid, "gc_x"] == pytest.approx(g.xpred.mean()) and t.loc[sid, "gc_y"] == pytest.approx(g.ypred.mean())
        assert abs(t.loc[sid, "kd_x"] - x) < 0.2 and abs(t.loc[sid, "kd_y"] - y) < 0.2
        assert ((g.xpred == t.loc[sid, "kd_x"]) & (g.ypred == t.loc[sid, "kd_y"])).any()  # a member of the set
    assert abs(t.loc["c", "gc_x"] - 10.0) > 2.0
    # brute-force density check for one sample
    g = allp[allp.sampleID == "a"]
    xs, ys = g.xpred.to_numpy(), g.ypred.to_numpy()
    dens = [np.exp(-((xs - a) ** 2 + (ys - b) ** 2) / (2 * 0.2 ** 2)).sum() for a, b in zip(xs, ys)]
    assert (xs[int(np.argmax(dens))], ys[int(np.argmax(dens))]) == (t.loc["a", "kd_x"], t.loc["a", "kd_y"])


def test_native_vcf_parser_matches_python_reader(tmp_path, monkeypatch):
    """loc_vcf_parse_gt (multithreaded host parser in the library) vs the per-field Python reader on the
    cases allel.read_vcf handles: phased / unphased, missing, haploid, multi-digit alleles, GT not first in
    FORMAT, CRLF line ends, polyploid calls (first two alleles), short lines."""
    import gzip

    from locator_b200 import io

    rng = np.random.default_rng(8)
    n = 7
    lines = ["##fileformat=VCFv4.2", "##source=test",
             "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(f"s{i}" for i in range(n))]
    calls = ["0|1", "1/1", "./.", ".|.", "0", ".", "10/2", "1|0|1", "0/1:35:99", "./.:.:."]
    for v in range(300):
        fmt = "GT" if v % 3 else "GT:DP:GQ"
        row = [str(rng.choice(calls[:8] if fmt == "GT" else calls)) for _ in range(n)]
        if fmt != "GT":
            row = [c if ":" in c else c + ":7:50" for c in row]
        if v % 50 == 7:
            fmt, row = "DP:GT", ["12:" + c.split(":")[0] for c in row]
        lines.append(f"1\t{100 + 13 * v}\t.\tA\tC,G\t.\tPASS\t.\t{fmt}\t" + "\t".join(row))
    lines.append("1\t99999\t.\tA\tC\t.\tPASS\t.\tGT\t0|1\t1|1")  # fewer sample columns: the rest stay missing
    text = ("\r\n".join(lines[:40]) + "\r\n" + "\n".join(lines[40:]) + "\n").encode()
    p = tmp_path / "odd.vcf.gz"
    with gzip.open(p, "wb") as fh:
        fh.write(text)
    fast = io.read_vcf(str(p))
    monkeypatch.setenv("LOC_PY_VCF", "1")
    slow = io.read_vcf(str(p))
    monkeypatch.delenv("LOC_PY_VCF")
    assert fast["calldata/GT"].shape == (301, n, 2) and fast["calldata/GT"].dtype == np.int8
    for k in ("calldata/GT", "samples", "variants/POS"):
        assert np.array_equal(fast[k], slow[k]), k
    assert fast["calldata/GT"].max() == 10 and fast["calldata/GT"].min() == -1
    assert (fast["calldata/GT"][-1, 2:] == -1).all() and list(fast["calldata/GT"][-1, 0]) == [0, 1]
    # a line the native parser declines (no GT key) is left to the Python reader, which raises
    bad = tmp_path / "bad.vcf"
    bad.write_text("\n".join(lines[:3] + ["1\t5\t.\tA\tC\t.\tPASS\t.\tDP\t" + "\t".join(["3"] * n)]) + "\n")
    assert io._read_vcf_native(bad.read_bytes()) is None
    with pytest.raises(ValueError):
        io.read_vcf(str(bad))


def test_lazy_zarr_rows_and_genotype_slices(tmp_path):
    """--windows reads: a variant slice of a zarr-backed Genotypes decodes only the chunks it overlaps and
    equals the slice of the fully loaded array (ragged last chunk, slices inside / across chunks, empty)."""
    from locator_b200 import io

    rng = np.random.default_rng(0)
    gt = rng.integers(-1, 2, size=(1000, 17, 2)).astype(np.int8)
    z = str(tmp_path / "t.zarr")
    io.write_zarr(z, gt, [f"s{i}" for i in range(17)], np.arange(1000) * 3, chunk_variants=128)
    lz = io.read_zarr(z, lazy=True)
    g = io.Genotypes(lz["calldata/GT"], lz["samples"], lz["variants/POS"])
    assert g.shape == (1000, 17, 2) and len(g) == 1000 and g.lazy == (z, "calldata/GT", 0, 1000)
    for a, b in [(0, 1000), (5, 6), (100, 400), (127, 129), (990, 1000), (500, 500)]:
        sub = g[a:b]
        assert sub.lazy == (z, "calldata/GT", a, b) and sub.shape == (b - a, 17, 2)
        assert np.array_equal(sub.gt, gt[a:b]) and sub.lazy is None
        assert np.array_equal(sub.positions, np.arange(1000)[a:b] * 3)
    assert np.array_equal(g[100:400][10:20].gt, gt[110:120])
    # only the overlapping chunk files are opened
    os.remove(os.path.join(z, "calldata", "GT", "0.0.0"))
    assert np.array_equal(g[128:256].gt, gt[128:256])
    assert np.array_equal(g.gt[128:], gt[128:]) and (g.gt[:128] == 0).all()  # missing chunk -> fill value


def test_jacknife_draws_follow_the_reference_stream():
    """The threaded, vectorised draws of the jacknife sweep are the reference's per-site scalar-p draws
    (locator.py:722-727 restated in oracle/ingest_ref.jacknife_replace), replicate after replicate, and leave
    numpy's global stream where the reference's loop leaves it."""
    from locator_b200 import locator as L
    from oracle import ingest_ref

    rng = np.random.default_rng(8)
    n_pred, K = 23, 1200
    predgen = rng.integers(0, 3, size=(n_pred, K), dtype=np.uint8)
    af = rng.uniform(0, 1, size=K)
    af[:40] = 0.0
    af[40:80] = 1.0
    L.set_args(L.build_parser().parse_args(["--out", "x", "--jacknife", "--nboots", "5", "--jacknife_prop", "0.07"]))
    np.random.seed(4242)
    want = [ingest_ref.jacknife_replace(predgen, af, 0.07) for _ in range(5)]
    after_ref = np.random.random()
    np.random.seed(4242)
    got = list(L._jacknife_draws(af, K, n_pred))
    after = np.random.random()
    assert len(got) == 5 and after == after_ref
    for (ref_matrix, ref_sites), (sites, vals) in zip(want, got):
        assert np.array_equal(sites, ref_sites) and vals.shape == (int(K * 0.07), n_pred) and vals.dtype == np.uint8
        mine = predgen.copy()
        mine[:, sites] = vals.T
        assert np.array_equal(mine, ref_matrix)
    # no sites to replace: replicates still come out, the stream still advances like choice(K, 0)
    L.set_args(L.build_parser().parse_args(["--out", "x", "--jacknife", "--nboots", "2", "--jacknife_prop", "0.0"]))
    got = list(L._jacknife_draws(af, K, n_pred))
    assert [v.shape for _, v in got] == [(0, n_pred)] * 2


def test_legacy_binomial_reproduces_numpy_global_stream():
    """nprandom.legacy_binomial (loc_np_legacy_binomial: MT19937 + numpy's inversion sampler restated in the
    library) returns exactly what np.random.binomial returns for scalar-p calls in order, and leaves numpy's
    global stream -- position and cached gaussian included -- where numpy would have left it."""
    from locator_b200.nprandom import legacy_binomial

    rng = np.random.default_rng(21)
    for n in (0, 1, 2, 5, 16, 17, 60, 255):
        hi = min(1.0, 30.0 / max(n, 1))
        p = np.concatenate([rng.uniform(0, hi, 300), 1 - rng.uniform(0, hi, 300),
                            [0.0, 1.0, 0.5, np.nextafter(0.5, 1), 1e-300, 1 - 1e-16]])
        p = p[np.minimum(p, 1 - p) * n <= 30]
        np.random.seed(1000 + n)
        np.random.normal()           # leaves a cached gaussian in the state
        np.random.random(5)          # and a position inside the block of 624
        want = np.stack([np.random.binomial(n, pi, 11) for pi in p])
        after_want = (np.random.normal(), np.random.random())
        np.random.seed(1000 + n)
        np.random.normal()
        np.random.random(5)
        got = legacy_binomial(n, p, 11)
        after_got = (np.random.normal(), np.random.random())
        assert got.dtype == np.uint8 and np.array_equal(got, want) and after_got == after_want
    # several refills of the 624-word state, the config-5 shape of one jacknife replicate (scaled)
    af = rng.uniform(0, 1, 4000)
    np.random.seed(3)
    want = np.random.binomial(2, np.repeat(af, 250)).reshape(-1, 250)
    x = np.random.random()
    np.random.seed(3)
    assert np.array_equal(legacy_binomial(2, af, 250), want) and np.random.random() == x
    # numpy's BTPE branch and wide counts are left to numpy itself -- same values, same stream
    np.random.seed(4)
    want = np.random.binomial(100, np.repeat([0.4, 0.6], 5)).reshape(2, 5)
    x = np.random.random()
    np.random.seed(4)
    assert np.array_equal(legacy_binomial(100, [0.4, 0.6], 5), want) and np.random.random() == x
    assert legacy_binomial(2, [], 7).shape == (0, 7) and legacy_binomial(2, [0.3], 0).shape == (1, 0)
    with pytest.raises(ValueError):
        legacy_binomial(2, [0.2, np.nan], 3)
    with pytest.raises(ValueError):
        legacy_binomial(2, [1.5], 3)


def test_predict_locs_writes_the_reference_bytes(tmp_path, golden_dir, capsys, monkeypatch):
    """Output boundary: tests/golden/ref_out/* and the printed summaries were produced by the REFERENCE'S
    predict_locs (compiled from its source by tests/golden/make_reference_vectors.py) around a stand-in model
    with fixed predictions.  The mirror writes the same bytes -- predlocs / history file names per driver,
    comma vs tab separators, float formatting -- prints the same text and returns the same distances."""
    import json
    from locator_b200 import locator as L

    vec = json.load(open(os.path.join(golden_dir, "reference_vectors.json")))["predict_locs"]
    arr = np.load(os.path.join(golden_dir, "reference_vectors.npz"))
    pg, tg = object(), object()

    class StubModel:
        def predict(self, x):
            return arr["out_p_pred"] if x is pg else arr["out_p_val"]

    class StubHistory:
        history = vec["history"]

    names = np.array([f"msp_{i:02d}" for i in range(30)])
    meanlong, sdlong, meanlat, sdlat = (np.float64(v) for v in vec["norm"])
    monkeypatch.chdir(tmp_path)
    for name, c in vec["cases"].items():
        flags = ["--out", name] + (["--bootstrap"] if c["bootstrap"] else []) + (["--jacknife"] if c["jacknife"] else []) \
            + (["--windows", "--window_start", "0", "--window_size", "250000"] if c["windows"] else [])
        L.set_args(L.build_parser().parse_args(flags))
        capsys.readouterr()
        dists = L.predict_locs(StubModel(), pg, sdlong, meanlong, sdlat, meanlat, arr["out_testlocs"], arr["out_pred_idx"],
                               names, tg, StubHistory(), c["boot"])
        assert capsys.readouterr().out == vec["printed"][name]["stdout"]
        assert [float(d) for d in dists] == vec["printed"][name]["dists"]
    written = sorted(os.listdir(tmp_path))
    assert written == vec["files"]
    for f in written:
        assert open(tmp_path / f, "rb").read() == open(os.path.join(golden_dir, "ref_out", f), "rb").read(), f


def test_command_line_matches_the_reference_parser(golden_dir):
    """The reference's own argparse definition (compiled from its source by make_reference_vectors.py) parsed a set of
    command lines and dumped args.__dict__ the way the reference writes *_params.json (locator.py:181-184): the
    mirror produces the same text -- same flags, defaults, types, key order -- and knows every reference flag."""
    import json
    from locator_b200 import locator as L

    vec = json.load(open(os.path.join(golden_dir, "reference_vectors.json")))
    for case in vec["cli"]:
        ns = L.build_parser().parse_args(case["argv"])
        assert json.dumps(L._params_dict(ns), indent=2) == case["params_json"], case["argv"]
    ours = {a.option_strings[0] for a in L.build_parser()._actions if a.option_strings}
    assert set(vec["cli_help_flags"]) <= ours
    assert ours - set(vec["cli_help_flags"]) == {"--gpus", "--replicates_per_gpu", "--load_weights"}


def test_matrix_reader_matches_the_reference_branch(golden_dir):
    """--matrix: the reference's load_genotypes branch (count table -> haplotype pairs -> genotype cube,
    locator.py:200-227, run by make_reference_vectors.py) against io.read_matrix on the same file."""
    import json
    from locator_b200 import io

    vec = json.load(open(os.path.join(golden_dir, "reference_vectors.json")))["matrix"]
    arr = np.load(os.path.join(golden_dir, "reference_vectors.npz"))
    g = io.read_matrix(os.path.join(golden_dir, "matrix_input.txt"))
    assert list(g.gt.shape) == vec["shape"] and np.array_equal(g.gt, arr["matrix_gt"])
    assert [str(s) for s in g.samples] == vec["samples"]


def test_summariser_matches_the_reference_functions(golden_dir):
    """locator_py/plot_locator.py's kdepred / centroid / distance / distance_km (run with scikit-learn's KernelDensity
    by make_reference_vectors.py on positional arrays) against locator_b200.summarize: same density peak (a member of
    the prediction set), same centroid and distances."""
    import json
    from locator_b200 import summarize as S

    for c in json.load(open(os.path.join(golden_dir, "reference_vectors.json")))["summarize"]:
        xs, ys = np.array(c["x"]), np.array(c["y"])
        tx, ty = c["truth"]
        kx, ky = S.kde_peak(xs, ys)
        assert [kx, ky] == c["kd"]
        gx, gy = S.centroid(xs, ys)
        assert gx == pytest.approx(c["gc"][0], rel=1e-13, abs=1e-13) and gy == pytest.approx(c["gc"][1], rel=1e-13, abs=1e-13)
        assert float(np.hypot(kx - tx, ky - ty)) == pytest.approx(c["kd_dist"], rel=1e-13)
        assert float(np.hypot(gx - tx, gy - ty)) == pytest.approx(c["gc_dist"], rel=1e-12)
        assert float(S.distance_km(kx, ky, tx, ty)) == pytest.approx(c["kd_dist_km"], rel=1e-12)


def test_mirror_asks_its_model_for_what_the_reference_asks_keras_for(golden_dir, capsys, tmp_path):
    """load_callbacks / train_network of the reference, run around recording stand-ins (make_reference_vectors.py):
    callback settings and checkpoint file names per driver, the fit() arguments, the reload of the best weights.
    The mirror passes the same settings to its model (the checkpoint lives in device memory; the weights file,
    when kept, is .npz instead of .h5)."""
    import json
    from locator_b200 import locator as L

    req = json.load(open(os.path.join(golden_dir, "reference_vectors.json")))["keras_requests"]
    for cb in req["callbacks"]:
        flags = ["--out", "o/run", "--patience", str(cb.get("patience", 100))] + (["--bootstrap"] if cb["bootstrap"] else []) \
            + (["--jacknife"] if cb["jacknife"] else [])
        L.set_args(L.build_parser().parse_args(flags))
        ck, es, rl = L.load_callbacks(cb["boot"])
        rck, res, rrl = cb["callbacks"]
        assert ck.filepath == rck["filepath"].replace(".weights.h5", ".weights.npz")
        assert (ck.monitor, ck.save_best_only, ck.save_weights_only) == (rck["monitor"], rck["save_best_only"], rck["save_weights_only"])
        assert (es.monitor, es.min_delta, es.patience) == (res["monitor"], res["min_delta"], res["patience"])
        assert (rl.monitor, rl.factor, rl.patience, rl.min_delta, rl.cooldown, rl.min_lr) == \
            (rrl["monitor"], rrl["factor"], rrl["patience"], rrl["min_delta"], rrl["cooldown"], rrl["min_lr"])

    class StubModel:
        def __init__(self):
            self.kw, self.restored, self.saved = None, 0, []

        def fit(self, x, y, **kw):
            self.kw = kw
            return "HISTORY"

        def restore_best(self):
            self.restored += 1

        def save_weights(self, path):
            self.saved.append(path)

    for tr in req["train_network"]:
        flags = ["--out", str(tmp_path / "run")] + (["--bootstrap"] if tr["bootstrap"] else []) \
            + (["--jacknife"] if tr["jacknife"] else []) + (["--keep_weights"] if tr["keep_weights"] else [])
        L.set_args(L.build_parser().parse_args(flags))
        m = StubModel()
        cbs = L.load_callbacks(tr["boot"])
        hist, back = L.train_network(m, "TRAINGEN", "TESTGEN", "TRAINLOCS", "TESTLOCS", cbs, tr["boot"])
        assert (hist == "HISTORY" and back is m) == tr["returns_history_and_model"]
        want = tr["fit_kwargs"]
        assert m.kw["epochs"] == want["epochs"] and m.kw["batch_size"] == want["batch_size"] and m.kw["shuffle"] is want["shuffle"]
        assert m.kw["validation_data"] == ("TESTGEN", "TESTLOCS") and m.kw["callbacks"] == cbs
        assert m.restored == len(tr["loaded"]) == 1          # model.load_weights(best checkpoint)
        kept = [cbs[0].filepath] if tr["keep_weights"] else []   # the reference deletes the file unless --keep_weights
        assert m.saved == kept and bool(tr["shell"]) == (not tr["keep_weights"])
        assert "run time " in capsys.readouterr().out


def test_legacy_permutation_reproduces_numpy_global_stream():
    """nprandom.legacy_permutation / legacy_choice_without_replacement (numpy's legacy Fisher-Yates restated in the
    library) against np.random.permutation / choice(replace=False), values and stream position."""
    from locator_b200.nprandom import legacy_choice_without_replacement, legacy_permutation

    for n in (0, 1, 2, 3, 7, 100, 624, 625, 5830, 70001):
        np.random.seed(n + 1)
        np.random.normal()
        want, after_want = np.random.permutation(n), np.random.random()
        np.random.seed(n + 1)
        np.random.normal()
        got, after_got = legacy_permutation(n), np.random.random()
        assert got.dtype == np.int64 and np.array_equal(got, want) and after_got == after_want
    np.random.seed(12345)
    want, x = np.random.choice(5830, 291, replace=False), np.random.random()
    np.random.seed(12345)
    assert np.array_equal(legacy_choice_without_replacement(5830, 291), want) and np.random.random() == x
    with pytest.raises(ValueError):
        legacy_choice_without_replacement(10, 11)


def test_keras_weights_converter_host_side(tmp_path):
    """locator_b200.keras_weights: Keras-order npz files, shape checks against the reference network
    (load_network, locator.py:317-326), and a clear refusal where Keras itself is missing."""
    from locator_b200 import keras_weights as kw
    from oracle import model_ref

    ws = model_ref.init_weights(300, width=64, nlayers=4, seed=3)
    assert [tuple(w.shape) for w in ws] == kw.expected_shapes(300, 4, 64)
    p = str(tmp_path / "m.weights.npz")
    kw.write_npz(p, ws)
    back = kw.read_npz(p)
    assert kw.describe(back) == (300, 4, 64)
    assert all(np.array_equal(a, b) for a, b in zip(ws, back))
    with pytest.raises(ValueError):
        kw.describe(ws[:-2] + [np.zeros((3, 2), np.float32), ws[-1]])
    assert kw.main(["describe", p]) == 0
    if kw._keras() is None:
        assert kw.main(["to-h5", p, str(tmp_path / "m.weights.h5")]) == 2


def test_validate_args_limits_of_this_build():
    """Argument limits are checked before any data is read (locator.py:69,371 passes any --batch_size to model.fit;
    here 1..256 -- steps above 32 rows take the chunked path of csrc/bigbatch.cu -- and a clear refusal beyond)."""
    from locator_b200 import locator as L

    def ns(*extra):
        return L.build_parser().parse_args(["--vcf", "x.vcf", "--sample_data", "s.txt", "--out", "o"] + list(extra))

    for ok in ([], ["--batch_size", "1"], ["--batch_size", "64"], ["--batch_size", "256"], ["--width", "96"],
               ["--nlayers", "2"], ["--dropout_prop", "0"], ["--nlayers", "21"], ["--width", "320", "--nlayers", "13"],
               ["--jacknife", "--load_weights", "f"]):
        L.validate_args(ns(*ok))
    for bad, word in ((["--batch_size", "0"], "batch_size"), (["--batch_size", "257"], "batch_size"),
                      (["--width", "100"], "width"), (["--nlayers", "1"], "nlayers"), (["--dropout_prop", "1.0"], "dropout_prop"),
                      (["--max_epochs", "0"], "max_epochs"), (["--windows", "--window_size", "2e5"], "window_size"),
                      # deepest stack per width: the CUDA-core hidden stack's shared-memory layout (loc_hidden_max_nlayers)
                      (["--nlayers", "22"], "at most 21"), (["--width", "512"], "width 512"),
                      (["--width", "224", "--nlayers", "11"], "at most 10"),
                      # replicate runs train every model they predict from
                      (["--bootstrap", "--load_weights", "f"], "load_weights"),
                      (["--windows", "--window_size", "100", "--load_weights", "f"], "load_weights")):
        with pytest.raises(SystemExit, match=word):
            L.validate_args(ns(*bad))
