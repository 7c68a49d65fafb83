#!/usr/bin/env python3
"""Benchmark of the Locator training hot path (BASELINE.json metric: train samples/s per model).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg2|cfg3|fixture]
                    [--dump-outputs DIR]

A "step" is one optimizer step of one model (batch 32) on BASELINE config[1]: 1,000 samples x
100,000 SNPs (810 train / 90 validation rows), nlayers=10, width=256.  The timed region runs exactly
K consecutive steps of model.fit's schedule through the C ABI (loc_train_steps: the production path
-- every first-layer backward also runs the next step's forward; whenever the K steps cross the end
of an epoch, that epoch's validation pass, callbacks and checkpoint are inside the timed region, as
in the reference's model.fit) on data already resident in HBM.  N > 1: every rank trains its own
model on its own GPU (replicates are independent; no collective on the training path) -> weak scaling.

--dump-outputs DIR: after the timed steps, rank 0 writes what they left in its model as float32 DIR/<name>.npy (see
dump_outputs).  The inputs depend only on the arguments (fixed seeds), so two builds can be compared output for output.

Printed JSON line (rank 0): the metric (`value`, samples/s), the run's settings and clocks, and extra objects:
  e2e          the public API end to end: LocatorModel(...) creation + init + fit() for >= 20 epochs on
               PAGEABLE host numpy matrices (H2D, 2-bit pack, epochs incl. validation, history D2H)
  roofline     the first-layer backward + Adam kernel (24*K*H bytes per launch) timed alone, CUDA events
  work_queue   BASELINE config[3] (--bootstrap --nboots 64 on the same matrix, 20 epochs per model) through
               the replicate work queue of locator_b200.replicates, the ranks of this job as its workers
  replicate_group / tensor_parallel / large_batch   side measurements (several models per GPU; one model over N GPUs;
               --batch_size 64 and 256)
  cpu_baseline the oracle (torch-CPU fp32 restatement of the Keras path; TF is not installable on this
               image) on a bounded number of steps
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n_total, K)  -> 10% NA-location rows, train_split 0.9 (SURVEY.md section 8 table)
    "fixture": (500, 5830),
    "cfg2": (1000, 100_000),
    "cfg3": (2500, 200_000),
}
H, L, B = 256, 10, 32


def split_sizes(n_total):
    known = n_total - n_total // 10
    nval = round((1 - 0.9) * known)
    return known - nval, nval


def synth(n, K, seed):
    """Synthetic genotypes with spatial structure (SURVEY.md 8d), uint8 [n, K] + z-scored locations."""
    rng = np.random.default_rng(seed)
    loc = rng.uniform(0, 50, size=(n, 2))
    z = (loc - 25.0) / 14.0
    x = np.empty((n, K), dtype=np.uint8)
    for k0 in range(0, K, 20000):
        k1 = min(K, k0 + 20000)
        c = rng.normal(0, 1.5, k1 - k0)
        a = rng.normal(0, 0.5, k1 - k0)
        b = rng.normal(0, 0.5, k1 - k0)
        p = 1.0 / (1.0 + np.exp(-(c[None, :] + z[:, :1] * a[None, :] + z[:, 1:] * b[None, :])))
        x[:, k0:k1] = rng.binomial(2, p).astype(np.uint8)
    y = ((loc - loc.mean(0)) / loc.std(0)).astype(np.float32)
    return x, y


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.samples.append([t.strip() for t in line.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=10)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[1]))
                mx.append(float(s[2]))
                for nm, v in zip(names, s[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def max_over_ranks(value, device):
    """MAX over ranks of a per-rank scalar (step time): the job is as slow as its slowest rank."""
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return float(value)
    t = torch.tensor([float(value)], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def aggregate_value(world, steps, batch, ms):
    """Whole-job samples/s: every rank trains its own model (weak scaling), time = max over ranks."""
    return world * steps * batch / (ms / 1000.0)


def cpu_steps(x, y, xv, yv, nsteps, threads):
    """Oracle (reference restatement) timed on the host cores: nsteps optimizer steps."""
    import torch
    from oracle import model_ref

    torch.set_num_threads(threads)
    K = x.shape[1]
    rng = np.random.default_rng(0)
    ref = model_ref.RefLocator(K, H, L, dropout=0.25, seed=1)
    n = len(x)
    perm = rng.permutation(n)
    ref.train_step(x[perm[:B]], y[perm[:B]], rng.uniform(size=(B, H)) >= 0.25)  # warm-up
    t0 = time.perf_counter()
    done = 0
    while done < nsteps:
        perm = rng.permutation(n)
        for s in range(0, n, B):
            rows = perm[s:s + B]
            ref.train_step(x[rows], y[rows], rng.uniform(size=(len(rows), H)) >= 0.25)
            done += 1
            if done >= nsteps:
                break
    dt = time.perf_counter() - t0
    return done * B / dt, dt


def workload_string(workload):
    """config.workload, the same text in both arms."""
    n_total, K = WORKLOADS[workload]
    ntr, nva = split_sizes(n_total)
    return (f"{workload}: {n_total} samples x {K} SNPs ({ntr} train / {nva} val), 1 model per GPU, batch {B}, "
            f"nlayers {L}, width {H}")


W1_SAMPLE_ROWS = 16384  # W1 is K x 256 float32 (100 MB at cfg2): a fixed sample of its SNP rows is dumped


def dump_outputs(m, out_dir):
    """What a caller of the timed loc_train_steps calls receives from the model after the last step, as float32
    .npy files: every weight array in Keras order and the last step's loss.  Every array's shape depends on the
    workload only (the per-epoch history is left out: it is empty when the run ends inside its first epoch).  W1 is
    cut to W1_SAMPLE_ROWS rows drawn with default_rng(0), so that the whole dump stays below 64 MB at every workload."""
    os.makedirs(out_dir, exist_ok=True)
    out = {"last_loss": np.array([m.state().last_loss], np.float32)}
    for i, w in enumerate(m.get_weights()):
        if i < 4:
            name = ("bn_gamma", "bn_beta", "bn_moving_mean", "bn_moving_var")[i]
        else:
            d, isb = divmod(i - 4, 2)
            name = f"dense{d + 1:02d}_{'bias' if isb else 'kernel'}"
        if i == 4:
            rows = np.sort(np.random.default_rng(0).choice(m.K, min(m.K, W1_SAMPLE_ROWS), replace=False))
            w, name = w[rows], name + "_sampled_rows"
        out[f"w{i:02d}_{name}"] = w
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def run_reference(args, workload):
    """--impl reference: the reference's algorithm on the host CPU (oracle port; TF/Keras cannot be
    installed on this image -- no wheel, no network), all host threads, bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    n_total, K = WORKLOADS[workload]
    ntr, nva = split_sizes(n_total)
    x, y = synth(ntr + nva, K, 1002)
    threads = os.cpu_count() or 1
    # each bench "step" = a bounded sample of 4 optimizer steps, so the run ends within minutes
    per = 4
    total = (args.steps + args.warmup) * per
    total = min(total, 400)
    t_w = max(1, args.warmup * per)
    cpu_steps(x[:ntr], y[:ntr], x[ntr:], y[ntr:], min(t_w, 8), threads)
    nst = max(4, min(args.steps * per, 240))
    val, dt = cpu_steps(x[:ntr], y[:ntr], x[ntr:], y[ntr:], nst, threads)
    line = {
        "impl": "reference", "metric": "train_samples_per_sec", "value": val, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * B / val,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(workload)},
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{nst} optimizer steps of the oracle (torch-CPU fp32 restatement of the Keras "
                                   f"path; TensorFlow not installable here) in {dt:.1f} s"},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def work_queue_leg(rank, world, store, barrier, n_total, K, group):
    """BASELINE config[3]: `locator --bootstrap --nboots 64 --max_epochs 20 --patience 1000 --seed 12345` on the
    synthetic 1,000 x 100,000 matrix, from the packed matrix in HBM to the last replicate's output files,
    through the product's replicate work queue (locator_b200.replicates: serve() + RankQueue -- the ranks of
    this job are the queue's workers, one per GPU; `locator --gpus N` runs the same loop in spawned workers).
    Every rank derives the same split and bootstrap site orders from numpy's seeded legacy stream, as the
    reference's loop does (locator.py:609-681); no collective, the only shared state is the queue's counter."""
    import contextlib
    import glob
    import shutil

    import torch
    from locator_b200 import locator as Lmod, replicates
    from locator_b200.genotypes import PackedGenotypes

    nboots, epochs = 64, 20
    tmp = f"/tmp/locbench_{os.environ.get('MASTER_PORT', 'solo')}_{os.getppid() if world > 1 else os.getpid()}"
    if rank == 0:
        shutil.rmtree(tmp, ignore_errors=True)
        os.makedirs(tmp, exist_ok=True)
    barrier()
    argv = ["--matrix", "synthetic", "--sample_data", "synthetic", "--out", os.path.join(tmp, "cfg4"), "--bootstrap",
            "--nboots", str(nboots), "--max_epochs", str(epochs), "--patience", "1000", "--seed", "12345",
            "--plot_history", "", "--keras_verbose", "0", "--replicates_per_gpu", str(group)]
    Lmod.set_args(Lmod.build_parser().parse_args(argv))
    x, yz = synth(n_total, K, 1002)
    locs = yz.astype(np.float64)
    locs[: n_total // 10] = np.nan  # the first 10 % of the samples are the ones to predict
    samples = np.array([f"s{i:04d}" for i in range(n_total)])
    with contextlib.redirect_stdout(sys.stderr):  # the mirrored functions print like the reference
        np.random.seed(12345)
        meanlong, sdlong, meanlat, sdlat, nlocs = Lmod.normalize_locs(locs)
        ac = Lmod.AlleleCounts(PackedGenotypes.from_counts(x))
        train, test, traingen, testgen, trainlocs, testlocs, pred, predgen = Lmod.split_train_test(ac, nlocs)
        base = {"traingen": traingen, "testgen": testgen, "predgen": predgen, "trainlocs": trainlocs,
                "testlocs": testlocs, "norm": (meanlong, sdlong, meanlat, sdlat), "pred": pred, "samples": samples}
        orders = replicates.draw_bootstrap_orders(traingen.K, nboots)
        items = [{"kind": "full", "boot": "FULL"}] + [{"kind": "boot", "boot": b, "site_order": o}
                                                      for b, o in enumerate(orders)]
        # warm-up: one short group per rank (lazy imports, first launches, allocator growth)
        Lmod.args.max_epochs = 2
        replicates.run_items_ranked(Lmod, base, items[1:1 + min(group, 2)], 1, None)
        Lmod.args.max_epochs = epochs
        torch.cuda.synchronize()
        barrier()
        if rank == 0:
            for f in glob.glob(os.path.join(tmp, "*")):
                os.remove(f)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record()
        prof = None
        if os.environ.get("LOC_BENCH_PROFILE"):  # where does the host side of the queue spend its time?
            import cProfile

            prof = cProfile.Profile()
            prof.enable()
        taken = replicates.run_items_ranked(Lmod, base, items, world, store, key="bench_cfg4")
        if prof is not None:
            import pstats

            prof.disable()
            pstats.Stats(prof, stream=sys.stderr).sort_stats("cumulative").print_stats(45)
        ev1.record()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    dt_max = max_over_ranks(dt, "cuda")
    dev_max = max_over_ranks(ev0.elapsed_time(ev1) / 1000.0, "cuda")
    mine = float(sum(len(g) for g in taken))
    most = max_over_ranks(mine, "cuda")
    barrier()
    n_models = len(items)
    out = None
    if rank == 0:
        files = glob.glob(os.path.join(tmp, "cfg4_boot*_predlocs.txt"))
        assert len(files) == n_models, f"work queue: {len(files)} prediction files for {n_models} models"
        ntr = traingen.n
        out = {"workload": f"cfg4: --bootstrap --nboots {nboots} (+ the FULL model) on {n_total} x {K}, --max_epochs "
                           f"{epochs} --patience 1000 --seed 12345, {group} replicates per GPU side by side",
               "models": n_models, "epochs_per_model": epochs, "seconds": dt_max, "device_seconds": dev_max,
               "models_per_hour": n_models * 3600.0 / dt_max,
               "train_samples_per_sec": n_models * epochs * ntr / dt_max, "scaling": "strong",
               "models_on_busiest_gpu": int(most),
               "granularity_bound": n_models / (world * float(-(-n_models // world))),
               "what": "timed: packed matrix resident -> bootstrap column gathers, model creation, 20 epochs incl. "
                       "validation, best-epoch reload, prediction, *_predlocs.txt / *_history.txt written; wall "
                       "clock, max over ranks; queue = locator_b200.replicates.RankQueue (guided group sizes)"}
        shutil.rmtree(tmp, ignore_errors=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=520)
    ap.add_argument("--warmup", type=int, default=52)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=100)
    ap.add_argument("--no-tp", action="store_true", help="skip the sharded-model measurement at N > 1")
    ap.add_argument("--no-queue", action="store_true", help="skip the cfg4 work-queue measurement")
    ap.add_argument("--no-large-batch", action="store_true", help="skip the --batch_size 64 / 256 side measurement")
    ap.add_argument("--e2e-epochs", type=int, default=20)
    ap.add_argument("--group", type=int, default=4, help="replicates per GPU for the group / work-queue measurements (0/1 = skip the group leg)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed model's outputs after its last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the CUDA model of --impl b200")
    workload = args.workload
    if args.impl == "reference":
        run_reference(args, workload)
        return

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    store = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        store = dist.distributed_c10d._get_default_store()

    from locator_b200 import model, _cabi
    lib = _cabi.lib

    n_total, K = WORKLOADS[workload]
    ntr, nva = split_sizes(n_total)
    spe = (ntr + B - 1) // B  # steps per epoch
    x, y = synth(ntr + nva, K, 1002 + rank)
    xtr, ytr, xva, yva = x[:ntr], y[:ntr], x[ntr:], y[ntr:]

    steps, warm = args.steps, max(3, args.warmup)
    n_ep_total = (steps + warm) // spe + 3
    m = model.LocatorModel(K, width=H, nlayers=L, dropout_prop=0.25, batch_size=B, max_epochs=n_ep_total + 2,
                           seed=100 + rank)
    gtr = m.bind_train(xtr, ytr)
    m.bind_val(xva, yva)
    m.set_schedule(patience=10 ** 6)
    rng = np.random.default_rng(7 + rank)
    stream = torch.cuda.current_stream().cuda_stream

    # the run is model.fit's sequence of steps: epoch e visits perms[e] in slices of 32; warm-up = its first
    # `warm` steps, timed region = the next `steps` steps (continuing inside the epoch the warm-up stopped in)
    perms = torch.as_tensor(np.stack([rng.permutation(ntr) for _ in range(n_ep_total)]).astype(np.int32)).cuda()

    def segments(g0, g1):
        """global steps [g0, g1) -> [(epoch, first step, count)], at most one segment per epoch"""
        out = []
        g = g0
        while g < g1:
            e, s0 = divmod(g, spe)
            n = min(spe - s0, g1 - g)
            out.append((e, s0, n))
            g += n
        return out

    def run(segs):
        for e, s0, n in segs:
            _cabi.check(lib.loc_train_steps(m._h, perms[e].data_ptr(), s0, n, stream), "loc_train_steps")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    timed = segments(warm, warm + steps)
    epoch_ends = sum(1 for e, s0, n in timed if s0 + n == spe)
    run(segments(0, warm))
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = _cabi.launch_count()
    with ClockSampler(local) as clk:
        ev0.record()
        run(timed)
        ev1.record()
        torch.cuda.synchronize()
    launches = _cabi.launch_count() - l0
    ms = max_over_ranks(ev0.elapsed_time(ev1), "cuda")
    st = m.state()
    assert st.t == warm + steps, (st.t, warm, steps)
    assert st.nonfinite == 0 and np.isfinite(st.last_loss), "non-finite loss during the timed region"
    value = aggregate_value(world, steps, B, ms)
    if args.dump_outputs and rank == 0:
        dump_outputs(m, args.dump_outputs)  # before the roofline launches below change the model

    # ---- roofline: first-layer backward + Adam alone, CUDA events on the launching stream ----
    rows_dev = torch.as_tensor(rng.permutation(ntr)[:B].astype(np.int32)).cuda()
    for stage in (0, 1):
        _cabi.check(lib.loc_debug_stage(m._h, stage, rows_dev.data_ptr(), B, stream), "loc_debug_stage")
    reps = 20

    def time_stage(stage, warmups=0, as_in_training=False):
        """mean launch duration (ms) of one stage, CUDA events on the launching stream.  as_in_training: a hidden-stack
        launch (untimed) precedes every timed launch, as in a training step -- it advances the optimizer step, so
        the backward walks its tiles in alternating order and meets the previous launch's tail in L2."""
        for _ in range(warmups):
            _cabi.check(lib.loc_debug_stage(m._h, stage, rows_dev.data_ptr(), B, stream), "loc_debug_stage")
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in evs:
            if as_in_training:
                _cabi.check(lib.loc_debug_stage(m._h, 1, rows_dev.data_ptr(), B, stream), "loc_debug_stage")
            a.record()
            _cabi.check(lib.loc_debug_stage(m._h, stage, rows_dev.data_ptr(), B, stream), "loc_debug_stage")
            b.record()
        torch.cuda.synchronize()
        return float(np.mean([a.elapsed_time(b) for a, b in evs]))

    tc = m.impl == "tcgen05"
    bwd_back_to_back_ms = time_stage(2, 3)
    bwd_ms = time_stage(2, 3, as_in_training=True)
    fwd_ms = time_stage(0)
    hid_ms = time_stage(1)
    fus_ms = time_stage(4, 3, as_in_training=True) if tc else None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    alg_bytes = 24.0 * K * H
    # the launch the production schedule issues 25 times out of 26: backward + Adam + the NEXT step's forward
    # on the chunks it has just updated (tcgen05 path); algorithmic bytes stay those of the backward + Adam alone
    kern_ms = fus_ms if tc else bwd_ms
    achieved = alg_bytes / (kern_ms / 1000.0) / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "l1_backward_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            if tj.get("K") == K:
                traffic = tj.get("dram_bytes_per_launch")
                traffic_src = f"ncu --set full capture of commit {tj.get('commit', '?')} ({tj.get('source', tpath)})"
        except Exception:
            pass
    roofline = {"bound": "hbm",
                "kernel": ("tc::k_l1_bwd_tc: first-layer backward + Adam with the next step's forward fused in"
                           if tc else "l1_backward_adam(simt)"),
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": kern_ms,
                "timing": "CUDA events around each launch on its stream, mean of %d; a hidden-stack launch between "
                          "timed launches as in training (alternating tile walk)" % reps,
                "plain_backward": {"kernel_ms": bwd_ms, "achieved": alg_bytes / (bwd_ms / 1000.0) / 1e9,
                                   "frac": alg_bytes / (bwd_ms / 1000.0) / 1e9 / peak,
                                   "back_to_back_ms": bwd_back_to_back_ms},
                "fused_as_forward_plus_backward_frac": (28.0 * K * H / (kern_ms / 1000.0) / 1e9 / peak) if tc else None,
                "stage_ms": {"l1_forward": fwd_ms, "hidden": hid_ms, "l1_backward": bwd_ms,
                             "l1_backward_with_fused_next_forward": fus_ms},
                "step_roofline_frac": (28.0 * K * H / 1e9 / peak) / (ms / 1000.0 / steps)}
    del m

    # ---- e2e: the public API on PAGEABLE host arrays: model creation + init + fit + history ----
    ne = max(args.e2e_epochs, -(-steps // spe))
    mw = model.LocatorModel(K, width=H, nlayers=L, dropout_prop=0.25, batch_size=B, max_epochs=2, seed=299 + rank)
    mw.fit(xtr, ytr, epochs=1, validation_data=(xva, yva), patience=10 ** 6)  # warm-up of the same call
    del mw
    e2e_runs = []
    for rep in range(3):  # median of three whole calls: pageable host copies make single runs noisy
        barrier()
        t0 = time.perf_counter()
        m2 = model.LocatorModel(K, width=H, nlayers=L, dropout_prop=0.25, batch_size=B, max_epochs=ne, seed=300 + rank + rep)
        h = m2.fit(xtr, ytr, epochs=ne, validation_data=(xva, yva), patience=10 ** 6)
        torch.cuda.synchronize()
        e2e_runs.append(max_over_ranks(time.perf_counter() - t0, "cuda"))
        assert len(h.history["loss"]) == ne and np.isfinite(h.history["loss"][-1])
        del m2
    dt = float(np.median(e2e_runs))
    nst = ne * spe
    h2d = xtr.nbytes + xva.nbytes + ytr.nbytes + yva.nbytes + ne * ntr * 4
    n_state_reads = -(-ne // 16) + 1
    e2e = {"value": world * ne * ntr / dt, "unit": "samples/s", "h2d_bytes_per_step": h2d / nst,
           "d2h_bytes_per_step": (ne * 12 + 48 * n_state_reads) / nst, "epochs": ne, "seconds": dt,
           "host_memory": "pageable numpy arrays", "runs_seconds": e2e_runs, "seconds_is": "median of 3 whole calls",
           "replicate_models_per_hour_20_epochs": world * 3600.0 / (dt * 20.0 / ne),
           "what": "LocatorModel(...) creation + weight init + fit() on host uint8 matrices: H2D, 2-bit pack, "
                   f"{ne} epochs incl. validation / callbacks / checkpoints, history D2H (model buffers come from "
                   "the library's handle pool after the warm-up call, as for every replicate of a run)"}

    # ---- replicate group: G independent models side by side on this GPU (bootstrap / windows) ----
    group = None
    if args.group > 1 and lib.loc_l1_impl().decode() == "tcgen05":
        G = args.group
        gval = model.PackedGenotypes.from_counts(xva)

        def measure_group(l1_ctas, schedule):
            os.environ["LOC_GROUP_SCHEDULE"] = schedule
            gm = [model.LocatorModel(K, width=H, nlayers=L, dropout_prop=0.25, batch_size=B, max_epochs=16,
                                     seed=500 + rank * 16 + g, l1_ctas=l1_ctas) for g in range(G)]
            for q in gm:
                q.bind_train(gtr, ytr)
                q.bind_val(gval, yva)
                q.set_schedule(patience=10 ** 6)
            ne_g = max(2, min(6, steps // spe))
            prng = np.random.default_rng(77)
            perms_g = [torch.as_tensor(np.stack([prng.permutation(ntr) for _ in range(ne_g + 1)]).astype(np.int32)).cuda()
                       for _ in range(G)]
            handles = (ctypes.c_void_p * G)(*[q._h for q in gm])

            def run_group(ne, skip):
                pp = (ctypes.c_void_p * G)(*[p.data_ptr() + skip * ntr * 4 for p in perms_g])
                _cabi.check(lib.loc_group_train_epochs(handles, G, pp, ne, stream), "loc_group_train_epochs")
            run_group(1, 0)
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            run_group(ne_g, 1)
            g1.record()
            torch.cuda.synchronize()
            gms = max_over_ranks(g0.elapsed_time(g1), "cuda")
            loss = float(gm[0].state().last_loss)
            del gm
            os.environ.pop("LOC_GROUP_SCHEDULE", None)
            return {"epochs": ne_g, "value": world * G * ne_g * ntr / (gms / 1000.0),
                    "ms_per_step_per_replicate": gms / (ne_g * spe * G), "last_loss_model0": loss}

        ring = measure_group(model.spare_cluster_l1_ctas(), "ring")  # first-layer kernels on SMs - 16, as the CLI's replicate runs
        lock = measure_group(148, "lockstep")    # every SM for the first-layer kernels, hidden stacks in one launch
        group = {"replicates_per_gpu": G, "epochs": ring["epochs"], "value": ring["value"],
                 "unit": "samples/s (all replicates)", "ms_per_step_per_replicate": ring["ms_per_step_per_replicate"],
                 "schedule": "ring", "lockstep": lock, "ring": ring,
                 "step_roofline_frac": (28.0 * K * H / 1e9 / peak) / (ring["ms_per_step_per_replicate"] / 1000.0),
                 "note": "last_loss_model0 differs between the schedules because the first-layer CTA count (132 vs "
                         "148) changes the fp32 summation order and Adam amplifies rounding at K = 100k: "
                         "tests/test_gpu_baseline_shapes.py::test_divergence_is_rounding_chaos",
                 "what": "loc_group_train_epochs, ring schedule: hidden stack of model g concurrent with the "
                         "first-layer backward + Adam of model g-1 (132 CTAs); 'lockstep' = the grouped-launch schedule"}

    # ---- --batch_size above 32 (reference flag locator.py:69): whole epochs of model.fit's schedule ----
    large_batch = None
    if world == 1 and not args.no_large_batch:
        large_batch = {"unit": "samples/s", "what": "loc_train_epochs at batch sizes above 32 (csrc/bigbatch.cu: batch statistics "
                       "over the whole step, wide first-layer forward, 32-row chunks through the hidden stack, one "
                       "backward + Adam pass over W1 | m | v); whole epochs incl. validation pass and callbacks"}
        prng = np.random.default_rng(99)
        for bsz in (64, 256):
            bm = model.LocatorModel(K, width=H, nlayers=L, dropout_prop=0.25, batch_size=bsz, max_epochs=16, seed=700)
            bm.bind_train(gtr, ytr)
            bm.bind_val(xva, yva)
            bm.set_schedule(patience=10 ** 6)
            ne_b = 4
            bm.train_epochs(np.stack([prng.permutation(ntr) for _ in range(2)]).astype(np.int32))
            pb = np.stack([prng.permutation(ntr) for _ in range(ne_b)]).astype(np.int32)
            torch.cuda.synchronize()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            bm.train_epochs(pb)
            b1.record()
            torch.cuda.synchronize()
            bms = b0.elapsed_time(b1)
            large_batch[f"batch_{bsz}"] = {"value": ne_b * ntr / (bms / 1000.0), "epochs": ne_b,
                                           "ms_per_step": bms / (ne_b * -(-ntr // bsz)),
                                           "last_loss": float(bm.state().last_loss)}
            del bm

    # ---- cfg4 through the replicate work queue (strong scaling over the ranks) ----
    work_queue = None
    if not args.no_queue and workload == "cfg2" and lib.loc_l1_impl().decode() == "tcgen05":
        try:
            work_queue = work_queue_leg(rank, world, store, barrier, n_total, K, max(1, min(8, args.group or 1)))
        except Exception as exc:  # an extra: never lose the bench line over it
            import traceback

            traceback.print_exc()
            work_queue = {"error": f"{type(exc).__name__}: {exc}"}

    # ---- one model sharded over the ranks (SNP columns; one 32 KB exchange of the Z1 tile per forward) ----
    tp = None
    if world > 1 and lib.loc_l1_impl().decode() == "tcgen05" and not args.no_tp:
        xs, ys = (x, y) if rank == 0 else synth(ntr + nva, K, 1002)  # every shard sees the same samples
        k0, k1 = model.shard_bounds(K, rank, world)
        xt, xv = np.ascontiguousarray(xs[:ntr, k0:k1]), np.ascontiguousarray(xs[ntr:, k0:k1])
        ne_t = max(2, min(10, steps // spe))
        tp_error = None

        def run_tp(exchange):
            tm = model.LocatorModel(k1 - k0, width=H, nlayers=L, dropout_prop=0.25, batch_size=B, max_epochs=64,
                                    seed=900, shard=(k0, K), exchange=exchange)
            tm.bind_train(xt, ys[:ntr])
            tm.bind_val(xv, ys[ntr:])
            tm.set_schedule(patience=10 ** 6)
            prng = np.random.default_rng(4242)  # the same batch order on every shard
            pw = np.stack([prng.permutation(ntr) for _ in range(2)]).astype(np.int32)
            pt = np.stack([prng.permutation(ntr) for _ in range(ne_t)]).astype(np.int32)
            barrier()  # every shard is ready: nobody spins in the exchange while a peer is still setting up
            tm.train_epochs(pw)
            barrier()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            tm.train_epochs(pt)
            t1.record()
            torch.cuda.synchronize()
            tms = max_over_ranks(t0.elapsed_time(t1), "cuda")
            st_t = tm.state()
            assert st_t.nonfinite == 0 and np.isfinite(st_t.last_loss), "non-finite loss in the sharded run"
            barrier()
            del tm
            return {"value": ne_t * ntr / (tms / 1000.0), "ms_per_step": tms / (ne_t * spe)}

        try:
            peer = run_tp("peer")
            hook = run_tp(model.all_reduce_exchange())
        except Exception as exc:  # the sharded measurement is an extra: never lose the bench line over it
            peer = hook = None
            tp_error = f"{type(exc).__name__}: {exc}"
        tp = {"error": tp_error} if peer is None else {
            "shards": world, "epochs": ne_t, "value": peer["value"], "unit": "samples/s (one model)",
            "ms_per_step": peer["ms_per_step"], "scaling": "strong", "with_nccl_all_reduce_hook": hook,
            "what": "one cfg model sharded over SNP columns: W1 + Adam state K/N per GPU, hidden stack replicated; "
                    "per forward pass every shard pushes its reduced [32][256] first-layer tile into the peers' "
                    "buffers over NVLink (own kernels, cudaIpc peer memory) and the hidden kernel sums them"}

    impl = lib.loc_l1_impl().decode()
    line = {
        "metric": "train_samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": steps,
        "warmup": warm, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "tf32" if impl == "tcgen05" else "f32",
        "data": "synthetic",
        "config": {"workload": workload_string(workload),
                   "l2": "inputs larger than L2 (W1+m+v = %.0f MB per step)" % (12.0 * K * H / 1e6),
                   "steps_per_epoch": spe,
                   "schedule": "model.fit's step sequence through loc_train_steps (production path: fused next "
                               "forward, alternating tile walk); timed steps continue the epoch the warm-up stopped in",
                   "epoch_ends_in_timed_region": epoch_ends,
                   "validation_pass_and_callbacks": "at every epoch end inside the timed region (%d here)" % epoch_ends},
        "clocks": clk.summary(), "gpu_launches": int(launches), "roofline": roofline, "e2e": e2e,
        "work_queue": work_queue, "replicate_group": group, "tensor_parallel": tp, "large_batch": large_batch,
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        val, dt = cpu_steps(xtr, ytr, xva, yva, args.cpu_steps, os.cpu_count() or 1)
        line["cpu_baseline"] = {"value": val, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
                                "sample": f"{args.cpu_steps} optimizer steps of the oracle (torch-CPU fp32 restatement "
                                          f"of the Keras path) on the same workload, {dt:.1f} s"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
