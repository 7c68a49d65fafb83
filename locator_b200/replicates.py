"""Replicate drivers: --bootstrap and --windows runs of the reference are loops over independent
models (/root/reference/locator/locator.py:519-583 windows, :609-681 bootstrap).  Here the
independent models (and the folds of locator_b200.holdout) are work items handed to run_work, which
serves them in this process with one GPU and from one worker process per GPU with ``--gpus N``;
there is no collective on the training path.  Everything that consumes numpy's
global random stream (bootstrap reseeds + site orders, per-window imputation / subsample / split)
is drawn serially in the parent, in the reference's order, and shipped with the work item, so the
indices do not depend on the number of GPUs.
"""
from __future__ import annotations

import copy
import itertools
import os
import time
import traceback

import numpy as np

from . import sites

def _tick(what):
    """LOC_TIMING=1: wall-clock milestones of the replicate drivers on stderr (seconds since the epoch, so the
    lines of the parent and the workers interleave on one axis)."""
    if os.environ.get("LOC_TIMING"):
        import sys

        print(f"[loc-timing {time.time():.3f} pid {os.getpid()}] {what}", file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------------
# (de)serialisation of packed device matrices for the worker processes
# ---------------------------------------------------------------------------------------------
# the packed device matrices a base dict or a work item may hold ("genotypes": the whole filtered matrix of a
# k-fold holdout run, whose folds are row gathers of it)
_MATRICES = ("traingen", "testgen", "predgen", "genotypes")


def _to_host(g):
    return {"words": g.words.cpu().numpy(), "n": g.n, "K": g.K}


def _to_dev(h):
    import torch
    from .genotypes import PackedGenotypes

    return PackedGenotypes(torch.as_tensor(h["words"]).cuda(), h["n"], h["K"])


def _convert(d, fn):
    """Copy of a base dict or work item (or None) with its packed matrices converted by fn (_to_host / _to_dev)."""
    return None if d is None else {k: fn(v) if k in _MATRICES else v for k, v in d.items()}


def draw_bootstrap_orders(nsites, nboots):
    """The reference's draws for every replicate, in order (locator.py:637, :648-650):
    reseed from the stream, then resample the sites with replacement."""
    orders = []
    for _ in range(nboots):
        np.random.seed(np.random.choice(range(int(1e6)), 1))
        orders.append(np.random.choice(nsites, nsites, replace=True))
    return orders


def _prepare(L, item, base):
    """Work item -> dict with the replicate's matrices, targets and output naming."""
    args = L.args
    if item["kind"] == "boot":
        order = item["site_order"]
        print("starting bootstrap " + str(item["boot"]))
        return {"traingen": base["traingen"].take_cols(order), "testgen": base["testgen"].take_cols(order),
                "predgen": base["predgen"].take_cols(order), "trainlocs": base["trainlocs"],
                "testlocs": base["testlocs"], "norm": base["norm"], "pred": base["pred"], "samples": base["samples"],
                "boot": item["boot"], "cb_boot": item["boot"], "seed_tag": item["boot"] + 1, "out": args.out,
                "sites": None if base.get("sites") is None else sites.take(base["sites"], order)}
    if item["kind"] == "full":
        # the un-resampled model of a bootstrap run (locator.py:611-632), as a work item of its own
        return {"traingen": base["traingen"], "testgen": base["testgen"], "predgen": base["predgen"],
                "trainlocs": base["trainlocs"], "testlocs": base["testlocs"], "norm": base["norm"],
                "pred": base["pred"], "samples": base["samples"], "boot": "FULL", "cb_boot": "FULL", "seed_tag": 0,
                "out": args.out, "sites": base.get("sites")}
    if item["kind"] == "window_lazy":
        # the window's genotypes are still on disk: read its zarr chunks / .bed records, filter and gather here (on
        # this worker's GPU); the random split was drawn by the parent in the reference's order
        from . import io

        cache = _prepare.__dict__.setdefault("stores", {})  # zarr metadata / parsed .bim + .fam, once per process
        keep_sites = bool(getattr(args, "keep_sites", False))
        if item.get("format") == "bed":
            prefix, a, b = item["where"]
            if ("bed", prefix, keep_sites) not in cache:
                cache[("bed", prefix, keep_sites)] = io.read_bed(prefix, sites=keep_sites)
            cs = cache[("bed", prefix, keep_sites)]
            rows = cs["calldata/GT"].rows(a, b)
        else:
            root, name, a, b = item["where"]
            if (root, keep_sites) not in cache:
                cache[(root, keep_sites)] = io.read_zarr(root, lazy=True, sites=keep_sites)
            cs = cache[(root, keep_sites)]
            rows = io.ZarrRows(root, name, a, b)
        ids = io.variant_ids(cs)
        sub = io.Genotypes(rows, cs["samples"], cs["variants/POS"][a:b],
                           None if ids is None else {k: v[a:b] for k, v in ids.items()})
        ac = L.filter_snps(sub)
        locs = item["locs"]
        train, test, traingen, testgen, trainlocs, testlocs, pred, predgen = L.split_train_test(ac, locs, item["drawn"])
        return {"traingen": traingen, "testgen": testgen, "predgen": predgen, "trainlocs": trainlocs,
                "testlocs": testlocs, "norm": item["norm"], "pred": pred, "samples": item["samples"], "boot": 0,
                "cb_boot": None, "seed_tag": item["index"] + 1, "out": item["window_out"], "sites": ac.sites}
    if item["kind"] == "window":
        return {"traingen": item["traingen"], "testgen": item["testgen"], "predgen": item["predgen"],
                "trainlocs": item["trainlocs"], "testlocs": item["testlocs"], "norm": item["norm"],
                "pred": item["pred"], "samples": item["samples"], "boot": 0, "cb_boot": None,
                "seed_tag": item["index"] + 1, "out": item["window_out"], "sites": item["sites"]}
    if item["kind"] == "fold":
        # k-fold holdout (locator_b200.holdout): row gathers of the filtered matrix; "pred" is the held-out fold
        g, locs, f = base["genotypes"], base["locs"], item["fold"]
        print("starting fold " + str(f))
        return {"traingen": g.take_rows(item["train"]), "testgen": g.take_rows(item["val"]),
                "predgen": g.take_rows(item["held"]), "trainlocs": locs[item["train"]], "testlocs": locs[item["val"]],
                "norm": base["norm"], "pred": item["held"], "samples": base["samples"], "boot": f, "cb_boot": f,
                "seed_tag": f + 1, "out": item["fold_out"], "fold": f, "sites": base.get("sites")}
    raise ValueError(item["kind"])


def _run_items(L, items, reps):
    """Train + predict a list of replicates inside the current process / on the current device.

    One replicate: the reference's sequence (load_network, train_network, predict_locs).  Several:
    the models are trained side by side as one lockstep group (model.fit_group, at any batch size and
    training-set size; results are bit-identical to training them one after the other), then predicted
    one by one.  ``reps``: the items prepared by _prepare (a Prefetcher).
    Returns one result per item: (fold, held-out rows, de-normalised predictions) for a holdout fold, else None.
    """
    from .model import fit_group

    args = L.args
    t1 = time.time()
    models, callbacks = [], []
    for rep in reps:
        L._seed_tag[0] = rep["seed_tag"]
        original_out = args.out
        args.out = rep["out"]  # window runs: file names derive from the window-specific stem (locator.py:555-557)
        try:
            models.append(L.load_network(rep["traingen"], args.dropout_prop))
            callbacks.append(L.load_callbacks(rep["cb_boot"]))
        finally:
            args.out = original_out
    _tick(f"{len(models)} models created")
    same = len({(m.width, m.nlayers, m.batch_size) for m in models}) == 1  # training-set sizes may differ
    # groups need one kernel family for the first layer AND the hidden stack: tcgen05 (width 256, up to 14 layers)
    # or CUDA cores (other widths).  Width-256 models deeper than 14 layers run a tcgen05 first layer in front of a
    # CUDA-core hidden stack and train one after the other.
    family = {(m.impl, m.hidden_impl) for m in models}
    if len(reps) > 1 and same and family in ({("tcgen05", "tcgen05")}, {("simt", "simt")}):
        start = time.time()
        histories = fit_group(models, [r["traingen"] for r in reps], [r["trainlocs"] for r in reps],
                              [(r["testgen"], r["testlocs"]) for r in reps], epochs=args.max_epochs,
                              patience=args.patience, verbose=1 if args.keras_verbose == 2 else 0)
        for m, cb in zip(models, callbacks):
            m.restore_best()
            if args.keep_weights:
                m.save_weights(cb[0].filepath)
        print("run time " + str((time.time() - start) / 60) + " minutes (" + str(len(reps)) + " replicates side by side)")
        _tick("group trained, best weights restored")
    else:
        histories = []
        for m, cb, rep in zip(models, callbacks, reps):
            h, _ = L.train_network(m, rep["traingen"], rep["testgen"], rep["trainlocs"], rep["testlocs"], cb, rep["boot"])
            histories.append(h)
    for cb, rep in zip(callbacks, reps):
        L.save_sites(cb[0].filepath, rep["sites"], rep["norm"])
    results = []
    for m, h, rep in zip(models, histories, reps):
        meanlong, sdlong, meanlat, sdlat = rep["norm"]
        if "fold" in rep:
            from .holdout import predict_fold

            results.append(predict_fold(m, h, rep))
            continue
        results.append(None)
        original_out = args.out
        args.out = rep["out"]
        try:
            dists = L.predict_locs(m, rep["predgen"], sdlong, meanlong, sdlat, meanlat, rep["testlocs"], rep["pred"],
                                   rep["samples"], rep["testgen"], h, rep["boot"])
        finally:
            args.out = original_out
        if args.plot_history:
            L.plot_history(h, dists)
    _tick("group predicted, files written")
    if items and items[0]["kind"] == "window":
        print(f"Window run time {(time.time() - t1) / 60:.2f} minutes")
    return results


class Prefetcher:
    """Prepares the NEXT group of replicates (zarr chunk decode, upload, filter, pack, gathers) in a helper
    thread on a side stream while the current group trains on the main stream.  Nothing in _prepare draws
    from numpy's global stream (the parent did), so the overlap cannot change any index."""

    def __init__(self, L, base):
        import torch
        from concurrent.futures import ThreadPoolExecutor

        self.L, self.base = L, base
        self.device = torch.cuda.current_device()
        self.side = torch.cuda.Stream()
        self.pool = ThreadPoolExecutor(1)

    def _work(self, items):
        import torch

        torch.cuda.set_device(self.device)
        with torch.cuda.stream(self.side):
            reps = [_prepare(self.L, it, self.base) for it in items]
        self.side.synchronize()  # everything the group needs is in device memory before it is handed over
        return reps

    def submit(self, items):
        return self.pool.submit(self._work, items)

    @staticmethod
    def collect(future):
        import torch

        reps = future.result()
        cur = torch.cuda.current_stream()
        for rep in reps:  # allocated on the side stream, used (and eventually freed) on this one
            for k in ("traingen", "testgen", "predgen"):
                rep[k].words.record_stream(cur)
        return reps

    def close(self):
        self.pool.shutdown(wait=True)


def _group_size(args):
    return max(1, min(8, int(getattr(args, "replicates_per_gpu", 1) or 1)))


def _n_gpus(args):
    return max(1, int(getattr(args, "gpus", 1) or 1))


def _resolve(runner):
    """'package.module:function' -> callable (test hook: a CPU stand-in for _run_item)."""
    import importlib

    mod, fn = runner.split(":")
    return getattr(importlib.import_module(mod), fn)


def serve(L, base, take_group, queue_is_deep, done, who="worker"):
    """The serving loop of one GPU: take a group of work items, prepare it (helper thread, side stream), train
    and predict it; while the queue is deep the NEXT group is taken and prepared meanwhile.

    take_group(block) -> list of items, or None when there is nothing (block=False) / the queue has ended;
    queue_is_deep() -> prefetching cannot starve another GPU; done(items, results) reports completion.
    Shared by one-GPU runs (run_work), the worker processes of ``--gpus N`` (ReplicatePool) and the ranks of a
    torch.distributed job (RankQueue)."""
    pf = Prefetcher(L, base)
    try:
        ahead = None
        while True:
            if ahead is None:
                items = take_group(True)
                if items is None:
                    break
                fut = pf.submit(items)
            else:
                items, fut = ahead
                ahead = None
            if queue_is_deep():
                nxt = take_group(False)
                if nxt is not None:
                    ahead = (nxt, pf.submit(nxt))
            _tick(f"{who}: group of {len(items)} taken")
            reps = Prefetcher.collect(fut)
            _tick(f"{who}: group prepared")
            results = _run_items(L, items, reps)
            _tick(f"{who}: group done")
            done(items, results)
    finally:
        pf.close()


class RankQueue:
    """Work queue for the ranks of ONE torch.distributed job (``torchrun --nproc-per-node N``, one rank per
    GPU): the items are known to every rank (they are drawn deterministically from --seed), and a single
    atomic counter in the job's key-value store hands out their indices -- no collective, no tensor traffic.
    Group sizes shrink towards the end of the queue (guided self-scheduling: about remaining / ranks items,
    at most `group`) so that the last round does not leave GPUs idle behind one full group.
    store = None: a single process (world 1) with a local counter."""

    def __init__(self, items, world=1, store=None, key="loc_queue", group=4):
        self.items, self.world, self.store, self.key = list(items), max(1, int(world)), store, key
        self.group = max(1, int(group))
        self._local = 0
        self.taken = []

    def _next(self):
        if self.store is None:
            self._local += 1
            return self._local - 1
        return int(self.store.add(self.key, 1)) - 1

    def take_group(self, block=True):
        n = len(self.items)
        first = self._next()
        if first >= n:
            return None
        remaining = n - first  # items not yet handed out, this one included
        want = max(1, min(self.group, -(-remaining // self.world)))
        idx = [first]
        while len(idx) < want:
            i = self._next()
            if i >= n:
                break
            idx.append(i)
        self.taken.append(idx)
        return [self.items[i] for i in idx]

    def queue_is_deep(self):
        """Prefetch only while every rank could still take a full group after this one."""
        if self.store is None:
            done = self._local
        else:
            done = int(self.store.add(self.key, 0))
        return len(self.items) - done >= self.world * self.group


def run_items_ranked(L, base, items, world=1, store=None, key="loc_queue"):
    """Rank mode of the replicate drivers: this process (one GPU) serves `items` together with the other
    ranks of the job.  Returns the indices this rank ran, in groups."""
    q = RankQueue(items, world, store, key, _group_size(L.args))
    serve(L, base, q.take_group, q.queue_is_deep, lambda its, res: None, who=f"rank {os.environ.get('RANK', '0')}")
    return q.taken


def _worker(rank, n_gpus, args, init_q, task_q, result_q, runner=None):
    try:
        if runner is not None:  # host-logic tests: no CUDA, no base; the runner consumes the raw item
            run = _resolve(runner)
            for item in iter(task_q.get, None):
                result_q.put(("done", rank, (item["seq"], run(rank, args, item))))
            result_q.put(("exit", rank, None))
            return
        _tick(f"worker {rank}: process up")
        import torch

        torch.cuda.set_device(rank % max(1, torch.cuda.device_count()))
        torch.zeros(1, device="cuda")  # create the CUDA context now, while the parent is still busy
        from . import locator as L

        _tick(f"worker {rank}: torch + CUDA context ready")

        L.set_args(copy.copy(args))
        # the pool is started before the parent has the run's matrices (so that this start-up -- import torch, CUDA
        # context: seconds -- overlaps the parent's own): they arrive here, once
        base = _convert(init_q.get(), _to_dev)
        _tick(f"worker {rank}: base matrices received")
        import queue as _queue

        G = _group_size(args)
        state = {"finished": False}

        def take_group(block):
            """Up to G queued items; None when there is nothing (block=False) or the queue has ended."""
            if state["finished"]:
                return None
            try:
                item = task_q.get() if block else task_q.get_nowait()
            except _queue.Empty:
                return None
            if item is None:
                state["finished"] = True
                return None
            items = [item]
            while len(items) < G:  # take what is already queued, up to a group
                try:
                    nxt = task_q.get_nowait()
                except _queue.Empty:
                    break
                if nxt is None:
                    state["finished"] = True
                    break
                items.append(nxt)
            return [_convert(it, _to_dev) for it in items]

        def queue_is_deep():
            """Prefetch only while every worker could still fill a group of its own (no starving at the tail)."""
            try:
                return task_q.qsize() >= n_gpus * G
            except NotImplementedError:
                return False

        def done(items, results):
            for it, res in zip(items, results):
                result_q.put(("done", rank, (it["seq"], res)))

        serve(L, base, take_group, queue_is_deep, done, who=f"worker {rank}")
        _tick(f"worker {rank}: exiting")
        result_q.put(("exit", rank, None))
    except BaseException:  # surface the failure (SystemExit / KeyboardInterrupt included) in the parent
        result_q.put(("error", rank, traceback.format_exc()))
        raise


class ReplicatePool:
    """One worker process per GPU pulling work items from a shared queue.  The workers start at once and wait for
    the run's base matrices (send_base); close() returns the items' results (see _run_items) in submission order."""

    def __init__(self, n_gpus, args, runner=None):
        import multiprocessing as mp

        ctx = mp.get_context("spawn")
        self.n = n_gpus
        self.task_q = ctx.Queue()
        self.result_q = ctx.Queue()
        self.init_qs = [ctx.Queue() for _ in range(n_gpus)]
        self.procs = [ctx.Process(target=_worker,
                                  args=(r, n_gpus, args, self.init_qs[r], self.task_q, self.result_q, runner))
                      for r in range(n_gpus)]
        for p in self.procs:
            p.start()
        self.submitted = 0
        self.closed = False

    def send_base(self, base):
        base_host = _convert(base, _to_host)
        for q in self.init_qs:
            q.put(base_host)

    def abort(self):
        """The parent failed before close(): do not leave workers waiting on their queues."""
        if not self.closed:
            self.closed = True
            for p in self.procs:
                p.terminate()
            for p in self.procs:
                p.join()

    def submit(self, item):
        self.task_q.put(dict(_convert(item, _to_host), seq=self.submitted))
        self.submitted += 1

    def close(self):
        self.closed = True
        _tick("parent: all items submitted, waiting for the workers")
        for _ in self.procs:
            self.task_q.put(None)
        import queue as _queue

        results = {}
        exited = 0
        errors = []
        exited_ranks = set()
        while exited < self.n and not errors:
            try:
                kind, rank, payload = self.result_q.get(timeout=2.0)
            except _queue.Empty:
                # a worker that died without a message (SIGSEGV / abort inside the CUDA library, a device-side
                # assert, the OOM killer) would leave this loop waiting forever
                for r, p in enumerate(self.procs):
                    if r not in exited_ranks and not p.is_alive():
                        errors.append((r, f"worker process exited with code {p.exitcode} without reporting"))
                        break
                continue
            if kind == "done":
                seq, res = payload
                results[seq] = res
            elif kind == "exit":
                exited += 1
                exited_ranks.add(rank)
            else:
                errors.append((rank, payload))
        for p in self.procs:
            if errors:
                p.terminate()
            p.join()
        _tick("parent: workers joined")
        if errors:
            raise RuntimeError(f"replicate worker {errors[0][0]} failed:\n{errors[0][1]}")
        if len(results) != self.submitted:
            raise RuntimeError(f"{self.submitted - len(results)} replicates were not completed")
        return [results[seq] for seq in range(self.submitted)]


# ---------------------------------------------------------------------------------------------
# drivers called from locator.main() and holdout.main()
# ---------------------------------------------------------------------------------------------
_early = {"pool": None}


def start_pool_early(args):
    """Called by main() right after the arguments are known: with several GPUs the worker processes of a
    --windows / --bootstrap / k-fold holdout run boot (import torch, create their CUDA context) while the parent is
    still importing, reading metadata and drawing indices."""
    n_gpus = _n_gpus(args)
    if n_gpus > 1 and (args.windows or args.bootstrap or getattr(args, "folds", None)) and _early["pool"] is None:
        _tick("parent: starting the worker pool")
        _early["pool"] = ReplicatePool(n_gpus, args)
    return _early["pool"]


def abort_early_pool():
    """End of main(): a pool that was never handed over (the run failed before its driver started) is torn down."""
    pool, _early["pool"] = _early["pool"], None
    if pool is not None:
        pool.abort()


def run_work(L, items, base=None):
    """Train and predict every work item; returns one result per item (see _run_items), in item order.

    ``items`` is consumed lazily, in order and in this thread, so whatever draws from numpy's global stream while
    producing them keeps the reference's order.  One GPU: this process serves the items in groups of
    --replicates_per_gpu, the next group prepared while one trains.  Several: the worker pool (started early by
    start_pool_early, or now) receives ``base`` and then every item as it is produced."""
    args = L.args
    n_gpus = _n_gpus(args)
    if n_gpus == 1:
        items, G, results = iter(items), _group_size(args), []
        serve(L, base, lambda block: list(itertools.islice(items, G)) or None, lambda: True,
              lambda its, res: results.extend(res), who="parent")
        return results
    pool, _early["pool"] = _early["pool"], None
    if pool is None:
        pool = ReplicatePool(n_gpus, args)
    try:
        _tick("parent: sending the base matrices")
        pool.send_base(base)
        for item in items:
            pool.submit(item)
        return pool.close()
    finally:
        pool.abort()


def run_bootstrap(L, traingen, testgen, trainlocs, testlocs, predgen, norm, pred, samples, site_table=None):
    """The un-resampled FULL model (locator.py:611-632) and every replicate, all work items.  Training draws nothing
    from numpy's global stream, so every replicate's draws are taken first (full groups form at once).
    ``site_table``: --keep_sites, the sites of the filtered matrix (replicate b gets them in its site order)."""
    base = {"traingen": traingen, "testgen": testgen, "predgen": predgen, "trainlocs": trainlocs,
            "testlocs": testlocs, "norm": norm, "pred": pred, "samples": samples, "sites": site_table}
    orders = draw_bootstrap_orders(traingen.K, L.args.nboots)
    boots = [{"kind": "boot", "boot": boot, "site_order": order} for boot, order in enumerate(orders)]
    run_work(L, [{"kind": "full", "boot": "FULL"}] + boots, base)


def window_bounds(positions, start, stop, size):
    """(i, a, b) per window; the slice is gt[a:b] -- SNP b itself is excluded, as in locator.py:531-538."""
    positions = np.asarray(positions)
    for i in np.arange(start, stop, size):
        mask = np.logical_and(positions >= i, positions < i + size)
        w = np.argwhere(mask)
        yield int(i), int(np.min(w)), int(np.max(w))


def run_windows(L, genotypes, samples):
    from . import io

    args = L.args
    positions = np.array(genotypes.positions)
    start = int(args.window_start)
    stop = np.max(positions) if args.window_stop == None else int(args.window_stop)  # noqa: E711
    size = int(args.window_size)  # validate_args: int() accepts it, as the reference requires
    # Recipes instead of matrices whenever no draw depends on the genotypes: whoever runs the window (a
    # worker process, or this process's prefetch thread) reads, filters and packs it.
    # LOC_WINDOWS_PARENT_INGEST=1 keeps the serial reference order of work (parity tests compare the two).
    recipes_ok = L.windows_are_data_independent() and not os.environ.get("LOC_WINDOWS_PARENT_INGEST")

    def items():
        for index, (i, a, b) in enumerate(window_bounds(positions, start, stop, size)):
            print(f"\nProcessing window {i}-{i+size}")
            print(f"SNPs {a}-{b}")
            sub = genotypes[a:b]
            sample_data, locs = L.sort_samples(samples, sub)
            meanlong, sdlong, meanlat, sdlat, locs = L.normalize_locs(locs)
            if sub.lazy is not None and recipes_ok:
                yield {"kind": "window_lazy", "index": index, "window_out": f"{args.out}_{i}-{i+size-1}",
                       "where": sub.lazy, "format": "bed" if isinstance(sub.rows_on_disk, io.BedRows) else "zarr",
                       "locs": locs, "drawn": L.draw_split(locs),
                       "norm": (meanlong, sdlong, meanlat, sdlat), "samples": samples}
                continue
            ac = L.filter_snps(sub)
            train, test, traingen, testgen, trainlocs, testlocs, pred, predgen = L.split_train_test(ac, locs)
            yield {"kind": "window", "index": index, "window_out": f"{args.out}_{i}-{i+size-1}", "traingen": traingen,
                   "testgen": testgen, "predgen": predgen, "trainlocs": trainlocs, "testlocs": testlocs,
                   "norm": (meanlong, sdlong, meanlat, sdlat), "pred": pred, "samples": samples, "sites": ac.sites}

    run_work(L, items())
