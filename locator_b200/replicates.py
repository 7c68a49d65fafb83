"""Replicate drivers: --bootstrap and --windows runs of the reference are loops over independent
models (/root/reference/locator/locator.py:519-583 windows, :609-681 bootstrap).  Here the
independent models are work items of a dynamic queue served by one worker process per GPU
(``--gpus N``); there is no collective on the training path.  Everything that consumes numpy's
global random stream (bootstrap reseeds + site orders, per-window imputation / subsample / split)
is drawn serially in the parent, in the reference's order, and shipped with the work item, so the
indices do not depend on the number of GPUs.
"""
from __future__ import annotations

import copy
import os
import time
import traceback

import numpy as np


def _tick(what):
    """LOC_TIMING=1: wall-clock milestones of the replicate drivers on stderr (seconds since the epoch, so the
    lines of the parent and the workers interleave on one axis)."""
    if os.environ.get("LOC_TIMING"):
        import sys

        print(f"[loc-timing {time.time():.3f} pid {os.getpid()}] {what}", file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------------
# (de)serialisation of packed device matrices for the worker processes
# ---------------------------------------------------------------------------------------------
def _to_host(g):
    return {"words": g.words.cpu().numpy(), "n": g.n, "K": g.K}


def _to_dev(h):
    import torch
    from .genotypes import PackedGenotypes

    return PackedGenotypes(torch.as_tensor(h["words"]).cuda(), h["n"], h["K"])


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
                "boot": item["boot"], "cb_boot": item["boot"], "seed_tag": item["boot"] + 1, "out": args.out}
    if item["kind"] == "full":
        # the un-resampled model of a bootstrap run (locator.py:611-632), as a work item of its own
        return {"traingen": base["traingen"], "testgen": base["testgen"], "predgen": base["predgen"],
                "trainlocs": base["trainlocs"], "testlocs": base["testlocs"], "norm": base["norm"],
                "pred": base["pred"], "samples": base["samples"], "boot": "FULL", "cb_boot": "FULL", "seed_tag": 0,
                "out": args.out}
    if item["kind"] == "window_lazy":
        # the window's genotypes are still on disk: decode its chunks, filter and gather here (on this
        # worker's GPU); the random split was drawn by the parent in the reference's order
        from . import io

        root, name, a, b = item["where"]
        cache = _prepare.__dict__.setdefault("stores", {})
        if root not in cache:
            cache[root] = io.read_zarr(root, lazy=True)
        cs = cache[root]
        sub = io.Genotypes(io.ZarrRows(root, name, a, b), cs["samples"], cs["variants/POS"][a:b])
        ac = L.filter_snps(sub)
        locs = item["locs"]
        train, test, traingen, testgen, trainlocs, testlocs, pred, predgen = L.split_train_test(ac, locs, item["drawn"])
        return {"traingen": traingen, "testgen": testgen, "predgen": predgen, "trainlocs": trainlocs,
                "testlocs": testlocs, "norm": item["norm"], "pred": pred, "samples": item["samples"], "boot": 0,
                "cb_boot": None, "seed_tag": item["index"] + 1, "out": item["window_out"]}
    if item["kind"] == "window":
        return {"traingen": item["traingen"], "testgen": item["testgen"], "predgen": item["predgen"],
                "trainlocs": item["trainlocs"], "testlocs": item["testlocs"], "norm": item["norm"],
                "pred": item["pred"], "samples": item["samples"], "boot": 0, "cb_boot": None,
                "seed_tag": item["index"] + 1, "out": item["window_out"]}
    raise ValueError(item["kind"])


def _run_items(L, items, base, reps=None):
    """Train + predict a list of replicates inside the current process / on the current device.

    One replicate: the reference's sequence (load_network, train_network, predict_locs).  Several:
    the models are trained side by side as one lockstep group (model.fit_group, at any batch size;
    results are bit-identical to training them one after the other), then predicted one by one.
    ``reps``: the items' matrices when a Prefetcher has already prepared them.
    """
    from .model import fit_group

    args = L.args
    t1 = time.time()
    if reps is None:
        reps = [_prepare(L, it, base) for it in items]
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
    same = len({(r["traingen"].n, m.width, m.nlayers, m.batch_size) for r, m in zip(reps, models)}) == 1
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
    for m, h, rep in zip(models, histories, reps):
        meanlong, sdlong, meanlat, sdlat = rep["norm"]
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


def _run_pipelined(L, groups, base):
    """groups: iterable of work-item lists.  Group i+1 is prepared while group i trains."""
    pf = Prefetcher(L, base)
    try:
        cur = None
        for items in groups:
            nxt = (items, pf.submit(items))
            if cur is not None:
                _run_items(L, cur[0], base, Prefetcher.collect(cur[1]))
            cur = nxt
        if cur is not None:
            _run_items(L, cur[0], base, Prefetcher.collect(cur[1]))
    finally:
        pf.close()


def _group_size(args):
    return max(1, min(8, int(getattr(args, "replicates_per_gpu", 1) or 1)))


def _resolve(runner):
    """'package.module:function' -> callable (test hook: a CPU stand-in for _run_item)."""
    import importlib

    mod, fn = runner.split(":")
    return getattr(importlib.import_module(mod), fn)


def serve(L, base, take_group, queue_is_deep, done, who="worker"):
    """The serving loop of one GPU: take a group of work items, prepare it (helper thread, side stream), train
    and predict it; while the queue is deep the NEXT group is taken and prepared meanwhile.

    take_group(block) -> list of items, or None when there is nothing (block=False) / the queue has ended;
    queue_is_deep() -> prefetching cannot starve another GPU; done(items) reports completion.
    Shared by the worker processes of ``locator --gpus N`` (ReplicatePool) and by the ranks of a
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
            _run_items(L, items, base, reps)
            _tick(f"{who}: group done")
            done(items)
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
    serve(L, base, q.take_group, q.queue_is_deep, lambda its: None, who=f"rank {os.environ.get('RANK', '0')}")
    return q.taken


def _worker(rank, n_gpus, args, base_host, task_q, result_q, runner=None, init_q=None):
    try:
        if runner is not None:  # host-logic tests: no CUDA, the runner consumes the raw item
            run = _resolve(runner)
            while True:
                item = task_q.get()
                if item is None:
                    break
                run(rank, args, item)
                result_q.put(("done", rank, item.get("boot", item.get("index"))))
            result_q.put(("exit", rank, None))
            return
        _tick(f"worker {rank}: process up")
        import torch

        torch.cuda.set_device(rank % max(1, torch.cuda.device_count()))
        torch.zeros(1, device="cuda")  # create the CUDA context now, while the parent is still busy
        from . import locator as L

        _tick(f"worker {rank}: torch + CUDA context ready")

        L.set_args(copy.copy(args))
        base = None
        if init_q is not None:
            # the pool was started before the parent had the run's matrices (so that this start-up -- import
            # torch, CUDA context: seconds -- overlaps the parent's own): they arrive here, once
            base_host = init_q.get()
            _tick(f"worker {rank}: base matrices received")
        if base_host is not None:
            base = dict(base_host)
            for k in ("traingen", "testgen", "predgen"):
                base[k] = _to_dev(base_host[k])
        import queue as _queue

        G = _group_size(args)
        state = {"finished": False}

        def to_dev(it):
            for k in ("traingen", "testgen", "predgen"):
                if k in it and isinstance(it[k], dict):
                    it[k] = _to_dev(it[k])
            return it

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
            return [to_dev(it) for it in items]

        def queue_is_deep():
            """Prefetch only while every worker could still fill a group of its own (no starving at the tail)."""
            try:
                return task_q.qsize() >= n_gpus * G
            except NotImplementedError:
                return False

        def done(items):
            for it in items:
                result_q.put(("done", rank, it.get("boot", it.get("index"))))

        serve(L, base, take_group, queue_is_deep, done, who=f"worker {rank}")
        _tick(f"worker {rank}: exiting")
        result_q.put(("exit", rank, None))
    except BaseException:  # surface the failure (SystemExit / KeyboardInterrupt included) in the parent
        result_q.put(("error", rank, traceback.format_exc()))
        raise


class ReplicatePool:
    """One worker process per GPU pulling work items from a shared queue."""

    def __init__(self, n_gpus, args, base=None, runner=None, deferred_base=False):
        """deferred_base: the workers are started now and wait for the run's matrices (``send_base``)."""
        import multiprocessing as mp

        ctx = mp.get_context("spawn")
        self.n = n_gpus
        self.task_q = ctx.Queue()
        self.result_q = ctx.Queue()
        self.init_qs = [ctx.Queue() for _ in range(n_gpus)] if deferred_base else None
        base_host = self._host(base)
        self.procs = [ctx.Process(target=_worker,
                                  args=(r, n_gpus, args, base_host, self.task_q, self.result_q, runner,
                                        self.init_qs[r] if deferred_base else None))
                      for r in range(n_gpus)]
        for p in self.procs:
            p.start()
        self.submitted = 0
        self.closed = False

    @staticmethod
    def _host(base):
        if base is None:
            return None
        base_host = dict(base)
        for k in ("traingen", "testgen", "predgen"):
            base_host[k] = _to_host(base[k])
        return base_host

    def send_base(self, base):
        base_host = self._host(base)
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
        item = dict(item)
        for k in ("traingen", "testgen", "predgen"):
            if k in item and not isinstance(item[k], dict):
                item[k] = _to_host(item[k])
        self.task_q.put(item)
        self.submitted += 1

    def close(self):
        self.closed = True
        _tick("parent: all items submitted, waiting for the workers")
        for _ in self.procs:
            self.task_q.put(None)
        import queue as _queue

        done = exited = 0
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
                done += 1
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
        if done != self.submitted:
            raise RuntimeError(f"{self.submitted - done} replicates were not completed")


# ---------------------------------------------------------------------------------------------
# drivers called from locator.main()
# ---------------------------------------------------------------------------------------------
_early = {"pool": None, "taken": None}


def start_pool_early(args):
    """Called by main() right after the arguments are known: with several GPUs the worker processes of a
    --windows / --bootstrap run boot (import torch, create their CUDA context) while the parent is still
    importing, reading metadata and drawing indices."""
    n_gpus = max(1, int(getattr(args, "gpus", 1) or 1))
    if n_gpus > 1 and (args.windows or args.bootstrap) and _early["pool"] is None:
        _tick("parent: starting the worker pool")
        _early["pool"] = ReplicatePool(n_gpus, args, deferred_base=bool(args.bootstrap) and not args.windows)
    return _early["pool"]


def abort_early_pool():
    """End of main(): a pool that was never handed over, or whose driver failed before close(), is torn down."""
    for key in ("pool", "taken"):
        pool, _early[key] = _early[key], None
        if pool is not None:
            pool.abort()


def _take_pool(n_gpus, args, base=None):
    pool, _early["pool"] = _early["pool"], None
    if pool is None:
        pool = ReplicatePool(n_gpus, args, base)
    elif pool.init_qs is not None:
        _tick("parent: sending the base matrices")
        pool.send_base(base)
    _early["taken"] = pool
    return pool


def run_bootstrap(L, traingen, testgen, trainlocs, testlocs, predgen, norm, pred, samples):
    args = L.args
    base = {"traingen": traingen, "testgen": testgen, "predgen": predgen, "trainlocs": trainlocs,
            "testlocs": testlocs, "norm": norm, "pred": pred, "samples": samples}
    n_gpus = max(1, int(getattr(args, "gpus", 1) or 1))
    if n_gpus == 1:
        # 1. initial full run (locator.py:611-632)
        L._seed_tag[0] = 0
        L._run_one(traingen, testgen, trainlocs, testlocs, predgen, norm, pred, samples, "FULL", "FULL")
        # 2. every replicate's draws, serially, as the reference's loop would take them
        orders = draw_bootstrap_orders(traingen.K, args.nboots)
        G = _group_size(args)
        items = [{"kind": "boot", "boot": boot, "site_order": order} for boot, order in enumerate(orders)]
        _run_pipelined(L, (items[i:i + G] for i in range(0, len(items), G)), base)
        return
    # Several GPUs: the full model is one more independent work item (training draws nothing from numpy's
    # global stream, so the replicates' draws do not have to wait for it), and the workers start up while
    # the parent draws: no GPU idles through the full run.
    orders = draw_bootstrap_orders(traingen.K, args.nboots)  # before the first submit: full groups form at once
    pool = _take_pool(n_gpus, args, base)
    pool.submit({"kind": "full", "boot": "FULL"})
    for boot, order in enumerate(orders):
        pool.submit({"kind": "boot", "boot": boot, "site_order": order})
    pool.close()


def window_bounds(positions, start, stop, size):
    """(i, a, b) per window; the slice is gt[a:b] -- SNP b itself is excluded, as in locator.py:531-538."""
    positions = np.asarray(positions)
    for i in np.arange(start, stop, size):
        mask = np.logical_and(positions >= i, positions < i + size)
        w = np.argwhere(mask)
        yield int(i), int(np.min(w)), int(np.max(w))


def run_windows(L, genotypes, samples):
    args = L.args
    positions = np.array(genotypes.positions)
    start = int(args.window_start)
    stop = np.max(positions) if args.window_stop == None else int(args.window_stop)  # noqa: E711
    size = int(args.window_size)  # validate_args: int() accepts it, as the reference requires
    n_gpus = max(1, int(getattr(args, "gpus", 1) or 1))
    pool = _take_pool(n_gpus, args) if n_gpus > 1 else None
    # Recipes instead of matrices whenever no draw depends on the genotypes: whoever runs the window (a
    # worker process, or this process's prefetch thread) reads, filters and packs it.
    # LOC_WINDOWS_PARENT_INGEST=1 keeps the serial reference order of work (parity tests compare the two).
    recipes_ok = L.windows_are_data_independent() and not os.environ.get("LOC_WINDOWS_PARENT_INGEST")
    pending, recipes = [], []
    for index, (i, a, b) in enumerate(window_bounds(positions, start, stop, size)):
        print(f"\nProcessing window {i}-{i+size}")
        print(f"SNPs {a}-{b}")
        sub = genotypes[a:b]
        sample_data, locs = L.sort_samples(samples, sub)
        meanlong, sdlong, meanlat, sdlat, locs = L.normalize_locs(locs)
        if sub.lazy is not None and recipes_ok:
            item = {"kind": "window_lazy", "index": index, "window_out": f"{args.out}_{i}-{i+size-1}",
                    "where": sub.lazy, "locs": locs, "drawn": L.draw_split(locs),
                    "norm": (meanlong, sdlong, meanlat, sdlat), "samples": samples}
            if pool is not None:
                pool.submit(item)
            else:
                recipes.append(item)
            continue
        ac = L.filter_snps(sub)
        train, test, traingen, testgen, trainlocs, testlocs, pred, predgen = L.split_train_test(ac, locs)
        item = {"kind": "window", "index": index, "window_out": f"{args.out}_{i}-{i+size-1}", "traingen": traingen,
                "testgen": testgen, "predgen": predgen, "trainlocs": trainlocs, "testlocs": testlocs,
                "norm": (meanlong, sdlong, meanlat, sdlat), "pred": pred, "samples": samples}
        if pool is None:
            pending.append(item)
            if len(pending) >= _group_size(args):
                _run_items(L, pending, None)
                pending = []
        else:
            pool.submit(item)
    if pending:
        _run_items(L, pending, None)
    if recipes:
        G = _group_size(args)
        _run_pipelined(L, (recipes[j:j + G] for j in range(0, len(recipes), G)), None)
    if pool is not None:
        pool.close()
