"""GPU box: replicate groups of large-batch models (loc_group_train_epochs) against the same models trained alone.

Workload: BASELINE config[1] (cfg2, 1,000 x 100,000), --batch_size 64 / 128 / 256, groups of G = 1 (model.fit's
schedule, loc_train_epochs), 2 and 4 models.  Whole epochs including the validation pass and callbacks, timed with
CUDA events after two warm-up epochs.  One JSON line per (B, G) and round: ms per replicate-step (elapsed time over
epochs x steps x G), summed samples/s over the G models, library launches.  For every group, model 1 is then trained
alone on the same batch orders and must end bit-identical (weights and history): "same_as_solo".

    python scripts/bigbatch_group_bench.py [cfg2] [--epochs E] [--rounds R]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from locator_b200 import model, _cabi  # noqa: E402
from locator_b200.genotypes import PackedGenotypes, _stream  # noqa: E402

WARMUP = 2


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name()


def orders(seed, ntr, epochs):
    rng = np.random.default_rng(seed)
    return [torch.tensor(np.stack([rng.permutation(ntr) for _ in range(e)]).astype(np.int32), device="cuda")
            for e in (WARMUP, epochs)]


def make(K, B, seed, data, max_epochs):
    m = model.LocatorModel(K, batch_size=B, seed=seed, max_epochs=max_epochs)
    m.bind_train(*data[0])
    m.bind_val(*data[1])
    m.set_schedule(patience=100000)
    return m


def run_group(ms, perms, ne):
    if len(ms) == 1:
        _cabi.check(_cabi.lib.loc_train_epochs(ms[0]._h, perms[0].data_ptr(), ne, _stream()), "loc_train_epochs")
        return
    handles = (C.c_void_p * len(ms))(*[m._h for m in ms])
    pptrs = (C.c_void_p * len(ms))(*[p.data_ptr() for p in perms])
    _cabi.check(_cabi.lib.loc_group_train_epochs(handles, len(ms), pptrs, ne, _stream()), "loc_group_train_epochs")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workload", nargs="?", default="cfg2")
    ap.add_argument("--epochs", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=1)
    a = ap.parse_args()
    n_total, K = bench.WORKLOADS[a.workload]
    ntr, nva = bench.split_sizes(n_total)
    x, y = bench.synth(ntr + nva, K, 1002)
    data = ((PackedGenotypes.from_counts(x[:ntr]), y[:ntr]), (PackedGenotypes.from_counts(x[ntr:]), y[ntr:]))
    print(json.dumps({"card": card(), "workload": a.workload, "n_train": ntr, "n_val": nva, "K": K}), flush=True)
    max_epochs = WARMUP + a.epochs
    for rnd in range(a.rounds):
        for B in (64, 128, 256):
            spe = -(-ntr // B)
            for G in (1, 2, 4):
                ms = [make(K, B, 1 + g, data, max_epochs) for g in range(G)]
                perms = [orders(1 + g, ntr, a.epochs) for g in range(G)]
                run_group(ms, [p[0] for p in perms], WARMUP)
                torch.cuda.synchronize()
                l0 = _cabi.launch_count()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run_group(ms, [p[1] for p in perms], a.epochs)
                e1.record()
                torch.cuda.synchronize()
                ms_total = e0.elapsed_time(e1)
                launches = _cabi.launch_count() - l0
                res = {"round": rnd, "batch_size": B, "G": G, "epochs": a.epochs, "steps_per_epoch": spe,
                       "ms_per_replicate_step": round(ms_total / (a.epochs * spe * G), 4),
                       "samples_per_s": round(G * ntr * a.epochs / (ms_total * 1e-3), 1), "launches": launches}
                if G > 1:
                    # model 1 of the group against the same model trained alone on the same batch orders
                    w_g, h_g = ms[1].get_weights(), ms[1].history_rows(max_epochs)
                    del ms
                    solo = make(K, B, 2, data, max_epochs)
                    run_group([solo], [perms[1][0]], WARMUP)
                    run_group([solo], [perms[1][1]], a.epochs)
                    w_s, h_s = solo.get_weights(), solo.history_rows(max_epochs)
                    res["same_as_solo"] = bool(np.array_equal(h_g, h_s) and all(np.array_equal(u, v) for u, v in zip(w_g, w_s)))
                    del solo
                else:
                    del ms
                print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
