"""GPU box: replicate groups of CUDA-core models (widths other than 256, loc_group_train_epochs) against the same
models trained alone.

Workload: BASELINE config[1] (cfg2, 1,000 x 100,000) at width 128 x 10 and 64 x 4 layers, --batch_size 32 (lockstep:
one hidden-stack launch per step for the group) and 64 (two 32-row chunks: one launch per chunk for the group); groups
of G = 1 (model.fit's schedule, loc_train_epochs), 2 and 4 models.  Whole epochs including the validation pass and
callbacks, after two warm-up epochs, timed with the host clock around the call and a device synchronise.  One JSON line
per (shape, B, G) and round: us per replicate-step (elapsed time over epochs x steps x G), summed samples/s over the G
models, library launches.  For every group, model 1 is then trained alone on the same batch orders and must end
bit-identical (weights and history): "same_as_solo".  The first line names the card, its power limit and SM clock.
--kernels: then, at 32 rows and G = 1 / 4, three epochs under torch.profiler (a run of its own, after the timed ones):
mean device time and count of every kernel, to show which passes a group shortens and which it lengthens.

    python scripts/simt_group_bench.py [cfg2] [--epochs E] [--rounds R] [--kernels]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from locator_b200 import model, _cabi  # noqa: E402
from locator_b200.genotypes import PackedGenotypes, _stream  # noqa: E402

WARMUP = 2
SHAPES = [(128, 10), (64, 4)]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name()


def orders(seed, ntr, epochs):
    rng = np.random.default_rng(seed)
    return [torch.tensor(np.stack([rng.permutation(ntr) for _ in range(e)]).astype(np.int32), device="cuda")
            for e in (WARMUP, epochs)]


def make(K, H, L, B, seed, data, max_epochs):
    m = model.LocatorModel(K, width=H, nlayers=L, batch_size=B, seed=seed, max_epochs=max_epochs)
    assert (m.impl, m.hidden_impl) == ("simt", "simt"), (H, L)
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
    ap.add_argument("--epochs", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=1)
    ap.add_argument("--kernels", action="store_true")
    a = ap.parse_args()
    n_total, K = bench.WORKLOADS[a.workload]
    ntr, nva = bench.split_sizes(n_total)
    x, y = bench.synth(ntr + nva, K, 1002)
    data = ((PackedGenotypes.from_counts(x[:ntr]), y[:ntr]), (PackedGenotypes.from_counts(x[ntr:]), y[ntr:]))
    print(json.dumps({"card": card(), "workload": a.workload, "n_train": ntr, "n_val": nva, "K": K}), flush=True)
    max_epochs = WARMUP + a.epochs
    for rnd in range(a.rounds):
        for H, L in SHAPES:
            for B in (32, 64):
                spe = -(-ntr // B)
                for G in (1, 2, 4):
                    ms = [make(K, H, L, B, 1 + g, data, max_epochs) for g in range(G)]
                    perms = [orders(1 + g, ntr, a.epochs) for g in range(G)]
                    run_group(ms, [p[0] for p in perms], WARMUP)
                    torch.cuda.synchronize()
                    l0 = _cabi.launch_count()
                    t0 = time.perf_counter()
                    run_group(ms, [p[1] for p in perms], a.epochs)
                    torch.cuda.synchronize()
                    sec = time.perf_counter() - t0
                    launches = _cabi.launch_count() - l0
                    res = {"round": rnd, "width": H, "nlayers": L, "batch_size": B, "G": G, "epochs": a.epochs,
                           "steps_per_epoch": spe, "us_per_replicate_step": round(sec * 1e6 / (a.epochs * spe * G), 1),
                           "samples_per_s": round(G * ntr * a.epochs / sec, 1), "launches": launches}
                    if G > 1:
                        # model 1 of the group against the same model trained alone on the same batch orders
                        w_g, h_g = ms[1].get_weights(), ms[1].history_rows(max_epochs)
                        del ms
                        solo = make(K, H, L, B, 2, data, max_epochs)
                        run_group([solo], [perms[1][0]], WARMUP)
                        run_group([solo], [perms[1][1]], a.epochs)
                        w_s, h_s = solo.get_weights(), solo.history_rows(max_epochs)
                        res["same_as_solo"] = bool(np.array_equal(h_g, h_s) and
                                                   all(np.array_equal(u, v) for u, v in zip(w_g, w_s)))
                        del solo
                    else:
                        del ms
                    print(json.dumps(res), flush=True)
    if a.kernels:
        kernel_times(K, ntr, data)


def kernel_times(K, ntr, data, epochs=3):
    from torch.profiler import ProfilerActivity, profile

    for H, L in SHAPES:
        for G in (1, 4):
            ms = [make(K, H, L, 32, 1 + g, data, WARMUP + epochs) for g in range(G)]
            perms = [orders(1 + g, ntr, epochs) for g in range(G)]
            run_group(ms, [p[0] for p in perms], WARMUP)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run_group(ms, [p[1] for p in perms], epochs)
                torch.cuda.synchronize()
            kernels = {}
            for e in prof.key_averages():
                t = e.device_time_total
                if e.count and t:
                    kernels[e.key.split("(")[0]] = {"count": e.count, "mean_us": round(t / e.count, 1)}
            print(json.dumps({"profile": "kernels", "width": H, "nlayers": L, "batch_size": 32, "G": G, "epochs": epochs,
                              "kernels": kernels}), flush=True)
            del ms


if __name__ == "__main__":
    main()
