"""GPU box: k-fold holdout models (python -m locator_b200.holdout) trained one at a time and in replicate groups.

Workload: BASELINE config[1] (cfg2, 1,000 x 100,000 synthetic genotypes), the first 900 samples located; folds and
inner validation splits drawn by locator_b200.holdout.draw_folds (numpy seed 1), fold matrices gathered from one
packed matrix on the device, models created as the command creates them (first-layer kernels on SMs - 16 at this K).
k = 10 (training sets of 729 rows each: equal) and k = 7 (694 / 695 rows: ragged groups), --batch_size 32 and 64,
G = 1 (model.fit, one fold after the other) and G = 4 (model.fit_group over folds 0-3, 4-7, 8-9 / 4-6).  20 epochs per
fold with patience 1000 (no early stop), after one untimed warm-up pass of the same configuration.  Timed with the host
clock around all folds and a device synchronise: model creation, training with validation passes and callbacks, and
the best-weight restore; no prediction or file output.  One JSON line per (k, B, G) and round: models per hour, us per replicate-step (elapsed over
the folds' summed optimizer steps).  The first line names the card, its power limit and SM clock.

    python scripts/holdout_bench.py [--epochs 20] [--rounds 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from locator_b200 import holdout, model  # noqa: E402
from locator_b200.genotypes import PackedGenotypes  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name()


def run(g, locs, folds, B, G, epochs):
    """Train every fold, G side by side; returns (seconds, summed optimizer steps)."""
    K = g.K
    ctas = model.spare_cluster_l1_ctas()
    mats = [(g.take_rows(tr), locs[tr], g.take_rows(va), locs[va]) for _, tr, va in folds]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for f0 in range(0, len(folds), G):
        part = list(range(f0, min(len(folds), f0 + G)))
        ms = [model.LocatorModel(K, batch_size=B, max_epochs=epochs, seed=1000 + f, l1_ctas=ctas) for f in part]
        if G == 1:
            x, y, xv, yv = mats[f0]
            ms[0].fit(x, y, epochs=epochs, batch_size=B, validation_data=(xv, yv), patience=1000)
        else:
            model.fit_group(ms, [mats[f][0] for f in part], [mats[f][1] for f in part],
                            [(mats[f][2], mats[f][3]) for f in part], epochs=epochs, patience=1000)
        for m in ms:
            m.restore_best()
    torch.cuda.synchronize()
    steps = sum(epochs * -(-len(tr) // B) for _, tr, _ in folds)
    return time.perf_counter() - t0, steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    n_total, K = bench.WORKLOADS["cfg2"]
    x, y = bench.synth(n_total, K, 1002)
    n_known = 900
    locs = np.full((n_total, 2), np.nan)
    locs[:n_known] = y[:n_known]
    g = PackedGenotypes.from_counts(x)
    print(json.dumps({"card": card(), "workload": "cfg2", "n": n_total, "located": n_known, "K": K,
                      "epochs": a.epochs}), flush=True)
    for k in (10, 7):
        np.random.seed(1)
        folds = holdout.draw_folds(locs, k, 0.9)
        sizes = sorted({len(tr) for _, tr, _ in folds})
        for B in (32, 64):
            for G in (1, 4):
                run(g, locs, folds[:G], B, G, 1)  # warm-up: module loads, first launches of this shape
                for rnd in range(a.rounds):
                    sec, steps = run(g, locs, folds, B, G, a.epochs)
                    print(json.dumps({"k": k, "train_rows": sizes, "B": B, "G": G, "round": rnd, "seconds": round(sec, 3),
                                      "models_per_hour": round(k * 3600 / sec, 1),
                                      "us_per_replicate_step": round(1e6 * sec / steps, 2)}), flush=True)


if __name__ == "__main__":
    main()
