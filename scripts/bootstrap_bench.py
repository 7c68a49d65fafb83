"""--bootstrap through the real CLI at BASELINE config 4 shape (GPU box): 1,000 samples x 100,000 SNPs,
--nboots R replicates of E epochs each (throughput schedule: --patience 1000), on 1 and N GPUs.
Wall time of each CLI run is measured from process start to exit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=2)
    ap.add_argument("--nboots", type=int, default=16)
    ap.add_argument("--epochs", type=int, default=20)
    ap.add_argument("--snps", type=int, default=100000)
    ap.add_argument("--samples", type=int, default=1000)
    ap.add_argument("--batch_size", type=int, default=None, help="passed to the CLI (default: the CLI's own)")
    ap.add_argument("--replicates_per_gpu", type=int, default=None, help="passed to the CLI (default: the CLI's own)")
    a = ap.parse_args()
    import bench
    from locator_b200 import io

    t0 = time.time()
    x, y = bench.synth(a.samples, a.snps, 1002)
    gt = np.stack([(x.T >= 1), (x.T >= 2)], axis=2).astype(np.int8)
    os.makedirs("/tmp/bb", exist_ok=True)
    z = "/tmp/bb/g.zarr"
    samples = [f"s{i}" for i in range(a.samples)]
    io.write_zarr(z, gt, samples, np.arange(len(gt)) * 10, chunk_variants=16384, compress=False)
    rng = np.random.default_rng(1)
    loc = rng.uniform(0, 50, size=(a.samples, 2))
    loc[rng.choice(a.samples, a.samples // 10, replace=False)] = np.nan
    with open("/tmp/bb/samples.txt", "w") as fh:
        fh.write("sampleID\tx\ty\n")
        for s, (u, v) in zip(samples, loc):
            fh.write(f"{s}\t{'NA' if np.isnan(u) else u}\t{'NA' if np.isnan(v) else v}\n")
    print(f"store: {gt.nbytes / 1e9:.2f} GB int8 built in {time.time() - t0:.1f} s", flush=True)
    res, outs = {}, {}
    for n in sorted({1, a.gpus}):
        out = f"/tmp/bb/run{n}"
        cmd = [sys.executable, "-m", "locator_b200", "--zarr", z, "--sample_data", "/tmp/bb/samples.txt", "--out", out,
               "--seed", "12345", "--bootstrap", "--nboots", str(a.nboots), "--max_epochs", str(a.epochs),
               "--patience", "1000", "--keras_verbose", "0", "--gpus", str(n)]
        for flag in ("batch_size", "replicates_per_gpu"):
            if getattr(a, flag) is not None:
                cmd += [f"--{flag}", str(getattr(a, flag))]
        t = time.time()
        r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=1500)
        dt = time.time() - t
        files = sorted(f for f in os.listdir("/tmp/bb") if f.startswith(f"run{n}_boot") and f.endswith("predlocs.txt"))
        outs[n] = {f[len(f"run{n}_"):]: open(os.path.join("/tmp/bb", f)).read() for f in files}
        res[n] = {"seconds": dt, "models_done": len(files), "models_per_hour": 3600.0 * len(files) / dt, "rc": r.returncode}
        if r.returncode != 0:
            print(r.stdout[-1500:], r.stderr[-3000:])
        if os.environ.get("LOC_TIMING"):
            print(f"process started at {t:.3f}")
            print("\n".join(l for l in r.stderr.splitlines() if "loc-timing" in l), flush=True)
        print(n, "GPU(s):", json.dumps(res[n]), flush=True)
    same = all(outs[1] == outs[n] for n in outs)
    print(json.dumps({"workload": f"bootstrap: FULL + {a.nboots} replicates x {a.samples} samples x {a.snps} SNPs, "
                                  f"{a.epochs} epochs each", "batch_size": a.batch_size,
                      "replicates_per_gpu": a.replicates_per_gpu, "results": res,
                      "outputs_identical_across_gpu_counts": same}))


if __name__ == "__main__":
    main()
