"""python -m locator_b200.predict on a GPU, stage by stage.

Workload: one model of BASELINE config 2's shape (K = 100,000 sites, width 256, 10 layers; weights as initialised:
the arithmetic does not depend on their values) and a query of 10,000 samples:
  * a 400,000-record .bed (1 GB of records), of which the model's sites are 100,000 (1 % of them absent from the
    query, 10 % with REF / ALT swapped) -- the .bed path never builds a GT cube;
  * a zarr store (raw chunks) holding only the model's 100,000 records (a 2 GB int8 cube; 400,000 records would be
    8 GB of cube to write for every call).
Both are written to a temporary directory just before they are read (so they come from the page cache) and removed
at the end.

Stages, each synchronised: query upload (read + host-to-device copy), host join (sites.join), mapped pack (CUDA
events, median of 20 launches; bytes/s over the record bytes the kernel must read), predict (LocatorModel creation,
load_weights and predict of all 10,000 rows), and the whole command (predict.main in this process: torch and the
library are already loaded).  One JSON line per query format to --out, with the card's name and power limit read in
the same call.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from locator_b200 import genotypes as G, io, predict, sites  # noqa: E402
from locator_b200.model import LocatorModel  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(", ")
    return {"gpu": name or torch.cuda.get_device_name(), "power_limit": power or None}


def wall(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, time.perf_counter() - t


def kernel_ms(fn, reps=20):
    fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in ev]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_predict.jsonl"))
    ap.add_argument("--records", type=int, default=400_000)
    ap.add_argument("--samples", type=int, default=10_000)
    ap.add_argument("--sites", type=int, default=100_000)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "predict_bench needs a CUDA device"
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    rng = np.random.default_rng(0)
    tmp = tempfile.mkdtemp(prefix="predict_bench_")
    try:
        run(a, rng, tmp)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run(a, rng, tmp):
    nvar, N, K = a.records, a.samples, a.sites
    samples = np.array([f"s{i}" for i in range(N)])
    pos = np.arange(1, nvar + 1, dtype=np.int64) * 10
    # .bed records from random bytes, with code 1 (missing) turned into 0: a query with a quarter of its calls
    # missing would not be realistic
    rb = (N + 3) // 4
    rec = rng.integers(0, 256, size=(nvar, rb), dtype=np.uint8)
    rec &= ~np.uint8(0x55) | (rec >> 1) & np.uint8(0x55)  # code 1 (missing) -> 0
    with open(os.path.join(tmp, "q.bed"), "wb") as fh:
        fh.write(io.BED_MAGIC + b"\x01")
        fh.write(rec.tobytes())
    with open(os.path.join(tmp, "q.bim"), "w") as fh:
        fh.writelines(f"1\t.\t0\t{p}\tT\tA\n" for p in pos)
    with open(os.path.join(tmp, "q.fam"), "w") as fh:
        fh.writelines(f"{s}\t{s}\t0\t0\t0\t-9\n" for s in samples)
    # the model: K of the records, 1 % absent (positions the query lacks), 10 % with swapped alleles
    pick = np.sort(rng.choice(nvar, K, replace=False))
    table = sites.table({"chrom": np.full(nvar, "1"), "ref": np.full(nvar, "A"), "alt": np.full(nvar, "T")}, pos, pick)
    absent = rng.uniform(size=K) < 0.01
    table["pos"][absent] += 5
    swap = rng.uniform(size=K) < 0.1
    table["ref"][swap], table["alt"][swap] = "T", "A"
    m = LocatorModel(K, seed=1)
    wpath = os.path.join(tmp, "cfg2.weights.npz")
    m.save_weights(wpath)
    sites.write(sites.sidecar_path(wpath), table, 256, 10, (0.0, 1.0, 0.0, 1.0))
    del m
    # zarr: the model's records only, as an int8 cube (raw chunks)
    gt_model = io.decode_bed(rec[pick], N)
    io.write_zarr(os.path.join(tmp, "q.zarr"), gt_model, samples, pos[pick], chunk_variants=4096, compress=False,
                  chrom="1", ref="A", alt="T")
    del gt_model
    info = card()
    for fmt, path in (("bed", os.path.join(tmp, "q")), ("zarr", os.path.join(tmp, "q.zarr"))):
        ns = predict.build_parser().parse_args(["--weights", wpath, f"--{fmt}", path, "--out", os.path.join(tmp, fmt)])
        models = predict.check_models(ns.weights)
        (cs, query, smp), t_read = wall(lambda: predict.read_query(ns))
        dev, t_up = wall(lambda: predict.upload_query(cs))
        (src, flip), t_join = wall(lambda: sites.join(models[0][1], query))
        s_dev = torch.as_tensor(src).cuda()
        f_dev = torch.as_tensor(flip).cuda()
        pack_ms = kernel_ms(lambda: G.pack_sites_mapped(dev, s_dev, f_dev))
        nrec = int((src >= 0).sum())
        rec_bytes = nrec * (rb if fmt == "bed" else 2 * N)
        (xy, packed), t_pred = wall(lambda: predict.predict_model(dev, src, flip, wpath, models[0][2], models[0][3]))
        del dev, packed
        torch.cuda.empty_cache()
        _, t_cmd = wall(lambda: predict.main(["--weights", wpath, f"--{fmt}", path, "--out", os.path.join(tmp, fmt)]))
        row = dict(info, format=fmt, records=int(len(query["pos"])), samples=N, K=K, matched=nrec,
                   flipped=int(flip.sum()), query_read_s=round(t_read, 3), query_upload_s=round(t_up, 3),
                   join_s=round(t_join, 3), mapped_pack_ms=round(pack_ms, 3),
                   mapped_pack_record_GBps=round(rec_bytes / pack_ms / 1e6, 1), predict_s=round(t_pred, 3),
                   command_s=round(t_cmd, 3))
        print(json.dumps(row), flush=True)
        with open(a.out, "a") as fh:
            fh.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
