"""--bed ingest on the GPU box: the .bed kernels against the int8 kernels, and filter_snps from files on disk.

1. Device time (CUDA events, median of repeated launches) of loc_bed_site_stats / loc_bed_pack_sites /
   loc_bed_missing_calls next to loc_site_stats / loc_pack_sites at ingest_bench.py's shape (400k sites x 2,500
   samples), as GB/s of the bytes each kernel must move and as a fraction of a device-to-device copy measured in
   the same run.  The inputs (2 GB cube, 250 MB of records) are larger than L2.
2. Wall time of the whole filter_snps (read, host-to-device copy, statistics, compaction, pack; synchronised) from
   files on disk: a .bed fileset against a raw (uncompressed) zarr store of the same cube, at a shape whose int8
   cube is >= 10 GB.  Both are written just before, so they are read from the page cache.

One JSON line per measurement to --out, each with the card's name and power limit read in the same call.
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
from locator_b200 import genotypes as G, io, locator as L  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(", ")
    return {"gpu": name or torch.cuda.get_device_name(), "power_limit": power or None}


def timed(fn, reps=20):
    fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in ev]))


def encode_bed(gt):
    """Device GT int8 [nvar, N, 2] (biallelic, whole-call missing) -> .bed records uint8 [nvar, ceil(N/4)]."""
    nvar, n, _ = gt.shape
    alt = (gt == 1).sum(dim=2)
    code = torch.full((nvar, n), 3, dtype=torch.uint8, device=gt.device)
    code[alt == 1] = 2
    code[alt == 2] = 0
    code[gt[:, :, 0] < 0] = 1
    rb = (n + 3) // 4
    pad = torch.zeros((nvar, rb * 4), dtype=torch.uint8, device=gt.device)
    pad[:, :n] = code
    q = pad.view(nvar, rb, 4)
    return q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6)


def random_cube(nvar, n, gen, miss=0.01):
    p = torch.rand(nvar, 1, 1, device="cuda", generator=gen) ** 2
    gt = (torch.rand(nvar, n, 2, device="cuda", generator=gen) < p).to(torch.int8)
    gt = torch.sort(gt, dim=2).values
    gt[(torch.rand(nvar, n, device="cuda", generator=gen) < miss)] = -1
    return gt


def kernels(emit, nvar, n):
    gen = torch.Generator(device="cuda").manual_seed(1)
    gt = random_cube(nvar, n, gen)
    bed = G.BedRecords(encode_bed(gt).contiguous(), n)
    rb = bed.records.shape[1]
    big = torch.empty(gt.numel(), dtype=torch.uint8, device="cuda")
    t = timed(lambda: big.copy_(gt.view(torch.uint8).view(-1)))
    peak = 2 * gt.numel() / t / 1e6  # GB/s: read + write
    emit({"what": "d2d_copy", "bytes": 2 * gt.numel(), "ms": t, "GBps": peak})

    def row(what, ms, nbytes, **kw):
        emit({"what": what, "shape": [nvar, n], "ms": ms, "bytes": nbytes, "GBps": nbytes / ms / 1e6,
              "of_d2d_copy": nbytes / ms / 1e6 / peak, **kw})

    _, na, alt, miss, keep = G.site_stats(gt, 2)
    na2, alt2, miss2, keep2 = G.bed_site_stats(bed, 2)
    assert torch.equal(alt, alt2) and torch.equal(keep, keep2) and torch.equal(miss, miss2)
    row("site_stats (int8 cube)", timed(lambda: G.site_stats(gt, 2)), gt.numel())
    row("bed_site_stats", timed(lambda: G.bed_site_stats(bed, 2)), nvar * rb)
    idx = G.compact_sites(keep)
    K = int(idx.numel())
    rw = G.row_words_for(K)
    assert torch.equal(G.pack_sites(gt, idx).words, G.bed_pack_sites(bed, idx).words)
    row("pack_sites (int8 cube)", timed(lambda: G.pack_sites(gt, idx)), 2 * K * n + n * rw * 4, K=K)
    row("bed_pack_sites", timed(lambda: G.bed_pack_sites(bed, idx)), K * rb + n * rw * 4, K=K)
    ks, _ = G.bed_missing_calls(bed, idx, miss2)
    row("bed_missing_calls (both phases)", timed(lambda: G.bed_missing_calls(bed, idx, miss2)),
        K * rb + 16 * int(ks.numel()), K=K, missing_calls=int(ks.numel()))
    row("missing_calls (int8 cube, both phases)", timed(lambda: G.missing_calls(gt, idx, miss)),
        2 * K * n + 16 * int(ks.numel()), K=K, missing_calls=int(ks.numel()))
    del gt, bed, big
    torch.cuda.empty_cache()


def files_on_disk(emit, nvar, n, rounds, chunk=65536):
    """filter_snps wall time, .bed against a raw zarr store of the same cube (written chunk by chunk)."""
    d = tempfile.mkdtemp(prefix="bed_ingest_")
    try:
        gen = torch.Generator(device="cuda").manual_seed(2)
        samples = [f"s{i}" for i in range(n)]
        pos = np.arange(nvar, dtype=np.int64) * 10 + 1
        z = os.path.join(d, "g.zarr")
        prefix = os.path.join(d, "g")
        t0 = time.time()
        os.makedirs(os.path.join(z, "calldata", "GT"))
        for name in (z, os.path.join(z, "calldata")):
            with open(os.path.join(name, ".zgroup"), "w") as fh:
                json.dump({"zarr_format": 2}, fh)
        with open(os.path.join(z, "calldata", "GT", ".zarray"), "w") as fh:
            json.dump({"zarr_format": 2, "shape": [nvar, n, 2], "chunks": [chunk, n, 2], "dtype": "|i1",
                       "compressor": None, "fill_value": 0, "order": "C", "filters": None}, fh)
        io.write_zarr(os.path.join(d, "meta.zarr"), np.zeros((1, n, 2), np.int8), samples, pos[:1])
        shutil.move(os.path.join(d, "meta.zarr", "samples"), os.path.join(z, "samples"))
        io.write_zarr(os.path.join(d, "pos.zarr"), np.zeros((nvar, 1, 2), np.int8)[:1], ["x"], pos, chunk_variants=nvar)
        shutil.move(os.path.join(d, "pos.zarr", "variants"), os.path.join(z, "variants"))
        with open(prefix + ".bed", "wb") as bed_fh:
            bed_fh.write(io.BED_MAGIC + b"\x01")
            for c, a in enumerate(range(0, nvar, chunk)):
                b = min(nvar, a + chunk)
                gt = random_cube(b - a, n, gen)
                cube = np.zeros((chunk, n, 2), np.int8)
                cube[: b - a] = gt.cpu().numpy()
                with open(os.path.join(z, "calldata", "GT", f"{c}.0.0"), "wb") as fh:
                    fh.write(cube.tobytes())
                bed_fh.write(encode_bed(gt).cpu().numpy().tobytes())
        with open(prefix + ".bim", "w") as fh:
            fh.writelines(f"1\tv{i}\t0\t{p}\tT\tA\n" for i, p in enumerate(pos))
        with open(prefix + ".fam", "w") as fh:
            fh.writelines(f"{s}\t{s}\t0\t0\t0\t-9\n" for s in samples)
        emit({"what": "inputs written", "shape": [nvar, n], "cube_GB": nvar * n * 2 / 1e9,
              "bed_GB": os.path.getsize(prefix + ".bed") / 1e9, "s": time.time() - t0})
        words = {}
        for r in range(rounds):
            for src in ("zarr", "bed"):
                L.set_args(L.command_parser().parse_args([f"--{src}", z if src == "zarr" else prefix, "--out",
                                                        os.path.join(d, "o"), "--min_mac", "2"]))
                genotypes, _ = L.load_genotypes()
                torch.cuda.synchronize()
                t = time.time()
                ac = L.filter_snps(genotypes)
                torch.cuda.synchronize()
                wall = time.time() - t
                words.setdefault(src, ac.packed.words)
                emit({"what": f"filter_snps from {src}", "round": r, "shape": [nvar, n], "K": ac.shape[0], "s": wall,
                      "file_GB": (nvar * n * 2 if src == "zarr" else os.path.getsize(prefix + ".bed")) / 1e9})
                del ac, genotypes
                torch.cuda.empty_cache()
        emit({"what": "filter_snps zarr == bed", "equal": bool(torch.equal(words["zarr"], words["bed"]))})
    finally:
        shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_bed_ingest.jsonl"))
    ap.add_argument("--kernel-shape", type=int, nargs=2, default=[400_000, 2500])
    ap.add_argument("--file-shape", type=int, nargs=2, default=[2_100_000, 2500])  # 10.5 GB int8 cube
    ap.add_argument("--rounds", type=int, default=2)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    info = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        def emit(d):
            line = json.dumps({**d, **info})
            print(line, flush=True)
            fh.write(line + "\n")
            fh.flush()

        kernels(emit, *a.kernel_shape)
        files_on_disk(emit, *a.file_shape, a.rounds)


if __name__ == "__main__":
    main()
