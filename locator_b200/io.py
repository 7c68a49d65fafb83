"""Genotype readers of the product path (no scikit-allel / zarr dependency).

Reference: ``load_genotypes`` /root/reference/locator/locator.py:187-228 --
``allel.read_vcf`` (calldata/GT int8 [nvar, N, 2], missing = -1, samples),
``zarr.open_group`` (calldata/GT, samples, variants/POS) and the ``--matrix`` table.
The readers only produce the int8 GT cube on the host; filtering, allele counting and
packing happen on the GPU (locator_b200.genotypes).  PLINK 1 .bed files (``--bed``, an extension of
this build) are not turned into a cube at all: their 2-bit records go to the device as they are.
"""
from __future__ import annotations

import gzip
import json
import os
import re
import zlib

import numpy as np


class Genotypes:
    """GT int8 [nvar, N, 2] (missing = -1) + sample IDs (+ positions), as allel.GenotypeArray is used.

    ``gt`` may be a ZarrRows (chunked store on disk) or a BedRows (PLINK 1 .bed records): nothing is decoded
    until ``.gt`` is read, and a variant slice ``g[a:b]`` only reads the rows that overlap it (the windows
    driver, locator.py:538).  ``ids``: optional {"chrom", "ref", "alt"} string arrays per variant (site identity:
    REF is allele index 0, ALT allele index 1), needed to record or match a model's sites (locator_b200.sites).
    """

    def __init__(self, gt, samples=None, positions=None, ids=None):
        if isinstance(gt, (ZarrRows, BedRows)):
            self._lazy, self._gt = gt, None
            assert len(gt.shape) == 3 and gt.shape[2] == 2
        else:
            self._lazy, self._gt = None, np.ascontiguousarray(gt, dtype=np.int8)
            assert self._gt.ndim == 3 and self._gt.shape[2] == 2
        self.samples = None if samples is None else np.asarray(samples)
        self.positions = None if positions is None else np.asarray(positions)
        self.ids = ids

    @property
    def gt(self):
        if self._gt is None:
            lazy = self._lazy
            cube = decode_bed(lazy.read(), lazy.nsamp) if isinstance(lazy, BedRows) else lazy.read()
            self._gt = np.ascontiguousarray(cube, dtype=np.int8)
        return self._gt

    @property
    def rows_on_disk(self):
        """The ZarrRows / BedRows behind this object while nothing has been decoded on the host, else None."""
        return self._lazy if self._gt is None else None

    @property
    def lazy(self):
        """While nothing has been decoded: where the rows are -- (store path, array name, first row, end row) of a
        zarr store, (file prefix, first row, end row) of a .bed file; else None."""
        return None if self._gt is not None or self._lazy is None else self._lazy.where()

    @property
    def shape(self):
        return self._gt.shape if self._gt is not None else self._lazy.shape

    def __len__(self):
        return self.shape[0]

    def __getitem__(self, key):
        """Variant slicing (gt[a:b] / gt[a:b, :, :]) as the windows driver does (locator.py:538)."""
        if isinstance(key, tuple):
            key = key[0]
        pos = None if self.positions is None else self.positions[key]
        ids = None if self.ids is None else {k: v[key] for k, v in self.ids.items()}
        if self._gt is None and isinstance(key, slice) and key.step in (None, 1):
            a, b, _ = key.indices(self._lazy.shape[0])
            return Genotypes(self._lazy.rows(a, max(a, b)), self.samples, pos, ids)
        return Genotypes(self.gt[key], self.samples, pos, ids)


def variant_ids(callset):
    """{"chrom", "ref", "alt"} of a reader's dict (read_vcf(sites=True) / read_zarr / read_bed), or None when the
    input does not name its alleles."""
    keys = ("variants/CHROM", "variants/REF", "variants/ALT")
    if not all(k in callset for k in keys):
        return None
    return {n: np.asarray(callset[k]) for n, k in zip(("chrom", "ref", "alt"), keys)}


def _open_bytes(path):
    with open(path, "rb") as fh:
        magic = fh.read(2)
    if magic == b"\x1f\x8b":
        with gzip.open(path, "rb") as fh:
            return fh.read()
    with open(path, "rb") as fh:
        return fh.read()


def _parse_allele(tok):
    return -1 if tok in (b".", b"") else int(tok)


def _read_vcf_native(data):
    """The library's multithreaded parser (loc_vcf_parse_gt); None when it declines a line (the Python
    parser below then either handles the oddity or raises the error a user should see)."""
    from ._cabi import lib

    h = data.find(b"#CHROM")
    if h < 0 or (h > 0 and data[h - 1:h] != b"\n"):
        return None
    e = data.find(b"\n", h)
    header = data[h:e if e >= 0 else len(data)].rstrip(b"\r").rstrip(b"\t").split(b"\t")
    samples = np.array([s.decode() for s in header[9:]], dtype=str)
    n = len(samples)
    nvar = int(lib.loc_vcf_count(data, len(data)))
    if nvar < 0:
        return None
    gt = np.empty((nvar, n, 2), dtype=np.int8)
    pos = np.empty(nvar, dtype=np.int64)
    if nvar and lib.loc_vcf_parse_gt(data, len(data), n, nvar, gt.ctypes.data, pos.ctypes.data, min(16, os.cpu_count() or 1)) != 0:
        return None
    return {"calldata/GT": gt, "samples": samples, "variants/POS": pos}


_VCF_IDS = re.compile(rb"^([^#\n][^\t\n]*)\t[^\t\n]*\t[^\t\n]*\t([^\t\n]*)\t([^\t\n,]*)", re.M)


def _vcf_ids(data, nvar, path):
    """CHROM, REF and the first ALT allele (allele index 1) of every data line."""
    rows = _VCF_IDS.findall(data)
    if len(rows) != nvar:
        raise ValueError(f"{path}: {len(rows)} data lines with CHROM / REF / ALT columns for {nvar} variants")
    cols = list(zip(*rows)) if rows else [(), (), ()]
    return {k: np.array([x.decode() for x in c], dtype=str) for k, c in
            zip(("variants/CHROM", "variants/REF", "variants/ALT"), cols)}


def read_vcf(path, sites=False):
    """VCF / VCF.gz -> dict like allel.read_vcf: 'calldata/GT', 'samples', 'variants/POS'; with sites=True also
    'variants/CHROM', 'variants/REF' and 'variants/ALT' (the first ALT allele: the one GT index 1 names).

    Fast path: FORMAT is exactly GT and every call is 3 bytes (``0|1``, ``./.``) -- one numpy view
    per line.  Anything else goes through a per-field parser (multi-digit alleles, extra FORMAT
    keys, haploid calls -> second allele -1).
    """
    data = _open_bytes(path)
    out = _read_vcf(data, path)
    if sites:
        out.update(_vcf_ids(data, len(out["variants/POS"]), path))
    return out


def _read_vcf(data, path):
    if not os.environ.get("LOC_PY_VCF"):
        fast = _read_vcf_native(data)
        if fast is not None:
            return fast
    samples = None
    gts, pos = [], []
    for line in data.split(b"\n"):
        if not line or line.startswith(b"##"):
            continue
        line = line.rstrip(b"\r")
        if line.startswith(b"#CHROM"):
            samples = np.array([s.decode() for s in line.rstrip(b"\t").split(b"\t")[9:]], dtype=str)
            continue
        f = line.rstrip(b"\t").split(b"\t")
        n = len(samples)
        calls = f[9:9 + n]
        pos.append(int(f[1]))
        g = None
        if f[8] == b"GT":
            try:
                arr = np.array(calls, dtype="S3")
                if arr.shape[0] == n and all(len(c) == 3 for c in calls):
                    b3 = arr.view(np.uint8).reshape(n, 3)
                    a0 = b3[:, 0].astype(np.int16) - 48
                    a1 = b3[:, 2].astype(np.int16) - 48
                    ok = ((b3[:, 1] == 124) | (b3[:, 1] == 47)).all() and \
                        (((a0 >= 0) & (a0 <= 9)) | (b3[:, 0] == 46)).all() and \
                        (((a1 >= 0) & (a1 <= 9)) | (b3[:, 2] == 46)).all()
                    if ok:
                        a0[b3[:, 0] == 46] = -1
                        a1[b3[:, 2] == 46] = -1
                        g = np.stack([a0, a1], axis=1).astype(np.int8)
            except ValueError:
                g = None
        if g is None:
            gi = f[8].split(b":").index(b"GT")
            g = np.full((n, 2), -1, dtype=np.int8)
            for s, field in enumerate(calls):
                alle = field.split(b":")[gi].replace(b"|", b"/").split(b"/")
                g[s, 0] = _parse_allele(alle[0])
                if len(alle) > 1:
                    g[s, 1] = _parse_allele(alle[1])
        gts.append(g)
    if samples is None:
        raise ValueError(f"{path}: no #CHROM header line")
    gt = np.stack(gts) if gts else np.zeros((0, len(samples), 2), np.int8)
    return {"calldata/GT": gt, "samples": samples, "variants/POS": np.array(pos, dtype=np.int64)}


def read_matrix(path):
    """--matrix table: first column sampleID, then one column per site with counts 0/1/2
    (locator.py:200-227 turns count c into haplotypes (c>=1, c>=2))."""
    import pandas as pd

    gmat = pd.read_csv(path, sep="\t")
    samples = np.array(gmat["sampleID"])
    counts = np.array(gmat.drop(labels="sampleID", axis=1), dtype="int8")  # [N, nsites]
    if np.any((counts < 0) | (counts > 2)):
        raise ValueError("matrix entries must be 0, 1 or 2")
    h1 = (counts >= 1).astype(np.int8)
    h2 = (counts >= 2).astype(np.int8)
    gt = np.stack([h1.T, h2.T], axis=2)
    return Genotypes(gt, samples)


# ---------------------------------------------------------------------------------------------
# zarr v2 directory store (what scripts/vcf_to_zarr.py / allel.vcf_to_zarr writes)
# ---------------------------------------------------------------------------------------------
def _blosc_decompress_array(raw):
    """One Blosc frame -> uint8 array, through the C ABI (loc_blosc_decompress; LZ4 + byte shuffle).
    ctypes drops the GIL for the call, so chunks decode in parallel from a thread pool."""
    from ._cabi import lib, check

    nbytes = int.from_bytes(raw[4:8], "little")
    out = np.empty(nbytes, dtype=np.uint8)
    src = np.frombuffer(raw, dtype=np.uint8)
    n = lib.loc_blosc_decompress(src.ctypes.data, len(raw), out.ctypes.data, nbytes)
    if n < 0:
        check(1, "loc_blosc_decompress")
    return out


def _zstd_decompress_array(raw, nbytes):
    """One Zstandard frame of known decoded size -> uint8 array (loc_zstd_decompress: the system's libzstd)."""
    from ._cabi import lib, check

    if nbytes <= 0:
        raise ValueError("zstd chunks of object arrays are not supported")
    out = np.empty(nbytes, dtype=np.uint8)
    src = np.frombuffer(raw, dtype=np.uint8)
    n = lib.loc_zstd_decompress(src.ctypes.data, len(raw), out.ctypes.data, nbytes)
    if n < 0:
        check(1, "loc_zstd_decompress")
    return out[:n]


def _blosc_decompress(raw, nbytes_hint=None):
    """One Blosc frame -> bytes."""
    return _blosc_decompress_array(raw).tobytes()


def _decode_vlen_utf8(buf):
    """numcodecs VLenUTF8: uint32 item count, then (uint32 length, bytes) per item."""
    n = int.from_bytes(buf[:4], "little")
    out, pos = [], 4
    for _ in range(n):
        ln = int.from_bytes(buf[pos:pos + 4], "little")
        pos += 4
        out.append(buf[pos:pos + ln].decode("utf-8"))
        pos += ln
    return np.array(out, dtype=object)


_PARALLEL_MIN_BYTES = 1 << 22  # smaller reads are not worth a thread pool


def _io_threads():
    """Host threads for chunk decoding (LOC_IO_THREADS overrides; default: the cores, at most 16)."""
    env = os.environ.get("LOC_IO_THREADS")
    if env:
        return max(1, int(env))
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(16, n))


class ZarrRows:
    """Rows [a, b) of a chunked zarr-v2 array, decoded on demand."""

    def __init__(self, root, name, a=None, b=None):
        self.root, self.name = root, name
        with open(os.path.join(root, name, ".zarray")) as fh:
            meta = json.load(fh)
        full = tuple(meta["shape"])
        self.a = 0 if a is None else int(a)
        self.b = full[0] if b is None else int(b)
        self.shape = (self.b - self.a,) + full[1:]
        self.dtype = np.dtype(meta["dtype"])
        self.stored_shape, self.stored_dtype = self.shape, self.dtype  # what read(out=) fills

    def rows(self, a, b):
        return ZarrRows(self.root, self.name, self.a + a, self.a + b)

    def where(self):
        return (self.root, self.name, self.a, self.b)

    def read(self, out=None):
        """Decode the rows; with ``out`` (C-contiguous array of this shape and dtype, e.g. a view of pinned
        memory) the chunks are decoded straight into it."""
        return _zarr_array(self.root, self.name, rows=(self.a, self.b), out=out)


def _zarr_array(root, name, rows=None, out=None):
    """The whole array, or (rows = (a, b)) only its first-axis range [a, b): just the chunks that overlap.
    ``out``: optional destination (shape / dtype of the result, C-contiguous)."""
    adir = os.path.join(root, name)
    with open(os.path.join(adir, ".zarray")) as fh:
        meta = json.load(fh)
    if meta.get("order", "C") != "C":
        raise ValueError(f"{name}: only C-order zarr arrays are supported")
    shape, chunks = tuple(meta["shape"]), tuple(meta["chunks"])
    dtype = np.dtype(meta["dtype"])
    comp = meta.get("compressor")
    sep = meta.get("dimension_separator", ".")
    fill = meta.get("fill_value", 0)
    is_obj = dtype.kind == "O"
    filters = meta.get("filters") or []
    if is_obj and [f.get("id") for f in filters] != ["vlen-utf8"]:
        raise ValueError(f"{name}: object arrays are only supported with the vlen-utf8 filter")
    if not is_obj and filters:
        raise ValueError(f"{name}: zarr filters {filters!r} are not supported")
    r0, r1 = (0, shape[0]) if (rows is None or not shape) else (max(0, int(rows[0])), min(shape[0], int(rows[1])))
    out_shape = ((max(0, r1 - r0),) + shape[1:]) if shape else shape
    if out is None:
        out = np.empty(out_shape, dtype=dtype)
    elif out.shape != out_shape or out.dtype != dtype or not out.flags.c_contiguous:
        raise ValueError(f"{name}: destination must be a C-contiguous {dtype} array of shape {out_shape}")
    fill_value = ("" if is_obj else 0) if fill in (None, "") or is_obj else fill
    grid = [(-(-s // c)) for s, c in zip(shape, chunks)]
    if shape and r1 > r0:
        first = range(r0 // chunks[0], -(-r1 // chunks[0]))
        indices = [(i,) + rest for i in first for rest in np.ndindex(*grid[1:])]
    elif shape:
        indices = []
    else:
        indices = [()]
    if comp is not None and comp.get("id") not in ("zlib", "gzip", "blosc", "zstd"):
        raise ValueError(f"{name}: zarr compressor {comp.get('id')!r} is not available in this build "
                         "(supported: none, zlib, gzip, zstd, blosc with lz4 / zstd)")
    chunk_nbytes = int(np.prod(chunks, dtype=np.int64)) * dtype.itemsize if not is_obj else 0
    row_bytes = int(np.prod(shape[1:], dtype=np.int64)) * dtype.itemsize if shape else 0

    def load(idx):
        """Decode chunk idx into its part of ``out`` (disjoint parts: safe from several threads)."""
        fn = os.path.join(adir, sep.join(str(i) for i in idx) if shape else "0")
        if shape:
            sl = tuple(slice(i * c, min((i + 1) * c, s)) for i, c, s in zip(idx, chunks, shape))
            lo, hi = max(sl[0].start, r0), min(sl[0].stop, r1)  # rows of this chunk inside the requested range
            dst = (slice(lo - r0, hi - r0),) + sl[1:]
        if not os.path.exists(fn):  # a chunk that was never written holds the fill value
            out[dst if shape else ...] = fill_value
            return
        whole_rows = bool(shape) and not is_obj and chunks[1:] == shape[1:]
        with open(fn, "rb") as fh:
            if comp is None and whole_rows:
                # raw chunk spanning whole rows: read the wanted rows straight into the output
                fh.seek((lo - sl[0].start) * row_bytes)
                want = (hi - lo) * row_bytes
                if fh.readinto(memoryview(out[lo - r0:hi - r0]).cast("B")) != want:
                    raise ValueError(f"{fn}: truncated chunk")
                return
            raw = fh.read()
        if comp is None:
            buf = raw
        elif comp.get("id") in ("zlib", "gzip"):
            buf = zlib.decompress(raw, 15 + 32)
        elif comp.get("id") == "zstd":
            buf = _zstd_decompress_array(raw, chunk_nbytes)
        else:
            buf = _blosc_decompress_array(raw)
        if is_obj:
            chunk = _decode_vlen_utf8(bytes(buf)).reshape(chunks)
        else:
            chunk = np.frombuffer(buf, dtype=dtype).reshape(chunks)
        if not shape:
            out[...] = chunk.reshape(())
            return
        src = (slice(lo - sl[0].start, hi - sl[0].start),) + tuple(slice(0, x.stop - x.start) for x in sl[1:])
        out[dst] = chunk[src]

    nthreads = min(len(indices), _io_threads())
    if nthreads > 1 and not is_obj and out.nbytes >= _PARALLEL_MIN_BYTES:
        # file reads, zlib / Blosc decoding and the numpy copies all drop the GIL
        from concurrent.futures import ThreadPoolExecutor

        with ThreadPoolExecutor(nthreads) as pool:
            list(pool.map(load, indices))
    else:
        for idx in indices:
            load(idx)
    return out


def _zarr_strings(path, name):
    """A string array of the store as str (fixed-width bytes or vlen-utf8); 2-D (allel's variants/ALT): column 0."""
    a = _zarr_array(path, name)
    if a.ndim == 2:
        a = a[:, 0]
    return np.array([x.decode() if isinstance(x, bytes) else str(x) for x in a], dtype=str)


def read_zarr(path, lazy=False, sites=False):
    """zarr v2 group with calldata/GT, samples, variants/POS -> dict (arrays fully loaded, like gt[:]; with
    lazy=True calldata/GT is a ZarrRows that decodes row ranges on demand).  sites=True: variants/CHROM, REF and
    ALT (its first column: allele index 1) too, as str arrays, when the store has them."""
    out = {
        "calldata/GT": ZarrRows(path, "calldata/GT") if lazy else _zarr_array(path, "calldata/GT"),
        "samples": _zarr_array(path, "samples"),
        "variants/POS": _zarr_array(path, "variants/POS"),
    }
    for name in ("variants/CHROM", "variants/REF", "variants/ALT") if sites else ():
        if os.path.exists(os.path.join(path, name, ".zarray")):
            out[name] = _zarr_strings(path, name)
    return out


def write_zarr(path, gt, samples, positions, chunk_variants=65536, compress=True, chrom=None, ref=None, alt=None):
    """Minimal zarr v2 writer (the vcf_to_zarr equivalent of this build): zlib-compressed chunks.  chrom / ref /
    alt: optional per-variant strings, written as variants/CHROM, REF and ALT."""
    os.makedirs(path, exist_ok=True)
    with open(os.path.join(path, ".zgroup"), "w") as fh:
        json.dump({"zarr_format": 2}, fh)

    def put(name, arr, chunks):
        adir = os.path.join(path, name)
        os.makedirs(adir, exist_ok=True)
        parent = os.path.dirname(adir)
        if parent != path and not os.path.exists(os.path.join(parent, ".zgroup")):
            with open(os.path.join(parent, ".zgroup"), "w") as fh:
                json.dump({"zarr_format": 2}, fh)
        meta = {"zarr_format": 2, "shape": list(arr.shape), "chunks": list(chunks), "dtype": arr.dtype.str,
                "compressor": {"id": "zlib", "level": 1} if compress else None, "fill_value": 0, "order": "C",
                "filters": None}
        with open(os.path.join(adir, ".zarray"), "w") as fh:
            json.dump(meta, fh)
        grid = [(-(-s // c)) for s, c in zip(arr.shape, chunks)]
        for idx in np.ndindex(*grid):
            sl = tuple(slice(i * c, min((i + 1) * c, s)) for i, c, s in zip(idx, chunks, arr.shape))
            chunk = np.zeros(chunks, dtype=arr.dtype)
            chunk[tuple(slice(0, s.stop - s.start) for s in sl)] = arr[sl]
            raw = chunk.tobytes()
            with open(os.path.join(adir, ".".join(str(i) for i in idx)), "wb") as fh:
                fh.write(zlib.compress(raw, 1) if compress else raw)

    gt = np.ascontiguousarray(gt, dtype=np.int8)
    put("calldata/GT", gt, (min(chunk_variants, max(1, gt.shape[0])), gt.shape[1], 2))
    s = np.asarray(samples)
    s = s.astype("S" + str(max(1, max((len(str(x)) for x in s), default=1)))) if s.dtype.kind in "UO" else s
    put("samples", s, (max(1, s.shape[0]),))
    p = np.asarray(positions, dtype=np.int64)
    put("variants/POS", p, (min(chunk_variants, max(1, p.shape[0])),))
    for name, v in (("CHROM", chrom), ("REF", ref), ("ALT", alt)):
        if v is not None:
            v = np.broadcast_to(np.asarray(v, dtype=str), p.shape)
            b = v.astype("S" + str(max(1, max((len(x.encode()) for x in v), default=1))))
            put("variants/" + name, b, (min(chunk_variants, max(1, b.shape[0])),))


# ---------------------------------------------------------------------------------------------
# PLINK 1 binary fileset (PREFIX.bed / .bim / .fam), SNP-major
# ---------------------------------------------------------------------------------------------
BED_MAGIC = b"\x6c\x1b"
BED_HEADER = 3  # magic bytes + mode byte (0x01: SNP-major)
# 2-bit code -> GT row; A1 (.bim column 5) is allele index 1, A2 (column 6) allele index 0
BED_CODE_GT = np.array([[1, 1], [-1, -1], [0, 1], [0, 0]], dtype=np.int8)


def read_fam(path):
    """Sample IDs of a .fam file: column 2 (IID); the family ID is ignored."""
    with open(path) as fh:
        return np.array([line.split()[1] for line in fh if line.strip()], dtype=str)


def read_bim(path):
    """(chromosome, position) per variant of a .bim file: columns 1 and 4."""
    import pandas as pd

    if os.path.getsize(path) == 0:
        return np.array([], dtype=str), np.array([], dtype=np.int64)
    t = pd.read_csv(path, sep=r"\s+", header=None, usecols=[0, 3], dtype={0: str, 3: np.int64})
    return t[0].to_numpy(dtype=str), t[3].to_numpy(dtype=np.int64)


def read_bim_alleles(path):
    """(A1, A2) per variant of a .bim file: columns 5 and 6."""
    import pandas as pd

    if os.path.getsize(path) == 0:
        return np.array([], dtype=str), np.array([], dtype=str)
    t = pd.read_csv(path, sep=r"\s+", header=None, usecols=[4, 5], dtype=str, keep_default_na=False)
    return t[4].to_numpy(dtype=str), t[5].to_numpy(dtype=str)


def check_bed(path, nvar, nsamp):
    """Refuse a .bed file this build cannot read for nvar variants and nsamp samples; reads only its header."""
    with open(path, "rb") as fh:
        head = fh.read(BED_HEADER)
    if len(head) < BED_HEADER or head[:2] != BED_MAGIC:
        raise ValueError(f"{path}: not a PLINK 1 .bed file (magic bytes 6c 1b expected, found {head[:2].hex(' ') or 'none'})")
    if head[2] == 0:
        raise ValueError(f"{path}: sample-major .bed (mode byte 0) is not supported; write it SNP-major (mode byte 1), "
                         "as PLINK does by default")
    if head[2] != 1:
        raise ValueError(f"{path}: unknown .bed mode byte {head[2]:#04x} (1 = SNP-major expected)")
    want = BED_HEADER + nvar * ((nsamp + 3) // 4)
    size = os.path.getsize(path)
    if size != want:
        raise ValueError(f"{path}: {size} bytes, but the {nvar} variants of the .bim and {nsamp} samples of the .fam need "
                         f"3 + {nvar} x ceil({nsamp}/4) = {want} bytes")


class BedRows:
    """Records [a, b) of a SNP-major .bed file; ``shape`` is that of the GT cube [b - a, N, 2] they stand for.
    read() gives the raw records, uint8 [b - a, ceil(N/4)] (``stored_shape``); nothing is read before."""

    def __init__(self, prefix, nvar, nsamp, a=None, b=None):
        self.prefix, self.path = prefix, prefix + ".bed"
        self.nvar, self.nsamp = int(nvar), int(nsamp)
        self.record_bytes = (self.nsamp + 3) // 4
        self.a = 0 if a is None else int(a)
        self.b = self.nvar if b is None else int(b)
        self.shape = (self.b - self.a, self.nsamp, 2)
        self.dtype = np.dtype(np.int8)  # of the cube
        self.stored_shape, self.stored_dtype = (self.b - self.a, self.record_bytes), np.dtype(np.uint8)

    def rows(self, a, b):
        return BedRows(self.prefix, self.nvar, self.nsamp, self.a + a, self.a + b)

    def where(self):
        return (self.prefix, self.a, self.b)

    def read(self, out=None):
        """The records; with ``out`` (C-contiguous uint8 array of ``stored_shape``, e.g. a view of pinned memory)
        they are read straight into it, by positioned reads from a few threads."""
        if out is None:
            out = np.empty(self.stored_shape, dtype=np.uint8)
        elif out.shape != self.stored_shape or out.dtype != np.uint8 or not out.flags.c_contiguous:
            raise ValueError(f"{self.path}: destination must be a C-contiguous uint8 array of shape {self.stored_shape}")
        nbytes = out.nbytes
        if nbytes == 0:
            return out
        buf = memoryview(out).cast("B")
        offset = BED_HEADER + self.a * self.record_bytes
        fd = os.open(self.path, os.O_RDONLY)
        try:
            def load(span):
                lo, hi = span
                while lo < hi:
                    n = os.preadv(fd, [buf[lo:hi]], offset + lo)
                    if n <= 0:
                        raise ValueError(f"{self.path}: truncated file")
                    lo += n

            piece = 1 << 26
            spans = [(lo, min(nbytes, lo + piece)) for lo in range(0, nbytes, piece)]
            nthreads = min(len(spans), _io_threads())
            if nthreads > 1:
                from concurrent.futures import ThreadPoolExecutor

                with ThreadPoolExecutor(nthreads) as pool:  # os.preadv drops the GIL
                    list(pool.map(load, spans))
            else:
                for span in spans:
                    load(span)
        finally:
            os.close(fd)
        return out


def decode_bed(records, nsamp):
    """uint8 records [nvar, ceil(N/4)] -> GT int8 [nvar, N, 2] (host; the GPU path never builds the cube)."""
    records = np.asarray(records, dtype=np.uint8)
    codes = (records[:, :, None] >> np.array([0, 2, 4, 6], dtype=np.uint8)) & 3
    return BED_CODE_GT[codes.reshape(records.shape[0], -1)[:, :nsamp]]


def read_bed(prefix, sites=False):
    """PLINK 1 fileset -> dict like read_zarr(lazy=True): 'calldata/GT' (a BedRows: no genotype byte is read
    here), 'samples' (.fam IIDs), 'variants/POS' and 'variants/CHROM' (.bim); sites=True: 'variants/REF' = A2 and
    'variants/ALT' = A1 too (allele indices 0 and 1).  The .bed header and size are checked against the .bim / .fam."""
    samples = read_fam(prefix + ".fam")
    chrom, pos = read_bim(prefix + ".bim")
    check_bed(prefix + ".bed", len(pos), len(samples))
    out = {"calldata/GT": BedRows(prefix, len(pos), len(samples)), "samples": samples, "variants/POS": pos,
           "variants/CHROM": chrom}
    if sites:
        out["variants/ALT"], out["variants/REF"] = read_bim_alleles(prefix + ".bim")
    return out


def write_bed(prefix, gt, samples, positions, chrom="1"):
    """GT int8 [nvar, N, 2] -> PREFIX.bed (SNP-major) / .bim / .fam, the write_zarr of PLINK input.  Refuses what a
    .bed cannot hold: allele indices >= 2 and calls with one allele missing.  Allele 1 is written as A1."""
    gt = np.asarray(gt, dtype=np.int8)
    if gt.ndim != 3 or gt.shape[2] != 2:
        raise ValueError("write_bed: GT must be [nvar, N, 2]")
    if (gt >= 2).any():
        raise ValueError("write_bed: allele indices >= 2 do not fit a .bed (biallelic) file")
    miss = gt < 0
    if (miss[:, :, 0] != miss[:, :, 1]).any():
        raise ValueError("write_bed: half-missing calls do not fit a .bed file")
    nvar, n = gt.shape[:2]
    alt = (gt == 1).sum(axis=2)
    code = np.where(miss[:, :, 0], 1, np.where(alt == 2, 0, np.where(alt == 1, 2, 3))).astype(np.uint8)
    rb = (n + 3) // 4
    padded = np.zeros((nvar, rb * 4), dtype=np.uint8)  # pad fields 0
    padded[:, :n] = code
    q = padded.reshape(nvar, rb, 4)
    records = q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6)
    with open(prefix + ".bed", "wb") as fh:
        fh.write(BED_MAGIC + b"\x01")
        fh.write(np.ascontiguousarray(records).tobytes())
    positions = np.asarray(positions, dtype=np.int64)
    chroms = np.broadcast_to(np.asarray(chrom, dtype=str), positions.shape)
    with open(prefix + ".bim", "w") as fh:
        fh.writelines(f"{c}\t{c}:{p}\t0\t{p}\tT\tA\n" for c, p in zip(chroms, positions))
    with open(prefix + ".fam", "w") as fh:
        fh.writelines(f"{s}\t{s}\t0\t0\t0\t-9\n" for s in np.asarray(samples).astype(str))
