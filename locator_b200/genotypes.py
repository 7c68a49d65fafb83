"""2-bit packed genotype matrices resident in HBM, and the ingest kernels over them.

Host mirror of the integer half of the reference's ingest
(``/root/reference/locator/locator.py``: filter_snps :265-281, split_train_test
:295-308, bootstrap gather :648-653, jacknife replacement :721-727).  Every
function here calls the CUDA library through the C ABI; torch only owns the
device buffers.
"""
from __future__ import annotations

import threading

import numpy as np
import torch

from . import _cabi
from ._cabi import lib, check


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _dev():
    if not torch.cuda.is_available():
        raise _cabi.LocatorCudaError("locator_b200 needs a CUDA device (no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


def row_words_for(K: int) -> int:
    """uint32 words per packed row: ceil(K/16) rounded up to a multiple of 4 (16-byte rows)."""
    w = (int(K) + 15) // 16
    return max(4, (w + 3) // 4 * 4)


def _idx(x):
    """Index array (host or device) -> int64 device tensor."""
    if isinstance(x, torch.Tensor):
        return x.to(device=_dev(), dtype=torch.int64).contiguous()
    return torch.as_tensor(np.ascontiguousarray(np.asarray(x, dtype=np.int64))).to(_dev())


def _as_dev(x, dtype):
    if isinstance(x, torch.Tensor):
        return x.to(device=_dev(), dtype=dtype).contiguous()
    return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype).to(_dev())


class PackedGenotypes:
    """[n, K] alt-allele counts (0/1/2), sample-major, 2 bits each, in device memory."""

    def __init__(self, words: torch.Tensor, n: int, K: int):
        self.words = words  # int32 [n, row_words] (bit pattern of uint32)
        self.n = int(n)
        self.K = int(K)
        self.row_words = int(words.shape[1]) if words.dim() == 2 else row_words_for(K)
        self.version = 0  # bumped by the in-place edits (replace_cols / patch)

    @property
    def ptr(self):
        return self.words.data_ptr()

    @property
    def shape(self):
        """(n samples, K SNPs) -- the orientation of the reference's traingen / testgen / predgen."""
        return (self.n, self.K)

    def to_numpy(self):
        return self.to_counts().cpu().numpy()

    @staticmethod
    def empty(n, K):
        rw = row_words_for(K)
        return PackedGenotypes(torch.zeros((max(int(n), 0), rw), dtype=torch.int32, device=_dev()), n, K)

    # ---- uint8 [n, K] <-> packed -------------------------------------------------
    @staticmethod
    def from_counts(counts) -> "PackedGenotypes":
        """counts: uint8 [n, K] array/tensor (host or device) -> packed on the GPU."""
        if isinstance(counts, np.ndarray) and counts.ndim == 2 and counts.size:
            # host matrix: pinned double-buffered upload + pack (no pageable copy of the whole matrix)
            h = np.ascontiguousarray(counts, dtype=np.uint8)
            n, K = h.shape
            out = PackedGenotypes.empty(n, K)
            check(lib.loc_upload_pack_counts(h.ctypes.data, n, K, out.ptr, out.row_words, _stream()),
                  "loc_upload_pack_counts")
            return out
        c = _as_dev(counts, torch.uint8)
        n, K = c.shape
        out = PackedGenotypes.empty(n, K)
        for r0 in range(0, n, 65535):
            r1 = min(n, r0 + 65535)
            check(lib.loc_pack_counts(c[r0:r1].data_ptr(), r1 - r0, K, out.words[r0:r1].data_ptr(), out.row_words,
                                      _stream()), "loc_pack_counts")
        return out

    def to_counts(self) -> torch.Tensor:
        out = torch.empty((self.n, self.K), dtype=torch.uint8, device=self.words.device)
        for r0 in range(0, self.n, 65535):
            r1 = min(self.n, r0 + 65535)
            check(lib.loc_unpack_counts(self.words[r0:r1].data_ptr(), r1 - r0, self.K, self.row_words,
                                        out[r0:r1].data_ptr(), _stream()), "loc_unpack_counts")
        return out

    # ---- gathers ---------------------------------------------------------------------
    def take_rows(self, rows) -> "PackedGenotypes":
        """out[r] = self[rows[r]]  (ac[:, idx] transposed, locator.py:303-307)."""
        idx = _idx(rows)
        n_out = int(idx.numel())
        out = PackedGenotypes.empty(n_out, self.K)
        for r0 in range(0, n_out, 65535):
            r1 = min(n_out, r0 + 65535)
            check(lib.loc_gather_rows(self.ptr, self.row_words, idx[r0:r1].data_ptr(), r1 - r0,
                                      out.words[r0:r1].data_ptr(), _stream()), "loc_gather_rows")
        return out

    def take_cols(self, cols) -> "PackedGenotypes":
        """out[:, k] = self[:, cols[k]]  (bootstrap site_order :651-653, max_SNPs :279)."""
        idx = _idx(cols)
        K_out = int(idx.numel())
        out = PackedGenotypes.empty(self.n, K_out)
        for r0 in range(0, self.n, 65535):
            r1 = min(self.n, r0 + 65535)
            check(lib.loc_gather_cols(self.words[r0:r1].data_ptr(), r1 - r0, self.row_words, idx.data_ptr(), K_out,
                                      out.words[r0:r1].data_ptr(), out.row_words, _stream()), "loc_gather_cols")
        return out

    def site_sums(self) -> torch.Tensor:
        """int64 [K] device tensor: sum over all rows of every SNP's allele count (locator.py:714-717)."""
        out = torch.empty(max(self.K, 1), dtype=torch.int64, device=self.words.device)
        check(lib.loc_site_sums(self.ptr, self.n, self.K, self.row_words, out.data_ptr(), _stream()), "loc_site_sums")
        return out[: self.K]

    def clone(self) -> "PackedGenotypes":
        return PackedGenotypes(self.words.clone(), self.n, self.K)

    def replace_cols(self, sites, vals) -> None:
        """self[:, sites[i]] = vals[i]  in place (jacknife :726-727); vals uint8 [nsites, n]."""
        s = _idx(sites)
        v = _as_dev(vals, torch.uint8)
        assert v.shape == (s.numel(), self.n)
        check(lib.loc_replace_cols(self.ptr, self.n, self.row_words, s.data_ptr(), int(s.numel()), v.data_ptr(),
                                   _stream()), "loc_replace_cols")
        self.version += 1

    def patch(self, ks, samps, vals) -> None:
        """self[samps[i], ks[i]] = vals[i]  (imputed calls of replace_md :258-261)."""
        k = _idx(ks)
        s = _idx(samps)
        v = _as_dev(np.asarray(vals, dtype=np.uint8), torch.uint8)
        check(lib.loc_patch_calls(self.ptr, self.row_words, k.data_ptr(), s.data_ptr(), v.data_ptr(), int(k.numel()),
                                  _stream()), "loc_patch_calls")
        self.version += 1


class _Staging(threading.local):
    """Per-thread pair of pinned host buffers the genotype rows are read into (reused across windows)."""
    bufs = None
    events = None


_staging = _Staging()
UPLOAD_BLOCK_BYTES = 1 << 29  # rows are staged in blocks of at most 512 MB


def _staging_buffers(nbytes):
    st = _staging
    if st.bufs is None or st.bufs[0].numel() < nbytes:
        for ev in (st.events or []):
            if ev is not None:
                ev.synchronize()  # nothing may still be reading the buffers that are about to be freed
        # windows differ in their SNP counts: leave headroom so that the next, slightly larger one fits
        cap = min(max(int(nbytes), UPLOAD_BLOCK_BYTES), int(nbytes) + int(nbytes) // 4)
        st.bufs = [torch.empty(cap, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
        st.events = [None, None]
    return st


_TORCH_DTYPES = {np.dtype(np.int8): torch.int8, np.dtype(np.uint8): torch.uint8}


def upload_rows(rows) -> torch.Tensor:
    """Rows of a genotype file on disk -> device tensor of ``rows.stored_shape``, without an intermediate pageable
    copy: io.ZarrRows (GT int8 [nvar, N, 2]) or io.BedRows (.bed records uint8 [nvar, ceil(N/4)]).

    Blocks of rows are read (zarr: chunks decoded by a thread pool, io._zarr_array; .bed: positioned reads) straight
    into one of two pinned staging buffers and copied to the device asynchronously: block i+1 is read while block i
    is in flight.
    """
    shape, dtype = tuple(rows.stored_shape), _TORCH_DTYPES[np.dtype(rows.stored_dtype)]
    nvar = shape[0]
    dev = _dev()
    out = torch.empty(shape, dtype=dtype, device=dev)
    if nvar == 0:
        return out
    row_bytes = int(np.prod(shape[1:], dtype=np.int64)) * out.element_size()
    block = max(1, min(nvar, UPLOAD_BLOCK_BYTES // row_bytes))
    st = _staging_buffers(block * row_bytes)
    stream = torch.cuda.current_stream()
    for i, a in enumerate(range(0, nvar, block)):
        b = min(nvar, a + block)
        slot = i & 1
        if st.events[slot] is not None:
            st.events[slot].synchronize()  # the previous copy out of this buffer has finished
        host = st.bufs[slot][:(b - a) * row_bytes].view(dtype).view((b - a,) + shape[1:])
        rows.rows(a, b).read(out=host.numpy())
        out[a:b].copy_(host, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(stream)
        st.events[slot] = ev
    return out


def site_stats(gt, min_mac=2):
    """Per-site allelism / alt count / missing calls / keep flag of GT int8 [nvar, N, 2] on the GPU.

    Returns (n_alleles, alt_count, n_missing, keep) as device tensors (locator.py:267-273).
    """
    g = _as_dev(gt, torch.int8)
    nvar, N, ploidy = g.shape
    assert ploidy == 2
    dev = g.device
    na = torch.empty(nvar, dtype=torch.int32, device=dev)
    alt = torch.empty(nvar, dtype=torch.int32, device=dev)
    miss = torch.empty(nvar, dtype=torch.int32, device=dev)
    keep = torch.empty(nvar, dtype=torch.uint8, device=dev)
    check(lib.loc_site_stats(g.data_ptr(), nvar, N, int(min_mac), na.data_ptr(), alt.data_ptr(), miss.data_ptr(),
                             keep.data_ptr(), _stream()), "loc_site_stats")
    return g, na, alt, miss, keep


def compact_sites(keep: torch.Tensor) -> torch.Tensor:
    """Ascending indices of the kept sites as an int64 device tensor (prefix sum + scatter on the GPU; the only
    thing the host reads is their number, which sizes the packed matrix)."""
    nvar = int(keep.numel())
    idx = torch.empty(max(nvar, 1), dtype=torch.int64, device=keep.device)
    count = torch.zeros(1, dtype=torch.int64, device=keep.device)
    check(lib.loc_compact_sites(keep.data_ptr(), nvar, idx.data_ptr(), count.data_ptr(), _stream()), "loc_compact_sites")
    return idx[: int(count.item())]


def missing_calls(g: torch.Tensor, site_idx: torch.Tensor, n_missing: torch.Tensor):
    """(k, sample) of every missing call of the kept sites, row-major (site, sample) order, as int64 device
    tensors -- np.nonzero(is_missing) of the filtered cube without touching it on the host."""
    nvar, N, _ = g.shape
    K = int(site_idx.numel())
    offsets = torch.zeros(K + 1, dtype=torch.int64, device=g.device)
    null = None
    check(lib.loc_missing_calls(g.data_ptr(), nvar, N, site_idx.data_ptr(), K, n_missing.data_ptr(),
                                offsets.data_ptr(), null, null, _stream()), "loc_missing_calls")
    total = int(offsets[K].item())
    ks = torch.empty(max(total, 1), dtype=torch.int64, device=g.device)
    samps = torch.empty(max(total, 1), dtype=torch.int64, device=g.device)
    if total:
        check(lib.loc_missing_calls(g.data_ptr(), nvar, N, site_idx.data_ptr(), K, n_missing.data_ptr(),
                                    offsets.data_ptr(), ks.data_ptr(), samps.data_ptr(), _stream()), "loc_missing_calls")
    return ks[:total], samps[:total]


def pack_sites(g: torch.Tensor, site_idx) -> PackedGenotypes:
    """Pack the listed sites of device GT int8 [nvar, N, 2] -> PackedGenotypes [N, K]."""
    idx = _idx(site_idx)
    nvar, N, _ = g.shape
    K = int(idx.numel())
    out = PackedGenotypes.empty(N, K)
    if K:
        check(lib.loc_pack_sites(g.data_ptr(), nvar, N, idx.data_ptr(), K, out.ptr, out.row_words, _stream()),
              "loc_pack_sites")
    return out


# ---- PLINK 1 .bed records on the device (the GT cube they stand for is never built) ----
class BedRecords:
    """SNP-major .bed records uint8 [nvar, ceil(N/4)] in device memory (header stripped); ``shape`` is that of
    the GT cube [nvar, N, 2] they stand for."""

    def __init__(self, records: torch.Tensor, nsamp: int):
        self.records = records
        self.nvar, self.nsamp = int(records.shape[0]), int(nsamp)
        assert records.dim() == 2 and records.shape[1] == (self.nsamp + 3) // 4

    @property
    def shape(self):
        return (self.nvar, self.nsamp, 2)

    @staticmethod
    def upload(rows) -> "BedRecords":
        """io.BedRows -> device (pinned double-buffered positioned reads, upload_rows)."""
        return BedRecords(upload_rows(rows), rows.nsamp)

    @staticmethod
    def from_host(records, nsamp) -> "BedRecords":
        return BedRecords(_as_dev(np.asarray(records, dtype=np.uint8), torch.uint8), nsamp)


def bed_site_stats(bed: BedRecords, min_mac=2):
    """site_stats on .bed records: (n_alleles, alt_count, n_missing, keep) device tensors of the cube they stand for
    (loc_bed_site_stats)."""
    dev = bed.records.device
    na = torch.empty(bed.nvar, dtype=torch.int32, device=dev)
    alt = torch.empty(bed.nvar, dtype=torch.int32, device=dev)
    miss = torch.empty(bed.nvar, dtype=torch.int32, device=dev)
    keep = torch.empty(bed.nvar, dtype=torch.uint8, device=dev)
    check(lib.loc_bed_site_stats(bed.records.data_ptr(), bed.nvar, bed.nsamp, int(min_mac), na.data_ptr(),
                                 alt.data_ptr(), miss.data_ptr(), keep.data_ptr(), _stream()), "loc_bed_site_stats")
    return na, alt, miss, keep


def bed_pack_sites(bed: BedRecords, site_idx) -> PackedGenotypes:
    """pack_sites on .bed records: the listed sites -> PackedGenotypes [N, K] (loc_bed_pack_sites)."""
    idx = _idx(site_idx)
    K = int(idx.numel())
    out = PackedGenotypes.empty(bed.nsamp, K)
    if K:
        check(lib.loc_bed_pack_sites(bed.records.data_ptr(), bed.nvar, bed.nsamp, idx.data_ptr(), K, out.ptr,
                                     out.row_words, _stream()), "loc_bed_pack_sites")
    return out


def bed_missing_calls(bed: BedRecords, site_idx: torch.Tensor, n_missing: torch.Tensor):
    """missing_calls on .bed records: (k, sample) of every missing call of the kept sites in row-major (site,
    sample) order (loc_bed_missing_calls)."""
    K = int(site_idx.numel())
    dev = bed.records.device
    offsets = torch.zeros(K + 1, dtype=torch.int64, device=dev)
    null = None
    check(lib.loc_bed_missing_calls(bed.records.data_ptr(), bed.nvar, bed.nsamp, site_idx.data_ptr(), K,
                                    n_missing.data_ptr(), offsets.data_ptr(), null, null, _stream()),
          "loc_bed_missing_calls")
    total = int(offsets[K].item())
    ks = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
    samps = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
    if total:
        check(lib.loc_bed_missing_calls(bed.records.data_ptr(), bed.nvar, bed.nsamp, site_idx.data_ptr(), K,
                                        n_missing.data_ptr(), offsets.data_ptr(), ks.data_ptr(), samps.data_ptr(),
                                        _stream()), "loc_bed_missing_calls")
    return ks[:total], samps[:total]


def pack_sites_mapped(g, src, flip) -> PackedGenotypes:
    """A query in a stored model's site order: PackedGenotypes [N, K] where column k is query record src[k] (-1:
    absent) of device GT int8 [nvar, N, 2] (GT cube) or BedRecords, allele roles swapped where flip[k]; missing
    calls, calls with an allele index >= 2 and absent sites are 3 (loc_pack_sites_mapped / loc_bed_pack_sites_mapped)."""
    s = _idx(src)
    f = _as_dev(flip, torch.uint8)
    K = int(s.numel())
    if isinstance(g, BedRecords):
        out = PackedGenotypes.empty(g.nsamp, K)
        if K:
            check(lib.loc_bed_pack_sites_mapped(g.records.data_ptr(), g.nvar, g.nsamp, s.data_ptr(), f.data_ptr(), K,
                                                out.ptr, out.row_words, _stream()), "loc_bed_pack_sites_mapped")
        return out
    nvar, N, _ = g.shape
    out = PackedGenotypes.empty(N, K)
    if K:
        check(lib.loc_pack_sites_mapped(g.data_ptr(), nvar, N, s.data_ptr(), f.data_ptr(), K, out.ptr, out.row_words,
                                        _stream()), "loc_pack_sites_mapped")
    return out
