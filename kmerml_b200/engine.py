"""Host-side driver of the dense counting path: torch owns device memory and the
stream, the work is done by libkmerml_b200.so through the C-ABI.

Replaces (reference tree) kmerml/kmers/generate.py:36-58 for k <= 14 and adds the
frequency rows the reference only gestures at (tests/test_ml.py:8).
"""
import ctypes
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _lib


def row_layout(k_list):
    """{k: (offset, length)} of the concatenated output row, in k_list order."""
    out, off = {}, 0
    for k in k_list:
        out[k] = (off, 4 ** k)
        off += 4 ** k
    return out, off


def _dedupe(k_values):
    ks = list(dict.fromkeys(int(k) for k in k_values))
    if not ks:
        raise ValueError("k_values is empty")
    return ks


@dataclass
class DenseResult:
    k_list: list
    counts: torch.Tensor      # [n_genomes, row_len] int32 storage of uint32 counts
    freq: torch.Tensor        # [n_genomes, row_len] float32 or None
    totals: torch.Tensor      # [n_genomes, nk] int64 (counted windows per k)

    def counts_of(self, g, k):
        lay, _ = row_layout(self.k_list)
        off, n = lay[k]
        return self.counts[g, off:off + n]

    def freq_of(self, g, k):
        lay, _ = row_layout(self.k_list)
        off, n = lay[k]
        return self.freq[g, off:off + n]

    def counts_numpy(self, g, k):
        return self.counts_of(g, k).cpu().numpy().view(np.uint32)


def _device_index(device):
    dev = torch.device(device if device is not None else "cuda")
    if dev.type != "cuda":
        raise _lib.KmermlError("kmerml_b200 runs on a CUDA device only (no CPU fallback)")
    return dev.index if dev.index is not None else torch.cuda.current_device()


def _flags(canonical, partition):
    """partition: True (default paths), False (global atomics for k = 9..12), "k8as9" (k = 8 counted as
    9-mers through the partition path instead of the packed shared histogram)."""
    f = _lib.FLAG_CANONICAL if canonical else 0
    if partition == "k8as9":
        return f | _lib.FLAG_K8_AS_9
    return f | (0 if partition else _lib.FLAG_NO_PARTITION)


def count_dense_device(fasta, offsets, k_values, *, min_record_len=None, canonical=False,
                       want_freq=True, out_counts=None, out_freq=None, out_totals=None, partition=True):
    """Count k-mers of genomes already resident in HBM.

    fasta    uint8 CUDA tensor holding the FASTA bytes of all genomes back to back
    offsets  n_genomes+1 byte offsets (host ints)
    """
    if not torch.cuda.is_available():
        raise _lib.KmermlError("no CUDA device: kmerml_b200 has no CPU fallback")
    if not (fasta.is_cuda and fasta.dtype == torch.uint8 and fasta.is_contiguous()):
        raise ValueError("fasta must be a contiguous uint8 CUDA tensor")
    ks = _dedupe(k_values)
    dev = fasta.device.index
    ctx = _lib.context(dev)
    L = _lib.load()
    n = len(offsets) - 1
    _, row_len = row_layout(ks)
    counts = out_counts if out_counts is not None else torch.empty((n, row_len), dtype=torch.int32, device=fasta.device)
    freq = None
    if want_freq:
        freq = out_freq if out_freq is not None else torch.empty((n, row_len), dtype=torch.float32, device=fasta.device)
    totals = out_totals if out_totals is not None else torch.zeros((n, len(ks)), dtype=torch.int64, device=fasta.device)
    offs = np.asarray(offsets, dtype=np.uint64)
    karr = np.asarray(ks, dtype=np.int32)
    stream = torch.cuda.current_stream(fasta.device).cuda_stream
    _lib.check(L.kmerml_count_dense_batch(
        ctx.handle, fasta.data_ptr(), offs.ctypes.data, n, karr.ctypes.data, len(ks),
        int(min_record_len or 0), _flags(canonical, partition),
        counts.data_ptr(), counts.stride(0), freq.data_ptr() if freq is not None else None,
        freq.stride(0) if freq is not None else 0, totals.data_ptr(), ctypes.c_void_p(stream)))
    return DenseResult(ks, counts, freq, totals)


class CompactDenseResult:
    """Host result of count_dense_host(..., compact=True): the count rows as they crossed PCIe (one byte per bin
    for k >= 10 plus an exception list, uint32 for k < 10; include/kmerml_b200.h, kmerml_count_dense_host_compact).
    Lossless; counts_numpy(g, k) widens one k of one genome on demand (host code of the library)."""

    def __init__(self, k_list, rows, freq, totals, overflow_rows):
        self.k_list, self.rows, self.freq, self.totals = k_list, rows, freq, totals
        self._wide = overflow_rows                       # {genome: uint32 row} for genomes whose exception list overflowed

    def counts_numpy(self, g, k):
        lay, _ = row_layout(self.k_list)
        off, n = lay[k]
        if g in self._wide:
            return self._wide[g][off:off + n]
        out = np.empty(n, dtype=np.uint32)
        karr = np.asarray(self.k_list, dtype=np.int32)
        row = self.rows[g]
        _lib.check(_lib.load().kmerml_compact_expand(karr.ctypes.data, len(self.k_list), row.data_ptr(),
                                                     self.k_list.index(k), out.ctypes.data))
        return out

    def counts_tensor(self):
        """[n_genomes, row_len] int32 tensor (uint32 storage) of all rows, widened (what count_dense_host returns)."""
        lay, row_len = row_layout(self.k_list)
        out = np.empty((self.rows.shape[0], row_len), dtype=np.uint32)
        karr = np.asarray(self.k_list, dtype=np.int32)
        L = _lib.load()
        for g in range(self.rows.shape[0]):
            if g in self._wide:
                out[g] = self._wide[g]
                continue
            for ki, k in enumerate(self.k_list):
                off, n = lay[k]
                _lib.check(L.kmerml_compact_expand(karr.ctypes.data, len(self.k_list), self.rows[g].data_ptr(), ki,
                                                   out[g, off:off + n].ctypes.data))
        return torch.from_numpy(out.view(np.int32))


def count_dense_host(buffers, k_values, *, min_record_len=None, canonical=False, want_freq=True,
                     device=None, out_counts=None, out_freq=None, out_totals=None, partition=True,
                     freq_on_device=False, wide_d2h=False, compact=False, out_rows=None, nibbles=True):
    """End to end from host byte buffers (numpy uint8 arrays / pinned torch tensors): H2D,
    counting and D2H all inside libkmerml_b200.so.  Returns host (pinned) torch tensors; with
    freq_on_device the frequency rows stay in HBM (a CUDA tensor) for the distance / ML stage."""
    if not torch.cuda.is_available():
        raise _lib.KmermlError("no CUDA device: kmerml_b200 has no CPU fallback")
    ks = _dedupe(k_values)
    dev = _device_index(device)
    ctx = _lib.context(dev)
    L = _lib.load()
    n = len(buffers)
    _, row_len = row_layout(ks)
    ptrs = (ctypes.c_void_p * max(n, 1))()
    sizes = np.zeros(max(n, 1), dtype=np.uint64)
    keep = []
    for i, b in enumerate(buffers):
        if isinstance(b, torch.Tensor):
            assert b.dtype == torch.uint8 and not b.is_cuda and b.is_contiguous()
            ptrs[i] = b.data_ptr() if b.numel() else None
            sizes[i] = b.numel()
        else:
            a = np.ascontiguousarray(np.frombuffer(b, dtype=np.uint8) if not isinstance(b, np.ndarray) else b)
            keep.append(a)
            ptrs[i] = a.ctypes.data if a.size else None
            sizes[i] = a.size
    pin = True
    karr = np.asarray(ks, dtype=np.int32)
    if compact:
        row_bytes = int(L.kmerml_compact_row_bytes(karr.ctypes.data, len(ks)))
        counts = out_rows if out_rows is not None else torch.empty((n, row_bytes), dtype=torch.uint8, pin_memory=pin)
    else:
        counts = out_counts if out_counts is not None else torch.empty((n, row_len), dtype=torch.int32, pin_memory=pin)
    freq = None
    if want_freq:
        if out_freq is not None:
            freq = out_freq
            freq_on_device = freq.is_cuda
        elif freq_on_device:
            freq = torch.empty((n, row_len), dtype=torch.float32, device=torch.device("cuda", dev))
        else:
            freq = torch.empty((n, row_len), dtype=torch.float32, pin_memory=pin)
    totals = out_totals if out_totals is not None else torch.zeros((n, len(ks)), dtype=torch.int64, pin_memory=pin)
    flags = _flags(canonical, partition) | (_lib.FLAG_FREQ_ON_DEVICE if (freq is not None and freq.is_cuda) else 0)
    if wide_d2h:                     # uint32 rows over PCIe as they are (default: bytes / nibbles + exceptions for k >= 10)
        flags |= _lib.FLAG_WIDE_D2H
    if not nibbles:                  # keep every level of k >= 10 at one byte per bin
        flags |= _lib.FLAG_NO_NIBBLES
    if compact:
        _lib.check(L.kmerml_count_dense_host_compact(
            ctx.handle, ptrs, sizes.ctypes.data, n, karr.ctypes.data, len(ks), int(min_record_len or 0),
            flags, counts.data_ptr(), counts.stride(0),
            freq.data_ptr() if freq is not None else None, freq.stride(0) if freq is not None else 0,
            totals.data_ptr()))
        # genomes whose exception list overflowed (too many bins at 255 / 15 or more): counted again, uint32 rows
        over = []
        for g in range(n):
            r = L.kmerml_compact_row_overflowed(karr.ctypes.data, len(ks), counts[g].data_ptr())
            if r < 0:
                _lib.check(r)
            if r:
                over.append(g)
        wide = {}
        if over:
            sub = count_dense_host([buffers[g] for g in over], ks, min_record_len=min_record_len, canonical=canonical,
                                   want_freq=False, device=device, partition=partition, wide_d2h=True)
            for j, g in enumerate(over):
                wide[g] = sub.counts[j].numpy().view(np.uint32)
        return CompactDenseResult(ks, counts, freq, totals, wide)
    _lib.check(L.kmerml_count_dense_host(
        ctx.handle, ptrs, sizes.ctypes.data, n, karr.ctypes.data, len(ks), int(min_record_len or 0),
        flags, counts.data_ptr(), counts.stride(0),
        freq.data_ptr() if freq is not None else None, freq.stride(0) if freq is not None else 0,
        totals.data_ptr()))
    return DenseResult(ks, counts, freq, totals)


def first_occurrence_device(fasta, k, *, min_record_len=None):
    """uint32[4^k] (as int64 tensor view-safe int32 storage) end offset of each k-mer's first window."""
    ctx = _lib.context(fasta.device.index)
    L = _lib.load()
    out = torch.empty(4 ** k, dtype=torch.int32, device=fasta.device)
    stream = torch.cuda.current_stream(fasta.device).cuda_stream
    _lib.check(L.kmerml_first_occurrence(ctx.handle, fasta.data_ptr(), fasta.numel(), int(k),
                                         int(min_record_len or 0), out.data_ptr(), ctypes.c_void_p(stream)))
    return out


def revcomp_codes(k):
    """numpy int64[4^k]: index of the reverse complement of every k-mer (A0 C1 G2 T3)."""
    idx = np.arange(4 ** k, dtype=np.int64)
    rc = np.zeros_like(idx)
    t = idx.copy()
    for _ in range(k):
        rc = (rc << 2) | (3 - (t & 3))
        t >>= 2
    return rc


def static_features_device(k, *, compat=False, device=None):
    """int32 [4^k, 8] CUDA tensor: n, A/C/G/T counts, cpg_count, has_repeat, first base."""
    dev = _device_index(device)
    ctx = _lib.context(dev)
    out = torch.empty((4 ** k, 8), dtype=torch.int32, device=torch.device("cuda", dev))
    stream = torch.cuda.current_stream(out.device).cuda_stream
    _lib.check(_lib.load().kmerml_static_features(ctx.handle, int(k), 1 if compat else 0, out.data_ptr(),
                                                  ctypes.c_void_p(stream)))
    return out


def normalize_rows_device(counts, totals):
    """float32 frequencies of uint32 count rows (int32 storage) given int64 row totals."""
    ctx = _lib.context(counts.device.index)
    out = torch.empty(counts.shape, dtype=torch.float32, device=counts.device)
    stream = torch.cuda.current_stream(counts.device).cuda_stream
    totals = totals.to(torch.int64).contiguous()
    _lib.check(_lib.load().kmerml_normalize_rows(ctx.handle, counts.data_ptr(), counts.stride(0), totals.data_ptr(),
                                                 counts.shape[0], counts.shape[1], out.data_ptr(), out.stride(0),
                                                 ctypes.c_void_p(stream)))
    return out


_DTYPE_CODE = {torch.float32: 0, torch.int32: 1, torch.float64: 2}
_METRIC_CODE = {"cosine": 0, "euclidean": 1}


def pairwise_distance_device(x, metric="cosine", *, out_dtype=torch.float32):
    """n x n distance matrix of the rows of the CUDA tensor x (float32, float64, or int32
    holding uint32 counts); float64 accumulation."""
    if metric not in _METRIC_CODE:
        raise ValueError(f"metric must be one of {sorted(_METRIC_CODE)}")
    if x.dtype not in _DTYPE_CODE or not x.is_cuda or x.dim() != 2 or x.stride(1) != 1:
        raise ValueError("x must be a 2-D CUDA tensor (float32 / float64 / int32) with contiguous rows")
    ctx = _lib.context(x.device.index)
    n, m = x.shape
    out = torch.empty((n, n), dtype=out_dtype, device=x.device)
    stream = torch.cuda.current_stream(x.device).cuda_stream
    o32 = out.data_ptr() if out_dtype == torch.float32 else None
    o64 = out.data_ptr() if out_dtype == torch.float64 else None
    _lib.check(_lib.load().kmerml_pairwise_distance(ctx.handle, x.data_ptr(), _DTYPE_CODE[x.dtype], x.stride(0), n, m,
                                                    _METRIC_CODE[metric], o32, o64, ctypes.c_void_p(stream)))
    return out


def pairwise_distance_rows_device(counts, row_begin, row_end, metric="cosine", *, out_dtype=torch.float32):
    """Rows [row_begin, row_end) of the n x n distance matrix of uint32 count rows (int32 storage; the row length
    a multiple of 64): one rank's block of a sharded distance computation, bit-identical to the same rows of
    pairwise_distance_device."""
    if metric not in _METRIC_CODE:
        raise ValueError(f"metric must be one of {sorted(_METRIC_CODE)}")
    if counts.dtype != torch.int32 or not counts.is_cuda or counts.dim() != 2 or counts.stride(1) != 1:
        raise ValueError("counts must be a 2-D int32 CUDA tensor with contiguous rows")
    ctx = _lib.context(counts.device.index)
    n, m = counts.shape
    out = torch.empty((max(row_end - row_begin, 0), n), dtype=out_dtype, device=counts.device)
    if out.numel() == 0:
        return out
    stream = torch.cuda.current_stream(counts.device).cuda_stream
    o32 = out.data_ptr() if out_dtype == torch.float32 else None
    o64 = out.data_ptr() if out_dtype == torch.float64 else None
    _lib.check(_lib.load().kmerml_pairwise_distance_rows(ctx.handle, counts.data_ptr(), counts.stride(0), n, m,
                                                         int(row_begin), int(row_end), _METRIC_CODE[metric], o32, o64,
                                                         ctypes.c_void_p(stream)))
    return out


def count_planes_device(counts, out_planes=None, n_rows=None):
    """Byte planes of uint32 count rows (int32 storage): (planes uint8 [4, n_rows, m], squared norms float64 [n_rows],
    largest count as a 1-element int32 device tensor).  n_rows >= counts.shape[0] pads with zero rows (equal blocks for
    an all_gather).  What one rank of a sharded distance computation runs on ITS rows before the gather."""
    if counts.dtype != torch.int32 or not counts.is_cuda or counts.dim() != 2 or counts.stride(1) != 1:
        raise ValueError("counts must be a 2-D int32 CUDA tensor with contiguous rows")
    n, m = counts.shape
    rows = n if n_rows is None else int(n_rows)
    if rows < n:
        raise ValueError("n_rows smaller than the number of rows")
    dev = counts.device
    planes = out_planes if out_planes is not None else torch.empty((4, rows, m), dtype=torch.uint8, device=dev)
    if planes.shape != (4, rows, m) or planes.dtype != torch.uint8 or not planes.is_contiguous():
        raise ValueError("out_planes must be a contiguous uint8 [4, n_rows, m] tensor")
    if rows > n:
        planes[:, n:].zero_()
    sumsq = torch.zeros(rows, dtype=torch.float64, device=dev)
    mx = torch.zeros(2, dtype=torch.int32, device=dev)
    if n:
        ctx = _lib.context(dev.index)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(_lib.load().kmerml_count_planes(ctx.handle, counts.data_ptr(), counts.stride(0), n, m, planes.data_ptr(),
                                                   rows * m, sumsq.data_ptr(), mx.data_ptr(), ctypes.c_void_p(stream)))
    return planes, sumsq, mx[:1]


def planes_needed(max_count):
    """How many byte planes hold every count up to max_count (uint32)."""
    max_count = int(max_count) & 0xFFFFFFFF
    return 4 if max_count >= 1 << 24 else 3 if max_count >= 1 << 16 else 2 if max_count >= 1 << 8 else 1


def distance_rows_planes_device(planes, n_planes, sumsq, row_begin, row_end, metric="cosine", *, out_dtype=torch.float32):
    """Rows [row_begin, row_end) of the n x n distance matrix from the first n_planes byte planes of ALL n count rows
    (uint8 [>= n_planes, n, m]) and their squared norms: bit-identical to pairwise_distance_device on the counts."""
    if metric not in _METRIC_CODE:
        raise ValueError(f"metric must be one of {sorted(_METRIC_CODE)}")
    if planes.dtype != torch.uint8 or not planes.is_cuda or planes.dim() != 3 or not planes[0].is_contiguous():
        raise ValueError("planes must be a uint8 CUDA tensor [planes, n, m] with contiguous planes")
    _, n, m = planes.shape
    out = torch.empty((max(row_end - row_begin, 0), n), dtype=out_dtype, device=planes.device)
    if out.numel() == 0:
        return out
    ctx = _lib.context(planes.device.index)
    stream = torch.cuda.current_stream(planes.device).cuda_stream
    o32 = out.data_ptr() if out_dtype == torch.float32 else None
    o64 = out.data_ptr() if out_dtype == torch.float64 else None
    _lib.check(_lib.load().kmerml_distance_rows_planes(ctx.handle, planes.data_ptr(), planes.stride(0), int(n_planes), n, m,
                                                       sumsq.data_ptr(), int(row_begin), int(row_end), _METRIC_CODE[metric],
                                                       o32, o64, ctypes.c_void_p(stream)))
    return out


def count_dense_range_device(fasta, begin, end, k_values, min_record_len=None, canonical=False, partition=True):
    """(counts int32[row_len], totals int64[nk]) of the windows of ONE genome whose last base
    lies in bytes [begin, end): the additive unit of intra-genome / multi-GPU parallelism."""
    ks = _dedupe(k_values)
    ctx = _lib.context(fasta.device.index)
    _, row_len = row_layout(ks)
    counts = torch.empty(row_len, dtype=torch.int32, device=fasta.device)
    totals = torch.zeros(len(ks), dtype=torch.int64, device=fasta.device)
    karr = np.asarray(ks, dtype=np.int32)
    stream = torch.cuda.current_stream(fasta.device).cuda_stream
    _lib.check(_lib.load().kmerml_count_dense_range(
        ctx.handle, fasta.data_ptr(), fasta.numel(), int(begin), int(end), karr.ctypes.data, len(ks),
        int(min_record_len or 0), _flags(canonical, partition), counts.data_ptr(), totals.data_ptr(),
        ctypes.c_void_p(stream)))
    return counts, totals


def _retry_after_cache_release(call):
    """The library's workspaces are its own device allocations: when one cannot grow because torch's caching
    allocator sits on freed blocks, release them and try once more (the workspace persists afterwards)."""
    try:
        return call()
    except _lib.KmermlError as exc:
        if "allocation" not in str(exc):
            raise
        torch.cuda.empty_cache()
        return call()


def count_sparse_device(fasta, k, *, min_record_len=None, canonical=False, want_first=True):
    """Distinct k-mers of ONE genome for any k <= 32 (meant for k > 14): returns
    (keys int64[n] -- uint64 2-bit packed, sorted --, counts int32[n], first int32[n] or None, windows)."""
    ctx = _lib.context(fasta.device.index)
    L = _lib.load()
    stream = ctypes.c_void_p(torch.cuda.current_stream(fasta.device).cuda_stream)
    cap = max(1024, min(int(fasta.numel()), 1 << 22))
    keys = torch.empty(cap, dtype=torch.int64, device=fasta.device)
    counts = torch.empty(cap, dtype=torch.int32, device=fasta.device)
    first = torch.empty(cap, dtype=torch.int32, device=fasta.device) if want_first else None
    nu, nw = ctypes.c_uint64(0), ctypes.c_uint64(0)
    _lib.check(L.kmerml_count_sparse(ctx.handle, fasta.data_ptr() if fasta.numel() else None, fasta.numel(), int(k),
                                     int(min_record_len or 0), _lib.FLAG_CANONICAL if canonical else 0,
                                     keys.data_ptr(), counts.data_ptr(), first.data_ptr() if want_first else None,
                                     cap, ctypes.byref(nu), ctypes.byref(nw), stream))
    n = int(nu.value)
    if n > cap:
        keys, counts, first = _sparse_fetch(ctx, L, n, fasta.device, want_first, stream)
    return keys[:n], counts[:n], (first[:n] if want_first else None), int(nw.value)


def _sparse_fetch(ctx, L, n, device, want_first, stream):
    """More distinct k-mers than the first guess: the reduced result is still in the workspace; size the
    outputs and copy it out (no second emit / sort / reduce)."""
    keys = torch.empty(n, dtype=torch.int64, device=device)
    counts = torch.empty(n, dtype=torch.int32, device=device)
    first = torch.empty(n, dtype=torch.int32, device=device) if want_first else None
    _lib.check(L.kmerml_sparse_fetch(ctx.handle, keys.data_ptr(), counts.data_ptr(),
                                     first.data_ptr() if want_first else None, n, stream))
    return keys, counts, first


SPARSE_RANGE_ALIGN = 131072


def count_sparse_range_device(fasta, begin, end, k, *, min_record_len=None, canonical=False):
    """count_sparse_device for the windows ending in the byte range [begin, end) (multiples of SPARSE_RANGE_ALIGN,
    or end == file size): the multi-GPU unit.  First offsets are relative to the file."""
    ctx = _lib.context(fasta.device.index)
    L = _lib.load()
    stream = ctypes.c_void_p(torch.cuda.current_stream(fasta.device).cuda_stream)
    cap = max(1024, min(int(end) - int(begin), 1 << 22))
    keys = torch.empty(cap, dtype=torch.int64, device=fasta.device)
    counts = torch.empty(cap, dtype=torch.int32, device=fasta.device)
    first = torch.empty(cap, dtype=torch.int32, device=fasta.device)
    nu, nw = ctypes.c_uint64(0), ctypes.c_uint64(0)
    _retry_after_cache_release(lambda: _lib.check(L.kmerml_count_sparse_range(
        ctx.handle, fasta.data_ptr() if fasta.numel() else None, fasta.numel(), int(begin), int(end), int(k),
        int(min_record_len or 0), _lib.FLAG_CANONICAL if canonical else 0, keys.data_ptr(), counts.data_ptr(),
        first.data_ptr(), cap, ctypes.byref(nu), ctypes.byref(nw), stream)))
    n = int(nu.value)
    if n > cap:
        keys, counts, first = _sparse_fetch(ctx, L, n, fasta.device, True, stream)
    return keys[:n], counts[:n], first[:n], int(nw.value)


def emit_sparse_range_device(fasta, begin, end, k, owner_bits, *, min_record_len=None, canonical=False):
    """Windows (k-mer int64 storage of uint64, end offset int32) ending in the byte range [begin, end), grouped by
    owner = the top owner_bits bits of the 2k-bit k-mer; returns (keys, ends, [windows per owner])."""
    ctx = _lib.context(fasta.device.index)
    L = _lib.load()
    stream = ctypes.c_void_p(torch.cuda.current_stream(fasta.device).cuda_stream)
    cap = max(int(end) - int(begin), 1)
    keys = torch.empty(cap, dtype=torch.int64, device=fasta.device)
    ends = torch.empty(cap, dtype=torch.int32, device=fasta.device)
    nw = ctypes.c_uint64(0)
    owners = np.zeros(1 << int(owner_bits), dtype=np.uint64)
    _retry_after_cache_release(lambda: _lib.check(L.kmerml_emit_sparse_range(
        ctx.handle, fasta.data_ptr() if fasta.numel() else None, fasta.numel(), int(begin), int(end), int(k),
        int(min_record_len or 0), _lib.FLAG_CANONICAL if canonical else 0, int(owner_bits), keys.data_ptr(), ends.data_ptr(),
        cap, ctypes.byref(nw), owners.ctypes.data, stream)))
    n = int(nw.value)
    return keys[:n], ends[:n], [int(x) for x in owners]


def reduce_sparse_windows_device(keys, ends, sort_bits):
    """Windows in any order -> (distinct k-mers ascending in their low sort_bits bits, counts, smallest end offset)."""
    ctx = _lib.context(keys.device.index)
    L = _lib.load()
    stream = ctypes.c_void_p(torch.cuda.current_stream(keys.device).cuda_stream)
    n = int(keys.numel())
    if n == 0:
        return keys, torch.zeros(0, dtype=torch.int32, device=keys.device), ends
    keys, ends = keys.contiguous(), ends.contiguous()
    cap = max(1024, min(n, 1 << 22))
    ok = torch.empty(cap, dtype=torch.int64, device=keys.device)
    oc = torch.empty(cap, dtype=torch.int32, device=keys.device)
    of = torch.empty(cap, dtype=torch.int32, device=keys.device)
    nu = ctypes.c_uint64(0)
    _retry_after_cache_release(lambda: _lib.check(L.kmerml_reduce_sparse_windows(
        ctx.handle, int(sort_bits), keys.data_ptr(), ends.data_ptr(), n, ok.data_ptr(), oc.data_ptr(), of.data_ptr(), cap,
        ctypes.byref(nu), stream)))
    m = int(nu.value)
    if m > cap:
        ok, oc, of = _sparse_fetch(ctx, L, m, keys.device, True, stream)
    return ok[:m], oc[:m], of[:m]


def merge_sparse_device(keys, counts, first, k):
    """(k-mer, count, first) triples in any order, duplicates allowed -> distinct k-mers ascending, counts added,
    smallest first offset kept (int64 / int32 / int32 storage of uint64 / uint32 / uint32)."""
    ctx = _lib.context(keys.device.index)
    L = _lib.load()
    stream = ctypes.c_void_p(torch.cuda.current_stream(keys.device).cuda_stream)
    n = int(keys.numel())
    if n == 0:
        return keys, counts, first
    keys, counts, first = keys.contiguous(), counts.contiguous(), first.contiguous()
    ok = torch.empty(n, dtype=torch.int64, device=keys.device)
    oc = torch.empty(n, dtype=torch.int32, device=keys.device)
    of = torch.empty(n, dtype=torch.int32, device=keys.device)
    nu = ctypes.c_uint64(0)
    _retry_after_cache_release(lambda: _lib.check(L.kmerml_merge_sparse(
        ctx.handle, int(k), keys.data_ptr(), counts.data_ptr(), first.data_ptr(), n,
        ok.data_ptr(), oc.data_ptr(), of.data_ptr(), n, ctypes.byref(nu), stream)))
    m = int(nu.value)
    return ok[:m], oc[:m], of[:m]


def genome_stats_device(fasta):
    """{"contigs", "total_size", "gc_content", "n_count"} of one FASTA file on the GPU
    (the tallies of kmerml/utils/genome_metadata.py:55-85)."""
    ctx = _lib.context(fasta.device.index)
    out = torch.zeros(4, dtype=torch.int64, device=fasta.device)
    stream = torch.cuda.current_stream(fasta.device).cuda_stream
    _lib.check(_lib.load().kmerml_genome_stats(ctx.handle, fasta.data_ptr() if fasta.numel() else None, fasta.numel(),
                                               out.data_ptr(), ctypes.c_void_p(stream)))
    contigs, total, gc, nn = (int(v) for v in out.cpu().tolist())
    return {"contigs": contigs, "total_size": total, "n_count": nn,
            "gc_content": (gc / total) * 100 if total > 0 else 0}


def encode_device(fasta, want_tallies=False):
    """Stage 1 on its own: uint8 symbols of one FASTA file on the GPU -- 0..3 (A C G T) where the byte is a base of a
    record, 255 elsewhere (kmerml/kmers/generate.py:39-41,55-56).  With want_tallies also the int64[4] device tensor
    (contigs, total_size, G+C, N) of genome_stats_device."""
    ctx = _lib.context(fasta.device.index)
    sym = torch.empty(fasta.numel(), dtype=torch.uint8, device=fasta.device)
    tallies = torch.zeros(4, dtype=torch.int64, device=fasta.device) if want_tallies else None
    stream = torch.cuda.current_stream(fasta.device).cuda_stream
    _lib.check(_lib.load().kmerml_encode(ctx.handle, fasta.data_ptr() if fasta.numel() else None, fasta.numel(),
                                         sym.data_ptr() if sym.numel() else None,
                                         tallies.data_ptr() if want_tallies else None, ctypes.c_void_p(stream)))
    return (sym, tallies) if want_tallies else sym


def kmer_count_stats_device(counts_row, k):
    """Summary of one k's count vector (int32 storage of uint32) as kmerml/utils/kmer_metadata.py:59-78 reports
    it for a k{k}.txt file: totals over the OBSERVED k-mers.  Reduction + radix-select kernels
    (kmerml_count_stats), one small device -> host read."""
    ctx = _lib.context(counts_row.device.index)
    row = counts_row.contiguous()
    out = torch.empty(8, dtype=torch.int64, device=row.device)
    stream = torch.cuda.current_stream(row.device).cuda_stream
    _lib.check(_lib.load().kmerml_count_stats(ctx.handle, row.data_ptr(), row.numel(), out.data_ptr(), ctypes.c_void_p(stream)))
    total, n, mx, mn, lo, hi = (int(v) for v in out[:6].cpu().tolist())
    if n == 0:
        return {"k_value": k, "total_kmers": 0, "unique_kmers": 0, "max_count": 0, "min_count": 0,
                "mean_count": float("nan"), "median_count": float("nan"), "estimated_genome_size": k - 1}
    return {"k_value": k, "total_kmers": total, "unique_kmers": n, "max_count": mx, "min_count": mn,
            "mean_count": total / n, "median_count": (float(lo) + float(hi)) / 2.0, "estimated_genome_size": total + k - 1}


def column_stats_device(x):
    """(rows with a non-zero entry int32[m], mean float64[m], population variance float64[m]) of the columns of a
    2-D CUDA tensor (float32 / float64 / int32 storage of uint32 counts)."""
    if x.dtype not in _DTYPE_CODE or not x.is_cuda or x.dim() != 2 or x.stride(1) != 1:
        raise ValueError("x must be a 2-D CUDA tensor (float32 / float64 / int32) with contiguous rows")
    ctx = _lib.context(x.device.index)
    n, m = x.shape
    nnz = torch.empty(m, dtype=torch.int32, device=x.device)
    mean = torch.empty(m, dtype=torch.float64, device=x.device)
    var = torch.empty(m, dtype=torch.float64, device=x.device)
    stream = torch.cuda.current_stream(x.device).cuda_stream
    _lib.check(_lib.load().kmerml_column_stats(ctx.handle, x.data_ptr(), _DTYPE_CODE[x.dtype], x.stride(0), n, m,
                                               nnz.data_ptr(), mean.data_ptr(), var.data_ptr(), ctypes.c_void_p(stream)))
    return nnz, mean, var


def format_kmer_file_device(counts_row, first, k, *, canonical=False):
    """uint8 tensor: the text of the reference's k{k}.txt for one genome (kmerml/kmers/generate.py:68-91) from
    its dense count row (int32 storage of uint32, 4^k) and first-occurrence offsets; lines in dict insertion order."""
    ctx = _lib.context(counts_row.device.index)
    L = _lib.load()
    stream = ctypes.c_void_p(torch.cuda.current_stream(counts_row.device).cuda_stream)
    max_lines = int(torch.count_nonzero(counts_row).item())
    text = torch.empty(max(max_lines * (k + 4), 16), dtype=torch.uint8, device=counts_row.device)
    while True:
        nlen, nlines = ctypes.c_uint64(0), ctypes.c_uint64(0)
        _lib.check(L.kmerml_format_kmer_file(ctx.handle, int(k), counts_row.data_ptr(), first.data_ptr(),
                                             _lib.FLAG_CANONICAL if canonical else 0, max(max_lines, 1), text.data_ptr(),
                                             text.numel(), ctypes.byref(nlen), ctypes.byref(nlines), stream))
        if nlines.value > max_lines:
            max_lines = int(nlines.value)
            continue
        if nlen.value > text.numel():                    # counts with many digits: exact size is known now
            text = torch.empty(int(nlen.value), dtype=torch.uint8, device=counts_row.device)
            continue
        return text[:int(nlen.value)]


def format_kmer_lines_device(codes, counts, k):
    """uint8 tensor: the same text from k-mers already in line order (int64 storage of uint64 codes, int32 counts)."""
    ctx = _lib.context(codes.device.index)
    L = _lib.load()
    stream = ctypes.c_void_p(torch.cuda.current_stream(codes.device).cuda_stream)
    n = int(codes.numel())
    text = torch.empty(max(n * (k + 4), 16), dtype=torch.uint8, device=codes.device)
    while True:
        nlen = ctypes.c_uint64(0)
        _lib.check(L.kmerml_format_kmer_lines(ctx.handle, int(k), codes.data_ptr() if n else None,
                                              counts.data_ptr() if n else None, n, text.data_ptr(), text.numel(),
                                              ctypes.byref(nlen), stream))
        if nlen.value > text.numel():
            text = torch.empty(int(nlen.value), dtype=torch.uint8, device=codes.device)
            continue
        return text[:int(nlen.value)]


@dataclass
class Sketches:
    """Bottom-s MinHash sketches of a batch of genomes (kmerml_sketch_batch): row g of `hashes` holds the filled[g]
    smallest distinct hashes of genome g's k-mers, ascending, then UINT64_MAX."""
    hashes: torch.Tensor      # [n, s] int64 storage of uint64
    filled: torch.Tensor      # [n] int32
    k: int
    s: int
    seed: int
    canonical: bool

    def __len__(self):
        return self.hashes.shape[0]

    def params(self):
        return (self.k, self.s, self.seed, self.canonical)


_SKETCH_METRIC = {"mash": _lib.SKETCH_METRIC_MASH, "jaccard": _lib.SKETCH_METRIC_JACCARD}


def sketch_batch_device(fasta, offsets, k, *, sketch_size=1000, seed=42, canonical=True, min_record_len=None):
    """MinHash sketches of genomes already resident in HBM (laid out as for count_dense_device), any k <= 32."""
    if not (fasta.is_cuda and fasta.dtype == torch.uint8 and fasta.is_contiguous()):
        raise ValueError("fasta must be a contiguous uint8 CUDA tensor")
    ctx = _lib.context(fasta.device.index)
    n = len(offsets) - 1
    s = int(sketch_size)
    hashes = torch.empty((n, max(s, 1)), dtype=torch.int64, device=fasta.device)
    filled = torch.zeros(n, dtype=torch.int32, device=fasta.device)
    offs = np.asarray(offsets, dtype=np.uint64)
    stream = torch.cuda.current_stream(fasta.device).cuda_stream
    _retry_after_cache_release(lambda: _lib.check(_lib.load().kmerml_sketch_batch(
        ctx.handle, fasta.data_ptr() if fasta.numel() else None, offs.ctypes.data, n, int(k), int(min_record_len or 0),
        _lib.FLAG_CANONICAL if canonical else 0, s, int(seed) & 0xFFFFFFFFFFFFFFFF, hashes.data_ptr(), hashes.stride(0),
        filled.data_ptr(), ctypes.c_void_p(stream))))
    return Sketches(hashes, filled, int(k), s, int(seed), bool(canonical))


def _check_sketches(*sketches):
    for sk in sketches[1:]:
        if sk.params() != sketches[0].params():
            raise ValueError("sketches differ in k, sketch size or scale, seed or canonical flag: "
                             f"{sketches[0].params()} vs {sk.params()}")


def sketch_distance_rows_device(sk, row_begin, row_end, metric="mash", *, out_dtype=torch.float32):
    """Rows [row_begin, row_end) of the Mash or Jaccard distance matrix of the sketches; bit-identical to the same
    rows of sketch_distance_device."""
    if metric not in _SKETCH_METRIC:
        raise ValueError(f"metric must be one of {sorted(_SKETCH_METRIC)}")
    if out_dtype not in (torch.float32, torch.float64):
        raise ValueError("out_dtype must be torch.float32 or torch.float64")
    h = sk.hashes
    n = h.shape[0]
    out = torch.empty((max(int(row_end) - int(row_begin), 0), n), dtype=out_dtype, device=h.device)
    if out.numel() == 0:
        return out
    ctx = _lib.context(h.device.index)
    stream = torch.cuda.current_stream(h.device).cuda_stream
    o32 = out.data_ptr() if out_dtype == torch.float32 else None
    o64 = out.data_ptr() if out_dtype == torch.float64 else None
    _lib.check(_lib.load().kmerml_sketch_distance_rows(
        ctx.handle, h.data_ptr(), h.stride(0), sk.filled.data_ptr(), n, sk.s, sk.k, int(row_begin), int(row_end),
        _SKETCH_METRIC[metric], o32, o64, ctypes.c_void_p(stream)))
    return out


def sketch_distance_device(sk, metric="mash", *, out_dtype=torch.float32):
    """n x n Mash (default) or Jaccard distance matrix of the sketches (kmerml_sketch_distance_rows)."""
    return sketch_distance_rows_device(sk, 0, len(sk), metric, out_dtype=out_dtype)


def concat_sketches(*sketches):
    """One Sketches of several batches (same k, s, seed and canonical flag), rows in argument order."""
    _check_sketches(*sketches)
    first = sketches[0]
    return Sketches(torch.cat([sk.hashes for sk in sketches]), torch.cat([sk.filled for sk in sketches]),
                    first.k, first.s, first.seed, first.canonical)


@dataclass
class ScaledSketches:
    """Scaled (FracMinHash) sketches of a batch of genomes (kmerml_fmh_batch): genome g's sketch is
    hashes[offsets[g]:offsets[g + 1]], every distinct hash <= (2^64 - 1) // scale of its k-mers, ascending.  With
    abundance tracking, abundances[i] is the number of windows of that genome whose k-mer hashes to hashes[i]."""
    hashes: torch.Tensor      # [total] int64 storage of uint64
    offsets: torch.Tensor     # [n + 1] int64
    k: int
    scale: int
    seed: int
    canonical: bool
    abundances: Optional[torch.Tensor] = None     # [total] int32, or None

    def __len__(self):
        return self.offsets.shape[0] - 1

    def sizes(self):
        """[n] int64: the number of hashes of each sketch."""
        return self.offsets[1:] - self.offsets[:-1]

    def params(self):
        return (self.k, self.scale, self.seed, self.canonical)


_FMH_METRIC = {"containment": _lib.FMH_CONTAINMENT, "max_containment": _lib.FMH_MAX_CONTAINMENT,
               "jaccard": _lib.FMH_JACCARD, "containment_ani": _lib.FMH_CONTAINMENT_ANI,
               "max_containment_ani": _lib.FMH_MAX_CONTAINMENT_ANI}
_FMH_WEIGHTED_METRIC = {"weighted_containment": _lib.FMH_WEIGHTED_CONTAINMENT,
                        "angular_similarity": _lib.FMH_ANGULAR_SIMILARITY}


def fmh_batch_device(fasta, offsets, k, *, scale=1000, seed=42, canonical=True, min_record_len=None,
                     track_abundance=False):
    """Scaled sketches of genomes already resident in HBM (laid out as for count_dense_device), any k <= 32.  The
    output is sized from a guess (1.25 hashes per `scale` bytes, + 256 per genome); a batch with more hashes than that
    is copied out of the library's workspace once its size is known (kmerml_fmh_fetch), never sketched twice.  With
    track_abundance, also the abundance of every hash (kmerml_fmh_fetch_abundances)."""
    if not (fasta.is_cuda and fasta.dtype == torch.uint8 and fasta.is_contiguous()):
        raise ValueError("fasta must be a contiguous uint8 CUDA tensor")
    ctx = _lib.context(fasta.device.index)
    L = _lib.load()
    n = len(offsets) - 1
    offs = np.asarray(offsets, dtype=np.uint64)
    scale = int(scale)
    guess = int(sum(int(offs[g + 1] - offs[g]) / max(scale, 1) * 1.25 + 256 for g in range(n)))
    hashes = torch.empty(max(guess, 1), dtype=torch.int64, device=fasta.device)
    sk_offsets = torch.empty(n + 1, dtype=torch.int64, device=fasta.device)
    total = ctypes.c_uint64(0)
    stream = ctypes.c_void_p(torch.cuda.current_stream(fasta.device).cuda_stream)
    _retry_after_cache_release(lambda: _lib.check(L.kmerml_fmh_batch(
        ctx.handle, fasta.data_ptr() if fasta.numel() else None, offs.ctypes.data, n, int(k), int(min_record_len or 0),
        (_lib.FLAG_CANONICAL if canonical else 0) | (_lib.FLAG_FMH_ABUNDANCE if track_abundance else 0), scale,
        int(seed) & 0xFFFFFFFFFFFFFFFF, hashes.data_ptr(), guess, sk_offsets.data_ptr(), ctypes.byref(total), stream)))
    if total.value > guess:
        hashes = torch.empty(int(total.value), dtype=torch.int64, device=fasta.device)
        _lib.check(L.kmerml_fmh_fetch(ctx.handle, hashes.data_ptr(), total.value, sk_offsets.data_ptr(), stream))
    abundances = None
    if track_abundance:
        abundances = torch.empty(max(int(total.value), 1), dtype=torch.int32, device=fasta.device)
        _lib.check(L.kmerml_fmh_fetch_abundances(ctx.handle, abundances.data_ptr(), total.value, stream))
        abundances = abundances[:int(total.value)]
    return ScaledSketches(hashes[:int(total.value)], sk_offsets, int(k), scale, int(seed), bool(canonical), abundances)


def fmh_compare_device(queries, references=None, metric="containment", *, out_dtype=torch.float32,
                       want_intersections=False):
    """[n_q, n_r] similarity of every query sketch to every reference sketch (the queries themselves when
    `references` is None): "containment" |Q n R| / |Q|, "max_containment" |Q n R| / min(|Q|, |R|), "jaccard",
    "containment_ani" and "max_containment_ani" (the containment to the power 1/k); 0 when |Q n R| = 0.
    With want_intersections, also the exact [n_q, n_r] int64 |Q n R|.
    Sketches with abundances (track_abundance) also give "weighted_containment", sum_{Q n R} a_Q / sum_Q a_Q (the
    share of the query's k-mer mass that R explains; needs the query abundances), and "angular_similarity",
    1 - 2 acos(cos) / pi of the abundance vectors (needs both); want_intersections then returns the exact integer
    numerators sum_{Q n R} a_Q and sum_{Q n R} a_Q a_R instead of |Q n R|."""
    if metric not in _FMH_METRIC and metric not in _FMH_WEIGHTED_METRIC:
        raise ValueError(f"metric must be one of {sorted(_FMH_METRIC) + sorted(_FMH_WEIGHTED_METRIC)}")
    if out_dtype not in (torch.float32, torch.float64):
        raise ValueError("out_dtype must be torch.float32 or torch.float64")
    refs = queries if references is None else references
    if not (isinstance(queries, ScaledSketches) and isinstance(refs, ScaledSketches)):
        raise ValueError("queries and references must be ScaledSketches")
    _check_sketches(queries, refs)
    if metric in _FMH_WEIGHTED_METRIC:
        return _fmh_compare_weighted(queries, refs, metric, out_dtype, want_intersections)
    dev = queries.hashes.device
    n_q, n_r = len(queries), len(refs)
    out = torch.empty((n_q, n_r), dtype=out_dtype, device=dev)
    inter = torch.empty((n_q, n_r), dtype=torch.int32, device=dev) if want_intersections else None
    if out.numel():
        ctx = _lib.context(dev.index)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(_lib.load().kmerml_fmh_compare(
            ctx.handle, queries.hashes.data_ptr(), queries.offsets.data_ptr(), n_q, refs.hashes.data_ptr(),
            refs.offsets.data_ptr(), n_r, queries.k, _FMH_METRIC[metric],
            inter.data_ptr() if inter is not None else None, out.data_ptr() if out_dtype == torch.float32 else None,
            out.data_ptr() if out_dtype == torch.float64 else None, ctypes.c_void_p(stream)))
    if want_intersections:
        return out, inter.to(torch.int64)
    return out


def _fmh_compare_weighted(queries, refs, metric, out_dtype, want_numerators):
    if queries.abundances is None or (metric == "angular_similarity" and refs.abundances is None):
        raise ValueError(f"{metric} needs sketches made with track_abundance=True "
                         f"({'queries' if metric == 'weighted_containment' else 'queries and references'})")
    dev = queries.hashes.device
    n_q, n_r = len(queries), len(refs)
    out = torch.empty((n_q, n_r), dtype=out_dtype, device=dev)
    num = torch.empty((n_q, n_r), dtype=torch.int64, device=dev) if want_numerators else None
    if out.numel():
        ctx = _lib.context(dev.index)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(_lib.load().kmerml_fmh_compare_weighted(
            ctx.handle, queries.hashes.data_ptr(), queries.offsets.data_ptr(), queries.abundances.data_ptr(), n_q,
            refs.hashes.data_ptr(), refs.offsets.data_ptr(),
            refs.abundances.data_ptr() if refs.abundances is not None else None, n_r, _FMH_WEIGHTED_METRIC[metric],
            num.data_ptr() if num is not None else None, out.data_ptr() if out_dtype == torch.float32 else None,
            out.data_ptr() if out_dtype == torch.float64 else None, ctypes.c_void_p(stream)))
    if want_numerators:
        return out, num
    return out


@dataclass
class GatherResult:
    """Gather of each query sketch into the reference sketches that cover it (kmerml_fmh_gather): row q lists its
    matches in pick order, n_matches[q] of them; the columns past that hold -1 (reference) and 0 (counts)."""
    n_matches: torch.Tensor   # [n_q] int32
    reference: torch.Tensor   # [n_q, m] int32: reference index of each match
    unique: torch.Tensor      # [n_q, m] int64: query hashes first assigned to that reference
    intersect: torch.Tensor   # [n_q, m] int64: |Q n R| of the whole query
    remaining: torch.Tensor   # [n_q, m] int64: query hashes still unassigned after the match
    # queries with abundances only (else None): over the hashes the match takes,
    unique_weighted: Optional[torch.Tensor] = None    # [n_q, m] int64: the sum of their query abundances
    unique_sumsq: Optional[torch.Tensor] = None       # [n_q, m] int64: the sum of their squares
    median_abund: Optional[torch.Tensor] = None       # [n_q, m] float64: their median


def fmh_gather_device(queries, references, *, threshold=1, max_matches=None):
    """Greedy, exact gather of every query into the references: repeatedly pick the reference that shares the most
    still-unassigned query hashes (ties: the smallest reference index) while that number is >= `threshold`, and
    assign those hashes to it.  The default `max_matches`, min(n_r, max_q |Q| // threshold), never truncates.  When
    the queries carry abundances, the picks are the same and each match also gets the sum, sum of squares and median
    of the query abundances of the hashes it takes (kmerml_fmh_gather_abundance)."""
    if not (isinstance(queries, ScaledSketches) and isinstance(references, ScaledSketches)):
        raise ValueError("queries and references must be ScaledSketches")
    _check_sketches(queries, references)
    threshold = int(threshold)
    if threshold < 1:
        raise ValueError("threshold must be >= 1")
    dev = queries.hashes.device
    n_q, n_r = len(queries), len(references)
    if max_matches is None:
        largest = int(queries.sizes().max()) if n_q else 0
        max_matches = min(n_r, largest // threshold)
    max_matches = int(max_matches)
    if max_matches < 0:
        raise ValueError("max_matches must be >= 0")
    n_matches = torch.zeros(n_q, dtype=torch.int32, device=dev)
    m = max(max_matches, 1)
    ref = torch.full((n_q, m), -1, dtype=torch.int32, device=dev)
    counts = torch.zeros((3, n_q, m), dtype=torch.int32, device=dev)       # uint32 unique | intersect | remaining
    weighted = queries.abundances is not None
    if weighted:
        sums = torch.zeros((2, n_q, m), dtype=torch.int64, device=dev)     # uint64 (< 2^63) unique_weighted | sumsq
        median = torch.zeros((n_q, m), dtype=torch.float64, device=dev)
    if n_q and max_matches:
        ctx = _lib.context(dev.index)
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        args = (ctx.handle, queries.hashes.data_ptr(), queries.offsets.data_ptr(), n_q, references.hashes.data_ptr(),
                references.offsets.data_ptr(), n_r, threshold, m, n_matches.data_ptr(), ref.data_ptr(),
                counts[0].data_ptr(), counts[1].data_ptr(), counts[2].data_ptr())
        if weighted:
            _retry_after_cache_release(lambda: _lib.check(_lib.load().kmerml_fmh_gather_abundance(
                *args, queries.abundances.data_ptr(), sums[0].data_ptr(), sums[1].data_ptr(), median.data_ptr(),
                stream)))
        else:
            _retry_after_cache_release(lambda: _lib.check(_lib.load().kmerml_fmh_gather(*args, stream)))
    wide = (counts[:, :, :max_matches].to(torch.int64) & 0xFFFFFFFF)
    res = GatherResult(n_matches, ref[:, :max_matches], wide[0], wide[1], wide[2])
    if weighted:
        res.unique_weighted, res.unique_sumsq = sums[0, :, :max_matches], sums[1, :, :max_matches]
        res.median_abund = median[:, :max_matches]
    return res


def concat_scaled_sketches(*sketches):
    """One ScaledSketches of several batches (same k, scale, seed and canonical flag), genomes in argument order.
    Abundances are kept when every batch has them; a mix of batches with and without them raises ValueError."""
    _check_sketches(*sketches)
    has = [sk.abundances is not None for sk in sketches]
    if any(has) and not all(has):
        raise ValueError("some sketches carry abundances and some do not")
    first = sketches[0]
    offs, base = [first.offsets[:1]], 0
    for sk in sketches:
        offs.append(sk.offsets[1:] + base)
        base += int(sk.offsets[-1])
    abundances = torch.cat([sk.abundances for sk in sketches]) if all(has) else None
    return ScaledSketches(torch.cat([sk.hashes for sk in sketches]), torch.cat(offs), first.k, first.scale, first.seed,
                          first.canonical, abundances)
