"""The dense path at k = 13 and 14 -- the largest rows it accepts (KMERML_MAX_DENSE_K) -- against exact references.

At these k every stage takes a route of its own: global-atomic counting one genome at a time, a cascade of up to 13
levels, the canonical fold and the first-occurrence select / sort / format over 4^14 bins, nibble levels on the host
wire, and Gram grids of tens of thousands of K splits.  A 4^14 uint64 dense reference is 2 GiB, so the references here
are built from the sparse C oracle (exact, any k): the GPU rows are compared in sparse form on the device, and the
references themselves are pinned to the dense oracle at k <= 8 by the CPU tests at the top of this file.

Memory: a k = 14 row is 1 GiB of uint32.  Every GPU test frees its tensors and the library's workspaces when it ends
(fixture `cuda`), and no test holds more than one 4^14 host array at a time."""
import contextlib
import functools
import gc
import io
import random

import numpy as np
import pytest

import oracle
from helpers import fuzz_fasta

FREQ_RTOL = 1e-6
GRAM_RTOL = 1e-13


# ---------------------------------------------------------------- references built from the sparse oracle
def sparse_ref(data, k, min_len=None):
    """(codes uint64 ascending, counts int64) of the k-mers the reference observes (oracle.count_sparse, sorted)."""
    codes, counts = oracle.count_sparse(data, k, min_len)
    order = np.argsort(codes, kind="stable")
    return codes[order], counts[order].astype(np.int64)


def revcomp_np(codes, k):
    codes = np.asarray(codes, np.uint64)
    rc = np.zeros_like(codes)
    t = codes.copy()
    for _ in range(k):
        rc = (rc << np.uint64(2)) | (np.uint64(3) - (t & np.uint64(3)))
        t >>= np.uint64(2)
    return rc


def canonical_ref(ref, k):
    """Canonical counts in sparse form: the counts of x and rc(x) summed on min(x, rc(x))."""
    codes, counts = ref
    key = np.minimum(codes, revcomp_np(codes, k))
    uniq, inv = np.unique(key, return_inverse=True)
    out = np.zeros(uniq.size, np.int64)
    np.add.at(out, inv, counts)
    return uniq, out


def freq_ref(ref):
    """float64 frequencies count / windows of the observed k-mers."""
    counts = ref[1].astype(np.float64)
    return counts / counts.sum() if counts.size else counts


def gram_ref(refs):
    """Exact n x n Gram matrix (int64) of count rows given in sparse form; a list of refs per row sums its levels
    (a concatenated row [k1, k2] has disjoint bins per level)."""
    rows = [r if isinstance(r, list) else [r] for r in refs]
    n = len(rows)
    g = np.zeros((n, n), np.int64)
    for i in range(n):
        for j in range(i, n):
            s = 0
            for (ci, ni), (cj, nj) in zip(rows[i], rows[j]):
                _, ia, ib = np.intersect1d(ci, cj, assume_unique=True, return_indices=True)
                s += int(np.dot(ni[ia], nj[ib]))
            g[i, j] = g[j, i] = s
    return g


def distance_ref(g, metric):
    """float64 cosine / Euclidean distances from an exact Gram matrix (the formulas of the distance kernels)."""
    g = g.astype(np.float64)
    d = np.diag(g)
    with np.errstate(divide="ignore", invalid="ignore"):
        if metric == "cosine":
            den = np.sqrt(d)[:, None] * np.sqrt(d)[None, :]
            out = np.where(den > 0, 1.0 - g / den, np.nan)
        else:
            d2 = d[:, None] + d[None, :] - 2.0 * g
            out = np.where(d2 > 0, np.sqrt(np.maximum(d2, 0)), 0.0)
    np.fill_diagonal(out, 0.0)
    return out


def stats_ref(values):
    """kmer_metadata.py:59-78 over the observed counts (values > 0), in exact integer arithmetic."""
    v = np.sort(np.asarray(values, np.uint64)[np.asarray(values, np.uint64) > 0])
    n = int(v.size)
    if n == 0:
        return None
    total = int(v.sum(dtype=np.uint64))
    lo, hi = int(v[(n - 1) // 2]), int(v[n // 2])
    return {"total_kmers": total, "unique_kmers": n, "max_count": int(v[-1]), "min_count": int(v[0]),
            "mean_count": total / n, "median_count": (float(lo) + float(hi)) / 2.0}


# ---------------------------------------------------------------- inputs
def _seq(rng, n):
    return np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].tobytes()


def _wrap(seq, width):
    return b"\n".join(seq[i:i + width] for i in range(0, len(seq), width))


@functools.lru_cache(maxsize=1)
def genomes():
    """Genomes whose k = 13 and 14 rows reach the edges of the dense path."""
    from kmerml_b200 import synth
    rng = np.random.default_rng(1314)
    # 4.2 Mbp wrapped at 60 bases (many slices), records of exactly 14, 13, 12 and 1 bases, N runs, soft-masked
    # lower case
    w = synth.fasta_bytes([2_400_000, 14, 13, 12, 1_100_001, 1, 700_000], seed=13, width=60).copy()
    for _ in range(40):
        i = int(rng.integers(100, w.size - 5000))
        seg = w[i:i + int(rng.integers(1, 3000))]
        seg[seg != 10] = ord("N")
    body = w >= 65
    body[:w.tolist().index(10)] = False                                       # keep the first header
    low = body & (w <= 90) & (rng.random(w.size) < 0.3)
    w[low] += 32
    wrapped = w.tobytes()
    # one unwrapped 1.5 Mbp chromosome with CRLF line ends, records of 1..20 bases, and runs of 1..20 bases between
    # N: run ends at every level of the cascade
    parts = [b">chr1 one line\r\n", _seq(rng, 1_500_000), b"\r\n"]
    for n in range(1, 21):
        parts += [f">s{n} short\r\n".encode(), _seq(rng, n), b"\r\n"]
    parts += [b">runs\r\n", b"N".join(_seq(rng, int(n)) for n in rng.integers(1, 21, 3000)), b"\r\n"]
    crlf = b"".join(parts)
    # A^13 C A^13 G repeated: the 13-mer of A counted 70 000 times (three byte planes) while no 14-mer reaches 65 536
    # (35 000: two planes); a homopolymer, a tandem array, then ordinary sequence
    poly = (b">poly\n" + _wrap((b"A" * 13 + b"C" + b"A" * 13 + b"G") * 35_000, 60) + b"\n>homo\n" + b"A" * 5000 +
            b"\n>tandem\n" + b"ACGTTGCAAT" * 3000 + b"\n>rand\n" + _wrap(_seq(rng, 200_000), 60) + b"\n")
    # a random 40 kb unit repeated 20 times: ~40 000 bins of k = 14 at 19..20, more than the 32 768 exceptions a
    # nibble level of the host wire holds
    over = b">sat\n" + _seq(rng, 40_000) * 20 + b"\n"
    # the same repeat, shorter (the 13-mer of A 40 000 times): a Gram entry with poly that needs poly's third plane
    poly2 = b">poly2\n" + _wrap((b"A" * 13 + b"G" + b"A" * 13 + b"T") * 20_000, 70) + b"\n>r\n" + _seq(rng, 50_000) + b"\n"
    return {"wrapped": wrapped, "crlf": crlf, "poly": poly, "poly2": poly2, "over": over, "empty": b"", "header": b">e\n"}


@functools.lru_cache(maxsize=None)
def ref_of(name, k, min_len):
    return sparse_ref(genomes()[name], k, min_len)


# ---------------------------------------------------------------- CPU: the references against the dense oracle
def test_sparse_reference_matches_dense_oracle():
    rng = random.Random(1314)
    datas = [fuzz_fasta(rng, max_len=3000) for _ in range(25)] + [b"", b">e\n", genomes()["poly"][:20_000]]
    for d in datas:
        for k in (1, 2, 5, 7, 8):
            for ml in (None, k + 3):
                dense = oracle.count_dense(d, k, ml)
                codes, counts = sparse_ref(d, k, ml)
                nz = np.nonzero(dense)[0]
                assert np.array_equal(codes, nz.astype(np.uint64)), (d[:40], k)
                assert np.array_equal(counts, dense[nz].astype(np.int64))
                assert int(np.count_nonzero(dense)) == codes.size
                assert np.allclose(freq_ref((codes, counts)), oracle.frequencies(dense)[nz], rtol=1e-15, atol=0)


def test_canonical_reference_matches_dense_oracle():
    rng = random.Random(7)
    for d in [fuzz_fasta(rng, max_len=3000) for _ in range(15)] + [genomes()["poly"][:30_000]]:
        for k in (1, 2, 3, 6, 7, 8):
            canon = oracle.canonical_from_forward(oracle.count_dense(d, k), k)
            codes, counts = canonical_ref(sparse_ref(d, k), k)
            nz = np.nonzero(canon)[0]
            assert np.array_equal(codes, nz.astype(np.uint64)), (d[:40], k)
            assert np.array_equal(counts, canon[nz].astype(np.int64))
            assert np.array_equal(revcomp_np(codes, k), [oracle.revcomp_code(int(c), k) for c in codes])


def test_gram_and_distance_reference_match_dense_oracle():
    rng = random.Random(11)
    datas = [fuzz_fasta(rng, max_len=4000) for _ in range(6)] + [b">e\n", genomes()["poly"][:30_000]]
    for ks in ([6], [8], [6, 3]):
        dense = np.stack([np.concatenate([oracle.count_dense(d, k, max(ks)) for k in ks]) for d in datas]).astype(np.int64)
        g = gram_ref([[sparse_ref(d, k, max(ks)) for k in ks] for d in datas])
        assert np.array_equal(g, dense @ dense.T), ks
        for metric in ("cosine", "euclidean"):
            want = oracle.pairwise_distance(dense, metric)
            got = distance_ref(g, metric)
            assert np.allclose(got, want, rtol=1e-12, atol=1e-12, equal_nan=True), (ks, metric)
            assert np.array_equal(np.isnan(got), np.isnan(want))


def test_stats_reference_matches_file_stats():
    rng = random.Random(3)
    for d in [fuzz_fasta(rng, max_len=3000) for _ in range(10)] + [genomes()["poly"][:30_000]]:
        for k in (2, 5, 8):
            text = oracle.kmer_file_text(d, k, 8)
            if not text:
                assert stats_ref(sparse_ref(d, k, 8)[1]) is None
                continue
            want = oracle.kmer_file_stats(text, k)
            got = stats_ref(sparse_ref(d, k, 8)[1])
            assert {key: want[key] for key in got} == got, (d[:40], k)


def test_inputs_reach_the_edges():
    """What the GPU tests rely on the inputs to contain, checked on the references."""
    g = genomes()
    poly13, poly14 = ref_of("poly", 13, 13), ref_of("poly", 14, 14)
    assert poly13[1].max() >= 65536 and 256 <= poly14[1].max() < 65536        # three planes at 13, two at 14
    assert gram_ref([poly13, ref_of("poly2", 13, 13)])[0, 1] >= 65536 * 40_000      # the third plane meets poly2
    over14 = ref_of("over", 14, 14)
    assert int((over14[1] >= 15).sum()) > 32768 and len(g["over"]) <= 5 * 4 ** 13      # nibbles that overflow
    assert all(len(g[n]) <= 5 * 4 ** 13 for n in g)                          # every genome's 13 / 14 levels as nibbles
    assert len(g["wrapped"]) > 4_000_000
    assert b"\r\n" in g["crlf"] and max(len(line) for line in g["crlf"].split(b"\r\n")) >= 1_500_000
    w = g["wrapped"]
    assert any(97 <= c <= 122 for c in w[100:10_000]) and w.count(b"N") > 10_000
    # synthetic count rows for the median: the middle values fall in each of the three radix passes
    for values, shift in SELECT_CASES:
        s = stats_ref(values)
        if s is not None and shift is not None:
            v = np.sort(np.asarray(values, np.uint64)[np.asarray(values, np.uint64) > 0])
            mid = int(v[(v.size - 1) // 2])
            assert mid >> shift and not mid >> (shift + (11 if shift else 10)), (values[:4], shift)


# values of synthetic count rows for kmerml_count_stats, and the radix pass (bit shift of its digit) whose digit is the
# highest non-zero one of the lower median (None: no observed bin or not applicable)
_R = np.random.default_rng(21)
SELECT_CASES = [
    ([1023, 1024, 1025, 1536, 2047], 10),                                     # around 2^10, odd
    ([1023, 1024, 1025, 3000], 10),                                           # even: the middles straddle 2^10
    ([2 ** 21 - 1, 2 ** 21, 2 ** 21 + 1, 2 ** 21 + 7, 5], 21),
    ([2 ** 21 - 1] * 3 + [2 ** 21] * 3, 10),                                  # ties across the pass-1 digit boundary
    ([0xFFFFFFFF, 0xFFFFFFFE, 0x80000000, 0xFFFFFFFF, 1, 0x7FFFFFFF], 21),
    ([0xFFFFFFFF] * 4, 21),                                                   # all equal, the largest count
    ([777] * 9, 0),                                                           # all equal, one digit
    ([2 ** 21 + 5], 21),                                                      # one observed bin
    ([3, 2 ** 11 - 1, 2 ** 11, 2 ** 22 - 1, 2 ** 22, 2 ** 32 - 1, 2 ** 10], 10),
    (list(_R.integers(1, 2 ** 32, 10_001)), 21),                              # random 32-bit counts, odd
    (list(_R.integers(2 ** 10, 2 ** 21, 4_000)), 10),                         # random, even, pass 2
    (list(_R.integers(1, 2 ** 10, 3_001)), 0),
    ([], None),                                                               # nothing observed
]


# ---------------------------------------------------------------- GPU
def release():
    """Free what dropped tensors left in torch's cache and the library's workspaces (they grow to the largest call
    and persist in the cached context): a k = 14 row is 1 GiB, and cached blocks of one case's sizes do not fit the
    next case's."""
    import torch
    from kmerml_b200 import _lib
    gc.collect()
    torch.cuda.synchronize()
    while _lib._contexts:
        _lib._contexts.popitem()[1].close()
    torch.cuda.empty_cache()


@pytest.fixture
def cuda():
    import torch
    yield torch
    release()


def to_device(torch, datas):
    from kmerml_b200 import synth
    arrs = [np.frombuffer(d, np.uint8) if len(d) else np.zeros(0, np.uint8) for d in datas]
    buf, offs = synth.pack(arrs)
    return torch.from_numpy(np.concatenate([buf, np.zeros(64, np.uint8)])).cuda(), offs


def observed(row):
    """(bins uint64 ascending, counts int64) of the non-zero entries of a uint32 count row (int32 storage), found
    on the device: only the observed bins come to the host."""
    import torch
    nz = torch.nonzero(row).flatten()
    return nz.cpu().numpy().astype(np.uint64), (row[nz].to(torch.int64) & 0xFFFFFFFF).cpu().numpy()


def assert_row(row, ref, what):
    import torch
    bins, counts = observed(row)
    assert int(torch.count_nonzero(row)) == ref[0].size, what
    assert np.array_equal(bins, ref[0]), (what, np.setxor1d(bins, ref[0])[:5])
    assert np.array_equal(counts, ref[1]), (what, np.nonzero(counts != ref[1])[0][:5])


def check_batch(torch, names, ks, min_record_len=None, canonical=False):
    from kmerml_b200 import engine
    datas = [genomes()[n] for n in names]
    dev, offs = to_device(torch, datas)
    res = engine.count_dense_device(dev, offs, ks, min_record_len=min_record_len, canonical=canonical)
    torch.cuda.synchronize()
    ml = min_record_len or max(ks)
    totals = res.totals.cpu().numpy()
    for g, name in enumerate(names):
        for ki, k in enumerate(ks):
            ref = ref_of(name, k, ml)
            if canonical:
                ref = canonical_ref(ref, k)
            what = (name, k, ks, min_record_len, canonical)
            assert_row(res.counts_of(g, k), ref, what)
            assert int(totals[g, ki]) == int(ref[1].sum()), what
            f = res.freq_of(g, k)
            nz = torch.from_numpy(ref[0].astype(np.int64)).cuda()
            got = f[nz].double().cpu().numpy()
            want = freq_ref(ref)
            assert np.all(np.abs(got - want) <= FREQ_RTOL * want), what
            assert int(torch.count_nonzero(f)) == ref[0].size, what
    del res, dev, f, nz
    release()


@pytest.mark.gpu
def test_batch_counts_k13_k14(cuda):
    """count_dense_device: k = 14 and 13 alone and together, levels cascaded down from them (12, 9, 3 from 14; 1 from
    13 and from 14 -- 13 levels, three cascade launches), a record filter above max(k), and canonical rows."""
    for names in (["wrapped", "empty", "poly"], ["crlf", "header", "poly"]):
        for ks in ([14], [13], [14, 13], [14, 12, 9, 3], [13, 1], [14, 1]):
            check_batch(cuda, names, ks)
        check_batch(cuda, names, [14, 13], min_record_len=20)
        check_batch(cuda, names, [14, 13, 7], canonical=True)


@pytest.mark.gpu
def test_host_call_modes_k13_k14(cuda, monkeypatch):
    """count_dense_host: narrow wire (default), uint32 wire, compact result, bytes instead of nibbles -- all equal to the
    device-resident rows; the 13 / 14 levels crossed as nibbles, and the genome with more than 32 768 bins at 15 or
    above comes back through the wide fallback / is reported by the compact call."""
    torch = cuda
    from kmerml_b200 import engine
    monkeypatch.setenv("KMERML_HOST_SLOTS", "2")              # read when the context is made: slots are reused
    release()
    names = ["wrapped", "over", "header", "poly"]
    ks = [14, 13, 5]
    datas = [genomes()[n] for n in names]
    dev, offs = to_device(torch, datas)
    dres = engine.count_dense_device(dev, offs, ks, want_freq=False)
    del dev
    for g, name in enumerate(names):
        for k in ks:
            assert_row(dres.counts_of(g, k), ref_of(name, k, 14), (name, k))

    def same_rows(counts_host, totals, what):
        for g in range(len(names)):
            assert torch.equal(counts_host[g].cuda(), dres.counts[g]), (what, names[g])
        assert torch.equal(totals, dres.totals.cpu()), what

    for what, kw in (("narrow", {}), ("wide_d2h", {"wide_d2h": True}), ("bytes", {"nibbles": False})):
        h = engine.count_dense_host(datas, ks, want_freq=False, **kw)
        same_rows(h.counts, h.totals, what)
        del h
    karr = np.asarray(ks, np.int32)
    for nibbles in (True, False):
        comp = engine.count_dense_host(datas, ks, want_freq=False, compact=True, nibbles=nibbles)
        head = comp.rows[:, :8].contiguous()
        assert all(bytes(head[g, :4].tolist()) == b"KMW2" for g in range(len(names)))
        mask = head.view(torch.int32)[:, 1].tolist()                 # bit i: level k_list[i] went as nibbles
        if nibbles:
            assert all(m & 3 == 3 and not m & 4 for m in mask), mask     # k = 14 and 13 as nibbles, k = 5 as uint32
        else:
            assert not any(mask), mask
        over = [g for g in range(len(names))
                if engine._lib.load().kmerml_compact_row_overflowed(karr.ctypes.data, len(ks), comp.rows[g].data_ptr())]
        assert over == ([1] if nibbles else []), over                # bins >= 255 stay few: bytes do not overflow
        assert sorted(comp._wide) == over
        for g in range(len(names)):
            for k in ks:
                got = torch.from_numpy(comp.counts_numpy(g, k).view(np.int32)).cuda()
                assert torch.equal(got, dres.counts_of(g, k)), (nibbles, names[g], k)
        assert torch.equal(comp.totals, dres.totals.cpu())
        del comp


@pytest.mark.gpu
def test_byte_ranges_k13_k14(cuda):
    """count_dense_range_device over dist.chunk_ranges for 2, 3 and 7 ranks sums to the whole-genome row."""
    torch = cuda
    from kmerml_b200 import dist as kdist
    from kmerml_b200 import engine
    for name in ("crlf", "wrapped"):
        data = genomes()[name]
        dev = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).cuda()
        for ks in ([14, 13, 5], [13]):
            whole = engine.count_dense_device(dev, [0, len(data)], ks, want_freq=False)
            for k in ks:
                assert_row(whole.counts_of(0, k), ref_of(name, k, max(ks)), (name, k, ks))
            want = whole.counts[0].to(torch.int64) & 0xFFFFFFFF
            for world in (2, 3, 7):
                acc = torch.zeros_like(want)
                tot = torch.zeros_like(whole.totals[0])
                for b, e in kdist.chunk_ranges(len(data), world):
                    c, t = engine.count_dense_range_device(dev, b, e, ks)
                    acc += c.to(torch.int64) & 0xFFFFFFFF
                    tot += t
                    del c
                assert torch.equal(acc, want), (name, ks, world)
                assert torch.equal(tot, whole.totals[0]), (name, ks, world)
                del acc
            del whole, want
        del dev


@pytest.mark.gpu
def test_text_k13_k14(cuda, tmp_path):
    """k{k}.txt text at k = 13 and 14: first occurrence + the GPU formatter, the drop-in extractor across the
    dense / sparse boundary and with a repeated k, canonical rows, and the sparse path on the same k."""
    torch = cuda
    from kmerml_b200 import engine
    from kmerml_b200.kmers.generate import KmerExtractor, format_kmer_lines
    for name in ("poly", "crlf"):
        data = genomes()[name]
        dev = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).cuda()
        res = engine.count_dense_device(dev, [0, len(data)], [14, 13], want_freq=False)
        for k in (14, 13):
            row = res.counts_of(0, k)
            first = engine.first_occurrence_device(dev, k, min_record_len=14)
            text = engine.format_kmer_file_device(row, first, k).cpu().numpy().tobytes()
            assert text == oracle.kmer_file_text(data, k, 14).encode(), (name, k)
            del first
            # two GPU routes, one answer: the sparse path at the same k (its own record filter: min length k)
            keys, counts, sfirst, windows = engine.count_sparse_device(dev, k)
            dk = engine.count_dense_device(dev, [0, len(data)], [k], want_freq=False)
            bins, dcounts = observed(dk.counts[0])
            assert np.array_equal(keys.cpu().numpy().view(np.uint64), bins), (name, k)
            assert np.array_equal(counts.cpu().numpy().view(np.uint32).astype(np.int64), dcounts), (name, k)
            assert windows == int(dcounts.sum()) == int(dk.totals[0, 0])
            dfirst = engine.first_occurrence_device(dev, k)
            assert torch.equal(sfirst, dfirst[torch.from_numpy(bins.astype(np.int64)).cuda()]), (name, k)
            del keys, counts, sfirst, dk, dfirst
        del res
        # canonical rows against the host formatter (a canonical bin first appears where either strand's k-mer does)
        res = engine.count_dense_device(dev, [0, len(data)], [14, 13], canonical=True, want_freq=False)
        for k in (14, 13):
            row = res.counts_of(0, k)
            first = engine.first_occurrence_device(dev, k, min_record_len=14)
            got = engine.format_kmer_file_device(row, first, k, canonical=True).cpu().numpy().tobytes()
            bins, counts = observed(row)
            assert np.array_equal(bins, canonical_ref(ref_of(name, k, 14), k)[0]), (name, k)
            fwd = first[torch.from_numpy(bins.astype(np.int64)).cuda()].cpu().numpy().view(np.uint32)
            rcf = first[torch.from_numpy(revcomp_np(bins, k).astype(np.int64)).cuda()].cpu().numpy().view(np.uint32)
            order = np.argsort(np.minimum(fwd, rcf), kind="stable")
            assert got == format_kmer_lines(bins[order], counts[order], k), (name, k)
            del first
        del res, dev
    # the drop-in extractor: dense rows for k <= 14, the sparse path for 15, and k listed twice
    for name in ("poly", "crlf"):
        fa = tmp_path / f"{name}.fa"
        fa.write_bytes(genomes()[name])
        for k_values in ([15, 14, 13, 3], [14, 14, 2]):
            out = tmp_path / f"out_{name}_{len(k_values)}_{k_values[0]}"
            with contextlib.redirect_stdout(io.StringIO()):
                org = KmerExtractor(output_dir=out, compress=False).extract_kmers_from_fasta(fa, k_values)
            for k in dict.fromkeys(k_values):
                want = oracle.kmer_file_text(genomes()[name], k, max(k_values), multiplicity=k_values.count(k))
                assert (out / org / f"k{k}.txt").read_bytes() == want.encode(), (name, k_values, k)
            gc.collect()


@pytest.mark.gpu
def test_count_stats_k13_k14_and_radix_passes(cuda):
    """kmerml_count_stats on k = 13 / 14 rows, and on synthetic rows whose median digits fall in each of the three
    radix-select passes (11 + 11 + 10 bits)."""
    torch = cuda
    from kmerml_b200 import engine

    def check(row, values, what):
        got = engine.kmer_count_stats_device(row, k)
        want = stats_ref(values)
        if want is None:
            assert got["unique_kmers"] == 0 and got["total_kmers"] == 0, what
            return
        assert {key: got[key] for key in want} == want, (what, got, want)
        assert got["estimated_genome_size"] == want["total_kmers"] + k - 1

    for name in ("wrapped", "poly"):
        data = genomes()[name]
        dev = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).cuda()
        res = engine.count_dense_device(dev, [0, len(data)], [14, 13], want_freq=False)
        for k in (14, 13):
            check(res.counts_of(0, k), ref_of(name, k, 14)[1], (name, k))
        del res, dev
    k = 12
    rng = np.random.default_rng(4)
    for values, _ in SELECT_CASES:
        v = np.asarray(values, np.uint64)
        for length in (max(64, 3 * v.size), 4 ** 12):
            row = np.zeros(length, np.uint32)
            row[np.sort(rng.choice(length, v.size, replace=False))] = v.astype(np.uint32)
            check(torch.from_numpy(row.view(np.int32)).cuda(), v, (values[:4], length))


def same(a, b):
    """Equal matrices, NaN (the cosine distance of an all-zero row) where the other has NaN."""
    import torch
    return torch.equal(a.isnan(), b.isnan()) and torch.equal(a.nan_to_num(0.0), b.nan_to_num(0.0))


def _distance_rows(torch, names, ks):
    from kmerml_b200 import engine
    datas = [genomes()[n] for n in names]
    dev, offs = to_device(torch, datas)
    res = engine.count_dense_device(dev, offs, ks, want_freq=False)
    del dev
    return res.counts


@pytest.mark.gpu
def test_distances_k13_k14_rows(cuda):
    """Gram / distances on k = 14 and 13 rows (counts >= 256 and >= 65 536: two and three byte planes, K splits
    of 4^14 / 8192): single call against the exact sparse Gram, row blocks and plane shards bit-identical to it."""
    torch = cuda
    from kmerml_b200 import engine
    names = ["poly", "crlf", "poly2", "header"]
    for ks, planes in (([14], 2), ([13], 3)):
        X = _distance_rows(torch, names, ks)
        g = gram_ref([ref_of(n, ks[0], ks[0]) for n in names])
        for metric in ("cosine", "euclidean"):
            full = engine.pairwise_distance_device(X, metric, out_dtype=torch.float64)
            ok = np.isclose(full.cpu().numpy(), distance_ref(g, metric), rtol=GRAM_RTOL, atol=0, equal_nan=True)
            assert ok.all(), (ks, metric)
            n = len(names)
            for world in (1, 2, 3):
                per = (n + world - 1) // world
                blocks = [engine.pairwise_distance_rows_device(X, min(r * per, n), min((r + 1) * per, n), metric,
                                                               out_dtype=torch.float64) for r in range(world)]
                assert same(torch.cat(blocks), full), (ks, metric, world)
            del blocks
            release()
            p, sumsq, mx = engine.count_planes_device(X)
            assert engine.planes_needed(int(mx.item())) == planes
            for world in (1, 3):
                per = (n + world - 1) // world
                blocks = [engine.distance_rows_planes_device(p, planes, sumsq, min(r * per, n), min((r + 1) * per, n),
                                                             metric, out_dtype=torch.float64) for r in range(world)]
                assert same(torch.cat(blocks), full), (ks, metric, world)
            del p, sumsq, mx, full, blocks
            release()
        del X
        release()
    # one concatenated row of both levels: m = 4^14 + 4^13 = 335 544 320
    X = _distance_rows(torch, names, [14, 13])
    g = gram_ref([[ref_of(n, 14, 14), ref_of(n, 13, 14)] for n in names])
    for metric in ("cosine", "euclidean"):
        full = engine.pairwise_distance_device(X, metric, out_dtype=torch.float64)
        ok = np.isclose(full.cpu().numpy(), distance_ref(g, metric), rtol=GRAM_RTOL, atol=0, equal_nan=True)
        assert ok.all(), metric
        blocks = [engine.pairwise_distance_rows_device(X, r, r + 1, metric, out_dtype=torch.float64) for r in range(4)]
        assert same(torch.cat(blocks), full), metric
