"""k-mer abundance in scaled sketches on the GPU (KMERML_FLAG_FMH_ABUNDANCE, kmerml_fmh_fetch_abundances,
kmerml_fmh_compare_weighted, kmerml_fmh_gather_abundance and their Python surface) against the numpy references of
abundance_oracle, exactly."""
import ctypes
import math

import numpy as np
import pytest
import torch

import abundance_oracle
import fmh_oracle
import oracle
import sketch_oracle
from kmerml_b200 import _lib, engine, synth
from test_gpu_fracminhash import _host, _rows
from test_gpu_sketch import _device, _genomes, _mutate, _random_seq, _wrap

pytestmark = pytest.mark.gpu

ERR_ARG = -1


def _abund(sk):
    """[int64 array per genome] of the abundances of ScaledSketches."""
    a = sk.abundances.cpu().numpy().astype(np.int64)
    o = sk.offsets.cpu().numpy()
    return [a[o[g]:o[g + 1]] for g in range(len(sk))]


def _rows_a(sk, r0, r1):
    """_rows with the abundances."""
    o = sk.offsets
    sub = _rows(sk, r0, r1)
    sub.abundances = sk.abundances[int(o[r0]):int(o[r1])]
    return sub


@pytest.mark.parametrize("k", [9, 15, 21, 31, 32])
@pytest.mark.parametrize("canonical", [True, False])
def test_abundance_batch_matches_reference(k, canonical):
    seed = 42
    named = _genomes(k, seed, canonical)
    names = [n for n, _ in named]
    genomes = [g for _, g in named]
    fasta, offs = _device(genomes)
    for scale in (1, 16, 1000):
        plain = engine.fmh_batch_device(fasta, offs, k, scale=scale, seed=seed, canonical=canonical)
        sk = engine.fmh_batch_device(fasta, offs, k, scale=scale, seed=seed, canonical=canonical, track_abundance=True)
        assert plain.abundances is None and sk.abundances.dtype == torch.int32
        assert torch.equal(sk.hashes, plain.hashes) and torch.equal(sk.offsets, plain.offsets)
        got_h, got_a = _host(sk), _abund(sk)
        for g, data in enumerate(genomes):
            want_h, want_a = abundance_oracle.fmh_abundances(data, k, scale, seed, canonical)
            assert np.array_equal(got_h[g], want_h), (names[g], scale)
            assert np.array_equal(got_a[g], want_a), (names[g], scale)
            assert int(got_a[g].sum()) == fmh_oracle.survivors(data, k, scale, seed, canonical), (names[g], scale)
    # the tandem repeat of a low-hash k-mer overflowed its first region at scale 1000 and ran again
    tg = names.index("tandem_low_hash")
    assert fmh_oracle.survivors(genomes[tg], k, 1000, seed, canonical) > fmh_oracle.region(len(genomes[tg]), 1000)
    assert got_a[tg].max() > 11_000


def test_abundance_matches_sparse_counts():
    """At scale 1 every k-mer is kept: the abundances are count_sparse_device's counts, mapped through the hash."""
    k, seed = 21, 42
    for name, data in _genomes(k, seed, True):
        if name in ("empty", "no_windows"):
            continue
        fasta, offs = _device([data])
        sk = engine.fmh_batch_device(fasta, offs, k, scale=1, seed=seed, track_abundance=True)
        keys, counts, _, _ = engine.count_sparse_device(fasta, k, canonical=True, want_first=False)
        keys = keys.cpu().numpy().view(np.uint64)
        counts = counts.cpu().numpy().astype(np.int64)
        h = sketch_oracle.sketch_hash(keys, seed)
        order = np.argsort(h)
        assert np.array_equal(_host(sk)[0], h[order]), name
        assert np.array_equal(_abund(sk)[0], counts[order]), name


def test_abundance_independent_of_batch_and_rounds():
    k, seed = 21, 42
    genomes = [g for _, g in _genomes(k, seed, True)]
    probe = genomes[1]
    rng = np.random.default_rng(5)
    big = [synth.fasta_bytes([150_000_000], seed=int(s)).tobytes() for s in rng.integers(0, 1000, 2)]
    assert fmh_oracle.region(len(big[0]), 1) + fmh_oracle.region(len(big[1]), 1) > 1 << 28     # two rounds
    batch = dict(scale=1, seed=seed, track_abundance=True)
    alone = _abund(engine.fmh_batch_device(*_device([probe]), k, **batch))[0]
    in_batch = _abund(engine.fmh_batch_device(*_device(genomes), k, **batch))[1]
    rounds = engine.fmh_batch_device(*_device([big[0], probe, big[1]]), k, **batch)
    assert np.array_equal(alone, abundance_oracle.fmh_abundances(probe, k, 1, seed, True)[1])
    assert np.array_equal(in_batch, alone)
    assert np.array_equal(_abund(_rows_a(rounds, 1, 2))[0], alone)
    for i, g in ((0, 0), (2, 1)):
        one = engine.fmh_batch_device(*_device([big[g]]), k, **batch)
        part = _rows_a(rounds, i, i + 1)
        assert torch.equal(part.hashes, one.hashes) and torch.equal(part.abundances, one.abundances)
        del one, part
    del rounds
    torch.cuda.empty_cache()


def test_fetch_abundances():
    L = _lib.load()
    ctx = _lib.context(torch.cuda.current_device()).handle
    genomes = [g for _, g in _genomes(21, 42, True)]
    fasta, offs = _device(genomes)
    offs = np.asarray(offs, np.uint64)
    n = len(genomes)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    want = [abundance_oracle.fmh_abundances(g, 21, 16, 42, True)[1] for g in genomes]
    total_want = sum(w.size for w in want)

    def batch(flags, cap, out, off):
        total = ctypes.c_uint64(0)
        rc = L.kmerml_fmh_batch(ctx, fasta.data_ptr(), offs.ctypes.data, n, 21, 0, flags, 16, 42, out.data_ptr(), cap,
                                off.data_ptr(), ctypes.byref(total), stream)
        return rc, total.value

    small = torch.zeros(100, dtype=torch.int64, device="cuda")
    off = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    rc, total = batch(_lib.FLAG_CANONICAL | _lib.FLAG_FMH_ABUNDANCE, 100, small, off)
    assert rc == 0 and total == total_want > 100
    ab = torch.full((total + 5,), -7, dtype=torch.int32, device="cuda")
    assert L.kmerml_fmh_fetch_abundances(ctx, ab.data_ptr(), total - 1, stream) == ERR_ARG
    assert L.kmerml_fmh_fetch_abundances(ctx, None, total, stream) == ERR_ARG
    assert L.kmerml_fmh_fetch_abundances(ctx, ab.data_ptr(), total, stream) == 0
    torch.cuda.synchronize()
    o = off.cpu().numpy()
    a = ab[:total].cpu().numpy().astype(np.int64)
    for g in range(n):
        assert np.array_equal(a[o[g]:o[g + 1]], want[g]), g
    assert torch.all(ab[total:] == -7)
    # engine.fmh_batch_device fetches hashes and abundances after a short first guess
    fetched = engine.fmh_batch_device(fasta, offs.tolist(), 21, scale=16, track_abundance=True)
    assert [x.tolist() for x in _abund(fetched)] == [w.tolist() for w in want]
    # without the flag there is nothing to fetch
    assert batch(_lib.FLAG_CANONICAL, 100, small, off)[0] == 0
    assert L.kmerml_fmh_fetch_abundances(ctx, ab.data_ptr(), total, stream) == ERR_ARG


def _check_weighted(q, r, metric):
    """fmh_compare_device of a weighted metric against the reference: numerators exact, weighted containment bit for
    bit, angular similarity within 4 ulp; float32 the rounding of float64.  Returns the float64 matrix."""
    qh, qa, rh = _host(q), _abund(q), _host(r)
    ra = _abund(r) if r.abundances is not None else [None] * len(rh)
    d64, num = engine.fmh_compare_device(q, r, metric, out_dtype=torch.float64, want_intersections=True)
    d32 = engine.fmh_compare_device(q, r, metric).cpu().numpy()
    d64, num = d64.cpu().numpy(), num.cpu().numpy()
    for i in range(len(qh)):
        for j in range(len(rh)):
            x = abundance_oracle.weighted_numerator(qh[i], qa[i], rh[j], ra[j], metric)
            assert int(num[i, j]) == x, (metric, i, j)
            want = abundance_oracle.weighted_metric_value(x, qa[i], ra[j] if ra[j] is not None else [], metric)
            if metric == "weighted_containment":
                assert d64[i, j] == want, (i, j)
            else:
                assert abs(d64[i, j] - want) <= 4 * math.ulp(max(abs(want), 1e-300)), (i, j, d64[i, j], want)
    assert np.array_equal(d32, d64.astype(np.float32))
    return d64


def test_weighted_compare_matches_reference():
    k, seed, scale = 21, 42, 16
    rng = np.random.default_rng(12)
    base = synth.fasta_bytes([300_000], seed=21)
    unit = _random_seq(3000, rng).tobytes()
    queries = [base.tobytes(), _mutate(base, 0.01, rng).tobytes(), b"", b">none\nACGT\n",
               b">rep\n" + _wrap(unit * 40) + b">tail\n" + _wrap(base[1000:60_000].tobytes())]
    queries += [g for _, g in _genomes(k, seed, True)][:6]
    refs = [base.tobytes(), b"", b">rep\n" + _wrap(unit * 3), queries[1], synth.fasta_bytes([50_000], seed=23).tobytes()]
    q = engine.fmh_batch_device(*_device(queries), k, scale=scale, seed=seed, track_abundance=True)
    r = engine.fmh_batch_device(*_device(refs), k, scale=scale, seed=seed, track_abundance=True)
    for metric in abundance_oracle.WEIGHTED_METRICS:
        _check_weighted(q, r, metric)
    # weighted containment needs only the query abundances
    r_plain = engine.fmh_batch_device(*_device(refs), k, scale=scale, seed=seed)
    assert torch.equal(engine.fmh_compare_device(q, r_plain, "weighted_containment", out_dtype=torch.float64),
                       engine.fmh_compare_device(q, r, "weighted_containment", out_dtype=torch.float64))
    # Q = R: symmetric bit for bit, and a diagonal of exactly 1 for every non-empty sketch
    a = engine.fmh_compare_device(q, None, "angular_similarity", out_dtype=torch.float64).cpu().numpy()
    assert np.array_equal(a, a.T)
    nonempty = q.sizes().cpu().numpy() > 0
    assert np.all(np.diag(a)[nonempty] == 1.0) and np.all(np.diag(a)[~nonempty] == 0.0)
    # a block of query rows is the same rows of the whole matrix
    for metric in abundance_oracle.WEIGHTED_METRICS:
        full = engine.fmh_compare_device(q, r, metric, out_dtype=torch.float64)
        for r0, r1 in ((0, 1), (3, 7), (5, len(queries))):
            assert torch.equal(engine.fmh_compare_device(_rows_a(q, r0, r1), r, metric, out_dtype=torch.float64),
                               full[r0:r1])


def test_weighted_compare_skewed_long_reference_and_many_queries():
    """A 2 Mbp reference at scale 1 (hundreds of chunks) with abundances, and 10^5 one-hash queries."""
    k, seed = 21, 42
    rng = np.random.default_rng(4)
    seq = _random_seq(2_000_000, rng).tobytes()
    ref = b">chr\n" + _wrap(seq + seq[500_000:530_000] * 3)        # a region present four times
    sub = b">part\n" + _wrap(seq[500_000:520_000] * 2, 70)
    other = b">other\n" + _wrap(_random_seq(20_000, rng).tobytes())
    q = engine.fmh_batch_device(*_device([sub, other, b""]), k, scale=1, seed=seed, track_abundance=True)
    r = engine.fmh_batch_device(*_device([ref, sub]), k, scale=1, seed=seed, track_abundance=True)
    assert int(r.sizes()[0]) > 100 * 8192
    for metric in abundance_oracle.WEIGHTED_METRICS:
        _check_weighted(q, r, metric)
    # 10^5 queries of one hash each (abundance 1..1000) against the two references
    rh, ra = _host(r), _abund(r)
    pool = np.concatenate([rh[0][::7], rh[1], rng.integers(0, 2 ** 63, 30_000, dtype=np.uint64)])
    n_q = 100_000
    pick = rng.integers(0, pool.size, n_q)
    qv, qa = pool[pick], rng.integers(1, 1000, n_q).astype(np.int32)
    big = engine.ScaledSketches(torch.from_numpy(qv.view(np.int64)).cuda(), torch.arange(n_q + 1, device="cuda"),
                                k, 1, seed, True, torch.from_numpy(qa).cuda())
    for metric in abundance_oracle.WEIGHTED_METRICS:
        _, num = engine.fmh_compare_device(big, r, metric, out_dtype=torch.float64, want_intersections=True)
        want = np.zeros((n_q, 2), np.int64)
        for j in range(2):
            at = np.searchsorted(rh[j], qv)
            hit = (at < rh[j].size) & (rh[j][np.minimum(at, rh[j].size - 1)] == qv)
            w = ra[j][np.minimum(at, rh[j].size - 1)] if metric == "angular_similarity" else 1
            want[:, j] = np.where(hit, qa.astype(np.int64) * w, 0)
        assert np.array_equal(num.cpu().numpy(), want), metric


def _seq_record(name, seq):
    return b">" + name + b"\n" + _wrap(seq)


def _check_gather(q, r, threshold, max_matches):
    """fmh_gather_device with abundances: the plain outputs equal the plain gather's, the weighted ones the
    reference exactly (the last match at max_matches included)."""
    plain_q = engine.ScaledSketches(q.hashes, q.offsets, q.k, q.scale, q.seed, q.canonical)
    res = engine.fmh_gather_device(q, r, threshold=threshold, max_matches=max_matches)
    plain = engine.fmh_gather_device(plain_q, r, threshold=threshold, max_matches=max_matches)
    assert plain.unique_weighted is None and plain.median_abund is None
    for name in ("n_matches", "reference", "unique", "intersect", "remaining"):
        assert torch.equal(getattr(res, name), getattr(plain, name)), name
    assert res.unique_weighted.dtype == res.unique_sumsq.dtype == torch.int64
    assert res.median_abund.dtype == torch.float64
    qh, qa, rh = _host(q), _abund(q), _host(r)
    n = res.n_matches.cpu().numpy()
    cols = [t.cpu().numpy() for t in (res.reference, res.unique, res.intersect, res.remaining, res.unique_weighted,
                                      res.unique_sumsq, res.median_abund)]
    for i in range(len(qh)):
        want = abundance_oracle.gather_abundance_one(qh[i], qa[i], rh, threshold, max_matches)
        got = [tuple(c[i, t].item() for c in cols) for t in range(n[i])]
        assert got == want, (i, threshold, max_matches)
    return res


@pytest.mark.parametrize("k", [21, 31])
def test_weighted_gather_from_fasta(k):
    rng = np.random.default_rng(70 + k)
    A, B, C = (_random_seq(n, rng).tobytes() for n in (300_000, 200_000, 150_000))
    novel = _random_seq(100_000, rng).tobytes()
    fa, fb, fc = _seq_record(b"a", A), _seq_record(b"b", B), _seq_record(b"c", C)
    mut_c = _mutate(np.frombuffer(fc, np.uint8), 0.01, rng).tobytes()
    queries = [fa + _seq_record(b"b_half", B[:100_000]) + mut_c + _seq_record(b"novel", novel),
               fb, b"", _seq_record(b"novel", novel), fa + fc, fa * 3 + fb + fc * 2]
    unrelated = [_seq_record(b"u%d" % i, _random_seq(120_000, rng).tobytes()) for i in range(2)]
    refs = [unrelated[0], fa, fb, fc, fa + fb, fc, b"", unrelated[1]]
    for scale in (16, 100):
        q = engine.fmh_batch_device(*_device(queries), k, scale=scale, track_abundance=True)
        r = engine.fmh_batch_device(*_device(refs), k, scale=scale)
        for threshold in (1, 5, 50):
            for max_matches in (1, 2, None):
                _check_gather(q, r, threshold, max_matches)


def test_abundance_biology(tmp_path):
    """A coverage-skewed sample: 12 random 200 kbp sources at copy numbers 1..12, one copy of a 1 % mutant of a
    reference that is not in the sample.  Every source is found with its copy number as mean and median abundance."""
    from kmerml_b200.ml.sketch import gather
    k, scale = 21, 16
    rng = np.random.default_rng(102)
    n_src = 12
    sources = [_random_seq(200_000, rng).tobytes() for _ in range(n_src)]
    copies = [int(c) for c in rng.integers(1, 13, n_src)]
    original = _random_seq(200_000, rng).tobytes()
    mutant = _mutate(np.frombuffer(_seq_record(b"m", original), np.uint8), 0.01, rng).tobytes()
    unrelated = [_random_seq(150_000, rng).tobytes() for _ in range(3)]
    # no 21-mer repeats within or across the sources (canonical keys), so a source's abundances are its copy number
    keys = []
    for src in sources:
        codes, counts = oracle.count_sparse(_seq_record(b"s", src), k)
        keys.append(np.repeat(np.minimum(codes, sketch_oracle.revcomp_codes64(codes, k)), counts.astype(np.int64)))
    allk = np.concatenate(keys)
    assert np.unique(allk).size == allk.size
    sample = b"".join(_seq_record(b"s%d_%d" % (i, c), sources[i]) for i in range(n_src) for c in range(copies[i]))
    sample += mutant
    qpath = tmp_path / "sample.fa"
    qpath.write_bytes(sample)
    ref_bytes = [_seq_record(b"src%d" % i, s) for i, s in enumerate(sources)] + [_seq_record(b"orig", original)]
    ref_bytes += [_seq_record(b"u%d" % i, u) for i, u in enumerate(unrelated)]
    ref_paths = []
    for i, g in enumerate(ref_bytes):
        p = tmp_path / f"ref{i:02d}.fna"
        p.write_bytes(g)
        ref_paths.append(p)
    df = gather([qpath], ref_paths, k=k, scale=scale, threshold_bp=20_000, track_abundance=True)
    q = engine.fmh_batch_device(*_device([sample]), k, scale=scale, track_abundance=True)
    r = engine.fmh_batch_device(*_device(ref_bytes), k, scale=scale)
    total_a = int(q.abundances.to(torch.int64).sum())
    total_bases = sum(copies) * 200_000 + 200_000
    found = {m: row for m, row in zip(df["match"], df.itertuples())}
    assert sorted(found) == sorted([f"ref{i:02d}" for i in range(n_src + 1)])    # the sources and the original
    uniq = {f"ref{i:02d}": int(r.sizes()[i]) for i in range(n_src)}
    for i in range(n_src):
        row = found[f"ref{i:02d}"]
        c = copies[i]
        assert row.average_abund == c and row.median_abund == c and row.std_abund == 0.0, (i, c)
        assert row.unique_bp / scale == uniq[f"ref{i:02d}"]
        assert row.f_unique_weighted == c * uniq[f"ref{i:02d}"] / total_a
        share = c * 200_000 / total_bases
        assert abs(row.f_unique_weighted - share) <= 0.1 * share, (i, row.f_unique_weighted, share)
    orig = found[f"ref{n_src:02d}"]
    assert orig.median_abund == 1.0 and orig.f_unique_weighted < 200_000 / total_bases


def test_public_surface_and_errors(tmp_path):
    from kmerml_b200.ml import clustering
    from kmerml_b200.ml.sketch import containment_matrix, gather
    rng = np.random.default_rng(3)
    paths = []
    for fam in range(3):
        base = synth.fasta_bytes([200_000], seed=300 + fam)
        for member in range(3):
            p = tmp_path / f"GCF_{fam}{member}.fna"
            _mutate(base, 0.01, rng).tofile(p)
            paths.append(p)
    df = containment_matrix(paths, k=21, scale=100, metric="angular_similarity")
    assert list(df.index) == [p.stem for p in paths] == list(df.columns)
    assert np.array_equal(df.values, df.values.T) and np.all(np.diag(df.values) == 1.0)
    labels, _ = clustering.hierarchical_clustering(None, n_clusters=3, method="average", distances=1 - df)
    assert len(set(labels[:3])) == len(set(labels[3:6])) == len(set(labels[6:])) == 1 and len(set(labels)) == 3
    wc = containment_matrix(paths[:2], paths[2:5], k=21, scale=100, metric="weighted_containment")
    assert wc.shape == (2, 3) and 0.0 < wc.iloc[0, 0] <= 1.0
    # gather: the default DataFrame is unchanged; track_abundance adds the weighted columns
    cols = ["query", "rank", "match", "intersect_bp", "unique_bp", "remaining_bp", "f_orig_query", "f_match",
            "f_unique_to_query", "match_containment_ani"]
    plain = gather([paths[0]], paths[3:], k=21, scale=100, threshold_bp=5000)
    weighted = gather([paths[0]], paths[3:], k=21, scale=100, threshold_bp=5000, track_abundance=True)
    assert list(plain.columns) == cols
    assert list(weighted.columns) == cols + ["n_unique_weighted_found", "f_unique_weighted", "average_abund",
                                             "median_abund", "std_abund"]
    assert weighted[cols].equals(plain)
    q = engine.fmh_batch_device(*_device([paths[0].read_bytes()]), 21, scale=100, track_abundance=True)
    r = engine.fmh_batch_device(*_device([p.read_bytes() for p in paths[3:]]), 21, scale=100)
    res = engine.fmh_gather_device(q, r, threshold=50)
    mass = int(q.abundances.to(torch.int64).sum())
    for t, row in enumerate(weighted.itertuples()):
        u, uw, usq = (int(x[0, t]) for x in (res.unique, res.unique_weighted, res.unique_sumsq))
        assert row.n_unique_weighted_found == uw and row.f_unique_weighted == uw / mass
        assert row.average_abund == uw / u and row.median_abund == float(res.median_abund[0, t])
        assert row.std_abund == math.sqrt(max(usq / u - (uw / u) ** 2, 0.0))
    # argument errors
    plain_q = engine.fmh_batch_device(*_device([paths[0].read_bytes()]), 21, scale=100)
    with pytest.raises(ValueError):
        engine.fmh_compare_device(plain_q, q, "weighted_containment")
    with pytest.raises(ValueError):
        engine.fmh_compare_device(q, plain_q, "angular_similarity")
    with pytest.raises(ValueError):
        engine.concat_scaled_sketches(q, plain_q)
    both = engine.concat_scaled_sketches(q, q)
    assert torch.equal(both.abundances, torch.cat([q.abundances, q.abundances]))
    assert engine.concat_scaled_sketches(plain_q, plain_q).abundances is None
    L = _lib.load()
    ctx = _lib.context(torch.cuda.current_device()).handle
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = torch.empty((1, 1), dtype=torch.float64, device="cuda")

    def compare(metric=_lib.FMH_ANGULAR_SIMILARITY, qa=q.abundances.data_ptr(), ra=q.abundances.data_ptr()):
        return L.kmerml_fmh_compare_weighted(ctx, q.hashes.data_ptr(), q.offsets.data_ptr(), qa, 1, q.hashes.data_ptr(),
                                             q.offsets.data_ptr(), ra, 1, metric, None, None, out.data_ptr(), stream)

    assert compare() == 0 and out.item() == 1.0
    assert compare(_lib.FMH_WEIGHTED_CONTAINMENT, ra=None) == 0 and out.item() == 1.0
    for kw in ({"metric": 0}, {"metric": 7}, {"qa": None}, {"ra": None}):
        assert compare(**kw) == ERR_ARG, kw
