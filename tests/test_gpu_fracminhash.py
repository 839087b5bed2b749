"""Scaled (FracMinHash) sketches and their query x reference comparison on the GPU (kmerml_fmh_batch,
kmerml_fmh_fetch, kmerml_fmh_compare) against the numpy reference, bit for bit."""
import ctypes

import numpy as np
import pytest
import torch

import fmh_oracle
import oracle
import sketch_oracle
from kmerml_b200 import _lib, engine, synth
from test_gpu_sketch import _device, _genomes, _mutate, _random_seq, _wrap

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1
ERR_ARG, ERR_RANGE = -1, -2


def _host(sk):
    """[uint64 array per genome] of ScaledSketches."""
    h = sk.hashes.cpu().numpy().view(np.uint64)
    o = sk.offsets.cpu().numpy()
    return [h[o[g]:o[g + 1]] for g in range(len(sk))]


def _rows(sk, r0, r1):
    """The sketches of genomes [r0, r1) as a ScaledSketches of their own."""
    o = sk.offsets
    return engine.ScaledSketches(sk.hashes[int(o[r0]):int(o[r1])], o[r0:r1 + 1] - o[r0], sk.k, sk.scale, sk.seed,
                                 sk.canonical)


def _check(sk, genomes, k, scale, seed, canonical, min_len=None):
    got = _host(sk)
    assert len(got) == len(genomes) and int(sk.offsets[0]) == 0
    for g, data in enumerate(genomes):
        want = fmh_oracle.fmh_sketch(data, k, scale, seed, canonical, min_len)
        assert np.array_equal(got[g], want), (g, k, scale, canonical, got[g].size, want.size)
    return got


def test_region_rule():
    """The first region of a genome (what decides whether an overflow retry happens): one slot per byte at scale 1,
    about twice the expected survivors otherwise."""
    assert fmh_oracle.region(150_000_000, 1) == 150_000_000
    assert fmh_oracle.region(5_000_000, 1000) == 2 * 4999 + 1024
    assert fmh_oracle.region(100, 16) == 100


@pytest.mark.parametrize("k", [9, 15, 21, 31, 32])
@pytest.mark.parametrize("canonical", [True, False])
def test_fmh_batch_matches_oracle(k, canonical):
    seed = 42
    named = _genomes(k, seed, canonical)
    names = [n for n, _ in named]
    genomes = [g for _, g in named]
    fasta, offs = _device(genomes)
    bottom = engine.sketch_batch_device(fasta, offs, k, sketch_size=1000, seed=seed, canonical=canonical)
    bh = bottom.hashes.cpu().numpy().view(np.uint64)
    bf = bottom.filled.cpu().numpy()
    for scale in (1, 16, 1000):
        sk = engine.fmh_batch_device(fasta, offs, k, scale=scale, seed=seed, canonical=canonical)
        torch.cuda.synchronize()
        got = _check(sk, genomes, k, scale, seed, canonical)
        assert torch.equal(sk.sizes().cpu(), torch.tensor([g.size for g in got]))
        # the first s values of a scaled sketch with at least s values are the bottom-s sketch
        for g, f in enumerate(got):
            if f.size >= 1000:
                assert bf[g] == 1000 and np.array_equal(f[:1000], bh[g, :1000]), (g, scale)
            elif scale == 1:                          # every distinct k-mer: the bottom-s sketch is all of it
                assert bf[g] == f.size and np.array_equal(f, bh[g, :f.size]), g
    # the tandem repeat of a low-hash k-mer overflows its first region at scale 1000, so that genome ran again
    tg = names.index("tandem_low_hash")
    assert fmh_oracle.survivors(genomes[tg], k, 1000, seed, canonical) > fmh_oracle.region(len(genomes[tg]), 1000)


def test_fmh_min_record_len():
    rng = np.random.default_rng(9)
    short = b"".join(b">r%d\n" % i + _wrap(_random_seq(int(n), rng).tobytes()) for i, n in enumerate(rng.integers(10, 400, 60)))
    genomes = [short, synth.fasta_bytes([40_000, 90, 250], seed=4).tobytes()]
    fasta, offs = _device(genomes)
    for k in (15, 21):
        for ml in (None, 200):
            sk = engine.fmh_batch_device(fasta, offs, k, scale=16, seed=7, canonical=True, min_record_len=ml)
            _check(sk, genomes, k, 16, 7, True, min_len=ml)


def test_fmh_independent_of_batch_composition():
    k, seed = 21, 42
    named = _genomes(k, seed, True)
    genomes = [g for _, g in named]
    probe = genomes[1]                                # "many_slices": 700 kbp, two records
    rng = np.random.default_rng(5)
    big = [synth.fasta_bytes([150_000_000], seed=int(s)).tobytes() for s in rng.integers(0, 1000, 2)]
    # at scale 1 each region is one slot per byte: the two big genomes do not fit one round of 2^28 slots
    assert fmh_oracle.region(len(big[0]), 1) + fmh_oracle.region(len(big[1]), 1) > 1 << 28
    alone = _host(engine.fmh_batch_device(*_device([probe]), k, scale=1, seed=seed))[0]
    in_batch = _host(engine.fmh_batch_device(*_device(genomes), k, scale=1, seed=seed))[1]
    rounds = engine.fmh_batch_device(*_device([big[0], probe, big[1]]), k, scale=1, seed=seed)
    assert np.array_equal(alone, fmh_oracle.fmh_sketch(probe, k, 1, seed, True))
    assert np.array_equal(in_batch, alone)
    assert np.array_equal(_host(_rows(rounds, 1, 2))[0], alone)
    for i, g in ((0, 0), (2, 1)):
        one = engine.fmh_batch_device(*_device([big[g]]), k, scale=1, seed=seed)
        assert torch.equal(_rows(rounds, i, i + 1).hashes, one.hashes)
        assert 0.99 * 150_000_000 < int(one.sizes()[0]) <= 150_000_000
        del one
    del rounds
    torch.cuda.empty_cache()


def test_fmh_output_capacity_and_fetch():
    L = _lib.load()
    ctx = _lib.context(torch.cuda.current_device()).handle
    genomes = [g for _, g in _genomes(21, 42, True)]
    fasta, offs = _device(genomes)
    offs = np.asarray(offs, np.uint64)
    n = len(genomes)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    want = [fmh_oracle.fmh_sketch(g, 21, 16, 42, True) for g in genomes]
    total_want = sum(w.size for w in want)

    def batch(cap, out, off):
        total = ctypes.c_uint64(0)
        rc = L.kmerml_fmh_batch(ctx, fasta.data_ptr(), offs.ctypes.data, n, 21, 0, _lib.FLAG_CANONICAL, 16, 42,
                                out.data_ptr(), cap, off.data_ptr(), ctypes.byref(total), stream)
        return rc, total.value

    small = torch.full((100,), -7, dtype=torch.int64, device="cuda")
    off_small = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    rc, total = batch(100, small, off_small)
    assert rc == 0 and total == total_want > 100
    assert torch.all(small == -7)                     # nothing written
    fetched = torch.full((total,), -7, dtype=torch.int64, device="cuda")
    off_fetch = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    assert L.kmerml_fmh_fetch(ctx, fetched.data_ptr(), total, off_fetch.data_ptr(), stream) == 0
    assert L.kmerml_fmh_fetch(ctx, fetched.data_ptr(), total - 1, off_fetch.data_ptr(), stream) == ERR_ARG
    roomy = torch.full((total + 10,), -7, dtype=torch.int64, device="cuda")
    off_roomy = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    rc, total2 = batch(total + 10, roomy, off_roomy)
    assert rc == 0 and total2 == total
    torch.cuda.synchronize()
    assert torch.equal(fetched, roomy[:total]) and torch.all(roomy[total:] == -7)
    assert torch.equal(off_fetch, off_roomy) and torch.equal(off_small, off_roomy)
    o = off_roomy.cpu().numpy()
    h = roomy.cpu().numpy().view(np.uint64)
    for g in range(n):
        assert np.array_equal(h[o[g]:o[g + 1]], want[g]), g
    # engine.fmh_batch_device fetches when its first guess (1.25 hashes per `scale` bytes + 256) is short: a genome
    # made of one-window records of low-hash k-mers has about one hash per 24 bytes at scale 1000
    keys = np.random.default_rng(2).integers(0, 1 << 42, 2_000_000, dtype=np.uint64)
    ck = np.minimum(keys, sketch_oracle.revcomp_codes64(keys, 21))
    low = np.unique(keys[sketch_oracle.sketch_hash(ck, 42) <= np.uint64(fmh_oracle.threshold(1000))])[:600]
    dense = b"".join(b">r\n" + oracle.code_to_kmer(int(c), 21).encode() + b"\n" for c in low)
    guess = len(dense) / 1000 * 1.25 + 256
    want = fmh_oracle.fmh_sketch(dense, 21, 1000, 42, True)
    assert want.size > guess
    sk = engine.fmh_batch_device(*_device([dense]), 21, scale=1000)
    assert np.array_equal(_host(sk)[0], want)


def _compare_all(q, r, k, inter):
    """Every metric in float64 and float32 against the reference."""
    qs, rs = q.sizes().cpu().numpy(), r.sizes().cpu().numpy()
    for metric in fmh_oracle.METRICS:
        d64, x = engine.fmh_compare_device(q, r, metric, out_dtype=torch.float64, want_intersections=True)
        d32 = engine.fmh_compare_device(q, r, metric).cpu().numpy()
        d64 = d64.cpu().numpy()
        assert np.array_equal(x.cpu().numpy(), inter)
        want = np.array([[fmh_oracle.metric_value(int(inter[i, j]), int(qs[i]), int(rs[j]), k, metric)
                          for j in range(len(rs))] for i in range(len(qs))]).reshape(d64.shape)
        if metric.endswith("ani"):
            assert np.all(np.abs(d64 - want) <= 1e-12 * np.abs(want)), metric
        else:
            assert np.array_equal(d64, want), metric
        assert np.array_equal(d32, d64.astype(np.float32)), metric


def test_fmh_compare_matches_oracle():
    k, seed, scale = 21, 42, 16
    rng = np.random.default_rng(12)
    base = synth.fasta_bytes([300_000], seed=21)
    queries = [base.tobytes()] + [_mutate(base, p, rng).tobytes() for p in (0.001, 0.01, 0.05)]
    queries += [b"", synth.fasta_bytes([80_000], seed=22).tobytes(), b">none\nACGT\n"]
    queries += [g for _, g in _genomes(k, seed, True)][:6]
    refs = [base.tobytes(), b"", synth.fasta_bytes([50_000], seed=23).tobytes(), queries[5], queries[2]]
    qsk = engine.fmh_batch_device(*_device(queries), k, scale=scale, seed=seed)
    rsk = engine.fmh_batch_device(*_device(refs), k, scale=scale, seed=seed)
    qh, rh = _host(qsk), _host(rsk)
    inter = fmh_oracle.intersections(qh, rh)
    assert inter.shape == (len(queries), len(refs)) and inter[0, 0] == qh[0].size > 0
    _compare_all(qsk, rsk, k, inter)
    # x(Q, R) = x(R, Q)
    _, xt = engine.fmh_compare_device(rsk, qsk, "jaccard", want_intersections=True)
    assert np.array_equal(xt.cpu().numpy(), inter.T)
    # a set against itself: the Jaccard matrix is exactly symmetric
    j = engine.fmh_compare_device(qsk, None, "jaccard", out_dtype=torch.float64).cpu().numpy()
    assert np.array_equal(j, j.T)
    # a block of query rows is the same rows of the whole matrix
    full = engine.fmh_compare_device(qsk, rsk, "containment_ani", out_dtype=torch.float64)
    for r0, r1 in ((0, 1), (3, 7), (5, len(queries))):
        blk = engine.fmh_compare_device(_rows(qsk, r0, r1), rsk, "containment_ani", out_dtype=torch.float64)
        assert torch.equal(blk, full[r0:r1])
    # concat_scaled_sketches keeps every sketch
    both = engine.concat_scaled_sketches(qsk, rsk)
    assert [x.tolist() for x in _host(both)] == [x.tolist() for x in qh + rh]


def test_fmh_compare_skewed_and_long_reference():
    """A 20 kbp query against a 2 Mbp reference at scale 1: the reference spans hundreds of shared-memory chunks."""
    k, seed = 21, 42
    rng = np.random.default_rng(4)
    seq = _random_seq(2_000_000, rng).tobytes()
    ref = b">chr\n" + _wrap(seq)
    sub = b">part\n" + _wrap(seq[700_000:720_000], 70)        # a record that is a substring of the reference
    other = b">other\n" + _wrap(_random_seq(20_000, rng).tobytes())
    qsk = engine.fmh_batch_device(*_device([sub, other, b""]), k, scale=1, seed=seed)
    rsk = engine.fmh_batch_device(*_device([ref, sub]), k, scale=1, seed=seed)
    qh, rh = _host(qsk), _host(rsk)
    assert rh[0].size > 100 * 8192
    inter = fmh_oracle.intersections(qh, rh)
    _compare_all(qsk, rsk, k, inter)
    c = engine.fmh_compare_device(qsk, rsk, "containment", out_dtype=torch.float64).cpu().numpy()
    assert np.all(np.isin(qh[0], rh[0])) and c[0, 0] == 1.0 and c[0, 1] == 1.0
    assert c[2, 0] == 0.0 and c[2, 1] == 0.0                   # an empty query


def test_fmh_compare_million_queries():
    """n_q = 10^6 queries (more CTA rows than a grid dimension holds) of one hash each against two references."""
    rng = np.random.default_rng(8)
    r0 = np.unique(rng.integers(0, 2 ** 63, 50_000, dtype=np.uint64))
    r1 = np.unique(rng.integers(0, 2 ** 63, 20_000, dtype=np.uint64))
    pool = np.concatenate([r0, r1, rng.integers(0, 2 ** 63, 70_000, dtype=np.uint64)])
    n_q = 1_000_000
    qv = pool[rng.integers(0, pool.size, n_q)]
    dev = "cuda"

    def sk(values, offsets):
        return engine.ScaledSketches(torch.from_numpy(values.view(np.int64)).to(dev),
                                     torch.from_numpy(np.asarray(offsets, np.int64)).to(dev), 21, 1000, 42, True)

    q = sk(qv, np.arange(n_q + 1))
    r = sk(np.concatenate([r0, r1]), [0, r0.size, r0.size + r1.size])
    out, x = engine.fmh_compare_device(q, r, "containment", want_intersections=True)
    want = np.stack([np.isin(qv, r0), np.isin(qv, r1)], axis=1)
    assert np.array_equal(x.cpu().numpy(), want.astype(np.int64))
    assert np.array_equal(out.cpu().numpy(), want.astype(np.float32))


def test_fmh_biology():
    k, seed = 21, 42
    rng = np.random.default_rng(31)
    base = synth.fasta_bytes([3_000_000], seed=41)
    rates = (0.001, 0.01, 0.05)
    mutants = [_mutate(base, p, rng).tobytes() for p in rates]
    qsk = engine.fmh_batch_device(*_device(mutants), k, scale=100, seed=seed)
    rsk = engine.fmh_batch_device(*_device([base.tobytes()]), k, scale=100, seed=seed)
    ani = engine.fmh_compare_device(qsk, rsk, "containment_ani", out_dtype=torch.float64).cpu().numpy()[:, 0]
    for p, a in zip(rates, ani):
        assert abs(a - (1 - p)) <= 0.2 * p + 1e-3, (p, a)
    # a 50 kbp insert, sketched from its own file, is contained exactly in the 3 Mbp genome that carries it, while its
    # bottom-s Jaccard distance to that genome is close to 1
    insert = _random_seq(50_000, rng).tobytes()
    host = bytes(_random_seq(3_000_000, rng).tobytes())
    carrier = b">genome\n" + _wrap(host[:1_200_000] + insert + host[1_200_000:])
    plasmid = b">insert\n" + _wrap(insert, 80)
    fasta, offs = _device([plasmid, carrier])
    sk = engine.fmh_batch_device(fasta, offs, k, scale=1000, seed=seed)
    c = engine.fmh_compare_device(_rows(sk, 0, 1), _rows(sk, 1, 2), "containment", out_dtype=torch.float64)
    assert c.item() == 1.0
    bottom = engine.sketch_batch_device(fasta, offs, k, sketch_size=1000, seed=seed)
    d = engine.sketch_distance_device(bottom, "jaccard", out_dtype=torch.float64).cpu().numpy()
    assert d[0, 1] > 0.9


def test_fmh_arguments():
    L = _lib.load()
    ctx = _lib.context(torch.cuda.current_device()).handle
    genome = synth.fasta_bytes([5000], seed=1)
    fasta, offs = _device([genome.tobytes()])
    offs = np.asarray(offs, np.uint64)
    out = torch.empty(10_000, dtype=torch.int64, device="cuda")
    off = torch.zeros(2, dtype=torch.int64, device="cuda")
    d32 = torch.empty((1, 1), dtype=torch.float32, device="cuda")
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    total = ctypes.c_uint64(0)

    def batch(k=21, scale=10, n=1, min_len=0, out_p=out.data_ptr(), off_p=off.data_ptr(), total_p=ctypes.byref(total)):
        return L.kmerml_fmh_batch(ctx, fasta.data_ptr(), offs.ctypes.data, n, k, min_len, 1, scale, 42, out_p,
                                  out.numel(), off_p, total_p, stream)

    def compare(k=21, metric=0, n_q=1, n_r=1, q=out.data_ptr(), o32=d32.data_ptr()):
        return L.kmerml_fmh_compare(ctx, q, off.data_ptr(), n_q, out.data_ptr(), off.data_ptr(), n_r, k, metric, None,
                                    o32, None, stream)

    assert batch() == 0 and compare() == 0
    assert batch(min_len=21) == 0 and batch(scale=1) == 0
    for kw in ({"scale": 0}, {"k": 0}, {"k": 33}, {"n": -1}, {"min_len": 20}, {"out_p": None}, {"off_p": None},
               {"total_p": None}):
        assert batch(**kw) == ERR_ARG, kw
    for kw in ({"k": 0}, {"k": 33}, {"metric": -1}, {"metric": 5}, {"n_q": -1}, {"n_r": -1}, {"q": None}, {"o32": None}):
        assert compare(**kw) == ERR_ARG, kw
    for metric in range(5):
        assert compare(metric=metric) == 0
    sk = engine.fmh_batch_device(fasta, offs.tolist(), 21, scale=10)
    with pytest.raises(ValueError):
        engine.fmh_compare_device(sk, sk, "mash")
    for other in (dict(k=15), dict(scale=11), dict(seed=1), dict(canonical=False)):
        args = dict(k=21, scale=10, seed=42, canonical=True)
        args.update(other)
        k = args.pop("k")
        with pytest.raises(ValueError):
            engine.fmh_compare_device(sk, engine.fmh_batch_device(fasta, offs.tolist(), k, **args))
        with pytest.raises(ValueError):
            engine.concat_scaled_sketches(sk, engine.fmh_batch_device(fasta, offs.tolist(), k, **args))
    with pytest.raises(_lib.KmermlError):
        engine.fmh_batch_device(fasta, offs.tolist(), 21, scale=0)


def test_containment_matrix_dataframe_and_clustering(tmp_path):
    from kmerml_b200.ml import clustering
    from kmerml_b200.ml.sketch import containment_matrix
    rng = np.random.default_rng(3)
    paths = []
    for fam in range(3):
        base = synth.fasta_bytes([200_000], seed=300 + fam)
        for member in range(3):
            p = tmp_path / f"GCF_{fam}{member}.fna"
            _mutate(base, 0.01, rng).tofile(p)
            paths.append(p)
    df = containment_matrix(paths, k=21, scale=100, metric="max_containment_ani")
    assert list(df.index) == [p.stem for p in paths] == list(df.columns)
    assert np.array_equal(df.values, df.values.T) and np.all(np.diag(df.values) == 1.0)
    labels, _ = clustering.hierarchical_clustering(None, n_clusters=3, method="average", distances=1 - df)
    assert len(set(labels[:3])) == len(set(labels[3:6])) == len(set(labels[6:])) == 1 and len(set(labels)) == 3
    rect = containment_matrix(paths[:2], paths[2:7], k=21, scale=100, reference_ids=list("abcde"))
    assert rect.shape == (2, 5) and list(rect.index) == [p.stem for p in paths[:2]] and list(rect.columns) == list("abcde")
    assert rect.iloc[0, 0] > 0.1 and rect.iloc[0, 1] == 0.0
    with pytest.raises(ValueError):
        containment_matrix(paths, query_ids=["x"])
