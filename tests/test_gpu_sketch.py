"""MinHash sketches and their Mash / Jaccard distances on the GPU (kmerml_sketch_batch, kmerml_sketch_distance_rows)
against the numpy oracle, bit for bit."""
import ctypes

import numpy as np
import pytest
import torch

import oracle
import sketch_oracle
from kmerml_b200 import _lib, engine, synth

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1
ACGT = np.frombuffer(b"ACGT", np.uint8)


def _random_seq(n, rng):
    return ACGT[rng.integers(0, 4, n)]


def _wrap(seq, width=60, eol=b"\n"):
    seq = bytes(seq)
    return eol.join(seq[i:i + width] for i in range(0, len(seq), width)) + eol


def _first_tau(nbytes, s):
    """The library's first threshold and region for a genome (api.cu: sketch_first_tau, sketch_region)."""
    if 3 * s >= nbytes:
        return M64, nbytes
    tau = ((3 * s) << 64) // nbytes
    return tau, min(nbytes, 2 * ((nbytes * tau) >> 64) + 1024)


def _low_hash_kmer(k, seed, canonical, limit, rng):
    """A random k-mer whose (canonical) key hashes below `limit`."""
    while True:
        keys = rng.integers(0, 2 ** 62, 200_000, dtype=np.uint64)
        if k < 32:
            keys &= np.uint64((1 << (2 * k)) - 1)
        ck = np.minimum(keys, sketch_oracle.revcomp_codes64(keys, k)) if canonical else keys
        hit = np.nonzero(sketch_oracle.sketch_hash(ck, seed) < np.uint64(limit))[0]
        if hit.size:
            return oracle.code_to_kmer(int(keys[hit[0]]), k)


def _genomes(k, seed, canonical):
    """The mixed batch: (name, bytes) pairs."""
    rng = np.random.default_rng(100 + k)
    gs = [("small_records", synth.fasta_bytes([40_000, 9, 25_000], seed=1).tobytes()),
          ("many_slices", synth.fasta_bytes([400_000, 300_000], seed=2).tobytes())]
    # CRLF lines, N runs, IUPAC codes, lower case
    seq = bytearray(_random_seq(90_000, rng).tobytes())
    for p in rng.integers(0, len(seq) - 300, 40):
        n_run = int(rng.integers(1, 200))
        seq[p:p + n_run] = b"N" * n_run
    for p in rng.integers(0, len(seq), 300):
        seq[p] = b"RYKMSWBDHV"[int(rng.integers(0, 10))]
    seq[5000:9000] = bytes(seq[5000:9000]).lower()
    gs.append(("crlf_n_iupac", b">crlf record one\r\n" + _wrap(seq[:50_000], 70, b"\r\n") + b">two\r\n"
               + _wrap(seq[50_000:], 61, b"\r\n")))
    # headers everywhere: many records of all lengths, so slices begin in headers and in sequence
    parts = []
    for i in range(400):
        n = int(rng.integers(1, 3000))
        parts.append(b">rec%d some description that is long enough to cross a chunk %s\n" % (i, b"x" * int(rng.integers(0, 300))))
        parts.append(_wrap(_random_seq(n, rng).tobytes(), int(rng.integers(20, 120))))
    gs.append(("headers_everywhere", b"".join(parts)))
    gs.append(("below_one_slice", b">tiny\n" + _wrap(_random_seq(3000, rng).tobytes())))
    gs.append(("empty", b""))
    gs.append(("no_windows", b">h1\nACGTNACG\n>h2\n\n>h3\nAC\n"))
    # few distinct k-mers in many bytes: the threshold is raised until every window is kept
    unit = _random_seq(500, rng).tobytes()
    gs.append(("few_distinct", b">rep\n" + _wrap(unit * 400)))
    # a tandem repeat of a low-hash k-mer: its windows overflow the first region
    kmer = _low_hash_kmer(k, seed, canonical, M64 // 100_000, rng).encode()
    gs.append(("tandem_low_hash", b">t\n" + _wrap(_random_seq(200_000, rng).tobytes() + (kmer + b"CA") * 12_000
                                                 + _random_seq(5000, rng).tobytes())))
    # a long poly-A run (its key is 0)
    gs.append(("poly_a", b">a\n" + _wrap(_random_seq(20_000, rng).tobytes() + b"A" * 300_000 + _random_seq(5000, rng).tobytes())))
    gs.append(("copy_of_small", gs[0][1]))
    return gs


def _device(genomes):
    buf, offs = synth.pack([np.frombuffer(g, np.uint8) for g in genomes])
    return (torch.from_numpy(buf).cuda() if buf.size else torch.zeros(0, dtype=torch.uint8, device="cuda")), offs


def _check_against_oracle(sk, genomes, k, s, seed, canonical, min_len=None, ref=None):
    h = sk.hashes.cpu().numpy().view(np.uint64)
    f = sk.filled.cpu().numpy()
    for g, data in enumerate(genomes):
        want, wf = ref[g] if ref is not None else sketch_oracle.sketch(data, k, s, seed, canonical, min_len)
        want, wf = want[:s], min(wf, s)
        assert int(f[g]) == wf, (g, k, s, canonical)
        assert np.array_equal(h[g, :wf], want), (g, k, s, canonical)
        assert np.all(h[g, wf:] == np.uint64(M64)), (g, k, s, canonical)


@pytest.mark.parametrize("k", [9, 15, 21, 31, 32])
@pytest.mark.parametrize("canonical", [True, False])
def test_sketch_batch_matches_oracle(k, canonical):
    seed = 42
    named = _genomes(k, seed, canonical)
    genomes = [g for _, g in named]
    fasta, offs = _device(genomes)
    ref = [sketch_oracle.sketch(g, k, 4096, seed, canonical) for g in genomes]
    for s in (1, 1000, 4096):
        sk = engine.sketch_batch_device(fasta, offs, k, sketch_size=s, seed=seed, canonical=canonical)
        torch.cuda.synchronize()
        _check_against_oracle(sk, genomes, k, s, seed, canonical, ref=ref)
    # the retries these genomes are there for really happen: more than 3 s bytes but fewer than s distinct k-mers;
    # more windows of the low-hash k-mer than the first region holds
    sizes = {n: len(g) for n, g in named}
    assert ref[[n for n, _ in named].index("few_distinct")][1] < 1000 and _first_tau(sizes["few_distinct"], 1000)[0] < M64
    assert 12_000 > _first_tau(sizes["tandem_low_hash"], 1000)[1]
    if k == 21 and canonical:
        # a seed change changes the sketch, and the new one is exact too
        sk2 = engine.sketch_batch_device(fasta, offs, k, sketch_size=1000, seed=seed + 1, canonical=canonical)
        sk1 = engine.sketch_batch_device(fasta, offs, k, sketch_size=1000, seed=seed, canonical=canonical)
        assert not torch.equal(sk1.hashes, sk2.hashes)
        _check_against_oracle(sk2, genomes, k, 1000, seed + 1, canonical)


def test_sketch_min_record_len_and_poly_a_overflow():
    rng = np.random.default_rng(9)
    short = b"".join(b">r%d\n" % i + _wrap(_random_seq(int(n), rng).tobytes()) for i, n in enumerate(rng.integers(10, 400, 60)))
    genomes = [short, synth.fasta_bytes([40_000, 90, 250], seed=4).tobytes()]
    # a seed under which poly-A (key 0) hashes low: a poly-A run then overflows the first region
    seeds = np.arange(1_000_000, dtype=np.uint64)
    with np.errstate(over="ignore"):
        h0 = sketch_oracle.fmix64(np.uint64(0x9E3779B97F4A7C15) * (seeds + np.uint64(1)))
    seed = int(np.nonzero(h0 < np.uint64(M64 // 20_000))[0][0])
    genomes.append(b">polyA\n" + _wrap(_random_seq(30_000, rng).tobytes() + b"A" * 200_000))
    assert 200_000 > _first_tau(len(genomes[-1]), 1000)[1]
    fasta, offs = _device(genomes)
    for k in (15, 21):
        for ml in (None, 200):
            sk = engine.sketch_batch_device(fasta, offs, k, sketch_size=1000, seed=seed, canonical=True, min_record_len=ml)
            _check_against_oracle(sk, genomes, k, 1000, seed, True, min_len=ml)


def _mutate(base, p, rng):
    g = base.copy()
    seq = np.nonzero(np.isin(g, ACGT))[0]
    seq = seq[seq > 20]
    hit = seq[rng.random(seq.size) < p]
    g[hit] = ACGT[(np.searchsorted(ACGT, g[hit]) + rng.integers(1, 4, hit.size)) % 4]
    return g


def test_sketch_distances_match_oracle():
    k, s, seed = 21, 1000, 42
    rng = np.random.default_rng(12)
    base = synth.fasta_bytes([600_000], seed=21)
    rates = (0.001, 0.01, 0.05)
    genomes = [base.tobytes()] + [_mutate(base, p, rng).tobytes() for p in rates]
    genomes += [synth.fasta_bytes([80_000], seed=22).tobytes(), synth.fasta_bytes([50_000], seed=23).tobytes(),
                base.tobytes(), b"", b">none\nACGT\n", b">few\nACGTACGTACGTACGTACGTACGTAAAC\n"]
    genomes += [g for _, g in _genomes(k, seed, True)]
    n = len(genomes)
    fasta, offs = _device(genomes)
    sk = engine.sketch_batch_device(fasta, offs, k, sketch_size=s, seed=seed)
    h = sk.hashes.cpu().numpy().view(np.uint64)
    f = sk.filled.cpu().numpy()
    for metric in ("jaccard", "mash"):
        d64 = engine.sketch_distance_device(sk, metric, out_dtype=torch.float64).cpu().numpy()
        d32 = engine.sketch_distance_device(sk, metric).cpu().numpy()
        want = np.array([[sketch_oracle.sketch_distance(h[i], f[i], h[j], f[j], s, k, metric) for j in range(n)] for i in range(n)])
        if metric == "jaccard":
            assert np.array_equal(d64, want)
        else:
            assert np.all(np.abs(d64 - want) <= 1e-12 * np.abs(want))
        assert np.array_equal(d32, d64.astype(np.float32))
        assert np.array_equal(d64, d64.T)
        for i in range(n):
            assert d64[i, i] == (0.0 if f[i] else 1.0)
        for r0, r1 in ((0, n), (0, 1), (n - 1, n), (3, 4), (2, 11), (5, n)):
            blk = engine.sketch_distance_rows_device(sk, r0, r1, metric, out_dtype=torch.float64).cpu().numpy()
            assert np.array_equal(blk, d64[r0:r1])
            blk32 = engine.sketch_distance_rows_device(sk, r0, r1, metric).cpu().numpy()
            assert np.array_equal(blk32, d32[r0:r1])
        # identical genomes; two genomes that share no hash
        assert d64[0, 6] == 0.0
        assert np.intersect1d(h[4, :f[4]], h[5, :f[5]]).size == 0 and d64[4, 5] == 1.0
        assert d64[7, 8] == 1.0                                   # two empty sketches
    d = engine.sketch_distance_device(sk, "mash", out_dtype=torch.float64).cpu().numpy()
    for i, p in enumerate(rates, start=1):                       # Mash distance estimates the mutation rate
        assert abs(d[0, i] - p) <= 0.3 * p + 1e-3, (p, d[0, i])


def test_sketch_distance_matrix_dataframe_and_clustering(tmp_path):
    from kmerml_b200.ml import clustering
    from kmerml_b200.ml.sketch import sketch_distance_matrix
    rng = np.random.default_rng(3)
    paths = []
    for fam in range(3):
        base = synth.fasta_bytes([60_000], seed=300 + fam)
        for member in range(3):
            p = tmp_path / f"GCF_{fam}{member}.fna"
            _mutate(base, 0.01, rng).tofile(p)
            paths.append(p)
    df = sketch_distance_matrix(paths, k=21, sketch_size=500)
    assert list(df.index) == [p.stem for p in paths] == list(df.columns)
    labels, _ = clustering.hierarchical_clustering(None, n_clusters=3, method="average", distances=df)
    assert len(set(labels[:3])) == len(set(labels[3:6])) == len(set(labels[6:])) == 1 and len(set(labels)) == 3
    db = clustering.dbscan_clustering(None, eps=0.05, min_samples=2, distances=df)
    assert len(set(db[:3])) == 1 and db[0] != -1


def test_sketch_arguments():
    L = _lib.load()
    ctx = _lib.context(torch.cuda.current_device()).handle
    genome = synth.fasta_bytes([5000], seed=1)
    fasta, offs = _device([genome.tobytes()])
    offs = np.asarray(offs, np.uint64)
    out = torch.empty((1, 20000), dtype=torch.int64, device="cuda")
    filled = torch.zeros(1, dtype=torch.int32, device="cuda")
    d = torch.empty((1, 1), dtype=torch.float32, device="cuda")
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def batch(k=21, s=100, stride=100):
        return L.kmerml_sketch_batch(ctx, fasta.data_ptr(), offs.ctypes.data, 1, k, 0, 1, s, 42, out.data_ptr(), stride,
                                     filled.data_ptr(), stream)

    def rows(k=21, s=100, stride=100, r1=1, metric=0):
        return L.kmerml_sketch_distance_rows(ctx, out.data_ptr(), stride, filled.data_ptr(), 1, s, k, 0, r1, metric,
                                             d.data_ptr(), None, stream)

    ERR = -1
    assert batch() == 0 and rows() == 0
    for kw in ({"s": 0}, {"s": 16385, "stride": 20000}, {"k": 0}, {"k": 33}, {"stride": 99}):
        assert batch(**kw) == ERR, kw
        assert rows(**kw) == ERR, kw
    assert rows(r1=2) == ERR
    assert rows(metric=2) == ERR and rows(metric=-1) == ERR
    assert batch(s=16384, stride=20000) == 0
    with pytest.raises(_lib.KmermlError):
        engine.sketch_batch_device(fasta, offs.tolist(), 21, sketch_size=0)
    with pytest.raises(ValueError):
        engine.sketch_distance_device(engine.sketch_batch_device(fasta, offs.tolist(), 21), "euclidean")
