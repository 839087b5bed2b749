"""Gather of scaled sketches on the GPU (kmerml_fmh_gather, engine.fmh_gather_device, ml.sketch.gather) against the
numpy reference of gather_oracle, bit for bit in every output."""
import ctypes

import numpy as np
import pytest
import torch

import gather_oracle
from kmerml_b200 import _lib, engine, synth
from test_gpu_fracminhash import _host, _rows
from test_gpu_sketch import _device, _mutate, _random_seq, _wrap

pytestmark = pytest.mark.gpu

ERR_ARG = -1


def _check(q, r, threshold=1, max_matches=None):
    """fmh_gather_device against the reference and the invariants; returns the result."""
    qh, rh = _host(q), _host(r)
    res = engine.fmh_gather_device(q, r, threshold=threshold, max_matches=max_matches)
    want = gather_oracle.gather(qh, rh, threshold, max_matches)
    if max_matches is None:                           # the default never truncates: pad the unbounded reference
        m = gather_oracle.default_max_matches([x.size for x in qh], len(rh), threshold)
        assert want[1].shape[1] <= m
        want = (want[0],) + tuple(np.pad(w, ((0, 0), (0, m - w.shape[1])), constant_values=fill)
                                  for w, fill in zip(want[1:], (-1, 0, 0, 0)))
    got = (res.n_matches, res.reference, res.unique, res.intersect, res.remaining)
    assert [x.dtype for x in got] == [torch.int32, torch.int32, torch.int64, torch.int64, torch.int64]
    for name, g, w in zip(("n_matches", "reference", "unique", "intersect", "remaining"), got, want):
        assert np.array_equal(g.cpu().numpy(), w), (name, threshold, max_matches)
    # invariants, and intersect equal to fmh_compare_device's intersections
    n, ref, unique, inter, remaining = want
    if len(qh) and len(rh):
        x = engine.fmh_compare_device(q, r, want_intersections=True)[1].cpu().numpy()
    for i in range(len(qh)):
        c = int(n[i])
        assert c <= min(len(rh), qh[i].size // threshold)
        assert len(set(ref[i, :c].tolist())) == c
        assert np.all(np.diff(unique[i, :c]) <= 0) and np.all(unique[i, :c] <= inter[i, :c])
        assert np.array_equal(inter[i, :c], x[i, ref[i, :c]])
        if c:
            assert remaining[i, c - 1] == qh[i].size - unique[i, :c].sum()
    return res


def _seq_record(name, seq):
    return b">" + name + b"\n" + _wrap(seq)


@pytest.mark.parametrize("k", [21, 31])
def test_gather_from_fasta(k):
    rng = np.random.default_rng(70 + k)
    A, B, C = (_random_seq(n, rng).tobytes() for n in (300_000, 200_000, 150_000))
    novel = _random_seq(100_000, rng).tobytes()
    fa, fb, fc = _seq_record(b"a", A), _seq_record(b"b", B), _seq_record(b"c", C)
    mut_c = _mutate(np.frombuffer(fc, np.uint8), 0.01, rng).tobytes()
    queries = [fa + _seq_record(b"b_half", B[:100_000]) + mut_c + _seq_record(b"novel", novel),
               fb, b"", _seq_record(b"novel", novel), fa + fc]
    unrelated = [_seq_record(b"u%d" % i, _random_seq(120_000, rng).tobytes()) for i in range(2)]
    refs = [unrelated[0], fa, fb, fc, fa + fb, fc, b"", unrelated[1]]
    for scale in (16, 100):
        q = engine.fmh_batch_device(*_device(queries), k, scale=scale)
        r = engine.fmh_batch_device(*_device(refs), k, scale=scale)
        for threshold in (1, 5, 50):
            for max_matches in (1, 2, None):
                res = _check(q, r, threshold, max_matches)
        ref = res.reference.cpu().numpy()
        assert ref[0, 0] == 4                         # A + B covers more of query 0 than A alone
        assert 3 in ref[0] and 5 not in ref[0]        # C and its exact duplicate: the lower index wins
        assert ref[1, 0] == 2 and ref[4, :2].tolist() == [1, 3] and res.n_matches[2] == 0


def _sketches(values, offsets, dev="cuda"):
    return engine.ScaledSketches(torch.from_numpy(np.asarray(values, np.uint64).view(np.int64)).to(dev),
                                 torch.from_numpy(np.asarray(offsets, np.int64)).to(dev), 21, 1000, 42, True)


def _csr(arrays):
    off = np.concatenate(([0], np.cumsum([a.size for a in arrays]))).astype(np.int64)
    vals = np.concatenate(arrays).astype(np.uint64) if arrays else np.zeros(0, np.uint64)
    return _sketches(vals, off)


def test_gather_heavy_overlap_ties_and_long_reference():
    rng = np.random.default_rng(5)
    pool = np.unique(rng.integers(0, 2 ** 64 - 1, 60_000, dtype=np.uint64))
    shared = pool[0]
    refs = []
    for i in range(3000):                             # one hash in every one of 3000 references
        own = rng.choice(pool[1:], int(rng.integers(0, 40)), replace=False)
        refs.append(np.unique(np.concatenate(([shared], own))))
    block = pool[1:33]
    for i in range(20):                               # 20 references with exactly the same 32-value block: ties
        refs.append(block.copy())
    refs.append(np.sort(rng.choice(pool, 20_000, replace=False)))   # longer than one 8192-value chunk
    big = refs[-1]
    queries = [np.unique(np.concatenate([big[::3], block, [shared]])),
               np.unique(np.concatenate([block, [shared], pool[-50:]])),
               np.array([shared], np.uint64), np.zeros(0, np.uint64),
               np.unique(np.concatenate([refs[7], refs[8], refs[9]]))]
    q, r = _csr(queries), _csr(refs)
    for threshold in (1, 2, 30):
        for max_matches in (None, 3):
            res = _check(q, r, threshold, max_matches)
    res = _check(q, r)
    assert res.reference[2, 0] == 0                   # the shared hash: a 3000-way tie, reference 0 wins


def test_gather_ten_thousand_queries_and_independence():
    rng = np.random.default_rng(8)
    pool = np.unique(rng.integers(0, 2 ** 63, 4000, dtype=np.uint64))
    refs = [np.sort(rng.choice(pool, int(rng.integers(10, 400)), replace=False)) for _ in range(30)]
    queries = [np.unique(rng.choice(pool, int(rng.integers(0, 25)), replace=False)) for _ in range(10_000)]
    q, r = _csr(queries), _csr(refs)
    full = _check(q, r, threshold=2)
    again = engine.fmh_gather_device(q, r, threshold=2)
    m = full.reference.shape[1]
    for r0, r1 in ((0, 1), (17, 517), (9_000, 10_000)):
        blk = engine.fmh_gather_device(_rows(q, r0, r1), r, threshold=2, max_matches=m)
        for a, b, c in zip((blk.n_matches, blk.reference, blk.unique, blk.intersect, blk.remaining),
                           (full.n_matches, full.reference, full.unique, full.intersect, full.remaining),
                           (again.n_matches, again.reference, again.unique, again.intersect, again.remaining)):
            assert torch.equal(a, b[r0:r1]) and torch.equal(b, c)


def _genome(i):
    return synth.fasta_bytes([100_000], seed=500 + i)


def test_gather_biology_and_dataframe(tmp_path):
    from kmerml_b200.ml.sketch import gather
    rng = np.random.default_rng(11)
    sources = [3, 50, 77, 120, 181]
    base = [_genome(i) for i in range(190)]
    refs = base + [_mutate(base[s], 0.02, rng) for s in sources] + [_mutate(base[i], 0.02, rng) for i in range(5)]
    ref_paths = []
    for i, g in enumerate(refs):
        p = tmp_path / f"ref{i:03d}.fna"
        g.tofile(p)
        ref_paths.append(p)
    qpath = tmp_path / "sample.fa"
    np.concatenate([base[s] for s in sources] + [synth.fasta_bytes([50_000], seed=9)]).tofile(qpath)
    other = tmp_path / "mag.fa"
    np.concatenate([_mutate(base[60], 0.005, rng), synth.fasta_bytes([60_000], seed=10)]).tofile(other)
    df = gather([qpath, other], ref_paths, k=21, scale=100, threshold_bp=20_000)
    assert list(df.columns) == ["query", "rank", "match", "intersect_bp", "unique_bp", "remaining_bp", "f_orig_query",
                                "f_match", "f_unique_to_query", "match_containment_ani"]
    q = engine.fmh_batch_device(*_device([qpath.read_bytes(), other.read_bytes()]), 21, scale=100)
    r = engine.fmh_batch_device(*_device([p.read_bytes() for p in ref_paths]), 21, scale=100)
    qs, rs = q.sizes().cpu().numpy(), r.sizes().cpu().numpy()
    # the 5 sources first, not their 2 % cousins, and nothing else; the unique fractions add up to what was assigned
    s = df[df["query"] == "sample"]
    assert sorted(s["match"]) == sorted(f"ref{i:03d}" for i in sources) and s["rank"].tolist() == list(range(5))
    assigned = 1 - s["remaining_bp"].iloc[-1] / 100 / qs[0]
    assert abs(s["f_unique_to_query"].sum() - assigned) < 1e-12 and 0.85 < assigned < 0.95
    m = df[df["query"] == "mag"]
    assert m["match"].tolist() == ["ref060"] and 0.99 < m["match_containment_ani"].iloc[0] <= 1.0

    # column values: the engine's integers, in bp and as fractions, with ids given explicitly
    res = engine.fmh_gather_device(q, r, threshold=200)
    ids = [f"R{i}" for i in range(len(ref_paths))]
    df2 = gather([qpath, other], ref_paths, k=21, scale=100, threshold_bp=19_950, query_ids=["x", "y"],
                 reference_ids=ids)
    assert df2["query"].tolist() == ["x"] * int(res.n_matches[0]) + ["y"] * int(res.n_matches[1])
    row = 0
    for i in range(2):
        for t in range(int(res.n_matches[i])):
            ref = int(res.reference[i, t])
            u, x, rem = (int(v[i, t]) for v in (res.unique, res.intersect, res.remaining))
            got = df2.iloc[row]
            assert got["match"] == ids[ref] and got["rank"] == t
            assert (got["intersect_bp"], got["unique_bp"], got["remaining_bp"]) == (x * 100.0, u * 100.0, rem * 100.0)
            assert got["f_orig_query"] == x / qs[i] and got["f_match"] == x / rs[ref]
            assert got["f_unique_to_query"] == u / qs[i]
            assert abs(got["match_containment_ani"] - (x / rs[ref]) ** (1 / 21)) <= 1e-15
            row += 1
    assert row == len(df2) == len(df)
    with pytest.raises(ValueError):
        gather([qpath], ref_paths, query_ids=["a", "b"])


def test_gather_keeps_the_fetch_result():
    L = _lib.load()
    ctx = _lib.context(torch.cuda.current_device()).handle
    genomes = [synth.fasta_bytes([60_000], seed=i).tobytes() for i in range(4)]
    fasta, offs = _device(genomes)
    sk = engine.fmh_batch_device(fasta, offs, 21, scale=16)
    res = engine.fmh_gather_device(_rows(sk, 0, 2), sk)
    assert res.reference[:, 0].tolist() == [0, 1]
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    total = int(sk.offsets[-1])
    hashes = torch.full((total,), -7, dtype=torch.int64, device="cuda")
    off = torch.zeros(len(genomes) + 1, dtype=torch.int64, device="cuda")
    assert L.kmerml_fmh_fetch(ctx, hashes.data_ptr(), total, off.data_ptr(), stream) == 0
    assert torch.equal(hashes, sk.hashes) and torch.equal(off, sk.offsets)


def test_gather_arguments():
    L = _lib.load()
    ctx = _lib.context(torch.cuda.current_device()).handle
    q = _csr([np.arange(1, 50, dtype=np.uint64)])
    r = _csr([np.arange(1, 30, dtype=np.uint64), np.arange(20, 40, dtype=np.uint64)])
    n = torch.full((1,), 7, dtype=torch.int32, device="cuda")
    out = [torch.zeros(4, dtype=torch.int32, device="cuda") for _ in range(4)]
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(n_q=1, n_r=2, threshold=1, max_matches=4, n_p=n.data_ptr(), ref_p=out[0].data_ptr(),
             rem_p=out[3].data_ptr()):
        return L.kmerml_fmh_gather(ctx, q.hashes.data_ptr(), q.offsets.data_ptr(), n_q, r.hashes.data_ptr(),
                                   r.offsets.data_ptr(), n_r, threshold, max_matches, n_p, ref_p, out[1].data_ptr(),
                                   out[2].data_ptr(), rem_p, stream)

    assert call() == 0 and n.item() == 2 and out[0][:2].tolist() == [0, 1] and out[1][:2].tolist() == [29, 10]
    for kw in ({"threshold": 0}, {"max_matches": 0}, {"max_matches": -1}, {"n_q": -1}, {"n_r": -1}, {"n_p": None},
               {"ref_p": None}, {"rem_p": None}):
        assert call(**kw) == ERR_ARG, kw
    assert call(n_q=0, n_p=None) == 0
    n.fill_(7)
    assert call(n_r=0) == 0 and n.item() == 0
    assert call(max_matches=1) == 0 and n.item() == 1
    assert call(threshold=11) == 0 and n.item() == 1 and out[2][0].item() == 29
    for other in (dict(k=15), dict(scale=11), dict(seed=1), dict(canonical=False)):
        args = dict(k=21, scale=1000, seed=42, canonical=True)
        args.update(other)
        bad = engine.ScaledSketches(r.hashes, r.offsets, **args)
        with pytest.raises(ValueError):
            engine.fmh_gather_device(q, bad)
    with pytest.raises(ValueError):
        engine.fmh_gather_device(q, r.hashes)
    with pytest.raises(ValueError):
        engine.fmh_gather_device(q, r, threshold=0)
    empty = engine.fmh_gather_device(q, _csr([]))
    assert empty.reference.shape == (1, 0) and empty.n_matches.tolist() == [0]
