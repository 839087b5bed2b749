"""MinHash sketches on the host: the hash, the numpy oracle of the sketch and of its distances, and the multi-rank
assembly of the sketch distance matrix (world-2 gloo, numpy in place of the device calls).  No GPU."""
import math
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle
import sketch_oracle
from kmerml_b200 import dist as kdist
from kmerml_b200 import engine, synth

M64 = (1 << 64) - 1


def py_fmix64(x):
    x ^= x >> 33
    x = (x * 0xff51afd7ed558ccd) & M64
    x ^= x >> 33
    x = (x * 0xc4ceb9fe1a85ec53) & M64
    x ^= x >> 33
    return x


def py_hash(key, seed):
    return py_fmix64((key + 0x9E3779B97F4A7C15 * (seed + 1)) & M64)


def test_hash_pinned_values():
    cases = [(0, 0, 0x9ca066f1a4ab2eea), (0, 42, 0xce1dccd6fa332be2), (1, 42, 0x0bdd1bac740d1ba2),
             (0x1B, 7, 0x094fffc9b371bb3e), (M64, 42, 0x220f7248a77f87d2), (0x0123456789ABCDEF, M64, 0x87cbfbfe89022cea)]
    for key, seed, want in cases:
        assert py_hash(key, seed) == want
        assert int(sketch_oracle.sketch_hash(np.array([key], np.uint64), seed)[0]) == want
    assert int(sketch_oracle.fmix64(np.array([0], np.uint64))[0]) == 0          # why the seed term is added before mixing


def test_hash_is_a_bijection_on_a_sample():
    rng = np.random.default_rng(11)
    keys = np.unique(rng.integers(0, 2 ** 63, 2_000_000, dtype=np.uint64) * np.uint64(2)
                     + rng.integers(0, 2, 2_000_000, dtype=np.uint64))
    keys = np.concatenate([keys, np.arange(0, 100_000, dtype=np.uint64)])      # small keys: poly-A and its neighbours
    keys = np.unique(keys)
    for seed in (0, 42):
        assert np.unique(sketch_oracle.sketch_hash(keys, seed)).size == keys.size


def brute_sketch(data, k, s, seed, canonical, min_len=None):
    """Every window of every record, one at a time, into a set of hashes."""
    hs = set()
    need = k if min_len is None else min_len
    for _, seq in oracle.parse(data):
        if len(seq) < need:
            continue
        text = seq.decode("latin-1").upper()
        for i in range(len(text) - k + 1):
            w = text[i:i + k]
            if any(c not in "ACGT" for c in w):
                continue
            key = oracle.kmer_to_code(w)
            if canonical:
                key = min(key, oracle.revcomp_code(key, k))
            hs.add(py_hash(key, seed))
    out = sorted(hs)[:s]
    return out, len(out)


def test_oracle_sketch_matches_brute_force():
    genomes = [synth.fasta_bytes([700, 9, 450], seed=3).tobytes(),
               b">x\r\nACGTNNACGTRYACGTTTTTTTTTTTTTACGATCGATCGGGGACCA\r\nacgtacgtaaaCGCGCG\n>y\nACG\n>z\nTTTTTTTTTTTTTTT\n",
               b"", b">only header\n", b"junk before\n>r\nAC GT\tACGTACGTAC\n"]
    for data in genomes:
        for k in (5, 9, 15, 21, 32):
            for canonical in (False, True):
                for s, seed, ml in ((1, 42, None), (64, 42, None), (5000, 7, None), (64, 42, 300)):
                    h, f = sketch_oracle.sketch(data, k, s, seed, canonical, ml)
                    want, wf = brute_sketch(data, k, s, seed, canonical, ml)
                    assert f == wf and [int(v) for v in h] == want, (k, canonical, s, seed, ml)


def merge_distance(a, b, s, k, metric):
    """The definition written out as a two-pointer merge of two ascending sketches."""
    i = j = u = x = 0
    while u < s and (i < len(a) or j < len(b)):
        if j == len(b) or (i < len(a) and a[i] < b[j]):
            i += 1
        elif i == len(a) or b[j] < a[i]:
            j += 1
        else:
            i += 1
            j += 1
            x += 1
        u += 1
    jac = x / u if u else 0.0
    if jac == 0.0:
        return 1.0
    if jac == 1.0:
        return 0.0
    return 1.0 - jac if metric == "jaccard" else -math.log(2.0 * jac / (1.0 + jac)) / k


def test_oracle_distance_matches_merge():
    rng = np.random.default_rng(5)
    pool = np.unique(rng.integers(0, 2 ** 63, 4000, dtype=np.uint64))
    for trial in range(300):
        s = int(rng.choice([1, 2, 7, 50, 300]))
        na, nb = (int(rng.integers(0, s + 1)) for _ in range(2))
        share = int(rng.integers(0, min(na, nb) + 1))
        common = rng.choice(pool[:2000], share, replace=False)
        a = np.unique(np.concatenate([common, rng.choice(pool[2000:3000], na - share, replace=False)]))[:s]
        b = np.unique(np.concatenate([common, rng.choice(pool[3000:], nb - share, replace=False)]))[:s]
        for metric in ("jaccard", "mash"):
            got = sketch_oracle.sketch_distance(a, a.size, b, b.size, s, 21, metric)
            want = merge_distance([int(v) for v in a], [int(v) for v in b], s, 21, metric)
            assert got == want, (trial, metric)
            assert sketch_oracle.sketch_distance(b, b.size, a, a.size, s, 21, metric) == got
    assert sketch_oracle.sketch_distance([], 0, [], 0, 10, 21, "mash") == 1.0
    assert sketch_oracle.sketch_distance([5], 1, [5], 1, 10, 21, "mash") == 0.0


def np_rows(sk, r0, r1, metric):
    """Stand-in for engine.sketch_distance_rows_device (numpy, float32 as the device call returns by default)."""
    h = sk.hashes.numpy().view(np.uint64)
    f = sk.filled.numpy()
    n = h.shape[0]
    out = np.zeros((r1 - r0, n), np.float64)
    for i in range(r0, r1):
        for j in range(n):
            out[i - r0, j] = sketch_oracle.sketch_distance(h[i], int(f[i]), h[j], int(f[j]), sk.s, sk.k, metric)
    return torch.from_numpy(out.astype(np.float32))


def host_sketches(genomes, k, s, seed, canonical=True):
    hashes = np.full((len(genomes), s), M64, np.uint64)
    filled = np.zeros(len(genomes), np.int32)
    for g, data in enumerate(genomes):
        h, f = sketch_oracle.sketch(data, k, s, seed, canonical)
        hashes[g, :f] = h
        filled[g] = f
    return engine.Sketches(torch.from_numpy(hashes.view(np.int64)), torch.from_numpy(filled), k, s, seed, canonical)


def _genomes():
    base = synth.fasta_bytes([6000], seed=31)
    out = [base.tobytes()]
    rng = np.random.default_rng(8)
    for p in (0.01, 0.05, 0.2):
        g = base.copy()
        seq = np.nonzero(np.isin(g, np.frombuffer(b"ACGT", np.uint8)))[0][10:]
        hit = seq[rng.random(seq.size) < p]
        g[hit] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, hit.size)]
        out.append(g.tobytes())
    out += [synth.fasta_bytes([3000], seed=32).tobytes(), b"", b">short\nACGT\n"]
    return out


def _worker(rank, world, port, results):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        genomes = _genomes()
        shards = [[0, 2, 3, 5, 6], [1, 4]]                          # uneven, interleaved
        full = host_sketches(genomes, 15, 200, 42)
        mine = shards[rank]
        local = engine.Sketches(full.hashes[mine], full.filled[mine], 15, 200, 42, True)
        ok = True
        for metric in ("mash", "jaccard"):
            got = kdist.sketch_distance_from_shards(local, shards, metric, rows_fn=np_rows)
            want = np_rows(full, 0, len(genomes), metric)
            ok &= bool(torch.equal(got, want))
        # a rank whose sketches were made with another seed is refused
        other = engine.Sketches(local.hashes, local.filled, 15, 200, 42 + rank, True)
        try:
            kdist.sketch_distance_from_shards(other, shards, "mash", rows_fn=np_rows)
            ok = False
        except ValueError:
            pass
        results[rank] = ok
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def test_sketch_distance_from_shards_gloo_world2():
    world = 2
    results = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), results), nprocs=world, join=True)
    assert all(results[r] for r in range(world))


def test_sketch_distance_from_shards_one_process_and_mutation_sanity():
    genomes = _genomes()
    full = host_sketches(genomes, 15, 200, 42)
    shards = [list(range(len(genomes)))]
    d = kdist.sketch_distance_from_shards(full, shards, "mash", rows_fn=np_rows)
    assert torch.equal(d, np_rows(full, 0, len(genomes), "mash"))
    d = d.numpy()
    assert np.array_equal(d, d.T) and np.all(np.diag(d)[:5] == 0)
    assert d[5, 5] == 1.0 and d[6, 6] == 1.0                     # empty sketches: 1, also on the diagonal
    assert d[0, 1] < d[0, 2] < d[0, 3]                              # more mutations, farther away


def test_concat_sketches_refuses_other_parameters():
    a = host_sketches(_genomes()[:2], 15, 50, 42)
    b = host_sketches(_genomes()[2:4], 15, 50, 42)
    c = engine.concat_sketches(a, b)
    assert torch.equal(c.hashes, host_sketches(_genomes()[:4], 15, 50, 42).hashes)
    for other in (host_sketches(_genomes()[2:4], 16, 50, 42), host_sketches(_genomes()[2:4], 15, 50, 43),
                  host_sketches(_genomes()[2:4], 15, 50, 42, canonical=False)):
        try:
            engine.concat_sketches(a, other)
            assert False, "mismatched sketches were combined"
        except ValueError:
            pass
