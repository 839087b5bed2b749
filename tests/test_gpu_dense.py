"""GPU parity of the dense counting path (through the C-ABI) against the oracle and
the golden fixtures of the unmodified reference.  Integer counts are bit-exact;
frequencies are float32 within 1e-6 relative of the float64 restatement."""
import random

import numpy as np
import pytest

import oracle
from helpers import fuzz_fasta, golden_extract_cases, parse_kmer_file

pytestmark = pytest.mark.gpu

FREQ_RTOL = 1e-6


def torch_mod():
    import torch
    return torch


def gpu_counts(datas, ks, **kw):
    torch = torch_mod()
    from kmerml_b200 import engine, synth
    arrs = [np.frombuffer(d, np.uint8) if len(d) else np.zeros(0, np.uint8) for d in datas]
    buf, offs = synth.pack(arrs)
    dev = torch.from_numpy(np.concatenate([buf, np.zeros(64, np.uint8)])).cuda()
    res = engine.count_dense_device(dev, offs, ks, **kw)
    torch.cuda.synchronize()
    return res


def check_against_oracle(datas, ks, min_record_len=None, canonical=False, partition=True):
    res = gpu_counts(datas, ks, min_record_len=min_record_len, canonical=canonical, partition=partition)
    ml = min_record_len or max(ks)
    totals = res.totals.cpu().numpy()
    for g, d in enumerate(datas):
        for ki, k in enumerate(res.k_list):
            ref = oracle.count_dense(d, k, ml)
            if canonical:
                ref = oracle.canonical_from_forward(ref, k)
            got = res.counts_numpy(g, k).astype(np.uint64)
            assert np.array_equal(ref, got), f"genome {g} k={k}: {np.nonzero(ref != got)[0][:5]}"
            assert int(totals[g, ki]) == int(ref.sum())
            f = res.freq_of(g, k).cpu().numpy().astype(np.float64)
            want = oracle.frequencies(ref)
            denom = np.maximum(np.abs(want), 1e-300)
            assert np.all(np.abs(f - want) / denom <= FREQ_RTOL)


def test_golden_files_from_gpu_counts():
    """counts + first-occurrence order reproduce the reference's k{k}.txt lines exactly."""
    torch = torch_mod()
    from kmerml_b200 import engine
    for c in golden_extract_cases():
        ks = [k for k in dict.fromkeys(c["k_values"]) if k <= 12]
        if not ks:
            continue
        ml = max(c["k_values"])
        res = gpu_counts([c["fasta"]], ks, min_record_len=ml)
        a = np.frombuffer(c["fasta"], np.uint8) if len(c["fasta"]) else np.zeros(0, np.uint8)
        dev = torch.from_numpy(np.concatenate([a, np.zeros(64, np.uint8)])).cuda()[:a.size]
        for k in ks:
            counts = res.counts_numpy(0, k)
            first = engine.first_occurrence_device(dev, k, min_record_len=ml).cpu().numpy().view(np.uint32)
            nz = np.nonzero(counts)[0]
            assert np.all(first[nz] != 0xFFFFFFFF) and np.all(first[counts == 0] == 0xFFFFFFFF)
            order = nz[np.argsort(first[nz], kind="stable")]
            got = [(oracle.file_digits(b, k), int(counts[b])) for b in order]
            assert got == parse_kmer_file(c["files"][str(k)]), (c["name"], k)


def test_golden_batch_all_cases_one_launch():
    cases = golden_extract_cases()
    check_against_oracle([c["fasta"] for c in cases], [1, 2, 3, 5, 7])
    check_against_oracle([c["fasta"] for c in cases], [8, 4])
    check_against_oracle([c["fasta"] for c in cases][:12], [12, 11, 3])
    check_against_oracle([c["fasta"] for c in cases][:12], [12, 11, 3], partition=False)
    check_against_oracle([c["fasta"] for c in cases], [9])
    check_against_oracle([c["fasta"] for c in cases], [10, 6, 1])


def test_fuzz_small():
    rng = random.Random(99)
    for it in range(12):
        datas = [fuzz_fasta(rng) for _ in range(rng.randint(1, 40))]
        ks = sorted(rng.sample(range(1, 13), rng.randint(1, 4)), reverse=rng.random() < 0.3)
        mr = None if rng.random() < 0.7 else max(ks) + rng.randint(1, 10)
        check_against_oracle(datas, ks, min_record_len=mr, partition=(it % 3 != 0))
    # at least 8 x SMs genomes: the shared-histogram paths (k <= 8) walk each genome with one CTA
    torch = torch_mod()
    n = 8 * torch.cuda.get_device_properties(0).multi_processor_count + 16
    datas = [fuzz_fasta(rng) for _ in range(n)]
    check_against_oracle(datas, [8, 3])
    check_against_oracle(datas, [7, 2])


def test_canonical_opt_in():
    rng = random.Random(5)
    datas = [fuzz_fasta(rng, max_len=2000) for _ in range(6)]
    check_against_oracle(datas, [4, 5, 6], canonical=True)
    check_against_oracle(datas, [12, 9], canonical=True)
    check_against_oracle(datas, [12, 9], canonical=True, partition=False)
    # the tiled fold (k >= 7: odd and even k, palindromic middles) beside the pairwise one (k < 7)
    check_against_oracle(datas, [7, 3, 8], canonical=True)
    check_against_oracle(datas, [10, 6, 11, 1], canonical=True)
    from kmerml_b200 import synth
    big = [synth.fasta_bytes([300_000, 150_001], seed=77).tobytes()]
    check_against_oracle(big, [7, 8, 9, 10, 11, 12, 2], canonical=True)


def test_medium_genomes_multi_slice():
    """1-3 Mbp genomes: many slices/tiles per genome, both the shared and the global path."""
    from kmerml_b200 import synth
    g1 = synth.fasta_bytes([700_000, 300_001, 11, 250_000], seed=42).tobytes()
    g2 = synth.config3_genome(7, scale=0.3).tobytes()
    # N runs and soft-masked lower case in a wrapped genome
    rng = np.random.default_rng(8)
    s = np.frombuffer(synth.fasta_bytes([400_000], seed=9).tobytes(), np.uint8).copy()
    for _ in range(50):
        i = int(rng.integers(100, len(s) - 5000))
        n = int(rng.integers(1, 3000))
        seg = s[i:i + n]
        seg[seg != 10] = ord("N")
    low = (s >= 65) & (s <= 90) & (rng.random(len(s)) < 0.3)
    s[low] += 32
    s[:s.tolist().index(10)] = np.frombuffer(b">chr1 synthetic record len=400000"[: s.tolist().index(10)], np.uint8)
    g3 = s.tobytes()
    check_against_oracle([g1, g2, g3], [6])
    check_against_oracle([g1, g2, g3], [1, 2, 3, 4, 5, 6, 7])
    check_against_oracle([g1, g2, g3], [8])
    check_against_oracle([g1, g2, g3], [8, 3], partition="k8as9")
    # k = 8 packed 16-bit histogram: a homopolymer drives one bin far past 16 bits
    poly = (">p\n" + ("A" * 80 + "\n") * 4000 + "ACGTTGCA" * 50 + "\n").encode()
    check_against_oracle([poly, g3], [8, 5])
    check_against_oracle([g1, g3], list(range(1, 13)))
    check_against_oracle([g1, g3], list(range(1, 13)), partition=False)
    check_against_oracle([g1, g2, g3], [11, 9])
    check_against_oracle([g2, g3], [10])
    check_against_oracle([g1, g2], [13])


def test_host_api_matches_device_api():
    torch = torch_mod()
    from kmerml_b200 import engine
    rng = random.Random(3)
    datas = [fuzz_fasta(rng, max_len=3000) for _ in range(7)]
    for ks in ([3, 6], [10, 2, 8]):
        dres = gpu_counts(datas, ks)
        hres = engine.count_dense_host(datas, ks)
        assert torch.equal(dres.counts.cpu(), hres.counts)
        assert torch.equal(dres.freq.cpu(), hres.freq)
        assert torch.equal(dres.totals.cpu(), hres.totals)


def test_host_api_narrow_wire_format():
    """The count rows of k >= 10 cross PCIe as bytes + an exception list and are widened on the host: same rows
    as the plain uint32 copy, also when the exception list overflows (> 65536 bins at or above 255) and for more
    genomes than pipeline slots."""
    torch = torch_mod()
    from kmerml_b200 import engine
    from kmerml_b200 import synth
    rng = np.random.default_rng(8)
    unit = "".join("ACGT"[i] for i in rng.integers(0, 4, 90_000))
    body = unit * 260                                                         # ~86 000 distinct 10-mers, 260 times each
    tandem = (">t\n" + body + "\n").encode()                                  # one unwrapped line, 23 Mbp
    mid = synth.fasta_bytes([400_000, 30], seed=21).tobytes()
    # small enough for 4-bit bins at k = 10..12, with a short tandem array: ~2000 bins beyond 15 -> exception list
    sat = "".join("ACGT"[i] for i in rng.integers(0, 4, 2_000)) * 40
    mixed = synth.fasta_bytes([3_000_000], seed=24).tobytes() + (">sat\n" + sat + "\n").encode()
    datas = [mid, tandem, synth.fasta_bytes([150_000], seed=22).tobytes(), b">e\n", mixed,
             synth.fasta_bytes([90_000], seed=23).tobytes(), mid]
    for ks in ([12, 3, 10], [11, 8]):
        narrow = engine.count_dense_host(datas, ks, want_freq=False)
        wide = engine.count_dense_host(datas, ks, want_freq=False, wide_d2h=True)
        dres = gpu_counts(datas, ks)
        assert torch.equal(narrow.counts, wide.counts), ks
        assert torch.equal(narrow.totals, wide.totals)
        assert torch.equal(narrow.counts, dres.counts.cpu())
        comp = engine.count_dense_host(datas, ks, want_freq=False, compact=True)      # result left as it crossed the bus
        assert torch.equal(comp.counts_tensor(), wide.counts) and torch.equal(comp.totals, wide.totals), ks
        head = comp.rows[:, :8].contiguous().view(torch.int32)
        assert int(head[4, 1]) != 0                                                   # genome 4 went as nibbles
        if ks[0] == 12:
            bytes_only = engine.count_dense_host(datas, ks, want_freq=False, compact=True, nibbles=False)
            assert torch.equal(bytes_only.counts_tensor(), wide.counts), ks
            assert int(bytes_only.rows[:, :8].contiguous().view(torch.int32)[4, 1]) == 0
            assert torch.equal(engine.count_dense_host(datas, ks, want_freq=False, nibbles=False).counts, wide.counts)
    big = (narrow.counts.to(torch.int64) & 0xFFFFFFFF)
    assert int((big[1] >= 255).sum()) > 65536            # the tandem genome did overflow the exception list
    assert 1 in comp._wide


def test_argument_errors():
    torch = torch_mod()
    from kmerml_b200 import _lib, engine
    dev = torch.zeros(128, dtype=torch.uint8, device="cuda")
    with pytest.raises(_lib.KmermlError):
        engine.count_dense_device(dev, [0, 64], [15])
    with pytest.raises(_lib.KmermlError):
        engine.count_dense_device(dev, [0, 64], [5], min_record_len=3)
    with pytest.raises(_lib.KmermlError):
        engine.count_dense_device(dev, [64, 0], [5])


def test_byte_ranges_are_additive():
    """kmerml_count_dense_range over ranges that tile the file sums to the whole-genome rows
    (the multi-GPU all-reduce invariant), on both the partition and the global-atomic path."""
    torch = torch_mod()
    from kmerml_b200 import dist as kdist
    from kmerml_b200 import engine, synth
    g = synth.fasta_bytes([400_000, 30, 250_000], seed=77)
    g[100_000:100_900] = ord("N")
    dev = torch.from_numpy(g).cuda()
    for ks, part in (([12, 5], True), ([10], True), ([12, 11], False), ([6, 2], True), ([8], True)):
        whole = engine.count_dense_device(dev, [0, g.size], ks, want_freq=False, partition=part)
        for world in (2, 3, 5, 7):          # 3 and 7: ranges that start at odd tiles (k = 8 walks 32 KB tiles)
            acc = torch.zeros_like(whole.counts[0], dtype=torch.int64)
            tot = torch.zeros_like(whole.totals[0])
            for b, e in kdist.chunk_ranges(g.size, world):
                c, t = engine.count_dense_range_device(dev, b, e, ks, partition=part)
                acc += c.to(torch.int64) & 0xFFFFFFFF
                tot += t
            assert torch.equal(acc, whole.counts[0].to(torch.int64) & 0xFFFFFFFF), (ks, part, world)
            assert torch.equal(tot, whole.totals[0])
        for k in ks:
            assert np.array_equal(whole.counts_numpy(0, k).astype(np.uint64), oracle.count_dense(g.tobytes(), k, max(ks)))


@pytest.mark.gpu
def test_unwrapped_fasta_long_lines():
    """Whole chromosomes on one line (and a very long header line): the slice-table passes settle what the
    bounded look-back leaves open.  Dense (shared / packed / partition paths), sparse and first occurrence."""
    import torch
    from kmerml_b200 import engine
    rng = np.random.default_rng(17)
    def seq(n):
        return np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].tobytes()
    g1 = b">chr1 one line\n" + seq(700_001) + b"\n>chr2\n" + seq(300_000) + b"N" + seq(5_000) + b"\n"
    g2 = b">" + seq(400_000) + b" header made of bases\n" + seq(200_003) + b"\r\n>x\r\n" + seq(150_000)
    wrapped = seq(240_000)
    g3 = b">w\n" + b"\n".join(wrapped[i:i + 70] for i in range(0, len(wrapped), 70)) + b"\n"
    files = [g1, g2, g3]
    data = b"".join(files)
    offs = np.cumsum([0] + [len(f) for f in files]).tolist()
    dev = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).cuda()
    for ks in ([3, 6], [8], [5, 10], [12]):
        res = engine.count_dense_device(dev, offs, ks, want_freq=False)
        for gi, f in enumerate(files):
            for k in ks:
                got = res.counts_of(gi, k).cpu().numpy().astype(np.int64) & 0xFFFFFFFF
                want = oracle.count_dense(f, k, max(ks))
                assert np.array_equal(got, want.astype(np.int64)), (gi, k, ks)
    for f in (g1, g2):
        d1 = torch.from_numpy(np.frombuffer(f, np.uint8).copy()).cuda()
        keys, counts, first, windows = engine.count_sparse_device(d1, 17)
        wk, wc = oracle.count_sparse(f, 17)
        order = np.argsort(wk)
        assert np.array_equal(keys.cpu().numpy().view(np.uint64), wk[order])
        assert np.array_equal(counts.cpu().numpy().astype(np.int64), wc[order].astype(np.int64))
        fo = engine.first_occurrence_device(d1, 9)
        dense = oracle.count_dense(f, 9)
        assert np.array_equal(fo.cpu().numpy() >= 0, dense > 0)


def test_run_end_tail_list_overflow_rescans():
    """A run end every dozen bytes overflows the partition path's per-genome tail list; the genome's run
    ends are then walked again.  One such genome sits between two ordinary ones."""
    rng = random.Random(91)
    def seq(n):
        return "".join(rng.choice("ACGT") for _ in range(n))
    parts = []
    for r in range(60):
        parts.append(f">r{r}")
        line = []
        for _ in range(rng.randint(20, 60)):
            line.append(seq(rng.randint(9, 30)))
        parts.append("N".join(line))
        for _ in range(rng.randint(0, 30)):
            parts.append(seq(rng.randint(8, 14)) + rng.choice(["", "N", "x"]) + seq(rng.randint(0, 13)))
    busy = ("\n".join(parts) + "\n").encode()
    calm1 = (">a\n" + "\n".join(seq(70) for _ in range(300)) + "\n").encode()
    calm2 = (">b\n" + seq(40_000) + "\n>c\n" + seq(33) + "\n").encode()
    assert busy.count(b"N") * 6 > len(busy) // 64 + 1024       # really overflows
    for ks in ([9, 10, 11, 12], [5, 12], [1, 2, 3, 4, 5, 6, 7, 8, 9], [10], [8, 11]):
        check_against_oracle([calm1, busy, calm2], ks)
    check_against_oracle([calm1, busy, calm2], [9, 12], canonical=True)
    check_against_oracle([busy], [7, 12], min_record_len=40)


def test_sparse_byte_ranges_and_merge():
    """The multi-GPU units of the sparse path in one process: windows ending in byte ranges
    (kmerml_count_sparse_range), routed by key range and merged (kmerml_merge_sparse) == the whole genome."""
    import torch
    from helpers import reduce_windows, unwrapped_fasta_with_windows
    from kmerml_b200 import dist as kdist
    from kmerml_b200 import engine
    rng = np.random.default_rng(123)
    seqs = [np.frombuffer(b"ACGTN", np.uint8)[rng.choice(5, n, p=[.24, .25, .25, .24, .02])].tobytes()
            for n in (700_000, 12, 400_000, 90_000)]
    for k, canonical in ((21, True), (16, False), (32, False)):
        fa, wk, we = unwrapped_fasta_with_windows(seqs, k, canonical)
        dev = torch.from_numpy(np.frombuffer(fa, np.uint8).copy()).cuda()
        whole = engine.count_sparse_device(dev, k, canonical=canonical)
        u, cnt, fst = reduce_windows(wk, we)
        assert np.array_equal(whole[0].cpu().numpy().view(np.uint64), u)
        assert np.array_equal(whole[1].cpu().numpy().astype(np.int64), cnt)
        assert np.array_equal(whole[2].cpu().numpy().view(np.uint32).astype(np.int64), fst)
        assert whole[3] == int(cnt.sum())
        world = 3
        parts, windows = [], 0
        for b, e in kdist.chunk_ranges(len(fa), world, tile=engine.SPARSE_RANGE_ALIGN):
            pk, pc, pf, pw = engine.count_sparse_range_device(dev, b, e, k, canonical=canonical)
            ru, rc, rf = reduce_windows(wk, we, b, e)
            assert np.array_equal(pk.cpu().numpy().view(np.uint64), ru), (k, b, e)
            assert np.array_equal(pc.cpu().numpy().astype(np.int64), rc)
            assert np.array_equal(pf.cpu().numpy().view(np.uint32).astype(np.int64), rf)
            parts.append((pk, pc, pf))
            windows += pw
        assert windows == whole[3]
        # owner r receives every rank's k-mers of key range r
        got = []
        splits = [kdist.key_owner_splits(p[0], k, world) for p in parts]
        for r in range(world):
            ks_, cs_, fs_ = [], [], []
            for p, sp in zip(parts, splits):
                lo = sum(sp[:r])
                ks_.append(p[0][lo:lo + sp[r]]); cs_.append(p[1][lo:lo + sp[r]]); fs_.append(p[2][lo:lo + sp[r]])
            got.append(engine.merge_sparse_device(torch.cat(ks_), torch.cat(cs_), torch.cat(fs_), k))
        assert torch.equal(torch.cat([g[0] for g in got]), whole[0])
        assert torch.equal(torch.cat([g[1] for g in got]), whole[1])
        assert torch.equal(torch.cat([g[2] for g in got]), whole[2])
        # RAW routing (kmerml_emit_sparse_range / kmerml_reduce_sparse_windows): windows grouped by owner = top bits
        # of the k-mer, every owner sorts + reduces what all ranges sent it once; owners in order == the whole genome
        for owner_bits, world in ((0, 1), (2, 4), (3, 8)):
            sent = []
            for b, e in kdist.chunk_ranges(len(fa), world, tile=engine.SPARSE_RANGE_ALIGN):
                ek, ee, oc = engine.emit_sparse_range_device(dev, b, e, k, owner_bits, canonical=canonical)
                sel = (we >= b) & (we < e)
                assert sum(oc) == int(sel.sum()) == ek.numel(), (k, owner_bits, b, e)
                own = (ek.cpu().numpy().view(np.uint64) >> np.uint64(2 * k - owner_bits)).astype(np.int64) if owner_bits else \
                    np.zeros(ek.numel(), np.int64)
                assert np.all(np.diff(own) >= 0) and np.bincount(own, minlength=1 << owner_bits).tolist() == oc
                sent.append((ek, ee, oc))
            outs = []
            for r in range(world):
                ks_ = torch.cat([p[0][sum(p[2][:r]):sum(p[2][:r + 1])] for p in sent])
                es_ = torch.cat([p[1][sum(p[2][:r]):sum(p[2][:r + 1])] for p in sent])
                outs.append(engine.reduce_sparse_windows_device(ks_, es_, 2 * k - owner_bits))
            assert torch.equal(torch.cat([o[0] for o in outs]), whole[0]), (k, owner_bits)
            assert torch.equal(torch.cat([o[1] for o in outs]), whole[1])
            assert torch.equal(torch.cat([o[2] for o in outs]), whole[2])


def test_several_payload_groups():
    """More genomes than one payload group holds: with KMERML_GROUP_PAYLOAD_MB=1 the 9 genomes below fall into several
    groups (tail lists and overflow lists are addressed per group).  Runs in a fresh process because the limit is
    read when the context is created."""
    import os
    import subprocess
    import sys
    code = r"""
import random, sys
import numpy as np
sys.path.insert(0, 'tests'); sys.path.insert(0, '.')
import oracle
from helpers import fuzz_fasta
from test_gpu_dense import gpu_counts
rng = random.Random(3)
datas = []
for i in range(9):
    seq = ''.join(rng.choice('ACGT') for _ in range(rng.randint(60_000, 150_000)))
    if i % 3 == 1:
        seq = seq[:20_000] + 'ACGTTGCAAT' * 3000 + seq[20_000:] + 'N' + seq[:500]
    datas.append(('>g%d\n' % i + '\n'.join(seq[j:j + 70] for j in range(0, len(seq), 70)) + '\n>tail\nACGTACGTACGTAC\n').encode())
ks = [5, 9, 12]
res = gpu_counts(datas, ks)
for g, d in enumerate(datas):
    for k in ks:
        ref = oracle.count_dense(d, k, max(ks))
        assert np.array_equal(ref, res.counts_numpy(g, k).astype(np.uint64)), (g, k)
print('groups ok')
"""
    env = dict(os.environ, KMERML_GROUP_PAYLOAD_MB="1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "groups ok" in out.stdout, out.stdout + out.stderr


def test_calls_on_different_streams_are_ordered():
    """The context's scratch buffers are shared by all device-resident calls: a call on another stream than the one
    before must wait for it (kmerml_b200.h, "streams"), so back-to-back calls on two streams stay exact."""
    torch = torch_mod()
    from kmerml_b200 import engine, synth
    ks = [12, 9]
    datas = [synth.fasta_bytes([1_500_000 + 77 * i], seed=300 + i).tobytes() for i in range(2)]
    devs = []
    for d in datas:
        buf, offs = synth.pack([np.frombuffer(d, np.uint8)])
        devs.append((torch.from_numpy(np.concatenate([buf, np.zeros(64, np.uint8)])).cuda(), offs))
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    results = []
    for rep in range(3):
        for i in (0, 1):
            with torch.cuda.stream(streams[i]):
                results.append((i, engine.count_dense_device(devs[i][0], devs[i][1], ks)))
    torch.cuda.synchronize()
    refs = [[oracle.count_dense(d, k, max(ks)) for k in ks] for d in datas]
    for i, res in results:
        for ki, k in enumerate(ks):
            assert np.array_equal(refs[i][ki], res.counts_numpy(0, k).astype(np.uint64)), (i, k)


def test_encode_symbols():
    """kmerml_encode (stage 1 on its own) against the byte-wise restatement in tests/helpers.py, itself pinned to the
    oracle's k = 1 counts: fuzzed corner cases, a multi-slice genome with N runs, and the tallies."""
    torch = torch_mod()
    from helpers import encode_reference
    from kmerml_b200 import engine, synth
    rng = random.Random(21)
    datas = [fuzz_fasta(rng) for _ in range(40)]
    big = np.frombuffer(synth.fasta_bytes([300_000, 5, 120_000], seed=5).tobytes(), np.uint8).copy()
    big[100_000:103_000][big[100_000:103_000] != 10] = ord("N")
    datas.append(big.tobytes())
    datas.append(b"")
    for d in datas:
        buf = np.concatenate([np.frombuffer(d, np.uint8), np.zeros(64, np.uint8)])
        dev = torch.from_numpy(buf).cuda()[:len(d)]
        sym, tallies = engine.encode_device(dev, want_tallies=True)
        torch.cuda.synchronize()
        want = encode_reference(d)
        got = sym.cpu().numpy()
        assert np.array_equal(got, want), (d[:60], np.nonzero(got != want)[0][:5])
        assert int(tallies[1]) >= int((want < 4).sum())          # total_size counts N / IUPAC symbols too
        st = engine.genome_stats_device(dev)
        t = tallies.cpu().tolist()
        assert (t[0], t[1], t[3]) == (st["contigs"], st["total_size"], st["n_count"])


def test_allreduce_counts_entry_point():
    """kmerml_allreduce_counts (SURVEY 8b) with a ncclComm_t made through NCCL's own API: a communicator of one rank
    here; tools/nccl_abi_check.py under torchrun is the same check on N GPUs (run with 2 and 8, profiles/)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "nccl_abi_check.py")], capture_output=True, text=True,
                       timeout=300, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert '"ok"' in r.stdout
