"""The references of abundance tracking in scaled sketches (abundance_oracle: fmh_abundances, weighted_*,
gather_abundance_one) against plain-Python brute force.  No GPU."""
import math

import numpy as np
import pytest

import abundance_oracle
import fmh_oracle
import gather_oracle
from sketch_oracle import M64, revcomp_codes64, sketch_hash

ENC = {ord(c): i for i, c in enumerate("ACGT")}
ENC.update({ord(c): i for i, c in enumerate("acgt")})


def _windows(data, k, min_len=None):
    """Every k-mer window of FASTA bytes as a 2-bit code, record by record: a window holds k consecutive ACGT bases
    (any case) of one record's sequence lines; other bytes break it; records shorter than min_len (default k) bases
    are skipped (the rules of oracle.count_sparse)."""
    min_len = k if min_len is None else min_len
    out = []
    for rec in data.replace(b"\r", b"").split(b">")[1:]:
        seq = b"".join(rec.split(b"\n")[1:])
        if len(seq) < min_len:
            continue
        run, code = 0, 0
        for ch in seq:
            v = ENC.get(ch)
            if v is None:
                run, code = 0, 0
                continue
            code = ((code << 2) | v) & ((1 << (2 * k)) - 1)
            run += 1
            if run >= k:
                out.append(code)
    return out


def _brute(data, k, scale, seed, canonical):
    """{hash: windows} for the hashes <= T, by a dict over windows."""
    t = M64 // scale
    d = {}
    for c in _windows(data, k):
        key = np.uint64(c)
        if canonical:
            key = min(key, revcomp_codes64(np.array([c], np.uint64), k)[0])
        h = int(sketch_hash(np.array([key], np.uint64), seed)[0])
        if h <= t:
            d[h] = d.get(h, 0) + 1
    return d


def _fasta(rng):
    """Small FASTA with N runs, lower case, short records, CRLF lines and a repeated unit (abundances above 1)."""
    acgt = np.frombuffer(b"ACGT", np.uint8)
    unit = acgt[rng.integers(0, 4, 40)].tobytes()
    seq = bytearray(acgt[rng.integers(0, 4, 3000)].tobytes() + unit * 30)
    for p in rng.integers(0, len(seq) - 20, 12):
        seq[p:p + int(rng.integers(1, 15))] = b"N" * int(rng.integers(1, 15))
    seq[100:300] = bytes(seq[100:300]).lower()
    lines = b"\r\n".join(bytes(seq[i:i + 70]) for i in range(0, len(seq), 70))
    return (b">one\r\n" + lines + b"\r\n>short\nACGTA\n>two\n" + acgt[rng.integers(0, 4, 500)].tobytes() + b"\n"
            + b">rc\n" + unit[::-1].translate(bytes.maketrans(b"ACGT", b"TGCA")) * 5 + b"\n")


@pytest.mark.parametrize("k", [5, 15, 21, 32])
@pytest.mark.parametrize("canonical", [True, False])
def test_abundance_reference_against_window_dict(k, canonical):
    rng = np.random.default_rng(k)
    data = _fasta(rng)
    for scale in (1, 4):
        h, a = abundance_oracle.fmh_abundances(data, k, scale, 42, canonical)
        want = _brute(data, k, scale, 42, canonical)
        assert h.tolist() == sorted(want) and a.tolist() == [want[x] for x in sorted(want)]
        assert np.array_equal(h, fmh_oracle.fmh_sketch(data, k, scale, 42, canonical))
        assert int(a.sum()) == fmh_oracle.survivors(data, k, scale, 42, canonical)
    if k <= 21:
        assert a.max() > 1                            # the repeated unit


def _family(rng, n, pool, with_empty=True):
    """n sorted, distinct uint64 sketches drawn from `pool` with abundances in 1..50 (a few large), one empty."""
    sets, abund = [], []
    for i in range(n):
        size = 0 if (with_empty and i == 0) else int(rng.integers(1, pool.size))
        h = np.sort(rng.choice(pool, size, replace=False))
        a = rng.integers(1, 50, size).astype(np.int64)
        if size:
            a[rng.integers(0, size)] = int(rng.integers(1, 2 ** 31 // max(size, 1)))
        sets.append(h)
        abund.append(a)
    return sets, abund


def test_weighted_metrics_against_brute_force():
    rng = np.random.default_rng(4)
    pool = np.unique(rng.integers(0, 2 ** 64 - 1, 60, dtype=np.uint64))
    sets, abund = _family(rng, 12, pool)
    sets.append(sets[3].copy())                       # a duplicate with the same abundances
    abund.append(abund[3].copy())
    sets.append(sets[3].copy())                       # the same set with proportional abundances
    abund.append(abund[3] * 3)
    for i in range(len(sets)):
        qa = dict(zip(sets[i].tolist(), abund[i].tolist()))
        for j in range(len(sets)):
            ra = dict(zip(sets[j].tolist(), abund[j].tolist()))
            shared = set(qa) & set(ra)
            x_w = abundance_oracle.weighted_numerator(sets[i], abund[i], sets[j], abund[j], "weighted_containment")
            x_a = abundance_oracle.weighted_numerator(sets[i], abund[i], sets[j], abund[j], "angular_similarity")
            assert x_w == sum(qa[h] for h in shared)
            assert x_a == sum(qa[h] * ra[h] for h in shared)
            wc = abundance_oracle.weighted_metric_value(x_w, abund[i], abund[j], "weighted_containment")
            assert wc == (x_w / sum(qa.values()) if shared else 0.0)
            ang = abundance_oracle.weighted_metric_value(x_a, abund[i], abund[j], "angular_similarity")
            if shared:
                cos = x_a / math.sqrt(sum(v * v for v in qa.values()) * sum(v * v for v in ra.values()))
                assert abs(ang - (1 - 2 * math.acos(min(1.0, cos)) / math.pi)) < 1e-6
                assert 0.0 <= ang <= 1.0
            else:
                assert ang == 0.0
            # symmetric bit for bit
            x_t = abundance_oracle.weighted_numerator(sets[j], abund[j], sets[i], abund[i], "angular_similarity")
            assert x_t == x_a
            assert abundance_oracle.weighted_metric_value(x_t, abund[j], abund[i], "angular_similarity") == ang
        if sets[i].size:
            x = abundance_oracle.weighted_numerator(sets[i], abund[i], sets[i], abund[i], "angular_similarity")
            assert abundance_oracle.weighted_metric_value(x, abund[i], abund[i], "angular_similarity") == 1.0
    # proportional abundance vectors on the same set: exactly 1 as well
    x = abundance_oracle.weighted_numerator(sets[3], abund[3], sets[-1], abund[-1], "angular_similarity")
    assert abundance_oracle.weighted_metric_value(x, abund[3], abund[-1], "angular_similarity") == 1.0


def test_weighted_gather_against_brute_force():
    rng = np.random.default_rng(9)
    pool = np.unique(rng.integers(0, 2 ** 64 - 1, 400, dtype=np.uint64))
    refs, _ = _family(rng, 25, pool)
    refs += [refs[5].copy(), refs[6].copy()]          # duplicates: ties go to the smaller index
    queries, qabund = _family(rng, 8, pool)
    queries.append(np.zeros(0, np.uint64))
    qabund.append(np.zeros(0, np.int64))
    for q, a in zip(queries, qabund):
        for threshold in (1, 3, 40):
            for max_matches in (None, 1, 2):
                got = abundance_oracle.gather_abundance_one(q, a, refs, threshold, max_matches)
                plain = gather_oracle.gather_one(q, refs, threshold, max_matches)
                assert [g[:4] for g in got] == plain
                # brute force over plain sets
                left = dict(zip(q.tolist(), a.tolist()))
                for r, unique, _, _, uw, usq, med in got:
                    taken = sorted(left[h] for h in set(refs[r].tolist()) & set(left))
                    for h in set(refs[r].tolist()) & set(left):
                        del left[h]
                    assert len(taken) == unique and uw == sum(taken) and usq == sum(v * v for v in taken)
                    assert med == float(np.median(np.array(taken, dtype=np.float64)))
    # ties in the abundances and an even count: the mean of the two middle values
    q = np.arange(1, 7, dtype=np.uint64)
    got = abundance_oracle.gather_abundance_one(q, [5, 1, 5, 2, 9, 2], [q], 1)
    assert got == [(0, 6, 6, 0, 24, 140, 3.5)]
