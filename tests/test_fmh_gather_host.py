"""The numpy reference of gather (gather_oracle) against a plain-Python brute force on sets, and the invariants of
the result, on small random set families with ties, duplicates, empty sets and every stopping rule.  No GPU."""
import numpy as np
import pytest

import gather_oracle


def _brute(query, references, threshold, max_matches):
    """Gather on Python sets, written from the definition."""
    q0 = set(query.tolist())
    rs = [set(r.tolist()) for r in references]
    left = set(q0)
    out = []
    while max_matches is None or len(out) < max_matches:
        best, best_u = None, -1
        for i, r in enumerate(rs):
            u = len(left & r)
            if u > best_u:                            # strictly greater: the first index wins a tie
                best, best_u = i, u
        if best is None or best_u < threshold:
            break
        left -= rs[best]
        out.append((best, best_u, len(q0 & rs[best]), len(left)))
    return out


def _family(rng, n_r, universe, dup=True):
    """n_r sorted distinct uint64 arrays over a small universe (so they overlap), with exact duplicates, an empty set
    and a subset of another set among them."""
    vals = np.unique(rng.integers(0, 2 ** 63, universe, dtype=np.uint64))
    refs = []
    for _ in range(n_r):
        size = int(rng.integers(0, universe // 2 + 1))
        refs.append(np.sort(rng.choice(vals, size, replace=False)))
    if dup and n_r >= 4:
        refs[2] = refs[0].copy()                      # an exact duplicate: index 0 wins the tie
        refs[3] = np.zeros(0, np.uint64)              # an empty reference
        refs[1] = np.sort(np.union1d(refs[1], refs[0][: refs[0].size // 2]))
    return vals, refs


def _queries(rng, vals, refs, n_q):
    qs = [np.zeros(0, np.uint64)]                     # an empty query
    for _ in range(n_q - 1):
        parts = [refs[int(i)] for i in rng.integers(0, len(refs), int(rng.integers(1, 4)))]
        parts.append(rng.choice(vals, int(rng.integers(0, 6)), replace=False))
        q = np.unique(np.concatenate(parts)).astype(np.uint64)
        keep = rng.random(q.size) < 0.8
        qs.append(q[keep])
    return qs


def _check_invariants(q, refs, matches, threshold, max_matches):
    picked = [m[0] for m in matches]
    assert len(set(picked)) == len(picked)                                   # no reference twice
    uniq = [m[1] for m in matches]
    assert all(a >= b for a, b in zip(uniq, uniq[1:]))                      # non-increasing
    assert all(m[1] <= m[2] for m in matches)                               # unique <= intersect
    assert all(m[1] >= threshold for m in matches)
    for m in matches:
        assert m[2] == np.intersect1d(q, refs[m[0]]).size
    if matches:
        assert matches[-1][3] == q.size - sum(uniq)
    assert len(matches) <= min(len(refs), q.size // threshold)
    if max_matches is not None:
        assert len(matches) <= max_matches


@pytest.mark.parametrize("seed", range(12))
def test_oracle_matches_brute_force(seed):
    rng = np.random.default_rng(seed)
    vals, refs = _family(rng, int(rng.integers(4, 12)), int(rng.integers(8, 60)))
    qs = _queries(rng, vals, refs, 6)
    for threshold in (1, 2, 5, 1000):
        for max_matches in (None, 1, 2, 100):
            for q in qs:
                got = gather_oracle.gather_one(q, refs, threshold, max_matches)
                assert got == _brute(q, refs, threshold, max_matches), (seed, threshold, max_matches)
                _check_invariants(q, refs, got, threshold, max_matches)


def test_forced_ties_and_duplicates():
    v = np.arange(1, 21, dtype=np.uint64) * np.uint64(1_000_003)
    q = v[:12]
    refs = [v[12:], v[:4], v[4:8], v[:4].copy(), v[8:12], v[2:6]]
    # u = 4 for references 1, 2, 3, 4 and 5: 1 wins; then 2 (4 left), then 4; 3 and 5 are covered by then
    assert gather_oracle.gather_one(q, refs) == [(1, 4, 4, 8), (2, 4, 4, 4), (4, 4, 4, 0)]
    assert gather_oracle.gather_one(q, refs, max_matches=1) == [(1, 4, 4, 8)]
    assert gather_oracle.gather_one(q, refs, threshold=5) == []
    assert gather_oracle.gather_one(q, refs, threshold=13) == []          # threshold > |Q|
    assert gather_oracle.gather_one(np.zeros(0, np.uint64), refs) == []   # empty query
    assert gather_oracle.gather_one(q, []) == []                          # no references
    # a superset is picked before its parts, and a part's later unique is what the superset left
    refs2 = [v[:6], v[:10], v[6:12]]
    assert gather_oracle.gather_one(q, refs2) == [(1, 10, 10, 2), (2, 2, 6, 0)]


def test_result_arrays():
    v = np.arange(1, 11, dtype=np.uint64)
    qs = [v[:6], v[6:], np.zeros(0, np.uint64)]
    refs = [v[:3], v[3:8], v[8:]]
    n, ref, unique, inter, remaining = gather_oracle.gather(qs, refs)
    assert n.tolist() == [2, 2, 0] and ref.shape == (3, 2)
    assert ref.tolist() == [[0, 1], [1, 2], [-1, -1]]                    # query 0: a tie at 3, index 0 first
    assert unique.tolist() == [[3, 3], [2, 2], [0, 0]]
    assert inter.tolist() == [[3, 3], [2, 2], [0, 0]]
    assert remaining.tolist() == [[3, 0], [2, 0], [0, 0]]
    assert gather_oracle.default_max_matches([6, 4, 0], 3, 1) == 3
    assert gather_oracle.default_max_matches([6, 4, 0], 3, 4) == 1
    assert gather_oracle.default_max_matches([], 3, 1) == 0
    with pytest.raises(ValueError):
        gather_oracle.gather_one(qs[0], refs, threshold=0)
