"""numpy reference of gather (kmerml_fmh_gather): the greedy, exact split of each query sketch into the reference
sketches that cover it, on sorted uint64 arrays.  Test infrastructure only, like the oracle package."""
import numpy as np


def gather_one(query, references, threshold=1, max_matches=None):
    """Matches of one query (sorted, distinct uint64 array) in pick order: a list of (reference, unique, intersect,
    remaining).  Round t picks the reference with the most still-unassigned query hashes, the smallest index on a
    tie, and stops without recording when that count is < threshold or max_matches matches are recorded."""
    if threshold < 1:
        raise ValueError("threshold must be >= 1")
    left = np.ones(query.size, bool)                  # query hashes not yet assigned
    hit = [_positions(query, r) for r in references]
    matches = []
    while max_matches is None or len(matches) < max_matches:
        u = np.array([int(np.count_nonzero(left[h])) for h in hit], dtype=np.int64)
        if u.size == 0:
            break
        r = int(np.argmax(u))                         # the first index of the maximum
        if u[r] < threshold:
            break
        left[hit[r]] = False
        matches.append((r, int(u[r]), int(hit[r].size), int(np.count_nonzero(left))))
    return matches


def _positions(query, ref):
    """Where the values of `ref` sit in `query` (both sorted and distinct), for those that are there."""
    at = np.searchsorted(query, ref)
    ok = at < query.size
    ok[ok] = query[at[ok]] == ref[ok]
    return at[ok]


def gather(queries, references, threshold=1, max_matches=None):
    """gather_one of every query, as the arrays of engine.GatherResult: n_matches [n_q] and reference / unique /
    intersect / remaining [n_q, m] (m = max_matches, or the longest list when it is None; -1 and 0 past the
    matches)."""
    lists = [gather_one(q, references, threshold, max_matches) for q in queries]
    m = max_matches if max_matches is not None else max((len(x) for x in lists), default=0)
    n_matches = np.array([len(x) for x in lists], dtype=np.int32)
    ref = np.full((len(lists), m), -1, dtype=np.int32)
    cols = np.zeros((3, len(lists), m), dtype=np.int64)
    for q, x in enumerate(lists):
        for t, (r, unique, inter, remaining) in enumerate(x):
            ref[q, t] = r
            cols[:, q, t] = (unique, inter, remaining)
    return n_matches, ref, cols[0], cols[1], cols[2]


def default_max_matches(query_sizes, n_r, threshold):
    """engine.fmh_gather_device's default: min(n_r, max_q |Q| // threshold), which never truncates."""
    return min(n_r, max((int(s) // threshold for s in query_sizes), default=0))
