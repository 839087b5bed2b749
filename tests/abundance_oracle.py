"""numpy reference of k-mer abundance in scaled sketches (KMERML_FLAG_FMH_ABUNDANCE, kmerml_fmh_compare_weighted,
kmerml_fmh_gather_abundance), built on the references of fmh_oracle and gather_oracle.  Test infrastructure only,
like the oracle package."""
import math

import numpy as np

import oracle
from fmh_oracle import threshold
from gather_oracle import _positions, gather_one
from sketch_oracle import revcomp_codes64, sketch_hash

WEIGHTED_METRICS = ("weighted_containment", "angular_similarity")


def fmh_abundances(data, k, scale, seed, canonical, min_len=None):
    """(hashes, abundances): the sketch of fmh_oracle.fmh_sketch and, for each hash, the number of windows whose
    (canonical) key hashes to it -- the C oracle's counts summed per hash (a forward k-mer and its reverse complement
    fold together)."""
    codes, counts = oracle.count_sparse(data, k, min_len)
    if canonical:
        codes = np.minimum(codes, revcomp_codes64(codes, k))
    h, inv = np.unique(sketch_hash(codes, seed), return_inverse=True)
    a = np.zeros(h.size, np.int64)
    np.add.at(a, inv.reshape(-1), counts.astype(np.int64))
    keep = h <= np.uint64(threshold(scale))
    return h[keep], a[keep]


def weighted_numerator(qh, qa, rh, ra, metric):
    """The exact integer numerator: sum over Q n R of a_Q (weighted containment) or a_Q a_R (angular similarity)."""
    _, iq, ir = np.intersect1d(qh, rh, assume_unique=True, return_indices=True)
    aq = [int(v) for v in np.asarray(qa)[iq]]
    if metric == "weighted_containment":
        return sum(aq)
    return sum(x * int(y) for x, y in zip(aq, np.asarray(ra)[ir]))


def weighted_metric_value(x, qa, ra, metric):
    """The metric in float64 from the integer numerator x and the two abundance vectors; 0 when x = 0 or a
    denominator is 0.  Angular: 1 - 2 acos(c) / pi, c = min(1, x / (sqrt(|a_Q|^2) sqrt(|a_R|^2))), and c = 1 when
    x^2 = |a_Q|^2 |a_R|^2 exactly."""
    if metric == "weighted_containment":
        den = sum(int(v) for v in qa)
        return x / den if x and den else 0.0
    qn, rn = sum(int(v) ** 2 for v in qa), sum(int(v) ** 2 for v in ra)
    if not x or not qn or not rn:
        return 0.0
    c = 1.0 if x * x == qn * rn else min(1.0, float(x) / (math.sqrt(float(qn)) * math.sqrt(float(rn))))
    return 1.0 - 2.0 * math.acos(c) / math.pi


def gather_abundance_one(query, abund, references, threshold=1, max_matches=None):
    """The matches of gather_oracle.gather_one, each with the sum, the sum of squares and the median of the query
    abundances over the hashes it takes: a list of (reference, unique, intersect, remaining, unique_weighted,
    unique_sumsq, median_abund).  The picks are made on the unweighted counts."""
    abund = np.asarray(abund, dtype=np.int64)
    left = np.ones(query.size, bool)
    hit = [_positions(query, r) for r in references]
    out = []
    for r, unique, inter, remaining in gather_one(query, references, threshold, max_matches):
        taken = hit[r][left[hit[r]]]
        left[taken] = False
        a = [int(v) for v in abund[taken]]
        assert len(a) == unique
        s = sorted(a)
        n = len(s)
        median = float(s[n // 2]) if n % 2 else (s[n // 2 - 1] + s[n // 2]) / 2.0
        out.append((r, unique, inter, remaining, sum(a), sum(v * v for v in a), median))
    return out
