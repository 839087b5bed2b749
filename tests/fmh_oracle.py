"""numpy reference of the scaled (FracMinHash) sketches and their comparison (kmerml_fmh_batch, kmerml_fmh_compare):
the sketch is built on the C oracle's sparse counts (oracle.count_sparse) plus the canonical fold and the hash of
sketch_oracle.  Test infrastructure only, like the oracle package."""
import numpy as np

import oracle
from sketch_oracle import M64, revcomp_codes64, sketch_hash

METRICS = ("containment", "max_containment", "jaccard", "containment_ani", "max_containment_ani")


def threshold(scale):
    """T = floor((2^64 - 1) / scale): a hash is kept when it is <= T."""
    return M64 // int(scale)


def region(nbytes, scale):
    """The library's first survivor region of a genome (api.cu: sketch_region at tau = T)."""
    t = threshold(scale)
    if t == M64:
        return nbytes
    return min(nbytes, 2 * ((nbytes * t) >> 64) + 1024)


def survivors(data, k, scale, seed, canonical, min_len=None):
    """Windows (not distinct k-mers) whose hash is <= T: what the emitter stores."""
    codes, counts = oracle.count_sparse(data, k, min_len)
    if canonical:
        codes = np.minimum(codes, revcomp_codes64(codes, k))
    return int(counts[sketch_hash(codes, seed) <= np.uint64(threshold(scale))].sum())


def fmh_sketch(data, k, scale, seed, canonical, min_len=None):
    """uint64 array: every distinct hash <= T of the genome's k-mers, ascending."""
    codes, _ = oracle.count_sparse(data, k, min_len)
    if canonical:
        codes = np.minimum(codes, revcomp_codes64(codes, k))
    h = np.unique(sketch_hash(codes, seed))
    return h[h <= np.uint64(threshold(scale))]


def metric_value(x, nq, nr, k, metric):
    """The metric of x = |Q n R| in float64; 0 when x = 0."""
    if x == 0:
        return 0.0
    if metric == "containment":
        return x / nq
    if metric == "max_containment":
        return x / min(nq, nr)
    if metric == "jaccard":
        return x / (nq + nr - x)
    if metric == "containment_ani":
        return (x / nq) ** (1.0 / k)
    if metric == "max_containment_ani":
        return (x / min(nq, nr)) ** (1.0 / k)
    raise ValueError(metric)


def intersections(queries, references):
    """int64 [n_q, n_r] matrix of |Q n R| for two lists of uint64 sketches."""
    return np.array([[np.intersect1d(q, r, assume_unique=True).size for r in references] for q in queries],
                    dtype=np.int64).reshape(len(queries), len(references))
