"""numpy reference of the MinHash sketches and their distances (kmerml_sketch_batch, kmerml_sketch_distance_rows):
the sketch is built on the C oracle's sparse counts (oracle.count_sparse) plus a numpy canonical fold and the hash.
Test infrastructure only, like the oracle package."""
import math

import numpy as np

import oracle

M64 = (1 << 64) - 1


def fmix64(x):
    """MurmurHash3's 64-bit finalizer on a uint64 numpy array (wrapping arithmetic)."""
    x = np.asarray(x, dtype=np.uint64).copy()
    with np.errstate(over="ignore"):
        x ^= x >> np.uint64(33)
        x *= np.uint64(0xff51afd7ed558ccd)
        x ^= x >> np.uint64(33)
        x *= np.uint64(0xc4ceb9fe1a85ec53)
        x ^= x >> np.uint64(33)
    return x


def sketch_hash(keys, seed):
    """h(key) = fmix64(key + 0x9E3779B97F4A7C15 * (seed + 1)) mod 2^64."""
    add = np.uint64((0x9E3779B97F4A7C15 * (int(seed) + 1)) & M64)
    with np.errstate(over="ignore"):
        return fmix64(np.asarray(keys, dtype=np.uint64) + add)


def revcomp_codes64(codes, k):
    """Reverse complements of 2-bit packed k-mers (uint64 numpy array)."""
    c = np.asarray(codes, dtype=np.uint64).copy()
    rc = np.zeros_like(c)
    for _ in range(k):
        rc = (rc << np.uint64(2)) | (np.uint64(3) - (c & np.uint64(3)))
        c >>= np.uint64(2)
    return rc


def sketch(data, k, s, seed, canonical, min_len=None):
    """(hashes uint64[filled], filled): the min(s, D) smallest distinct hashes of the genome's k-mers, ascending."""
    codes, _ = oracle.count_sparse(data, k, min_len)
    if canonical:
        codes = np.minimum(codes, revcomp_codes64(codes, k))
    h = np.unique(sketch_hash(codes, seed))
    return h[:s], int(min(s, h.size))


def sketch_distance(a, fa, b, fb, s, k, metric):
    """Distance of two sketches (Ondov et al. 2016): U = the min(s, |A u B|) smallest values of A u B,
    x = |U n A n B|, j = x / |U|; Jaccard 1 - j, Mash -ln(2j / (1 + j)) / k; 1 when j = 0, 0 when j = 1."""
    A = np.asarray(a, dtype=np.uint64)[:fa]
    B = np.asarray(b, dtype=np.uint64)[:fb]
    U = np.union1d(A, B)[:s]
    x = int(np.intersect1d(np.intersect1d(U, A), B).size)
    u = int(U.size)
    if x == 0:
        return 1.0
    if x == u:
        return 0.0
    j = x / u
    if metric == "jaccard":
        return 1.0 - j
    if metric == "mash":
        return -math.log(2.0 * j / (1.0 + j)) / k
    raise ValueError(metric)
