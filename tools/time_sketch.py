"""MinHash sketches on a C3-shaped workload: 1000 genomes of 5 Mbp (synth.config3_genome), k = 21, canonical, s = 1000.
Reports the sketch batch time and rate, how many genomes need a retry (too few distinct hashes below the first
threshold, or a survivor region overflow), the full Mash matrix and a 1/8 row block, count_sparse_device on one of
the genomes for scale, and the GPU's name and power limit; ends with an exact check of sampled sketches against the
oracle.
    python tools/time_sketch.py [n_genomes] [scale] [--json OUT]"""
import json
import os
import subprocess
import sys
import time
from multiprocessing import Pool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from kmerml_b200 import engine, synth  # noqa: E402

K, S, SEED = 21, 1000, 42
M64 = (1 << 64) - 1


def _genome(args):
    i, scale = args
    return synth.config3_genome(i, scale)


def timed(f, reps):
    f()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        f()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def _u64_le(a, b):
    """a <= b for int64 tensors holding uint64 values."""
    flip = torch.iinfo(torch.int64).min
    return (a ^ flip) <= (b ^ flip)


def _hash(keys):
    """The sketch hash on int64 storage of uint64 keys (wrapping arithmetic, logical shifts)."""
    def shr33(x):
        return (x >> 33) & ((1 << 31) - 1)
    add = (0x9E3779B97F4A7C15 * (SEED + 1)) & M64
    x = keys + (add - (1 << 64) if add >= 1 << 63 else add)
    x = x ^ shr33(x)
    x = x * (0xff51afd7ed558ccd - (1 << 64))
    x = x ^ shr33(x)
    x = x * (0xc4ceb9fe1a85ec53 - (1 << 64))
    return x ^ shr33(x)


def first_round(sizes, fasta, offs):
    """Genomes whose first round (the library's threshold and region rule, api.cu) runs again: too few distinct
    hashes below the threshold, or more surviving windows than the region holds.  From the exact sparse counts."""
    more = over = 0
    for g in range(len(sizes)):
        b = int(sizes[g])
        if 3 * S >= b:
            continue                                   # every window is kept from the start, in a region of b slots
        tau = ((3 * S) << 64) // b
        cap = min(b, 2 * ((b * tau) >> 64) + 1024)
        one = fasta[offs[g]:offs[g + 1]].clone()           # (16-byte aligned, as the library requires)
        keys, counts, _, _ = engine.count_sparse_device(one, K, canonical=True, want_first=False)
        tau_t = torch.tensor(tau - (1 << 64) if tau >= 1 << 63 else tau, dtype=torch.int64, device=keys.device)
        keep = _u64_le(_hash(keys), tau_t)
        distinct, windows = int(keep.sum()), int(counts[keep].to(torch.int64).sum())
        if windows > cap:
            over += 1
        elif distinct < S:
            more += 1
    return more, over


def main():
    argv = sys.argv[1:]
    out_json = None
    if "--json" in argv:
        i = argv.index("--json")
        out_json = argv[i + 1]
        del argv[i:i + 2]
    n = int(argv[0]) if argv else 1000
    scale = float(argv[1]) if len(argv) > 1 else 1.0
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    t0 = time.perf_counter()
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        genomes = pool.map(_genome, [(i, scale) for i in range(n)], chunksize=4)
    buf, offs = synth.pack(genomes)
    gen_s = time.perf_counter() - t0
    fasta = torch.from_numpy(buf).cuda()
    sizes = np.diff(offs)
    res = {"gpu": gpu, "n_genomes": n, "bytes": int(buf.size), "k": K, "s": S, "canonical": True,
           "generate_s": round(gen_s, 1)}
    batch = lambda: engine.sketch_batch_device(fasta, offs, K, sketch_size=S, seed=SEED)   # noqa: E731
    ms = timed(batch, 5)
    res["sketch_batch_ms"] = round(ms, 2)
    res["sketch_gbp_per_s"] = round(buf.size / ms / 1e6, 2)
    sk = batch()
    res["filled_min"] = int(sk.filled.min())
    res["sketch_distance_full_ms"] = round(timed(lambda: engine.sketch_distance_device(sk, "mash"), 10), 3)
    res["sketch_distance_rows_eighth_ms"] = round(timed(lambda: engine.sketch_distance_rows_device(sk, 0, n // 8, "mash"), 10), 3)
    full = engine.sketch_distance_device(sk, "mash", out_dtype=torch.float64)
    res["mash_min_offdiag"] = float((full + torch.eye(n, device=full.device, dtype=full.dtype) * 9).min())
    one = fasta[offs[0]:offs[1]].clone()
    res["count_sparse_one_genome_ms"] = round(timed(lambda: engine.count_sparse_device(one, K, canonical=True,
                                                                                        want_first=False), 10), 2)
    more, over = first_round(sizes, fasta, offs)
    res["retry_more_tau"] = more
    res["retry_overflow"] = over
    # exact check of a sample against the numpy reference of the tests
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import sketch_oracle
    h = sk.hashes.cpu().numpy().view(np.uint64)
    f = sk.filled.cpu().numpy()
    sample = sorted(set(np.random.default_rng(0).choice(n, min(n, 8), replace=False).tolist()) | {0, n - 1})
    for g in sample:
        want, wf = sketch_oracle.sketch(genomes[g].tobytes(), K, S, SEED, True)
        assert int(f[g]) == wf and np.array_equal(h[g, :wf], want), f"genome {g}: sketch differs from the oracle"
    res["oracle_checked"] = sample
    print(json.dumps(res))
    if out_json:
        with open(out_json, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
