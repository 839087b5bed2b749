"""Cost of k-mer abundance tracking in scaled sketches (KMERML_FLAG_FMH_ABUNDANCE), k = 21, canonical:
    batch:   1000 genomes of 5 Mbp (synth.config3_genome) at scale 1000 and 100, with and without abundance tracking,
             the two calls alternated in the same run;
    compare: the 1000 x 1000 weighted containment and angular similarity beside the unweighted containment (scale 1000);
    gather:  one coverage-skewed metagenome-like query -- sources of tools/time_fmh_gather.py's references repeated as
             whole records at copy numbers 1-30, over 1 GB of FASTA -- against those references (scale 1000, threshold
             50 hashes), the weighted gather beside the plain one, then an exact check against the numpy reference.
Times are CUDA-event times of single calls after a warm-up call: min / median / max over the repetitions.  The GPU's
name, power limit and max SM clock are read in the same run.
    python tools/time_fmh_abundance.py [n_genomes] [--json OUT]"""
import json
import os
import subprocess
import sys
import time
from multiprocessing import Pool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from kmerml_b200 import engine, synth  # noqa: E402
from time_fmh_gather import N_REF, THRESHOLD, _ref_batch, _sources_a, timed  # noqa: E402

K, SEED = 21, 42
N_SOURCES = 20                                        # x 5 Mbp x copy numbers 1-30: ~1.5 GB of FASTA


def _host(sk):
    h = sk.hashes.cpu().numpy().view(np.uint64)
    o = sk.offsets.cpu().numpy()
    return [h[o[g]:o[g + 1]] for g in range(len(sk))]


def _alternated(f_plain, f_abund, reps):
    """[min, median, max] ms of each of two calls, timed alternately after one warm-up call of each."""
    f_plain(), f_abund()
    torch.cuda.synchronize()
    ms = ([], [])
    for _ in range(reps):
        for f, out in ((f_plain, ms[0]), (f_abund, ms[1])):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            torch.cuda.synchronize()
            out.append(a.elapsed_time(b))
    res = []
    for m in ms:
        m.sort()
        res.append([round(m[0], 3), round(m[len(m) // 2], 3), round(m[-1], 3)])
    return res


def main():
    argv = sys.argv[1:]
    out_json = None
    if "--json" in argv:
        i = argv.index("--json")
        out_json = argv[i + 1]
        del argv[i:i + 2]
    n = int(argv[0]) if argv else 1000
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    res = {"gpu": gpu, "n_genomes": n, "k": K, "canonical": True}
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        genomes = pool.map(synth.config3_genome, range(n), chunksize=4)
    buf, offs = synth.pack(genomes)
    del genomes
    fasta = torch.from_numpy(buf).cuda()
    res["bytes"] = int(buf.size)

    # batch, with and without abundances, alternated
    for scale in (1000, 100):
        def batch(track):
            return lambda: engine.fmh_batch_device(fasta, offs, K, scale=scale, seed=SEED, track_abundance=track)
        plain, abund = _alternated(batch(False), batch(True), 5)
        res[f"batch_scale{scale}_ms"] = plain
        res[f"batch_scale{scale}_abundance_ms"] = abund
        res[f"batch_scale{scale}_abundance_cost_pct"] = round(100 * (abund[1] / plain[1] - 1), 1)
    sk = engine.fmh_batch_device(fasta, offs, K, scale=1000, seed=SEED, track_abundance=True)
    plain_sk = engine.fmh_batch_device(fasta, offs, K, scale=1000, seed=SEED)
    assert torch.equal(sk.hashes, plain_sk.hashes) and torch.equal(sk.offsets, plain_sk.offsets)
    res["hashes_per_genome_scale1000"] = round(float(sk.sizes().double().mean()), 1)
    res["abundance_sum_scale1000"] = int(sk.abundances.to(torch.int64).sum())
    del fasta

    # n x n comparison, weighted beside unweighted
    res["compare_containment_ms"] = timed(lambda: engine.fmh_compare_device(sk, None, "containment"), 5)
    res["compare_weighted_containment_ms"] = timed(lambda: engine.fmh_compare_device(sk, None, "weighted_containment"), 5)
    res["compare_angular_similarity_ms"] = timed(lambda: engine.fmh_compare_device(sk, None, "angular_similarity"), 5)
    ang = engine.fmh_compare_device(sk, None, "angular_similarity", out_dtype=torch.float64)
    assert torch.equal(ang, ang.T) and bool(torch.all(torch.diagonal(ang) == 1.0))
    del sk, plain_sk, ang

    # a coverage-skewed metagenome-like query against the gather script's references
    t0 = time.perf_counter()
    n_ref = N_REF
    n_all = n_ref + n_ref // 4
    rng = np.random.default_rng(40)
    sources = _sources_a(n_ref)[:N_SOURCES]
    copies = [int(c) for c in rng.integers(1, 31, len(sources))]
    parts = []
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        for b in range(0, n_all, 250):
            chunk = [(a, min(a + 8, b + 250, n_all), n_ref) for a in range(b, min(b + 250, n_all), 8)]
            gs = [g for x in pool.map(_ref_batch, chunk) for g in x]
            rb, ro = synth.pack(gs)
            parts.append(engine.fmh_batch_device(torch.from_numpy(rb).cuda(), ro, K, scale=1000, seed=SEED))
    refs = engine.concat_scaled_sketches(*parts)
    del parts
    query = np.concatenate([synth.config3_genome(s) for s, c in zip(sources, copies) for _ in range(c)])
    res["query_bytes"] = int(query.size)
    assert query.size >= 1 << 30
    qf = torch.from_numpy(query).cuda()
    del query
    q = engine.fmh_batch_device(qf, [0, int(qf.numel())], K, scale=1000, seed=SEED, track_abundance=True)
    del qf
    plain_q = engine.ScaledSketches(q.hashes, q.offsets, q.k, q.scale, q.seed, q.canonical)
    res["prepare_s"] = round(time.perf_counter() - t0, 1)
    res["copy_numbers"] = copies
    gplain, gweighted = _alternated(lambda: engine.fmh_gather_device(plain_q, refs, threshold=THRESHOLD),
                                    lambda: engine.fmh_gather_device(q, refs, threshold=THRESHOLD), 3)
    res["gather_plain_ms"], res["gather_weighted_ms"] = gplain, gweighted
    out = engine.fmh_gather_device(q, refs, threshold=THRESHOLD)
    n_m = int(out.n_matches[0])
    res["matches"] = n_m
    res["median_abund"] = out.median_abund[0, :n_m].tolist()

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import abundance_oracle
    want = abundance_oracle.gather_abundance_one(_host(q)[0], q.abundances.cpu().numpy(), _host(refs), THRESHOLD)
    cols = [t.cpu().numpy() for t in (out.reference, out.unique, out.intersect, out.remaining, out.unique_weighted,
                                      out.unique_sumsq, out.median_abund)]
    got = [tuple(c[0, t].item() for c in cols) for t in range(n_m)]
    assert got == want, "weighted gather differs from the reference"
    res["reference_checked"] = True
    print(json.dumps(res))
    if out_json:
        with open(out_json, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
