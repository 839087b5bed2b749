"""Gather of scaled sketches (engine.fmh_gather_device) on two workloads, k = 21, canonical, scale 1000, threshold 50
hashes (the 50 kbp default of ml.sketch.gather).  References: n_ref genomes of 5 Mbp (synth.config3_genome) plus
n_ref / 4 mutants (0.5, 1, 2 or 5 %) of the first n_ref / 8, so many hashes sit in several references.
    A: one metagenome-like query: 100 of the references (a third of them mutated 1 %) and 20 Mbp of novel sequence.
    B: 1000 MAG-like queries, each 1-3 Mbp cut from one or two references and mutated 0.5 %.
Sketching happens once, outside the timed window.  Per workload: the query x reference comparison that gather
prefetches (fmh_compare_device), the candidate references and the rounds, the whole gather call, and the time per
round derived as (gather - comparison) / rounds; then an exact check of sampled queries against the numpy reference
of the tests, and the GPU's name and power limit.  Times are CUDA-event times of single calls after a warm-up call:
min / median / max over the repetitions.
    python tools/time_fmh_gather.py [n_ref] [--json OUT]"""
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

K, SEED, SCALE, THRESHOLD = 21, 42, 1000, 50
RATES = (0.005, 0.01, 0.02, 0.05)
N_REF = 2000
ACGT = np.frombuffer(b"ACGT", np.uint8)


def _mutate(g, p, rng):
    """A copy of FASTA text `g` with a fraction p of its bases (past the first header) substituted."""
    g = g.copy()
    body = np.nonzero(np.isin(g, ACGT))[0]
    body = body[body > 80]
    hit = body[rng.random(body.size) < p]
    g[hit] = ACGT[(np.searchsorted(ACGT, g[hit]) + rng.integers(1, 4, hit.size)) % 4]
    return g


def _reference(i, n_ref):
    """Reference i: genome i for i < n_ref, then mutant j = i - n_ref of genome j % (n_ref // 8)."""
    if i < n_ref:
        return synth.config3_genome(i)
    j = i - n_ref
    return _mutate(synth.config3_genome(j % (n_ref // 8)), RATES[j * len(RATES) // (n_ref // 4)],
                   np.random.default_rng(10_000 + j))


def _ref_batch(args):
    return [_reference(i, args[2]) for i in range(args[0], args[1])]


def _sources_a(n_ref):
    return list(range(0, n_ref, n_ref // 100))[:100]


def _query_a_part(args):
    i, src = args
    g = synth.config3_genome(src)
    return _mutate(g, 0.01, np.random.default_rng(20_000 + i)) if i % 3 == 0 else g


def _query_b(args):
    """MAG-like query q: 1-3 Mbp of FASTA text cut from one or two references, mutated 0.5 %."""
    q, n_ref = args
    rng = np.random.default_rng(30_000 + q)
    total = int(rng.integers(1_000_000, 3_000_001))
    srcs = rng.choice(n_ref, int(rng.integers(1, 3)), replace=False)
    parts = [np.frombuffer(b">mag%d\n" % q, np.uint8)]
    for s in srcs:
        g = synth.config3_genome(int(s))
        n = total // len(srcs)
        a = int(rng.integers(100, g.size - n))
        parts += [g[a:a + n], np.frombuffer(b"\n>part\n", np.uint8)]
    return _mutate(np.concatenate(parts), 0.005, rng)


def timed(f, reps):
    """[min, median, max] ms of `reps` calls, each between two events."""
    f()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        f()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    ms.sort()
    return [round(ms[0], 3), round(ms[len(ms) // 2], 3), round(ms[-1], 3)]


def _host(sk):
    h = sk.hashes.cpu().numpy().view(np.uint64)
    o = sk.offsets.cpu().numpy()
    return [h[o[g]:o[g + 1]] for g in range(len(sk))]


def _sketch(genomes):
    buf, offs = synth.pack(genomes)
    return engine.fmh_batch_device(torch.from_numpy(buf).cuda(), offs, K, scale=SCALE, seed=SEED)


def _workload(name, q, refs, ref_host, reps, sample):
    import gather_oracle
    res = {}
    res["compare_ms"] = timed(lambda: engine.fmh_compare_device(q, refs, want_intersections=True), reps)
    x = engine.fmh_compare_device(q, refs, want_intersections=True)[1]
    res["candidates"] = int((x >= THRESHOLD).any(0).sum())
    res["gather_ms"] = timed(lambda: engine.fmh_gather_device(q, refs, threshold=THRESHOLD), reps)
    out = engine.fmh_gather_device(q, refs, threshold=THRESHOLD)
    n = out.n_matches.cpu().numpy()
    # every round ends in a select; the last one finds nothing unless a query reached max_matches
    res["rounds"] = int(n.max()) + (1 if int(n.max()) < out.reference.shape[1] else 0)
    res["ms_per_round_derived"] = round((res["gather_ms"][1] - res["compare_ms"][1]) / res["rounds"], 4)
    res["matches_total"] = int(n.sum())
    res["matches_per_query_max"] = int(n.max())
    res["query_hashes_total"] = int(q.offsets[-1])
    qh = _host(q)
    cols = [t.cpu().numpy() for t in (out.reference, out.unique, out.intersect, out.remaining)]
    for i in sample:
        want = gather_oracle.gather_one(qh[i], ref_host, THRESHOLD)
        got = [(int(cols[0][i, t]), int(cols[1][i, t]), int(cols[2][i, t]), int(cols[3][i, t])) for t in range(n[i])]
        assert got == want, f"{name}: query {i} differs from the reference"
    res["reference_checked"] = list(sample)
    return res


def main():
    argv = sys.argv[1:]
    out_json = None
    if "--json" in argv:
        i = argv.index("--json")
        out_json = argv[i + 1]
        del argv[i:i + 2]
    n_ref = int(argv[0]) if argv else N_REF
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    n_all = n_ref + n_ref // 4
    res = {"gpu": gpu, "k": K, "scale": SCALE, "threshold_hashes": THRESHOLD, "references": n_all}
    t0 = time.perf_counter()
    parts = []
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        step = 250
        for b in range(0, n_all, step):                 # sketched in batches, so host memory stays small
            chunk = [(a, min(a + 8, b + step, n_all), n_ref) for a in range(b, min(b + step, n_all), 8)]
            parts.append(_sketch([g for gs in pool.map(_ref_batch, chunk) for g in gs]))
        refs = engine.concat_scaled_sketches(*parts)
        del parts
        part_a = pool.map(_query_a_part, list(enumerate(_sources_a(n_ref))))
        qa = _sketch([np.concatenate(part_a + [synth.fasta_bytes([20_000_000], seed=77)])])
        del part_a
        qb = _sketch(pool.map(_query_b, [(q, n_ref) for q in range(1000)], chunksize=8))
    res["prepare_s"] = round(time.perf_counter() - t0, 1)
    res["reference_hashes_total"] = int(refs.offsets[-1])
    ref_host = _host(refs)
    res["A"] = _workload("A", qa, refs, ref_host, 5, [0])
    res["B"] = _workload("B", qb, refs, ref_host, 5, [0, 1, 500, 999])
    print(json.dumps(res))
    if out_json:
        with open(out_json, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
