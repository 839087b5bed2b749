"""Scaled (FracMinHash) sketches on a C3-shaped workload: 1000 genomes of 5 Mbp (synth.config3_genome), k = 21,
canonical, scale 1000.  Reports the sketch batch, the 1000 x 1000 containment matrix, a skewed comparison of the 1000
genomes against one 3.1 Gbp reference (the first 620 genomes concatenated as one pangenome file), the same
1000 x 1000 comparison at scale 100, and the GPU's name and power limit; ends with an exact check of sampled sketches
and intersections against the numpy reference of the tests.  Times are CUDA-event times of single calls after a
warm-up call: min / median / max over the repetitions.
    python tools/time_fracminhash.py [n_genomes] [--json OUT]"""
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

K, SEED = 21, 42
PANGENOME_GENOMES = 620                               # 620 x 5 Mbp = 3.1 Gbp


def _genome(i):
    return synth.config3_genome(i)


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
    t0 = time.perf_counter()
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        genomes = pool.map(_genome, range(n), chunksize=4)
    buf, offs = synth.pack(genomes)
    res = {"gpu": gpu, "n_genomes": n, "bytes": int(buf.size), "k": K, "canonical": True,
           "generate_s": round(time.perf_counter() - t0, 1)}
    fasta = torch.from_numpy(buf).cuda()

    batch = lambda scale: engine.fmh_batch_device(fasta, offs, K, scale=scale, seed=SEED)   # noqa: E731
    res["fmh_batch_scale1000_ms"] = timed(lambda: batch(1000), 5)
    res["fmh_batch_gbp_per_s"] = round(buf.size / res["fmh_batch_scale1000_ms"][1] / 1e6, 1)
    sk = batch(1000)
    res["hashes_per_genome_scale1000"] = round(float(sk.sizes().double().mean()), 1)
    res["compare_nxn_scale1000_ms"] = timed(lambda: engine.fmh_compare_device(sk, None, "containment"), 5)
    full, inter = engine.fmh_compare_device(sk, None, "containment", out_dtype=torch.float64, want_intersections=True)

    # skewed: every genome against one 3.1 Gbp pangenome file made of the first PANGENOME_GENOMES genomes
    n_pan = min(PANGENOME_GENOMES, n)
    pan = torch.from_numpy(buf[:offs[n_pan]]).cuda()
    ref = engine.fmh_batch_device(pan, [0, offs[n_pan]], K, scale=1000, seed=SEED)
    res["pangenome_bytes"] = int(offs[n_pan])
    res["pangenome_hashes"] = int(ref.sizes()[0])
    res["compare_skewed_nx1_ms"] = timed(lambda: engine.fmh_compare_device(sk, ref, "containment"), 5)
    skew, skew_x = engine.fmh_compare_device(sk, ref, "containment", out_dtype=torch.float64, want_intersections=True)
    res["skewed_contained_exactly"] = int((skew[:n_pan, 0] == 1.0).sum())
    del pan
    res["fmh_batch_scale100_ms"] = timed(lambda: batch(100), 3)
    sk100 = batch(100)
    res["hashes_per_genome_scale100"] = round(float(sk100.sizes().double().mean()), 1)
    res["compare_nxn_scale100_ms"] = timed(lambda: engine.fmh_compare_device(sk100, None, "containment"), 3)
    x100 = engine.fmh_compare_device(sk100, None, "containment", want_intersections=True)[1]

    # exact check of a sample against the numpy reference of the tests
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import fmh_oracle
    hs, hs100, hr = _host(sk), _host(sk100), _host(ref)[0]
    x, x100, sx = inter.cpu().numpy(), x100.cpu().numpy(), skew_x.cpu().numpy()
    sample = sorted(set(np.random.default_rng(0).choice(n, min(n, 6), replace=False).tolist()) | {0, n - 1})
    for g in sample:
        want = fmh_oracle.fmh_sketch(genomes[g].tobytes(), K, 1000, SEED, True)
        assert np.array_equal(hs[g], want), f"genome {g}: sketch differs from the reference"
        want100 = fmh_oracle.fmh_sketch(genomes[g].tobytes(), K, 100, SEED, True)
        assert np.array_equal(hs100[g], want100), f"genome {g}: scale-100 sketch differs from the reference"
        for j in sample:
            assert x[g, j] == np.intersect1d(want, hs[j]).size, (g, j)
            assert x100[g, j] == np.intersect1d(want100, hs100[j]).size, (g, j)
        assert sx[g, 0] == np.intersect1d(want, hr).size, g
    res["reference_checked"] = sample
    print(json.dumps(res))
    if out_json:
        with open(out_json, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
