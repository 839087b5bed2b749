#!/usr/bin/env python
"""bench.py -- k-mer count+feature throughput (Gbp/s) of the dense hot path.

Workload (BASELINE.json configs[1], "C2"): 100 synthetic fungal-sized genomes
(12-40 Mbp, 8-30 records, upper-case 80-column FASTA), k = 1..12 dense histograms
+ frequency rows, on each GPU (weak scaling: every rank counts its own 100 genomes,
no data-path collective).

One "step" = one pass of the hot path over the whole batch.  Printed JSON line:
  value     whole-job Gbp/s with the FASTA bytes already resident in HBM
  e2e       the same through the host-buffer C-ABI call (pinned host FASTA -> H2D ->
            count -> D2H of counts + frequencies), copies inside the timed region
  roofline  the dominant kernel (count_kernel) against the measured HBM copy peak
  cpu_baseline  the oracle port timed on this box's host cores on a bounded sample

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

K_LIST = list(range(1, 13))
METRIC = "kmer_count_feature_throughput"
UNIT = "Gbp/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--genomes", type=int, default=100, help="genomes per GPU")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink genome sizes (debug only)")
    ap.add_argument("--k", default=None, help="comma-separated k list (default 1..12)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-genomes", type=int, default=None)
    ap.add_argument("--extras", default="on", choices=["on", "off"],
                    help="also time the other BASELINE configs (c3, c4_strong, c5_sparse: bench_extras.py)")
    ap.add_argument("--extra-scale", type=float, default=1.0, help="shrink the extras' genomes (debug only)")
    ap.add_argument("--c5-single", action="store_true", help="run c5_sparse on one GPU too (> 100 GB of workspace)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0's genomes) to DIR/<name>.npy: a fixed sample "
                         "of the count and frequency rows, and the window totals")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    return args


# ------------------------------------------------------------------ workload
def genome_shape(i, scale):
    """Record lengths of C2 genome i (SURVEY 8d: seeds 1000+i, 12-40 Mbp, 8..30 records)."""
    from kmerml_b200 import synth
    rng = np.random.default_rng(1000 + i)
    total = int(rng.integers(12_000_000, 40_000_000) * scale)
    nrec = int(rng.integers(8, 31))
    return synth.split_lengths(max(total, nrec + 1), nrec, rng)


def make_genome_gpu(i, scale, device, torch):
    """FASTA bytes of genome i generated on the GPU (uniform ACGT, 80 columns)."""
    lens = genome_shape(i, scale)
    gen = torch.Generator(device=device)
    gen.manual_seed(1000 + i)
    lut = torch.tensor([65, 67, 71, 84], dtype=torch.uint8, device=device)
    nl = torch.tensor([10], dtype=torch.uint8, device=device)
    parts = []
    for r, L in enumerate(lens):
        hdr = f">chr{r + 1} synthetic genome {i} record len={L}\n".encode()
        parts.append(torch.tensor(list(hdr), dtype=torch.uint8, device=device))
        seq = lut[torch.randint(0, 4, (L,), device=device, generator=gen)]
        full = (L // 80) * 80
        if full:
            body = seq[:full].view(-1, 80)
            parts.append(torch.cat([body, nl.expand(body.shape[0], 1)], dim=1).reshape(-1))
        if L > full:
            parts.append(seq[full:])
            parts.append(nl)
    return torch.cat(parts), sum(lens)


# ------------------------------------------------------------------ --dump-outputs
DUMP_BINS_PER_K = 4096
DUMP_BUDGET_BYTES = 48 << 20          # what --dump-outputs writes stays below 64 MB


def dump_selection(n_gen, ks):
    """(genome rows, row columns) that --dump-outputs writes: every bin of a level with at most 4096 bins and a seeded
    sample of 4096 bins of each larger one, for every genome unless that would exceed the budget (then a seeded
    sample of the genomes).  It depends on the arguments only, so two builds write the same entries."""
    from kmerml_b200 import engine
    lay, _ = engine.row_layout(ks)
    cols = []
    for k, (off, n) in lay.items():
        if n <= DUMP_BINS_PER_K:
            cols.append(np.arange(off, off + n))
        else:
            cols.append(off + np.sort(np.random.default_rng(k).choice(n, DUMP_BINS_PER_K, replace=False)))
    cols = np.concatenate(cols)
    per_genome = cols.size * (8 + 4) + len(ks) * 8           # float64 counts, float32 frequencies, float64 totals
    n_rows = max(1, min(n_gen, DUMP_BUDGET_BYTES // per_genome))
    if n_rows == n_gen:
        return np.arange(n_gen), cols
    return np.sort(np.random.default_rng(n_gen).choice(n_gen, n_rows, replace=False)), cols


def dump_sample(counts, freq, totals, ks, torch):
    """The selected entries of the count rows (uint32 as float64), frequency rows (float32) and window totals
    (float64), copied to host numpy arrays."""
    rows, cols = dump_selection(counts.shape[0], ks)
    r = torch.from_numpy(rows).to(counts.device)
    c = torch.from_numpy(cols).to(counts.device)
    pick = lambda t: t.index_select(1, c).index_select(0, r)      # columns first: never copies whole rows
    return {"counts": (pick(counts).to(torch.int64) & 0xFFFFFFFF).cpu().numpy().astype(np.float64),
            "freq": pick(freq).cpu().numpy().astype(np.float32),
            "totals": totals.index_select(0, r).cpu().numpy().astype(np.float64)}


def write_dump(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def wait_ready(self, timeout=8.0):
        """Block until nvidia-smi has printed its first sample (its start-up can take seconds on a cold box)."""
        t = time.time()
        while self.proc and not self.lines and time.time() - t < timeout and self.proc.poll() is None:
            time.sleep(0.02)

    def samples_between(self, t0, t1):
        return sum(1 for ts, _ in self.lines if t0 - 0.05 <= ts <= t1 + 0.05)

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, cmax = float(f[1]), float(f[2])
            except ValueError:
                continue
            mx.append(cmax)
            if t0 - 0.05 <= ts <= t1 + 0.05:
                sm.append(clk)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": float(max(mx)) if mx else None,
                    "reasons": ["no nvidia-smi sample fell into the loaded window"], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------ CPU legs
def oracle_seconds(data, ks):
    import oracle
    t0 = time.perf_counter()
    oracle.count_dense_multi(data, ks)
    return time.perf_counter() - t0


def _unmodified_reference_worker(job):
    """(child process) the UNMODIFIED reference from baseline/_ref under the Bio.SeqIO shim: one genome, k list."""
    fasta_path, out_dir, ks = job
    sys.path.insert(0, os.path.join(ROOT, "tests", "_ref"))          # Bio.SeqIO shim (biopython is not installable offline)
    sys.path.insert(1, os.path.join(ROOT, "baseline", "_ref"))
    import contextlib
    import io
    from kmerml.kmers.generate import KmerExtractor
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        KmerExtractor(output_dir=out_dir, compress=False).extract_kmers_from_fasta(fasta_path, list(ks))
    return time.perf_counter() - t0


def time_unmodified_reference(ks, cores, bases_per_genome=300_000):
    """The unmodified Python reference (pip-installed into baseline/_ref from the reference tree, see DESIGN.md) on
    `cores` processes, one small C2-shaped genome each; None when baseline/_ref is absent."""
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "kmerml")):
        return None
    import multiprocessing as mp
    import tempfile
    from kmerml_b200 import synth
    with tempfile.TemporaryDirectory() as td:
        jobs = []
        for i in range(cores):
            g = synth.fasta_bytes([bases_per_genome // 2, bases_per_genome - bases_per_genome // 2], seed=5000 + i)
            path = os.path.join(td, f"GCF_90000{i:04d}_1.fa")
            g.tofile(path)
            jobs.append((path, os.path.join(td, f"out{i}"), ks))
        t0 = time.perf_counter()
        with mp.get_context("spawn").Pool(cores) as pool:
            pool.map(_unmodified_reference_worker, jobs)
        wall = time.perf_counter() - t0
    total = cores * bases_per_genome
    return {"value": total / wall / 1e9, "unit": UNIT, "cores": cores, "kind": "reference",
            "sample": f"{cores} genomes of {bases_per_genome} bp, k={ks[0]}..{ks[-1]}, KmerExtractor.extract_kmers_from_fasta of the "
                      f"unmodified reference (baseline/_ref) in {cores} processes, wall {wall:.1f} s incl. process start-up"}


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port: the reference itself is
    pure Python + biopython and cannot travel to the GPU box) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import oracle
    from concurrent.futures import ThreadPoolExecutor
    from kmerml_b200 import synth
    oracle.build()
    ks = [int(x) for x in args.k.split(",")] if args.k else K_LIST
    cores = max(1, min(os.cpu_count() or 1, 64))
    # The first 2 x `cores` genomes of the C2 batch at their real sizes (12-40 Mbp), largest first so that the threads
    # finish together (~17 s per step on 16 threads); only a run with many steps shrinks them so that the whole run
    # stays near two minutes.
    n_ref = 2 * cores
    est_step_s = 17.0 * args.scale
    frac = min(1.0, 130.0 / max((args.steps + args.warmup) * est_step_s, 1e-9))
    scale = args.scale * frac
    genomes = sorted((synth.config2_genome(i, scale=scale) for i in range(n_ref)), key=len, reverse=True)
    datas = [g.tobytes() for g in genomes]
    nbases = sum(int(oracle.count_dense(d, 1).sum()) for d in datas)

    def step():
        with ThreadPoolExecutor(cores) as ex:
            list(ex.map(lambda d: oracle.count_dense_multi(d, ks), datas))

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    value = nbases / dt / 1e9
    sample = (f"the first {n_ref} genomes of the C2 batch (same generator and size distribution, "
              f"{'full size' if frac >= 1.0 else f'lengths x {frac:.2f}'}: mean {nbases / n_ref / 1e6:.1f} Mbp), "
              f"k={ks[0]}..{ks[-1]}, {cores} threads taking whole genomes, largest first (ctypes releases the GIL)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "C2 sample on host cores: " + sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "oracle C port of kmerml/kmers/generate.py:36-58 (the conservative baseline: ~100x faster than the Python it "
                "restates); the unmodified Python reference measured 0.034 Mbp/s on one core for k=1..12 in the build "
                "container (tests/golden/ref_timing.json) and is timed on this box in `unmodified_reference`",
    }
    try:
        line["unmodified_reference"] = time_unmodified_reference(ks, cores)
    except Exception as exc:                                      # report, never fake
        line["unmodified_reference"] = {"error": repr(exc)[:200]}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------ GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from kmerml_b200 import _lib, engine
    from kmerml_b200 import dist as kdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    numa_node = kdist.bind_to_gpu_numa_node(local) if world > 1 else None     # before any pinned allocation
    device = torch.device("cuda", local)
    if world > 1:
        import datetime
        # (a rank that fails alone must not keep the others in a collective for NCCL's default ten minutes)
        dist.init_process_group("nccl", device_id=device, timeout=datetime.timedelta(seconds=240))
    ks = [int(x) for x in args.k.split(",")] if args.k else K_LIST
    n_gen = args.genomes

    # ---- synthetic batch, generated on the GPU, resident in HBM
    parts, offs, nbases = [], [0], 0
    for i in range(n_gen):
        t, nb = make_genome_gpu(rank * 1000 + i, args.scale, device, torch)
        parts.append(t)
        offs.append(offs[-1] + t.numel())
        nbases += nb
    fasta = torch.cat(parts)
    sizes = [p.numel() for p in parts]
    del parts
    torch.cuda.synchronize()
    _, row_len = engine.row_layout(ks)
    counts = torch.empty((n_gen, row_len), dtype=torch.int32, device=device)
    freq = torch.empty((n_gen, row_len), dtype=torch.float32, device=device)
    totals = torch.zeros((n_gen, len(ks)), dtype=torch.int64, device=device)
    ctx = _lib.context(local)
    # host threads that widen the narrow D2H format: this rank's share of the cores
    ctx.set_host_threads(max(2, min(8, (os.cpu_count() or 2) // max(int(os.environ.get("LOCAL_WORLD_SIZE", world)), 1))))

    def step():
        engine.count_dense_device(fasta, offs, ks, out_counts=counts, out_freq=freq, out_totals=totals)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks / throttle reasons are sampled under load: from the first warm-up step to the end of the timed region
    sampler = ClockSampler(local)
    sampler.start()
    sampler.wait_ready()
    time.sleep(0.05)
    t_load = time.time()
    for _ in range(max(args.warmup, 0)):
        step()
    barrier()
    ctx.profile_enable(True)
    ctx.profile_read(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    t0 = time.time()
    e0.record()
    marks[0].record()
    for i in range(args.steps):
        step()
        marks[i + 1].record()
    e1.record()
    barrier()
    t1 = time.time()
    dumped = dump_sample(counts, freq, totals, ks, torch) if args.dump_outputs and rank == 0 else None
    ms = e0.elapsed_time(e1)
    step_ms = sorted(marks[i].elapsed_time(marks[i + 1]) for i in range(args.steps))
    prof = ctx.profile_read(reset=True)
    ctx.profile_enable(False)
    t_clk = t1
    if sampler.samples_between(t_load, t1) < 3:
        # the warm-up + timed steps were over before nvidia-smi sampled three times: keep the same load running
        # (untimed steps) until it has, so that the clocks are still read under this workload
        t_more = time.time()
        while sampler.samples_between(t_load, time.time()) < 3 and time.time() - t_more < 1.0:
            step()
            torch.cuda.synchronize()
        t_clk = time.time()
    clocks = sampler.stop(t_load, t_clk)
    clocks["window"] = "warm-up + timed steps" + ("" if t_clk == t1 else " + untimed steps of the same load until 3 samples")
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        nb_all = torch.tensor([nbases], dtype=torch.float64, device=device)
        dist.all_reduce(nb_all, op=dist.ReduceOp.SUM)
        total_bases = float(nb_all.item())
    else:
        total_bases = float(nbases)
    ms_per_step = ms / args.steps
    value = total_bases / (ms_per_step * 1e-3) / 1e9

    # ---- parity gates on the measured outputs (oracle = checker only)
    parity = {}
    lay, _ = engine.row_layout(ks)
    u64 = lambda t: t.to(torch.int64) & 0xFFFFFFFF
    ok_tot = True
    for ki, k in enumerate(ks):
        off, n = lay[k]
        s = torch.stack([u64(counts[g, off:off + n]).sum() for g in range(n_gen)])
        ok_tot &= bool(torch.equal(s, totals[:, ki]))
    parity["sum_counts_equals_windows"] = ok_tot
    if 12 in ks and 11 in ks:
        # marginal property: c11[p] >= sum_b c12[4p+b], equality except for run-end tails
        o12, n12 = lay[12]
        o11, n11 = lay[11]
        m = u64(counts[0, o12:o12 + n12]).view(-1, 4).sum(dim=1)
        d = u64(counts[0, o11:o11 + n11]) - m
        parity["marginal_k12_to_k11_tails"] = int(d.sum().item())
        ok_tot &= bool((d >= 0).all().item())
    cpu_baseline = None
    if rank == 0 and not args.no_cpu:
        import oracle
        oracle.build()
        gi = int(np.argmin(sizes))
        data = fasta[offs[gi]:offs[gi + 1]].cpu().numpy().tobytes()
        t_cpu = time.perf_counter()
        ref = oracle.count_dense_multi(data, ks)
        t_cpu = time.perf_counter() - t_cpu
        exact = True
        for k in ks:
            off, n = lay[k]
            got = counts[gi, off:off + n].cpu().numpy().view(np.uint32).astype(np.uint64)
            exact &= bool(np.array_equal(got, ref[k]))
        parity["oracle_bit_exact_genome"] = gi
        parity["oracle_bit_exact"] = exact
        nb_g = int(ref[1].sum())
        cpu_baseline = {"value": nb_g / t_cpu / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
                        "sample": f"smallest genome of the batch ({nb_g / 1e6:.1f} Mbp), k={ks[0]}..{ks[-1]}, "
                                  f"oracle C port, 1 thread, {t_cpu:.1f} s"}
        if not exact or not ok_tot:
            print(json.dumps({"error": "parity gate failed", "parity": parity}))
            raise SystemExit(3)

    # ---- roofline of the dominant kernel, live CUDA-event timing (kmerml_profile_read)
    peak, peak_src = measured_peak()
    kmax = max(ks)
    F = float(fasta.numel())
    out_bytes = n_gen * row_len * 8.0                          # sum_k 4^k * (4 + 4) per genome
    step_alg = F + out_bytes                                   # SURVEY 8d: B_alg per step
    per_step = {k: prof[k] / args.steps for k in prof if k.startswith("ms_")}
    # algorithmic bytes each kernel family is responsible for, per step
    if per_step.get("ms_partition", 0) > 0:
        alg = {"ms_partition": F,                               # one read of the FASTA bytes
               "ms_bucket": n_gen * sum(4 ** k for k in ks if k >= max(kmax - 7, min(ks))) * 8.0,
               "ms_cascade": n_gen * sum(4 ** k for k in ks if k < max(kmax - 7, min(ks))) * 4.0,
               "ms_finalize": n_gen * sum(4 ** k for k in ks if k < max(kmax - 7, min(ks))) * 4.0}
        names = {"ms_partition": "partition_kernel", "ms_bucket": "bucket_kernel",
                 "ms_cascade": "cascade_kernel", "ms_finalize": "finalize_low_kernel"}
    else:
        alg = {"ms_count": F + n_gen * (4 ** kmax) * 4.0,       # FASTA read + the top-level count vector
               "ms_cascade": n_gen * sum(4 ** k for k in ks if k < kmax) * 4.0,
               "ms_finalize": n_gen * row_len * 4.0}
        names = {"ms_count": "count_kernel", "ms_cascade": "cascade_kernel", "ms_finalize": "finalize_kernel"}
    kernels = []
    for key, nm in names.items():
        t = per_step.get(key, 0.0) * 1e-3
        if t > 0:
            kernels.append({"kernel": nm, "ms_per_step": t * 1e3, "alg_bytes_per_step": alg[key],
                            "achieved": alg[key] / t / 1e9, "frac": alg[key] / t / 1e9 / peak,
                            "share_of_step": t * 1e3 / ms_per_step})
    dom = max(kernels, key=lambda d: d["ms_per_step"]) if kernels else None
    n_dom_launch = max(int(prof["count_launches"]) // max(args.steps, 1), 1) if dom and dom["kernel"] in ("partition_kernel", "count_kernel") else 1
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tj = json.load(f)
        if dom and dom["kernel"] in tj:
            # measured DRAM bytes per algorithmic byte (one ncu --set full capture on a 24-genome subset of this
            # workload), scaled to this launch
            traffic = tj[dom["kernel"]]["ratio"] * dom["alg_bytes_per_step"] / n_dom_launch
            traffic_src = tj["source"]
    except Exception:
        pass
    roofline = {
        "bound": "hbm", "kernel": dom["kernel"] if dom else None,
        "achieved": dom["achieved"] if dom else 0.0, "peak": peak, "unit": "GB/s",
        "frac": dom["frac"] if dom else 0.0, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
        "alg_bytes_per_launch": (dom["alg_bytes_per_step"] / n_dom_launch) if dom else None,
        "avg_launch_ms": (dom["ms_per_step"] / n_dom_launch) if dom else None,
        "kernel_share_of_step": dom["share_of_step"] if dom else None,
        "step_frac": step_alg / (ms_per_step * 1e-3) / 1e9 / peak, "step_alg_bytes": step_alg,
        "kernels": kernels,
    }
    if dom and dom["kernel"] == "partition_kernel":
        # the longest kernel of the step is not the HBM-bound one: say so, and put the HBM-bound kernel beside it
        bk = next((k for k in kernels if k["kernel"] == "bucket_kernel"), None)
        roofline["note"] = ("partition_kernel (the longest kernel) is bound by the shared-memory pipe, not by HBM (ncu r02: L1TEX "
                            "76-82 % busy, DRAM 16 %): its algorithmic bytes are only the FASTA read.  The HBM-bound kernel of the "
                            "step is bucket_kernel (87 % of the step's algorithmic bytes); step_frac is the whole step")
        if bk:
            btr = None
            try:
                btr = tj["bucket_kernel"]["ratio"] * bk["alg_bytes_per_step"]
            except Exception:
                pass
            roofline["hbm_bound_kernel"] = {"kernel": "bucket_kernel", "achieved": bk["achieved"], "frac": bk["frac"],
                                            "avg_launch_ms": bk["ms_per_step"], "alg_bytes_per_launch": bk["alg_bytes_per_step"],
                                            "traffic": btr}

    # ---- end to end through the host-buffer C-ABI call
    e2e = None
    if not args.no_e2e:
        n_e2e = args.e2e_genomes or n_gen
        try:
            avail = 0
            with open("/proc/meminfo") as f:
                for line in f:
                    if line.startswith("MemAvailable"):
                        avail = int(line.split()[1]) * 1024
            need = lambda n: sum(sizes[:n]) + n * row_len * 4
            while n_e2e > 1 and need(n_e2e) * 3 > avail:
                n_e2e //= 2
            host_bufs = [torch.empty(sizes[i], dtype=torch.uint8, pin_memory=True) for i in range(n_e2e)]
            for i in range(n_e2e):
                host_bufs[i].copy_(fasta[offs[i]:offs[i + 1]])
            karr = np.asarray(ks, dtype=np.int32)
            row_bytes = int(_lib.load().kmerml_compact_row_bytes(karr.ctypes.data, len(ks)))
            hrows = torch.empty((n_e2e, row_bytes), dtype=torch.uint8, pin_memory=True)
            hf = freq[:n_e2e]          # the feature matrix stays resident in HBM (what the ML stage consumes)
            ht = torch.zeros((n_e2e, len(ks)), dtype=torch.int64, pin_memory=True)
            torch.cuda.synchronize()
            n_e2e_steps = args.steps

            def timed(fn):
                fn()                                              # warm-up (allocates the slots)
                barrier()
                t_a = time.perf_counter()
                for _ in range(n_e2e_steps):
                    res = fn()
                torch.cuda.synchronize()
                dt = (time.perf_counter() - t_a) / n_e2e_steps
                if world > 1:
                    t = torch.tensor([dt], dtype=torch.float64, device=device)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    dt = float(t.item())
                return dt, res

            def whole_job(x):
                t = torch.tensor([float(x)], dtype=torch.float64, device=device)
                if world > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.SUM)
                return float(t.item())

            # (1) the headline: the host result in the form it crosses PCIe in (lossless: one byte per bin for
            # k >= 10 + exception list, uint32 for k < 10; widened per (genome, k) on access)
            dt, comp = timed(lambda: engine.count_dense_host(host_bufs, ks, device=device, out_rows=hrows, out_freq=hf,
                                                             out_totals=ht, compact=True))
            nb_e2e = whole_job(sum(int(x) for x in ht[:, 0].tolist()))        # k=1 windows = valid bases
            gi_chk = [0, n_e2e // 2, n_e2e - 1]
            same = all(np.array_equal(comp.counts_numpy(g, k), counts[g, lay[k][0]:lay[k][0] + lay[k][1]].cpu().numpy().view(np.uint32))
                       for g in gi_chk for k in ks)
            e2e = {"value": nb_e2e / dt / 1e9, "unit": UNIT,
                   "h2d_bytes_per_step": int(whole_job(sum(sizes[:n_e2e]))),
                   "d2h_bytes_per_step": int(whole_job(sum(int(_lib.load().kmerml_compact_row_used_bytes(
                       karr.ctypes.data, len(ks), hrows[g].data_ptr())) for g in range(n_e2e)) + n_e2e * len(ks) * 8)),
                   "genomes": n_e2e, "ms_per_step": dt * 1e3, "matches_device_path": bool(same),
                   "matches_checked_genomes": gi_chk, "exception_list_overflows": len(comp._wide), "numa_node": numa_node,
                   "api": "kmerml_count_dense_host_compact (engine.count_dense_host(compact=True)): pinned host FASTA -> H2D -> "
                          "count + frequency rows -> D2H of the count rows in the compact lossless form (1 byte per bin for "
                          "k >= 10 -- 4 bits where the genome's mean count is <= 5 -- + exception list, uint32 for k < 10) and the window totals; rows are widened to uint32 per "
                          "(genome, k) on access (kmerml_compact_expand); the float32 frequency matrix is computed per step "
                          "and left resident in HBM (KMERML_FLAG_FREQ_ON_DEVICE)"}
            del comp
            # (2) beside it: the same call delivering uint32 rows in host memory (narrow wire format widened by host
            # threads inside the call); bound by the host's memory write bandwidth (~60 GB/s measured on this pool)
            hc = torch.empty((n_e2e, row_len), dtype=torch.int32, pin_memory=True)
            dt32, _ = timed(lambda: engine.count_dense_host(host_bufs, ks, device=device, out_counts=hc, out_freq=hf, out_totals=ht))
            same32 = torch.equal(hc, counts[:n_e2e].cpu())
            e2e["uint32_rows"] = {"value": nb_e2e / dt32 / 1e9, "unit": UNIT, "ms_per_step": dt32 * 1e3,
                                  "host_bytes_written_per_step": int(whole_job(n_e2e * row_len * 4)),
                                  "matches_device_path": bool(same32),
                                  "api": "kmerml_count_dense_host: same pipeline, the rows widened to uint32 in the caller's host "
                                         "buffer by the library's host threads"}
            del hc
        except Exception as exc:                                  # report, never fake
            e2e = {"value": None, "unit": UNIT, "error": repr(exc)[:300]}

    extras = {}
    if args.extras == "on":
        import bench_extras
        del counts, freq, totals, fasta
        if not args.no_e2e:
            host_bufs = hrows = hf = ht = None
        torch.cuda.empty_cache()
        extras = bench_extras.run_extras(args, torch, dist, device, rank, world)
    if world > 1:
        dist.barrier()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "ms_per_step_best": step_ms[0],
            "ms_per_step_median": float(np.median(step_ms)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"C2: {n_gen} synthetic fungal-sized genomes per GPU (12-40 Mbp x {args.scale:g}), "
                                   f"k={ks[0]}..{ks[-1]} dense histograms + frequency rows",
                       "genomes_per_gpu": n_gen, "k_list": ks, "bases_per_gpu": nbases,
                       "fasta_bytes_per_gpu": int(F),
                       "l2_policy": "inputs (GBs) and outputs far exceed the 126 MB L2; no explicit flush"},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e,
            "gpu_launches": int(prof["launches"]), "clocks": clocks, "parity": parity,
        }
        line.update(extras)
        if dumped:
            write_dump(args.dump_outputs, dumped)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
