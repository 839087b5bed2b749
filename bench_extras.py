"""bench_extras.py -- the other BASELINE.json configurations, timed on the device next to bench.py's C2 line.

  c3          1000 synthetic bacterial-sized genomes (5 Mbp, GC 0.30-0.70), k = 8 count rows, sharded over the
              ranks, rows all-gathered, genome x genome cosine distances in row blocks (tensor cores), gathered
  c4_strong   ONE 3.1 Gbp genome, k = 12 canonical: byte ranges with k-1 look-back, one reduce-scatter of the
              dense rows to owner slices (strong scaling: the genome is the same at every N)
  c5_sparse   the same genome with N runs, k = 21 canonical: windows emitted per byte range and grouped by owner,
              all-to-all by key range, one sort + reduce per rank

Every section: W warm-up + K timed steps between barriers, CUDA events on the launching stream, MAX over ranks;
bit-exactness against the single-GPU result (c4 at full size on every rank's slice, c5 on a bounded prefix plus
full-size invariants), oracle spot checks (the oracle is the checker only).  Inputs are generated on the GPU.
"""
import os
import time

import numpy as np

HUMAN_MBP = [248, 242, 198, 190, 181, 171, 159, 145, 138, 133, 135, 133, 114, 107, 102, 90, 83, 80, 58, 64, 46, 50, 156, 57]


def _ascii_from_codes(c):
    """uint8 codes 0..3 (A C G T) -> ASCII, in uint8 arithmetic (no int64 index tensor)."""
    hi = c >> 1
    return 65 + 2 * c + 2 * hi + 11 * (hi & c)


def gpu_fasta(torch, device, rec_lens, seed, name, gc=None, n_runs=False):
    """FASTA bytes (upper case, 80 columns) of one synthetic genome, generated on the GPU.
    gc: G+C fraction (None: uniform); n_runs: telomeric / centromeric / scattered N runs (SURVEY 8d, C5)."""
    gen = torch.Generator(device=device)
    gen.manual_seed(int(seed))
    host_rng = np.random.default_rng(int(seed))
    nl = torch.tensor([10], dtype=torch.uint8, device=device)
    parts = []
    for r, L in enumerate(rec_lens):
        hdr = f">chr{r + 1} {name} len={L}\n".encode()
        parts.append(torch.tensor(list(hdr), dtype=torch.uint8, device=device))
        if gc is None:
            codes = torch.randint(0, 4, (L,), dtype=torch.uint8, device=device, generator=gen)
        else:
            u = torch.rand(L, device=device, generator=gen)
            t1, t2, t3 = (1 - gc) / 2, 0.5, 0.5 + gc / 2             # A | C | G | T
            codes = ((u >= t1).to(torch.uint8) + (u >= t2).to(torch.uint8) + (u >= t3).to(torch.uint8))
            del u
        seq = _ascii_from_codes(codes)
        del codes
        if n_runs and L > 200_000:
            tel = min(10_000, L // 20)
            seq[:tel] = 78
            seq[L - tel:] = 78
            cen = min(3_000_000, L // 10)
            c0 = int(host_rng.integers(L // 4, L // 2))
            seq[c0:c0 + cen] = 78
            for _ in range(200):
                n = int(host_rng.integers(100, 50_000))
                p = int(host_rng.integers(0, max(L - n, 1)))
                seq[p:p + n] = 78
        full = (L // 80) * 80
        if full:
            body = seq[:full].view(-1, 80)
            parts.append(torch.cat([body, nl.expand(body.shape[0], 1)], dim=1).reshape(-1))
        if L > full:
            parts.append(seq[full:])
            parts.append(nl)
        del seq
    out = torch.cat(parts)
    pad = (-out.numel()) % 16                                     # keep every genome 16-byte aligned in a batch
    if pad:
        out = torch.cat([out, nl.expand(pad)])
    return out


def human_lengths(scale):
    total = int(3.1e9 * scale)
    w = np.asarray(HUMAN_MBP, dtype=np.float64)
    lens = np.maximum((w / w.sum() * total).astype(np.int64), 1000)
    return [int(x) for x in lens]


class Timer:
    def __init__(self, torch, dist, device, world):
        self.torch, self.dist, self.device, self.world = torch, dist, device, world

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps, warmup):
        """ms per step (max over ranks) and the last result."""
        torch = self.torch
        out = None
        for _ in range(warmup):
            out = fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1) / steps
        return self.max_over_ranks(ms), out

    def max_over_ranks(self, v):
        if self.world > 1:
            t = self.torch.tensor([v], dtype=self.torch.float64, device=self.device)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return float(v)

    def all_true(self, flag):
        t = self.torch.tensor([1 if flag else 0], device=self.device)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item())

    def sum_over_ranks(self, v):
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.device)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())


def _event_ms(pairs):
    return sum(a.elapsed_time(b) for a, b in pairs)


# ----------------------------------------------------------------------------------------------- C3
def run_c3(torch, dist, device, rank, world, steps, warmup, n_genomes=1000, mbp=5.0, oracle_check=True):
    from kmerml_b200 import dist as kdist
    from kmerml_b200 import engine
    T = Timer(torch, dist, device, world)
    L = int(mbp * 1e6)
    shards = kdist.shard_genomes([L] * n_genomes, world)
    mine = shards[rank]
    gcs = {i: float(np.random.default_rng(2000 + i).uniform(0.30, 0.70)) for i in mine}
    parts, offs = [], [0]
    for i in mine:
        nrec = 1 + (i % 3)
        lens = [L // nrec] * (nrec - 1) + [L - (L // nrec) * (nrec - 1)]
        g = gpu_fasta(torch, device, lens, 2000 + i, f"bacterium {i}", gc=gcs[i])
        parts.append(g)
        offs.append(offs[-1] + g.numel())
    fasta = torch.cat(parts) if parts else torch.zeros(0, dtype=torch.uint8, device=device)
    del parts
    n_max = max(len(s) for s in shards)
    M = 4 ** 8
    counts = torch.zeros((max(len(mine), 1), M), dtype=torch.int32, device=device)
    totals = torch.zeros((max(len(mine), 1), 1), dtype=torch.int64, device=device)
    ev = {"count": [], "gather": [], "distance": []}
    info = {"planes": 0}

    def mark():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def step():
        a = mark()
        if mine:
            engine.count_dense_device(fasta, offs, [8], want_freq=False, out_counts=counts[:len(mine)],
                                      out_totals=totals[:len(mine)])
        b = mark()
        if world > 1:
            # the rows travel as byte planes (2 of 4 for these counts), the norms and the largest count in one small
            # all_gather before them; every rank then holds all rows in planar form and computes its genomes' block
            got = []
            D = kdist.distance_matrix_from_shards(counts[:len(mine)], shards, "cosine", info=info,
                                                  on_gathered=lambda: got.append(mark()))
            c = got[0]
        else:
            c = mark()
            D = kdist.distance_matrix_sharded(counts, "cosine")
        d = mark()
        ev["count"].append((a, b)); ev["gather"].append((b, c)); ev["distance"].append((c, d))
        return D

    def gather_rows():                                   # (untimed: the uint32 matrix in genome order, for the checks)
        if world == 1:
            return counts
        pad = torch.zeros((n_max, M), dtype=torch.int32, device=device)
        pad[:len(mine)] = counts[:len(mine)]
        allc = torch.empty((world * n_max, M), dtype=torch.int32, device=device)
        dist.all_gather_into_tensor(allc, pad)
        rows = torch.empty((n_genomes, M), dtype=torch.int32, device=device)
        for r, idxs in enumerate(shards):
            if idxs:
                rows[torch.tensor(idxs, device=device)] = allc[r * n_max:r * n_max + len(idxs)]
        return rows

    ms, D = T.timed(step, steps, warmup)
    torch.cuda.synchronize()
    rows = gather_rows()
    n_ev = len(ev["count"])
    parts_ms = {k: T.max_over_ranks(_event_ms(v[n_ev - steps:]) / steps) for k, v in ev.items()}
    # ---- checks
    ok_sum = bool(torch.equal((counts[:len(mine)].to(torch.int64) & 0xFFFFFFFF).sum(dim=1), totals[:len(mine), 0])) if mine else True
    D1 = engine.pairwise_distance_device(rows, "cosine")
    same_D = bool(torch.equal(D, D1))
    exact, dist_ok = None, None
    if rank == 0 and oracle_check and mine:
        import oracle
        oracle.build()
        g0 = fasta[offs[0]:offs[1]].cpu().numpy().tobytes()
        ref = oracle.count_dense(g0, 8, 8)
        exact = bool(np.array_equal(ref, counts[0].cpu().numpy().view(np.uint32).astype(np.uint64)))
        sub = rows[:16].cpu().numpy().view(np.uint32).astype(np.float64)
        want = oracle.pairwise_distance(sub, "cosine")
        got = D[:16, :16].cpu().numpy().astype(np.float64)
        dist_ok = bool(np.all(np.abs(got - want) <= 1e-6 * np.maximum(np.abs(want), 1e-30) + 1e-7))
    bases = float(n_genomes) * L
    return {"workload": f"C3: {n_genomes} genomes x {mbp:g} Mbp, k=8 count rows + cosine distance matrix, genomes sharded over "
                        f"{world} GPU(s)" + (", rows all-gathered as byte planes, row-block distances, blocks gathered" if world > 1 else ""), "ms": ms, "Gbp/s": bases / (ms * 1e-3) / 1e9,
            "count_ms": parts_ms["count"], "gather_ms": parts_ms["gather"], "distance_ms": parts_ms["distance"],
            "count_Gbp/s_per_gpu": (len(mine) * L) / (parts_ms["count"] * 1e-3) / 1e9 if parts_ms["count"] > 0 else None,
            "gathered_as": f"{info['planes']} byte plane(s) of the count rows + squared norms (not the uint32 rows)" if world > 1 else None,
            "nvlink_bytes": int((world - 1) * n_max * (M * info["planes"] + 8) + (world - 1) * n_max * world * n_max * 4) if world > 1 else 0,
            "parity": {"sum_counts_equals_windows": T.all_true(ok_sum), "sharded_distance_bit_exact_vs_single_gpu": T.all_true(same_D),
                       "oracle_bit_exact_genome0": exact, "distance_within_1e-6_of_float64": dist_ok}}


# ----------------------------------------------------------------------------------------------- C4
def run_c4(torch, dist, device, rank, world, steps, warmup, scale=1.0):
    from kmerml_b200 import dist as kdist
    from kmerml_b200 import engine
    T = Timer(torch, dist, device, world)
    lens = human_lengths(scale)
    fasta = gpu_fasta(torch, device, lens, 4, "synthetic human-sized")
    bases = float(sum(lens))
    k = 12
    coll = []

    def step():
        begin, end = kdist.chunk_ranges(int(fasta.numel()), world)[rank]
        counts, totals = engine.count_dense_range_device(fasta, begin, end, [k], None, True)
        if world == 1:
            return counts, 0, totals
        part = torch.empty(4 ** k // world, dtype=torch.int32, device=device)
        a = torch.cuda.Event(enable_timing=True); a.record()
        dist.reduce_scatter_tensor(part, counts, op=dist.ReduceOp.SUM)
        dist.all_reduce(totals, op=dist.ReduceOp.SUM)
        b = torch.cuda.Event(enable_timing=True); b.record()
        coll.append((a, b))
        freq = engine.normalize_rows_device(part.unsqueeze(0), totals[:1])          # the owner's frequency slice
        return part, rank * (4 ** k // world), totals, freq

    ms, out = T.timed(step, steps, warmup)
    torch.cuda.synchronize()
    coll_ms = T.max_over_ranks(_event_ms(coll[len(coll) - steps:]) / steps) if coll else 0.0
    part, off, totals = out[0], out[1], out[2]
    # single-GPU result of the whole genome on this rank: timed (the strong-scaling reference) and compared
    def single():
        return engine.count_dense_device(fasta, [0, int(fasta.numel())], [k], canonical=True, want_freq=False)
    ms1, whole = T.timed(single, steps, 1)
    n = part.numel()
    same = bool(torch.equal(part, whole.counts[0, off:off + n])) and int(totals[0]) == int(whole.totals[0, 0])
    slice_sum = T.sum_over_ranks(float((part.to(torch.int64) & 0xFFFFFFFF).sum().item()))
    return {"workload": f"C4: one {bases / 1e9:.2f} Gbp genome, k=12 canonical dense counts, byte ranges with k-1 look-back on "
                        f"{world} GPU(s) + reduce-scatter to owner slices", "ms": ms, "Gbp/s": bases / (ms * 1e-3) / 1e9,
            "collective": "ncclReduceScatter(sum, uint32[4^12]) + all-reduce of the window total" if world > 1 else None,
            "collective_ms": coll_ms, "nvlink_bytes": int((world - 1) * (4 ** k // world) * 4) if world > 1 else 0,
            "single_gpu_ms": ms1, "strong_scaling_efficiency": ms1 / (world * ms) if ms > 0 else None,
            "bit_exact_vs_single_gpu": T.all_true(same), "sum_of_slices_equals_windows": slice_sum == float(int(whole.totals[0, 0])),
            "limiter": "the partition kernel (per-rank byte range) then the fixed-size part: bucket kernel + 64 MB "
                       "reduce-scatter, which do not shrink with N"}


# ----------------------------------------------------------------------------------------------- C5
def run_c5(torch, dist, device, rank, world, steps, warmup, scale=1.0, check_scale=0.016):
    from kmerml_b200 import dist as kdist
    from kmerml_b200 import engine
    T = Timer(torch, dist, device, world)
    k = 21
    # bounded exactness check first: the same sharded pipeline on a ~50 Mbp genome against the single-GPU result
    small = gpu_fasta(torch, device, human_lengths(check_scale * scale), 5, "c5 check", n_runs=True)
    mk, mc, mf, w = kdist.count_sparse_sharded(small, k, canonical=True)
    k1, c1, f1, w1 = engine.count_sparse_device(small, k, canonical=True)
    bits = 2 * k
    top = (k1 >> (bits - 16)) & 0xFFFF
    sel = ((top * world) >> 16) == rank
    small_ok = bool(torch.equal(mk, k1[sel]) and torch.equal(mc, c1[sel]) and torch.equal(mf, f1[sel]) and w == w1)
    small_mbp = small.numel() / 1e6
    del small, mk, mc, mf, k1, c1, f1
    torch.cuda.empty_cache()
    lens = human_lengths(scale)
    fasta = gpu_fasta(torch, device, lens, 4, "synthetic human-sized with N runs", n_runs=True)
    bases = float(sum(lens))

    def step():
        return kdist.count_sparse_sharded(fasta, k, canonical=True)

    ms, (keys, counts, first, windows) = T.timed(step, steps, warmup)
    torch.cuda.synchronize()
    # one more, untimed, step with a synchronisation after every phase: where the time goes
    phases = {}
    del keys, counts, first
    keys, counts, first, windows = kdist.count_sparse_sharded(fasta, k, canonical=True, phase_ms=phases)
    phases.pop("start", None)
    phases = {name: T.max_over_ranks(v) for name, v in phases.items()}
    n_local = int(keys.numel())
    asc = bool((keys[1:] > keys[:-1]).all().item()) if n_local > 1 else True
    lo = int(keys[0].item()) if n_local else None
    hi = int(keys[-1].item()) if n_local else None
    ordered = True
    if world > 1:
        ends = torch.tensor([lo if lo is not None else -1, hi if hi is not None else -1], dtype=torch.int64, device=device)
        allends = [torch.empty_like(ends) for _ in range(world)]
        dist.all_gather(allends, ends)
        last = -1
        for e in allends:
            a, b = int(e[0]), int(e[1])
            if a >= 0:
                ordered &= a > last
                last = b
    total_counts = T.sum_over_ranks(float((counts.to(torch.int64) & 0xFFFFFFFF).sum().item()))
    distinct = T.sum_over_ranks(float(n_local))
    raw = world > 1 and world & (world - 1) == 0
    return {"workload": f"C5: one {bases / 1e9:.2f} Gbp genome with N runs, k=21 canonical on {world} GPU(s): " +
                        ("windows of a byte range emitted and grouped by owner, all-to-all by key range, ONE sort + reduce per rank"
                         if raw else "per-range sort-reduce, all-to-all of the distinct k-mers by key range, merge"),
            "ms": ms, "Gbp/s": bases / (ms * 1e-3) / 1e9,
            "collective": ("all_to_all_single x2 (k-mer u64, end offset u32) of raw windows" if raw else
                           "all_to_all_single x3 (k-mer u64, count u32, first offset u32) of pre-reduced triples") if world > 1 else None,
            "phase_ms_synchronised": phases, "windows": int(windows), "distinct_kmers": int(distinct),
            "nvlink_bytes": int((float(windows) * 12 if raw else distinct * 16) * (world - 1) / world) if world > 1 else 0,
            "bit_exact_vs_single_gpu": {"genome_mbp": round(small_mbp, 1), "ok": T.all_true(small_ok)},
            "full_size_invariants": {"sum_counts_equals_windows": total_counts == float(windows),
                                     "keys_ascending_within_and_across_ranks": T.all_true(asc and ordered)}}


def run_extras(args, torch, dist, device, rank, world):
    """Dict of extra keys for the bench line.  c3 at every N; c4_strong at every N (N = 1 is the strong-scaling
    reference); c5_sparse at N > 1 (the single-GPU sparse pass of 3.1 Gbp needs > 100 GB of workspace)."""
    out = {}
    t0 = time.time()
    sc = args.extra_scale
    steps = args.steps
    try:
        out["c3"] = run_c3(torch, dist, device, rank, world, steps, 1, n_genomes=max(8, int(1000 * min(sc, 1.0))), mbp=5.0)
    except Exception as exc:                                              # report, never fake
        out["c3"] = {"error": repr(exc)[:300]}
    torch.cuda.empty_cache()
    try:
        out["c4_strong"] = run_c4(torch, dist, device, rank, world, steps, 1, scale=sc)
    except Exception as exc:
        out["c4_strong"] = {"error": repr(exc)[:300]}
    torch.cuda.empty_cache()
    if world > 1 or args.c5_single:
        # memory guard, agreed by all ranks BEFORE any collective of the section (a rank that runs out of memory
        # alone would leave the others waiting in the all-to-all): per window of this rank's byte range the emit +
        # sort workspace takes 24 B, the exchanged triples 2 x 16 B, the merge workspace ~48 B, its outputs 16 B; they
        # are not all live at once (measured peak at N = 2: ~75 B per window)
        need = 3.1e9 * sc / world * 100.0
        free = torch.tensor([float(torch.cuda.mem_get_info(device)[0])], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(free, op=dist.ReduceOp.MIN)
        if need > 0.7 * float(free.item()):
            out["c5_sparse"] = {"skipped": f"needs ~{need / 1e9:.0f} GB per GPU at N={world} (sort + exchange + merge buffers of "
                                           f"{3.1 * sc / world:.2f} G windows); {float(free.item()) / 1e9:.0f} GB free: run with more GPUs"}
        else:
            try:
                out["c5_sparse"] = run_c5(torch, dist, device, rank, world, steps, 1, scale=sc)
            except Exception as exc:
                out["c5_sparse"] = {"error": repr(exc)[:300]}
        torch.cuda.empty_cache()
    out["extras_seconds"] = round(time.time() - t0, 1)
    return out
