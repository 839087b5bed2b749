"""Multi-GPU layer: one process per GPU (torchrun), torch.distributed for the plumbing.

Two levels, as in SURVEY 8e:
  * whole genomes are independent units -> sharded across ranks (longest-processing-time
    first on file size), no data-path collective; rows are gathered only when asked for;
  * one large genome is cut into byte ranges of whole 16 KB tiles; every rank counts the
    windows that END in its range (kmerml_count_dense_range reads the k-1 bases before the
    range from the file itself) and the dense uint32 rows are summed with ONE all-reduce
    (NCCL over NVLink on GPUs).  Integer sums are order-independent, so the result is
    bit-identical to the single-GPU one;
  * one large genome, sparse k (15..32): every rank sort-reduces the windows of its byte range,
    routes each distinct k-mer to the rank that owns its key range with ONE all-to-all
    (k-mer, count, first offset), and merges what it receives.  The result stays sharded by key
    range, ascending across ranks.
"""
import numpy as np

TILE_BYTES = 16384


def shard_genomes(sizes, world_size):
    """Longest-processing-time-first assignment of genomes (by byte size) to ranks.
    Returns a list of index lists, one per rank; deterministic for equal inputs."""
    order = sorted(range(len(sizes)), key=lambda i: (-int(sizes[i]), i))
    load = [0] * world_size
    shards = [[] for _ in range(world_size)]
    for i in order:
        r = min(range(world_size), key=lambda j: (load[j], j))
        shards[r].append(i)
        load[r] += int(sizes[i])
    for s in shards:
        s.sort()
    return shards


def chunk_ranges(nbytes, world_size, tile=TILE_BYTES):
    """world_size contiguous byte ranges [begin, end) that tile [0, nbytes); every begin is a
    multiple of the tile size (the kernels' slice granularity)."""
    tiles = (int(nbytes) + tile - 1) // tile
    out = []
    for r in range(world_size):
        t0 = tiles * r // world_size
        t1 = tiles * (r + 1) // world_size
        out.append((min(t0 * tile, int(nbytes)), min(t1 * tile, int(nbytes))))
    return out


def bind_to_gpu_numa_node(device_index):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off, so that the pinned host buffers it
    allocates afterwards (first touch) and the copies to and from them stay on that socket.  With one process per
    GPU on a two-socket host this is what keeps 8 ranks' PCIe streams from crossing the inter-socket link.
    Returns the node number, or None when the topology cannot be read (nothing is changed then)."""
    import os
    try:
        import torch
        p = torch.cuda.get_device_properties(device_index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


def _world():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def allreduce_counts(counts, totals=None):
    """In-place SUM all-reduce of partial count rows (int32 storage of uint32: the wrap-around
    sum is the uint32 sum) and of the window totals."""
    import torch.distributed as dist
    _, world = _world()
    if world > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
        if totals is not None:
            dist.all_reduce(totals, op=dist.ReduceOp.SUM)
    return counts, totals


def count_genome_chunked(fasta, k_values, *, min_record_len=None, canonical=False, want_freq=True,
                         count_range=None):
    """Dense counts of ONE genome resident on every rank's device, computed cooperatively:
    rank r counts byte range r, then one all-reduce.  Every rank returns the full result.

    `count_range(fasta, begin, end, ks, min_record_len, canonical) -> (counts, totals)` can be
    injected (the CPU tests use the thread emulator); by default it is the CUDA entry point.
    """
    import torch
    from . import engine
    rank, world = _world()
    ks = list(dict.fromkeys(int(k) for k in k_values))
    begin, end = chunk_ranges(int(fasta.numel()), world)[rank]
    fn = count_range if count_range is not None else engine.count_dense_range_device
    counts, totals = fn(fasta, begin, end, ks, min_record_len, canonical)
    allreduce_counts(counts, totals)
    freq = None
    if want_freq:
        if counts.is_cuda:
            lay, _ = engine.row_layout(ks)
            freq = torch.empty(counts.shape, dtype=torch.float32, device=counts.device)
            for ki, k in enumerate(ks):
                off, n = lay[k]
                freq[off:off + n] = engine.normalize_rows_device(counts[off:off + n].unsqueeze(0).contiguous(),
                                                                 totals[ki:ki + 1])[0]
        else:
            lay, _ = engine.row_layout(ks)
            c = counts.numpy().view(np.uint32).astype(np.float64)
            f = np.zeros_like(c)
            for ki, k in enumerate(ks):
                off, n = lay[k]
                t = float(totals[ki])
                f[off:off + n] = c[off:off + n] / t if t else 0.0
            freq = torch.from_numpy(f.astype(np.float32))
    return counts, freq, totals


def count_genome_chunked_scatter(fasta, k, *, min_record_len=None, canonical=False, count_range=None):
    """Dense counts of ONE genome resident on every rank's device, result SHARDED: rank r counts byte range r
    and ONE reduce-scatter (SUM) leaves it with slice r of the 4^k row, [r * 4^k / world, (r + 1) * 4^k / world).
    The canonical fold is linear, so it is applied to every rank's partial row BEFORE the reduction
    (kmerml_count_dense_range does it): no second exchange.  A reduce-scatter moves (world - 1) / world of a row
    per rank, half of what the all-reduce of count_genome_chunked moves; gather the slices only if one rank needs
    the whole row.  Returns (slice int32[4^k / world], slice offset, windows of the whole genome)."""
    import torch
    import torch.distributed as dist
    from . import engine
    rank, world = _world()
    k = int(k)
    n_bins = 4 ** k
    if n_bins % world:
        raise ValueError("4^k must be divisible by the number of ranks")
    begin, end = chunk_ranges(int(fasta.numel()), world)[rank]
    fn = count_range if count_range is not None else engine.count_dense_range_device
    counts, totals = fn(fasta, begin, end, [k], min_record_len, canonical)
    if world == 1:
        return counts, 0, int(totals[0])
    part = torch.empty(n_bins // world, dtype=counts.dtype, device=counts.device)
    dist.reduce_scatter_tensor(part, counts.contiguous(), op=dist.ReduceOp.SUM)
    dist.all_reduce(totals, op=dist.ReduceOp.SUM)
    return part, rank * (n_bins // world), int(totals[0])


def distance_matrix_sharded(counts, metric="cosine", rows_fn=None):
    """n x n distance matrix of count rows resident on every rank: rank r computes rows
    [r * n / world, (r + 1) * n / world) (kmerml_pairwise_distance_rows, exact Gram entries on the tensor
    cores) and one all_gather assembles the matrix everywhere."""
    import torch
    import torch.distributed as dist
    from . import engine
    rank, world = _world()
    n = counts.shape[0]
    per = (n + world - 1) // world
    r0, r1 = min(rank * per, n), min((rank + 1) * per, n)
    if world == 1 and rows_fn is None:
        return engine.pairwise_distance_device(counts, metric)      # one GPU: the symmetric call (upper triangle only)
    fn = rows_fn if rows_fn is not None else engine.pairwise_distance_rows_device
    block = fn(counts, r0, r1, metric)
    if world == 1:
        return block
    pad = torch.zeros((per, n), dtype=block.dtype, device=block.device)
    pad[:r1 - r0] = block
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad)
    return torch.cat(parts)[:n]


def _all_gather_rows(out, block):
    """out [world * b, ...] <- the ranks' equal blocks [b, ...], in rank order."""
    import torch
    import torch.distributed as dist
    if dist.get_backend() == "nccl":
        dist.all_gather_into_tensor(out, block)
    else:
        parts = [torch.empty_like(block) for _ in range(dist.get_world_size())]
        dist.all_gather(parts, block)
        b = block.shape[0]
        for r, p in enumerate(parts):
            out[r * b:(r + 1) * b] = p


_POS_CACHE = {}


def _gathered_positions(shards, device):
    """Position of genome i in the gathered order (rank-major, every rank padded to the largest shard)."""
    import torch
    key = (tuple(tuple(s) for s in shards), str(device))
    pos = _POS_CACHE.get(key)
    if pos is None:
        n_max = max(len(s) for s in shards)
        n = sum(len(s) for s in shards)
        host = np.zeros(n, dtype=np.int64)
        for r, idxs in enumerate(shards):
            for j, i in enumerate(idxs):
                host[i] = r * n_max + j
        pos = torch.from_numpy(host).to(device)
        if len(_POS_CACHE) > 16:
            _POS_CACHE.clear()
        _POS_CACHE[key] = pos
    return pos


def distance_matrix_from_shards(counts, shards, metric="cosine", planes_fn=None, rows_fn=None, info=None, on_gathered=None):
    """n x n distance matrix of genomes counted on several GPUs, WITHOUT gathering the uint32 rows: rank r holds the
    count rows of the genomes shards[r] (in that order).  Every rank turns its rows into byte planes
    (kmerml_count_planes), one small all_gather carries the squared norms and the largest count, the planes that
    count needs -- one byte per bin and plane instead of four -- are all-gathered, every rank computes the row block of
    its own genomes on the tensor cores (kmerml_distance_rows_planes) and one all_gather assembles the matrix, which
    is then put into genome order.  Bit-identical to the single-GPU matrix of the gathered rows."""
    import torch
    import torch.distributed as dist
    from . import engine
    rank, world = _world()
    planes_fn = planes_fn if planes_fn is not None else engine.count_planes_device
    rows_fn = rows_fn if rows_fn is not None else engine.distance_rows_planes_device
    n = sum(len(s) for s in shards)
    n_max = max(max(len(s) for s in shards), 1)
    planes_l, sumsq_l, mx = planes_fn(counts[:len(shards[rank])], n_rows=n_max)
    pos = _gathered_positions(shards, counts.device)
    top = (mx.to(torch.int64) & 0xFFFFFFFF).to(torch.float64)
    if world == 1:
        nd = engine.planes_needed(int(top.item()))
        block = rows_fn(planes_l, nd, sumsq_l, 0, n_max, metric)
        return block[pos][:, pos]
    meta = torch.cat([sumsq_l, top])
    metas = torch.empty((world * (n_max + 1),), dtype=torch.float64, device=counts.device)
    _all_gather_rows(metas, meta)
    metas = metas.view(world, n_max + 1)
    nd = engine.planes_needed(int(metas[:, -1].max().item()))
    sumsq_all = metas[:, :n_max].reshape(-1).contiguous()
    m = planes_l.shape[2]
    planes_all = torch.empty((nd, world * n_max, m), dtype=torch.uint8, device=counts.device)
    for p in range(nd):
        _all_gather_rows(planes_all[p], planes_l[p])
    if info is not None:
        info["planes"] = nd
    if on_gathered is not None:
        on_gathered()
    block = rows_fn(planes_all, nd, sumsq_all, rank * n_max, (rank + 1) * n_max, metric)
    Dg = torch.empty((world * n_max, world * n_max), dtype=block.dtype, device=block.device)
    _all_gather_rows(Dg, block)
    return Dg[pos][:, pos]


def sketch_distance_from_shards(sk_local, shards, metric="mash", rows_fn=None):
    """n x n Mash / Jaccard distance matrix of genomes sketched on several GPUs: rank r holds the sketches of the
    genomes shards[r] (in that order).  The sketches and fill counts of all ranks are all-gathered (every rank padded
    to the largest shard), every rank computes the row block of its own genomes (kmerml_sketch_distance_rows) and one
    all_gather assembles the matrix, which is then put into genome order.  Bit-identical to the single-GPU matrix.
    `rows_fn(sketches, row_begin, row_end, metric)` can be injected (the CPU tests use numpy)."""
    import torch
    from . import engine
    rank, world = _world()
    rows_fn = rows_fn if rows_fn is not None else engine.sketch_distance_rows_device
    n_max = max(max(len(s) for s in shards), 1)
    mine = len(shards[rank])
    dev = sk_local.hashes.device
    s = sk_local.s
    # k, s, seed and canonical travel with the fill counts: sketches made with other parameters are not comparable
    params = torch.tensor([sk_local.k, s, sk_local.seed, int(sk_local.canonical)], dtype=torch.int64, device=dev)
    hashes = torch.full((n_max, s), -1, dtype=torch.int64, device=dev)
    hashes[:mine] = sk_local.hashes[:mine, :s]
    meta = torch.zeros((n_max + 4,), dtype=torch.int64, device=dev)
    meta[:mine] = sk_local.filled[:mine].to(torch.int64)
    meta[n_max:] = params
    pos = _gathered_positions(shards, dev)
    if world == 1:
        block = rows_fn(engine.Sketches(hashes, meta[:n_max].to(torch.int32), *sk_local.params()), 0, n_max, metric)
        return block[pos][:, pos]
    metas = torch.empty((world * (n_max + 4),), dtype=torch.int64, device=dev)
    _all_gather_rows(metas, meta)
    metas = metas.view(world, n_max + 4)
    for r in range(world):
        if not torch.equal(metas[r, n_max:], params):
            raise ValueError(f"rank {r} sketched with other parameters (k, s, seed, canonical): "
                             f"{metas[r, n_max:].tolist()} vs {params.tolist()}")
    all_hashes = torch.empty((world * n_max, s), dtype=torch.int64, device=dev)
    _all_gather_rows(all_hashes, hashes)
    sk_all = engine.Sketches(all_hashes, metas[:, :n_max].reshape(-1).to(torch.int32).contiguous(), *sk_local.params())
    block = rows_fn(sk_all, rank * n_max, (rank + 1) * n_max, metric)
    Dg = torch.empty((world * n_max, world * n_max), dtype=block.dtype, device=block.device)
    _all_gather_rows(Dg, block)
    return Dg[pos][:, pos]


def count_genomes_sharded(fasta_list, k_values, *, min_record_len=None, canonical=False, gather=True, count_batch=None):
    """Dense counts of many genomes: this rank counts its LPT shard; with gather=True the rows
    of all ranks are assembled (in input order) on every rank with one all_gather per tensor.

    fasta_list: per-genome uint8 tensors (only this rank's shard needs to be on its device).
    Returns (indices of the rows held, counts [n, row_len], totals [n, nk])."""
    import torch
    import torch.distributed as dist
    from . import engine
    rank, world = _world()
    ks = list(dict.fromkeys(int(k) for k in k_values))
    sizes = [int(t.numel()) for t in fasta_list]
    shards = shard_genomes(sizes, world)
    mine = shards[rank]
    _, row_len = engine.row_layout(ks)
    if count_batch is not None:
        counts, totals = count_batch([fasta_list[i] for i in mine], ks, min_record_len, canonical)
    elif mine:
        dev = fasta_list[mine[0]].device
        buf = torch.cat([fasta_list[i].to(dev) for i in mine])
        offs = np.concatenate(([0], np.cumsum([sizes[i] for i in mine]))).tolist()
        res = engine.count_dense_device(buf, offs, ks, min_record_len=min_record_len, canonical=canonical,
                                        want_freq=False)
        counts, totals = res.counts, res.totals
    else:
        dev = fasta_list[0].device if fasta_list else torch.device("cpu")
        counts = torch.zeros((0, row_len), dtype=torch.int32, device=dev)
        totals = torch.zeros((0, len(ks)), dtype=torch.int64, device=dev)
    if not gather or world == 1:
        return mine, counts, totals
    n_max = max(len(s) for s in shards)
    pad_c = torch.zeros((n_max, row_len), dtype=torch.int32, device=counts.device)
    pad_t = torch.zeros((n_max, len(ks)), dtype=torch.int64, device=counts.device)
    pad_c[:len(mine)] = counts
    pad_t[:len(mine)] = totals
    all_c = [torch.empty_like(pad_c) for _ in range(world)]
    all_t = [torch.empty_like(pad_t) for _ in range(world)]
    dist.all_gather(all_c, pad_c)
    dist.all_gather(all_t, pad_t)
    out_c = torch.empty((len(sizes), row_len), dtype=torch.int32, device=counts.device)
    out_t = torch.empty((len(sizes), len(ks)), dtype=torch.int64, device=counts.device)
    for r, idxs in enumerate(shards):
        for j, i in enumerate(idxs):
            out_c[i] = all_c[r][j]
            out_t[i] = all_t[r][j]
    return list(range(len(sizes))), out_c, out_t


SPARSE_RANGE_ALIGN = 131072


def key_owner_splits(keys, k, world_size):
    """keys: int64 tensor holding ascending uint64 2-bit packed k-mers.  Rank r owns the k-mers whose top
    16 bits t satisfy (t * world_size) >> 16 == r, so owners are ascending along `keys`; returns the number
    of keys per owner (list of world_size ints).  The keys are sorted, so the owner boundaries are found by a
    binary search for the first key of every rank (no pass over the keys)."""
    import torch
    bits = 2 * int(k)
    if keys.numel() == 0:
        return [0] * world_size
    if 16 <= bits < 64:
        # owner(key) >= r  <=>  top16 >= ceil(r * 65536 / world)  <=>  key >= that << (bits - 16)
        firsts = [((r * 65536 + world_size - 1) // world_size) << (bits - 16) for r in range(1, world_size)]
        cut = torch.searchsorted(keys, torch.tensor(firsts, dtype=torch.int64, device=keys.device)).cpu().tolist() if firsts else []
        edges = [0] + cut + [int(keys.numel())]
        return [edges[i + 1] - edges[i] for i in range(world_size)]
    if bits >= 16:
        top = (keys >> (bits - 16)) & 0xFFFF
    else:
        top = (keys << (16 - bits)) & 0xFFFF
    owner = (top * world_size) >> 16
    return torch.bincount(owner, minlength=world_size).cpu().tolist()


def count_sparse_sharded(fasta, k, *, min_record_len=None, canonical=False, count_range=None, merge=None,
                         emit_range=None, reduce_windows=None, phase_ms=None):
    """Distinct k-mers (k <= 32) of ONE genome resident on every rank's device, counted cooperatively.
    Rank r counts byte range r, the partial results are exchanged with one all-to-all per tensor, and rank r
    returns the k-mers of key range r: (keys, counts, first, windows of the whole genome).  Concatenating the
    ranks' results in rank order gives exactly the single-GPU result.

    Two routes.  RAW (the default when the number of ranks is a power of two): rank r emits the windows of its byte
    range grouped by owner (kmerml_emit_sparse_range: the owner is the top log2(world) bits of the k-mer), ONE
    all-to-all per tensor moves every window to its owner, and each rank sorts + reduces what it received once
    (kmerml_reduce_sparse_windows, the owner bits left out of the sort).  PRE-REDUCED (any number of ranks): every rank
    sort-reduces its range first, the distinct k-mers travel, the owner merges (a second sort).  RAW does one sort per
    rank instead of two; PRE-REDUCED moves less when the ranges hold many repeats.

    `count_range(fasta, begin, end, k, min_record_len, canonical) -> (keys, counts, first, windows)` and
    `merge(keys, counts, first, k) -> (keys, counts, first)` (PRE-REDUCED) or `emit_range(fasta, begin, end, k,
    owner_bits, min_record_len, canonical) -> (keys, ends, per-owner counts)` and `reduce_windows(keys, ends,
    sort_bits) -> (keys, counts, first)` (RAW) can be injected (CPU tests); by default they are the CUDA entry points."""
    import torch
    import torch.distributed as dist
    from . import engine
    rank, world = _world()
    begin, end = chunk_ranges(int(fasta.numel()), world, tile=SPARSE_RANGE_ALIGN)[rank]
    default_count = count_range is None
    if count_range is None:
        count_range = lambda f, b, e, kk, ml, c: engine.count_sparse_range_device(f, b, e, kk, min_record_len=ml, canonical=c)
    merge_takes_sort_k = merge is None                    # (the injected CPU stand-ins sort whole keys)
    if merge is None:
        merge = engine.merge_sparse_device
    import time as _time

    def mark(name, t_prev):
        """(diagnostic only: phase_ms = {} makes every phase end with a device synchronisation)"""
        if phase_ms is None:
            return t_prev
        if fasta.is_cuda:
            torch.cuda.synchronize()
        now = _time.perf_counter()
        phase_ms[name] = phase_ms.get(name, 0.0) + (now - t_prev) * 1e3
        return now

    tm = mark("start", _time.perf_counter())
    raw = (emit_range is not None) or (merge_takes_sort_k and default_count and world > 1 and world & (world - 1) == 0
                                       and 2 * int(k) > world.bit_length())
    if raw:
        owner_bits = world.bit_length() - 1
        if emit_range is None:
            emit_range = lambda f, b, e, kk, ob, ml, c: engine.emit_sparse_range_device(f, b, e, kk, ob, min_record_len=ml, canonical=c)
        if reduce_windows is None:
            reduce_windows = engine.reduce_sparse_windows_device
        keys, ends, send = emit_range(fasta, begin, end, int(k), owner_bits, min_record_len, canonical)
        tm = mark("emit_group_by_owner", tm)
        dev = keys.device
        send_t = torch.tensor(send, dtype=torch.int64, device=dev)
        recv_t = torch.empty_like(send_t)
        dist.all_to_all_single(recv_t, send_t)
        recv = recv_t.cpu().tolist()
        total = int(sum(recv))
        w = torch.tensor([int(keys.numel())], dtype=torch.int64, device=dev)
        got = []
        parts = [keys, ends]
        del keys, ends
        for i in range(2):
            t = parts[i].contiguous()
            parts[i] = None
            r = torch.empty(total, dtype=t.dtype, device=dev)
            dist.all_to_all_single(r, t, output_split_sizes=recv, input_split_sizes=send)
            del t
            got.append(r)
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
        tm = mark("all_to_all", tm)
        mk, mc, mf = reduce_windows(got[0], got[1], 2 * int(k) - owner_bits)
        tm = mark("sort_reduce", tm)
        return mk, mc, mf, int(w.item())
    keys, counts, first, windows = count_range(fasta, begin, end, int(k), min_record_len, canonical)
    tm = mark("range_sort_reduce", tm)
    if world == 1:
        return keys, counts, first, windows
    send = key_owner_splits(keys, k, world)
    send_t = torch.tensor(send, dtype=torch.int64, device=keys.device)
    recv_t = torch.empty_like(send_t)
    dist.all_to_all_single(recv_t, send_t)
    recv = recv_t.cpu().tolist()
    total = int(sum(recv))
    tm = mark("owner_splits", tm)
    out = []
    dev = keys.device
    parts = [keys, counts, first]
    del keys, counts, first
    for i in range(3):                                   # (each send buffer is released as soon as it has been exchanged)
        t = parts[i].contiguous()
        parts[i] = None
        r = torch.empty(total, dtype=t.dtype, device=dev)
        dist.all_to_all_single(r, t, output_split_sizes=recv, input_split_sizes=send)
        del t
        out.append(r)
    w = torch.tensor([windows], dtype=torch.int64, device=dev)
    dist.all_reduce(w, op=dist.ReduceOp.SUM)
    tm = mark("all_to_all", tm)
    # all keys a rank receives share the bits that select the rank (world a power of two: the top log2(world)
    # bits), so the merge's radix sort can leave them out: 2 (k - 1) bits are 5 byte-passes instead of 6 at k = 21
    k_sort = int(k)
    if world & (world - 1) == 0 and 2 * int(k) >= 16 and merge_takes_sort_k:
        k_sort = int(k) - (world.bit_length() - 1) // 2
    mk, mc, mf = merge(out[0], out[1], out[2], k_sort)
    tm = mark("merge", tm)
    return mk, mc, mf, int(w.item())
