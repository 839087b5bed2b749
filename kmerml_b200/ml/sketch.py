"""Genome x genome Mash / Jaccard distances from MinHash sketches, for any k up to 32 (engine.sketch_batch_device,
engine.sketch_distance_device).  The matrix feeds `hierarchical_clustering(..., distances=...)` and
`dbscan_clustering(..., distances=...)` directly.  Query x reference containment, Jaccard and ANI from scaled
(FracMinHash) sketches (engine.fmh_batch_device, engine.fmh_compare_device): `containment_matrix`.  Which references make up each query,
and how much of it each explains (engine.fmh_gather_device): `gather`."""
from pathlib import Path

import numpy as np
import pandas as pd
import torch

from .. import engine


def _load_batch(paths, dev):
    data = [np.fromfile(str(p), dtype=np.uint8) for p in paths]
    offsets = np.concatenate(([0], np.cumsum([d.size for d in data]))).tolist()
    host = np.concatenate(data) if data else np.zeros(0, np.uint8)
    fasta = torch.from_numpy(host).to(dev) if host.size else torch.zeros(0, dtype=torch.uint8, device=dev)
    return fasta, offsets


def sketch_distance_matrix(fasta_paths, k=21, sketch_size=1000, seed=42, canonical=True, metric="mash",
                           organism_ids=None, device=None):
    """Square DataFrame of the sketch distances between the genomes of `fasta_paths` (one FASTA file each), indexed
    by organism id (the file stems, as KmerExtractor.extract_from_genome_list names them, unless given)."""
    paths = [Path(p) for p in fasta_paths]
    if organism_ids is None:
        organism_ids = [p.stem for p in paths]
    organism_ids = list(organism_ids)
    if len(organism_ids) != len(paths):
        raise ValueError("Number of organism IDs must match number of genome paths")
    dev = torch.device(device if device is not None else "cuda")
    data = [np.fromfile(str(p), dtype=np.uint8) for p in paths]
    offsets = np.concatenate(([0], np.cumsum([d.size for d in data]))).tolist()
    host = np.concatenate(data) if data else np.zeros(0, np.uint8)
    fasta = torch.from_numpy(host).to(dev) if host.size else torch.zeros(0, dtype=torch.uint8, device=dev)
    sk = engine.sketch_batch_device(fasta, offsets, k, sketch_size=sketch_size, seed=seed, canonical=canonical)
    d = engine.sketch_distance_device(sk, metric, out_dtype=torch.float64).cpu().numpy()
    return pd.DataFrame(d, index=organism_ids, columns=organism_ids)


def containment_matrix(query_paths, reference_paths=None, *, k=21, scale=1000, seed=42, canonical=True,
                       metric="containment", query_ids=None, reference_ids=None, device=None):
    """DataFrame of a similarity of every query genome to every reference genome (one FASTA file each) from scaled
    sketches: index = query ids, columns = reference ids (file stems unless given).  Without `reference_paths` the
    queries are compared with each other.  `metric` is one of engine.fmh_compare_device's; all are similarities, so
    with "max_containment_ani" or "angular_similarity" (symmetric) `1 - df` goes straight into
    `hierarchical_clustering(..., distances=...)`.  The abundance-weighted metrics ("weighted_containment",
    "angular_similarity") sketch with abundance tracking."""
    q_paths = [Path(p) for p in query_paths]
    r_paths = q_paths if reference_paths is None else [Path(p) for p in reference_paths]
    q_ids = [p.stem for p in q_paths] if query_ids is None else list(query_ids)
    if reference_ids is None:
        r_ids = q_ids if reference_paths is None else [p.stem for p in r_paths]
    else:
        r_ids = list(reference_ids)
    if len(q_ids) != len(q_paths) or len(r_ids) != len(r_paths):
        raise ValueError("Number of ids must match number of genome paths")
    dev = torch.device(device if device is not None else "cuda")
    params = dict(scale=scale, seed=seed, canonical=canonical,
                  track_abundance=metric in ("weighted_containment", "angular_similarity"))
    queries = engine.fmh_batch_device(*_load_batch(q_paths, dev), k, **params)
    refs = None if reference_paths is None else engine.fmh_batch_device(*_load_batch(r_paths, dev), k, **params)
    d = engine.fmh_compare_device(queries, refs, metric, out_dtype=torch.float64).cpu().numpy()
    return pd.DataFrame(d, index=q_ids, columns=r_ids)


def _ids(paths, ids):
    ids = [p.stem for p in paths] if ids is None else list(ids)
    if len(ids) != len(paths):
        raise ValueError("Number of ids must match number of genome paths")
    return ids


def gather(query_paths, reference_paths, *, k=21, scale=1000, seed=42, canonical=True, threshold_bp=50_000,
           query_ids=None, reference_ids=None, device=None, track_abundance=False):
    """Long DataFrame of the gather of every query genome into the reference genomes (one FASTA file each; ids are
    the file stems unless given): one row per (query, match) in pick order.  A reference is picked while it covers at
    least max(1, ceil(threshold_bp / scale)) still-unassigned query hashes.  Columns: query, rank (0-based), match,
    intersect_bp / unique_bp / remaining_bp (hash counts times `scale`), f_orig_query = intersect / |Q|,
    f_match = intersect / |R|, f_unique_to_query = unique / |Q| and match_containment_ani = (intersect / |R|)^(1/k),
    all in float64.  With track_abundance the queries are sketched with k-mer abundances and, over the hashes each
    match takes, the columns n_unique_weighted_found (the sum of their abundances), f_unique_weighted (that over the
    query's total abundance: the match's share of the query's k-mers, e.g. of a metagenome's reads),
    average_abund, median_abund and std_abund (population standard deviation) are added."""
    q_paths = [Path(p) for p in query_paths]
    r_paths = [Path(p) for p in reference_paths]
    q_ids, r_ids = _ids(q_paths, query_ids), _ids(r_paths, reference_ids)
    dev = torch.device(device if device is not None else "cuda")
    params = dict(scale=scale, seed=seed, canonical=canonical)
    queries = engine.fmh_batch_device(*_load_batch(q_paths, dev), k, track_abundance=track_abundance, **params)
    refs = engine.fmh_batch_device(*_load_batch(r_paths, dev), k, **params)
    threshold = max(1, -(-int(threshold_bp) // int(scale)))
    res = engine.fmh_gather_device(queries, refs, threshold=threshold)
    n = res.n_matches.cpu().numpy()
    q_of = np.repeat(np.arange(len(q_ids)), n)
    rank = np.concatenate([np.arange(c) for c in n]) if len(n) else np.zeros(0, np.int64)
    ref = res.reference.cpu().numpy()[q_of, rank]
    unique, inter, remaining = (x.cpu().numpy()[q_of, rank].astype(np.float64)
                                for x in (res.unique, res.intersect, res.remaining))
    q_size = queries.sizes().cpu().numpy().astype(np.float64)[q_of]
    r_size = refs.sizes().cpu().numpy().astype(np.float64)[ref]
    df = pd.DataFrame({
        "query": [q_ids[i] for i in q_of], "rank": rank.astype(np.int64), "match": [r_ids[i] for i in ref],
        "intersect_bp": inter * scale, "unique_bp": unique * scale, "remaining_bp": remaining * scale,
        "f_orig_query": inter / q_size, "f_match": inter / r_size, "f_unique_to_query": unique / q_size,
        "match_containment_ani": (inter / r_size) ** (1.0 / k)})
    if track_abundance:
        weighted = res.unique_weighted.cpu().numpy()[q_of, rank]
        sumsq = res.unique_sumsq.cpu().numpy()[q_of, rank].astype(np.float64)
        q_mass = torch.zeros(len(queries), dtype=torch.int64, device=dev).index_add_(
            0, torch.repeat_interleave(torch.arange(len(queries), device=dev), queries.sizes()),
            queries.abundances.to(torch.int64)).cpu().numpy().astype(np.float64)[q_of]
        avg = weighted / unique
        df["n_unique_weighted_found"] = weighted.astype(np.int64)
        df["f_unique_weighted"] = weighted / q_mass
        df["average_abund"] = avg
        df["median_abund"] = res.median_abund.cpu().numpy()[q_of, rank]
        df["std_abund"] = np.sqrt(np.maximum(sumsq / unique - avg * avg, 0.0))
    return df
