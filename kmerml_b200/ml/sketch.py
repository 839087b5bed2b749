"""Genome x genome Mash / Jaccard distances from MinHash sketches, for any k up to 32 (engine.sketch_batch_device,
engine.sketch_distance_device).  The matrix feeds `hierarchical_clustering(..., distances=...)` and
`dbscan_clustering(..., distances=...)` directly."""
from pathlib import Path

import numpy as np
import pandas as pd
import torch

from .. import engine


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
