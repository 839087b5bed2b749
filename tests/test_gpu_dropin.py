"""GPU drop-in surface: KmerExtractor writes the reference's files byte for byte, the CLI
behaves like scripts/extract_kmers.py, and the feature / distance kernels match float64
restatements within 1e-6 relative."""
import contextlib
import io

import numpy as np
import pytest

import oracle
from helpers import golden_dupk_cases, golden_extract_cases, golden_metadata_cases

pytestmark = pytest.mark.gpu
RTOL = 1e-6


def test_extractor_files_and_messages_match_reference(tmp_path):
    from kmerml_b200.kmers.generate import KmerExtractor
    n = 0
    for c in golden_extract_cases():
        fa = tmp_path / c["name"] / "GCF_900000001_1.fa"
        fa.parent.mkdir()
        fa.write_bytes(c["fasta"])
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            org = KmerExtractor(output_dir=tmp_path / c["name"] / "out", compress=False).extract_kmers_from_fasta(
                fa, list(c["k_values"]))
        assert org == c["organism_id"]
        assert buf.getvalue().splitlines() == c["stdout"], c["name"]
        for k, text in c["files"].items():
            got = (tmp_path / c["name"] / "out" / org / f"k{k}.txt").read_bytes()
            assert got == text.encode(), (c["name"], k)
        n += 1
    assert n >= 49


def test_duplicate_k_values_count_as_often(tmp_path):
    """k_values = [8, 2, 8]: the reference counts k = 8 twice (generate.py:36,49-58); fixtures from the reference."""
    from kmerml_b200.kmers.generate import KmerExtractor
    for c in golden_dupk_cases():
        fa = tmp_path / c["name"] / "GCF_900000001_1.fa"
        fa.parent.mkdir()
        fa.write_bytes(c["fasta"])
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            org = KmerExtractor(output_dir=tmp_path / c["name"] / "out", compress=False).extract_kmers_from_fasta(
                fa, list(c["k_values"]))
        assert buf.getvalue().splitlines() == c["stdout"], c["name"]
        for k, text in c["files"].items():
            assert (tmp_path / c["name"] / "out" / org / f"k{k}.txt").read_bytes() == text.encode(), (c["name"], k)


def test_extractor_gzip_and_genome_list(tmp_path, capsys):
    import gzip
    from kmerml_b200.kmers.generate import KmerExtractor
    cases = [c for c in golden_extract_cases() if c["name"] in ("G0", "rand03")]
    paths = []
    for c in cases:
        p = tmp_path / f"{c['name']}.fa"
        p.write_bytes(c["fasta"])
        paths.append(p)
    ex = KmerExtractor(output_dir=tmp_path / "o")            # compress=True is the reference default
    done = ex.extract_from_genome_list(paths + [tmp_path / "missing.fa"], [2, 8])
    out = capsys.readouterr().out
    assert done == ["G0", "rand03"]
    assert "Error processing missing" in out and "Completed processing 2 out of 3 genomes" in out
    g0 = cases[0]
    assert gzip.open(tmp_path / "o" / "G0" / "k8.txt.gz", "rt").read() == g0["files"]["8"]
    with pytest.raises(ValueError):
        ex.extract_from_genome_list(paths, [2], organism_ids=["only_one"])


def test_extract_cli(tmp_path, capsys):
    from kmerml_b200.scripts import extract_kmers
    c = next(c for c in golden_extract_cases() if c["name"] == "G0")
    (tmp_path / "raw").mkdir()
    (tmp_path / "raw" / "GCF_900000001_1.fa").write_bytes(c["fasta"])
    assert extract_kmers.main(["-i", str(tmp_path / "raw"), "-o", str(tmp_path / "k"), "-k", "a,b"]) == 1
    assert extract_kmers.main(["-i", str(tmp_path / "raw"), "-o", str(tmp_path / "k"), "-p", "*.nothing"]) == 1
    capsys.readouterr()
    assert extract_kmers.main(["-i", str(tmp_path / "raw"), "-o", str(tmp_path / "k"), "-k", "2,8"]) == 0
    out = capsys.readouterr().out
    assert "Found 1 genome files" in out and "Processing GCF_900000001_1 (1/1)" in out
    assert "K-mer extraction completed successfully" in out
    assert (tmp_path / "k" / "GCF_900000001_1" / "k2.txt").read_text() == c["files"]["2"]


def test_static_features_match_statistics_py():
    from kmerml_b200 import engine
    for k, compat in ((1, False), (4, False), (6, True), (8, True)):
        t = engine.static_features_device(k, compat=compat).cpu().numpy()
        rng = np.random.default_rng(k)
        for idx in list(range(min(4 ** k, 70))) + rng.integers(0, 4 ** k, 200).tolist():
            s = oracle.compat_kmer_string(idx, k) if compat else oracle.code_to_kmer(idx, k)
            f = oracle.kmer_features(s)
            want = [len(s), f["A_count"], f["C_count"], f["G_count"], f["T_count"], f["cpg_count"], f["has_repeat"],
                    "ACGT".index(s[0])]
            assert t[idx].tolist() == want, (k, compat, idx, s)


def test_normalize_and_distances():
    import torch
    from kmerml_b200 import engine, synth
    genomes = [synth.config3_genome(i, scale=0.02).tobytes() for i in range(12)]
    buf, offs = synth.pack([np.frombuffer(g, np.uint8) for g in genomes])
    res = engine.count_dense_device(torch.from_numpy(buf).cuda(), offs, [6, 8])
    counts = res.counts[:, 4 ** 6:].contiguous()
    ref_counts = np.stack([oracle.count_dense(g, 8) for g in genomes]).astype(np.float64)
    freq = engine.normalize_rows_device(counts, res.totals[:, 1]).cpu().numpy().astype(np.float64)
    want = ref_counts / ref_counts.sum(1, keepdims=True)
    assert np.all(np.abs(freq - want) <= RTOL * np.maximum(want, 1e-300))
    for metric in ("cosine", "euclidean"):
        ref = oracle.pairwise_distance(want, metric)
        for x in (counts if metric == "cosine" else None, torch.as_tensor(want, device="cuda"),
                  torch.as_tensor(want.astype(np.float32), device="cuda")):
            if x is None:
                continue
            d = engine.pairwise_distance_device(x, metric, out_dtype=torch.float64).cpu().numpy()
            tol = RTOL if x.dtype != torch.float32 else 2e-5      # float32 INPUT rounding, not accumulation
            off = ~np.eye(len(genomes), dtype=bool)
            assert np.all(np.abs(d - ref)[off] <= tol * np.abs(ref)[off]), (metric, x.dtype)
            assert np.all(np.diag(d) == 0)


def test_builder_from_counts_and_distance_matrix():
    import torch
    from kmerml_b200 import engine, synth
    from kmerml_b200.ml.features import KmerFeatureBuilder
    genomes = [synth.config3_genome(i, scale=0.004).tobytes() for i in range(5)]
    buf, offs = synth.pack([np.frombuffer(g, np.uint8) for g in genomes])
    res = engine.count_dense_device(torch.from_numpy(buf).cuda(), offs, [5])
    orgs = [f"GCF_90000000{i}_1" for i in range(5)]
    b = KmerFeatureBuilder()
    m = b.from_counts(res, orgs, 5)
    ref = np.stack([oracle.count_dense(g, 5) for g in genomes]).astype(np.int64)
    keep = ref.any(axis=0)
    assert list(m.columns) == [oracle.code_to_kmer(i, 5) for i in np.nonzero(keep)[0]]
    assert list(m.columns) == sorted(m.columns) and np.array_equal(m.to_numpy(), ref[:, keep])
    f = ref[:, keep] / ref[:, keep].sum(1, keepdims=True)
    np.testing.assert_allclose(b.normalize().to_numpy(), f, rtol=RTOL)
    for metric in ("cosine", "euclidean"):
        d = b.distance_matrix(metric).to_numpy()
        want = oracle.pairwise_distance(f, metric)
        off = ~np.eye(5, dtype=bool)
        assert np.all(np.abs(d - want)[off] <= RTOL * np.abs(want)[off])
    # filter_features / get_top_features (tests/test_ml.py:9-12 of the reference): column reductions on the GPU
    # against the float64 pandas restatement
    import pandas as pd
    frame = pd.DataFrame(ref[:, keep], index=orgs, columns=m.columns)
    prev, var = (frame != 0).mean(axis=0), frame.var(axis=0, ddof=0)
    nnz, mean, dvar = engine.column_stats_device(b._device_counts[0])
    assert np.array_equal(nnz.cpu().numpy(), (frame != 0).sum(axis=0).to_numpy())
    np.testing.assert_allclose(mean.cpu().numpy(), frame.mean(axis=0).to_numpy(), rtol=1e-12)
    np.testing.assert_allclose(dvar.cpu().numpy(), var.to_numpy(), rtol=1e-9, atol=1e-12)
    thr = float(np.median(var))
    got = b.filter_features(min_prevalence=0.6, min_variance=thr)
    want_cols = frame.columns[((prev >= 0.6) & (var >= thr * (1 - 1e-9))).to_numpy()]
    assert set(got.columns) <= set(frame.columns[(prev >= 0.6).to_numpy()]) and abs(len(got.columns) - len(want_cols)) <= 2
    top = b.get_top_features(n_features=20)
    assert top.shape == (5, 20)
    # the clustering entry points (stubs in the reference) on the GPU distance matrix
    from kmerml_b200.ml import clustering
    labels, z = clustering.hierarchical_clustering(m, n_clusters=2, method="average", metric="cosine")
    assert z.shape == (4, 4) and set(labels) <= {0, 1} and len(labels) == 5
    assert len(clustering.dbscan_clustering(m, eps=1.0, min_samples=2)) == 5
    assert float(var[top.columns].min()) >= float(np.sort(var.to_numpy())[-20]) * (1 - 1e-9)


def test_sparse_counts_match_oracle():
    import torch
    from kmerml_b200 import engine, synth
    g = synth.fasta_bytes([30_000, 20, 18_000], seed=31)
    g[10_000:10_400] = ord("N")
    dev = torch.from_numpy(g).cuda()
    for k, canonical in ((15, False), (21, False), (21, True), (32, False), (31, True), (8, False)):
        keys, counts, first, windows = engine.count_sparse_device(dev, k, canonical=canonical)
        ref_codes, ref_counts = oracle.count_sparse(g.tobytes(), k)
        if canonical:
            agg = {}
            for c, n in zip(ref_codes.tolist(), ref_counts.tolist()):
                cc = min(c, oracle.revcomp_code(c, k))
                agg[cc] = agg.get(cc, 0) + n
        else:
            agg = dict(zip(ref_codes.tolist(), ref_counts.tolist()))
        got = dict(zip(keys.cpu().numpy().view(np.uint64).tolist(), counts.cpu().numpy().view(np.uint32).tolist()))
        assert got == agg, (k, canonical)
        assert windows == sum(agg.values())
        if not canonical:                                  # first-occurrence order = dict insertion order
            order = np.argsort(first.cpu().numpy().view(np.uint32), kind="stable")
            assert keys.cpu().numpy().view(np.uint64)[order].tolist() == ref_codes.tolist()


def test_tensor_core_gram_is_exact():
    """tcgen05 kind::i8 Gram of count rows (uint8 digit planes): distances equal the int64/float64
    reference to the last bit of the final float64 arithmetic, also with 2-, 3- and 4-byte counts and ragged
    n; the float64 CUDA-core path (float input) agrees within 1e-12."""
    import torch
    from kmerml_b200 import engine
    rng = np.random.default_rng(5)
    for n, m, hi in ((3, 64, 255), (129, 1024, 256), (77, 4096, 70_000), (260, 16384, 1000), (40, 256, 1 << 26)):
        c = rng.integers(0, hi, size=(n, m), dtype=np.int64)
        c[rng.integers(0, n)] = 0                                     # an all-zero row -> nan cosine distances
        x = torch.from_numpy(c.astype(np.uint32).view(np.int32)).cuda()
        g = (c @ c.T).astype(np.float64)
        nrm = np.sqrt(np.diag(g))
        for metric in ("cosine", "euclidean"):
            got = engine.pairwise_distance_device(x, metric, out_dtype=torch.float64).cpu().numpy()
            with np.errstate(divide="ignore", invalid="ignore"):
                if metric == "cosine":
                    ref = 1.0 - g / (nrm[:, None] * nrm[None, :])
                else:
                    ref = np.sqrt(np.maximum(np.diag(g)[:, None] + np.diag(g)[None, :] - 2 * g, 0))
            np.fill_diagonal(ref, 0.0)
            ok = np.isclose(got, ref, rtol=1e-13, atol=0, equal_nan=True)
            assert ok.all(), (n, m, hi, metric, np.abs(got - ref)[~ok][:3])
            alt = engine.pairwise_distance_device(torch.as_tensor(c.astype(np.float64), device="cuda"), metric,
                                                  out_dtype=torch.float64).cpu().numpy()
            assert np.allclose(got, alt, rtol=1e-12, atol=1e-12, equal_nan=True)


def test_feature_csv_text_from_the_gpu(tmp_path):
    """KmerFeatureExtractor with the GPU text path (csrc/featcsv.cu: parse, classify by composition, size, write)
    writes the same bytes as its pandas path -- which tests/test_host_layer.py pins on the reference's own CSVs
    (statistics.py:95-251, leading-zero quirk included)."""
    import gzip
    import json
    import os
    from helpers import GOLDEN
    from kmerml_b200.kmers.statistics import KmerFeatureExtractor
    with open(os.path.join(GOLDEN, "stats_cases.json")) as f:
        stats = json.load(f)
    by_name = {c["name"]: c for c in golden_extract_cases()}
    n = 0
    for ci, case in enumerate(stats):
        src = by_name[case["name"]]
        kdir = tmp_path / f"c{ci}" / "kmers" / "GCF_900000001_1"
        kdir.mkdir(parents=True)
        paths = []
        for k, text in src["files"].items():
            p = kdir / f"k{k}.txt"
            p.write_text(text)
            paths.append(p)
        outs = {}
        for dev in ("auto", None):
            with contextlib.redirect_stdout(io.StringIO()):
                res = KmerFeatureExtractor(input_paths=paths, output_dir=tmp_path / f"c{ci}" / f"f_{dev}", device=dev
                                           ).extract_features(case["feature_set"])
            path = res["GCF_900000001_1"]
            outs[dev] = path.read_bytes() if path is not None else None
        assert outs["auto"] == outs[None], (case["name"], case["feature_set"])
        if case["csv"] is not None and outs["auto"].decode() == case["csv"]:
            n += 1
    assert n >= 15                                             # byte-identical to the reference's CSV (entropy ulps aside)
    # a larger file (every 8-mer, counts up to 10^6), gzip input, a genome_size column, and a file the GPU parser
    # hands back to pandas (letters instead of digits)
    rng = np.random.default_rng(5)
    kdir = tmp_path / "big" / "kmers" / "GCF_900000002_1"
    kdir.mkdir(parents=True)
    digits = np.array(["".join("0231"[(i >> (2 * (7 - j))) & 3] for j in range(8)) for i in range(4 ** 8)])
    order = rng.permutation(4 ** 8)
    text = "".join(f"{digits[i]}\t{int(c)}\n" for i, c in zip(order, rng.integers(1, 10 ** 6, 4 ** 8)))
    (kdir / "k8.txt").write_text(text)
    with gzip.open(kdir / "k5.txt.gz", "wt") as f:
        f.write("".join(f"{digits[i][:5]}\t{i + 1}\n" for i in order[:700]))
    (kdir / "k3.txt").write_text("ACG\t5\nTTT\t2\n")
    meta = tmp_path / "big" / "genome_metadata.json"
    meta.write_text(json.dumps({"GCF_900000002_1": {"total_size": 12157105}}))
    outs = {}
    for dev in ("auto", None):
        with contextlib.redirect_stdout(io.StringIO()):
            res = KmerFeatureExtractor(input_paths=[tmp_path / "big" / "kmers"], output_dir=tmp_path / "big" / f"f_{dev}",
                                       metadata_file=meta, device=dev).extract_features()
        outs[dev] = res["GCF_900000002_1"].read_bytes()
    assert outs["auto"] == outs[None] and outs["auto"].count(b"\n") == 1 + 4 ** 8 + 700 + 2


def test_distance_row_blocks_match_full_matrix():
    """kmerml_pairwise_distance_rows: the row blocks the ranks of a sharded distance computation own,
    concatenated, are bit-identical to the single-call matrix (exact integer Gram entries)."""
    import torch
    from kmerml_b200 import engine
    rng = np.random.default_rng(11)
    for n, m, hi in ((5, 64, 300), (131, 4096, 70000), (300, 65536, 40)):
        X = torch.from_numpy(rng.integers(0, hi, (n, m)).astype(np.int32)).cuda()
        for metric in ("cosine", "euclidean"):
            full = engine.pairwise_distance_device(X, metric, out_dtype=torch.float64)
            for world in (1, 3, 8):
                per = (n + world - 1) // world
                blocks = [engine.pairwise_distance_rows_device(X, min(r * per, n), min((r + 1) * per, n), metric,
                                                               out_dtype=torch.float64) for r in range(world)]
                assert torch.equal(torch.cat(blocks), full), (n, m, metric, world)
        want = oracle.pairwise_distance(X.cpu().numpy().astype(np.float64), "cosine")
        got = engine.pairwise_distance_rows_device(X, 0, n, "cosine", out_dtype=torch.float64).cpu().numpy()
        assert np.all(np.abs(got - want) <= RTOL * np.maximum(np.abs(want), 1e-30) + 1e-12)


def test_distance_from_plane_shards_matches_full_matrix():
    """kmerml_count_planes + kmerml_distance_rows_planes: the sharded C3 route (every rank splits ITS rows into byte
    planes, the planes are gathered, row blocks from the planes) emulated on one GPU -- bit-identical to the single-call
    matrix, for 1..4 planes, uneven shards with padding rows, strided input rows."""
    import torch
    from kmerml_b200 import engine
    from kmerml_b200 import dist as kdist
    rng = np.random.default_rng(12)
    for n, m, hi, world in ((5, 64, 200, 2), (131, 4096, 70000, 3), (300, 65536, 900, 8), (40, 256, 2 ** 26, 4), (9, 128, 2 ** 20, 1)):
        wide = torch.from_numpy(rng.integers(0, hi, (n, m + 8)).astype(np.int64).astype(np.uint32).view(np.int32)).cuda()
        X = wide[:, :m]                                            # row stride m + 8: not contiguous
        shards = kdist.shard_genomes([int(v) for v in rng.integers(1, 100, n)], world)
        n_max = max(len(s) for s in shards)
        for metric in ("cosine", "euclidean"):
            full = engine.pairwise_distance_device(X.contiguous(), metric, out_dtype=torch.float64)
            parts = [engine.count_planes_device(X[torch.tensor(s, dtype=torch.long, device="cuda")] if s else X[:0], n_rows=n_max)
                     for s in shards]
            top = max(int(p[2].item()) & 0xFFFFFFFF for p in parts)
            nd = engine.planes_needed(top)
            assert nd == engine.planes_needed(int(X.contiguous().view(-1).cpu().numpy().view(np.uint32).max()))
            planes = torch.cat([p[0] for p in parts], dim=1)[:nd].contiguous()          # what the all_gathers assemble
            sumsq = torch.cat([p[1] for p in parts])
            blocks = [engine.distance_rows_planes_device(planes, nd, sumsq, r * n_max, (r + 1) * n_max, metric,
                                                         out_dtype=torch.float64) for r in range(world)]
            pos = kdist._gathered_positions(shards, X.device)
            got = torch.cat(blocks)[pos][:, pos]
            assert torch.equal(got, full), (n, m, hi, world, metric)


def test_genome_and_kmer_metadata():
    """Genome tallies (genome_metadata.py:55-85) and k-mer file summaries (kmer_metadata.py:59-78) from the GPU."""
    import torch
    from kmerml_b200 import engine
    for c in golden_extract_cases():
        a = np.frombuffer(c["fasta"], np.uint8) if len(c["fasta"]) else np.zeros(0, np.uint8)
        dev = torch.from_numpy(a.copy()).cuda() if a.size else torch.zeros(0, dtype=torch.uint8, device="cuda")
        got = engine.genome_stats_device(dev)
        want = oracle.genome_stats(c["fasta"])
        assert got["contigs"] == want["contigs"] and got["total_size"] == want["total_size"], c["name"]
        assert got["n_count"] == want["n_count"] and got["gc_content"] == want["gc_content"], c["name"]
    # ... and against what the reference's own managers wrote (tests/golden/metadata_cases.json), including
    # 400 contigs whose long headers hold G / C / N letters and cross the kernel's warp spans
    cases, big = golden_metadata_cases()
    for c in cases + big:
        a = np.frombuffer(c["fasta"], np.uint8) if len(c["fasta"]) else np.zeros(0, np.uint8)
        dev = torch.from_numpy(a.copy()).cuda() if a.size else torch.zeros(0, dtype=torch.uint8, device="cuda")
        got = engine.genome_stats_device(dev)
        for key in ("contigs", "total_size", "n_count", "gc_content"):
            assert got[key] == c["genome"][key], (c["name"], key)
    for c in cases:
        ks = [int(k) for k in c["kmers"] if int(k) <= 12]
        if not ks:
            continue
        dev = torch.from_numpy(np.frombuffer(c["fasta"], np.uint8).copy()).cuda()
        ml = max(int(k) for k in c["files"])
        res = engine.count_dense_device(dev, [0, dev.numel()], ks, min_record_len=ml, want_freq=False)
        for k in ks:
            assert engine.kmer_count_stats_device(res.counts_of(0, k), k) == c["kmers"][str(k)], (c["name"], k)
    # the drop-in managers (same JSON layout as the reference's) give the same records from files
    import tempfile
    from pathlib import Path
    from kmerml_b200.utils.genome_metadata import GenomeMetadataManager
    from kmerml_b200.utils.kmer_metadata import KmerMetadataManager
    with tempfile.TemporaryDirectory() as td:
        raw = Path(td) / "raw"
        raw.mkdir()
        picks = [c for c in cases if c["genome"]["contigs"] > 0][:6]
        for i, c in enumerate(picks):
            (raw / f"GCF_90000000{i}_1.fa").write_bytes(c["fasta"])
            kdir = Path(td) / "kmers" / f"GCF_90000000{i}_1"
            kdir.mkdir(parents=True)
            for k, text in c["files"].items():
                if text:
                    (kdir / f"k{k}.txt").write_text(text)
        gm = GenomeMetadataManager(Path(td) / "meta" / "genome_metadata.json")
        meta = gm.collect_metadata(raw)
        km = KmerMetadataManager(Path(td) / "meta" / "genome_metadata.json")
        km.add_kmer_metadata(sorted((Path(td) / "kmers").glob("*/k*.txt")))
        for i, c in enumerate(picks):
            org = f"GCF_90000000{i}_1"
            for key in ("contigs", "total_size", "n_count", "gc_content"):
                assert meta[org][key] == c["genome"][key], (c["name"], key)
            assert gm.get_genome_size(org) == c["genome"]["total_size"]
            for k, want in c["kmers"].items():
                got = {key: km.metadata[org]["kmers"][k][key] for key in want}
                assert got == want, (c["name"], k)
    g0 = next(c for c in golden_extract_cases() if c["name"] == "rand07")
    ks = [k for k in g0["k_values"] if k <= 12]
    dev = torch.from_numpy(np.frombuffer(g0["fasta"], np.uint8).copy()).cuda()
    res = engine.count_dense_device(dev, [0, dev.numel()], ks, min_record_len=max(g0["k_values"]), want_freq=False)
    for k in ks:
        counts = np.array([int(line.split("\t")[1]) for line in g0["files"][str(k)].splitlines()])
        s = engine.kmer_count_stats_device(res.counts_of(0, k), k)
        assert s["total_kmers"] == counts.sum() and s["unique_kmers"] == counts.size
        assert s["max_count"] == counts.max() and s["min_count"] == counts.min()
        assert s["mean_count"] == float(counts.mean()) and s["median_count"] == float(np.median(counts))
        assert s["estimated_genome_size"] == counts.sum() + k - 1


def test_gpu_formatter_matches_golden_text():
    """kmerml_format_kmer_file / _lines: the k{k}.txt text straight from the GPU, byte-identical to the files the
    unmodified reference wrote (tests/golden) -- dense rows, canonical rows and the sparse path."""
    import torch
    from kmerml_b200 import engine
    from kmerml_b200.kmers.generate import format_kmer_lines
    for c in golden_extract_cases():
        if not len(c["fasta"]):
            continue
        dev = torch.from_numpy(np.frombuffer(c["fasta"], np.uint8).copy()).cuda()
        max_k = max(c["k_values"])
        ks = [k for k in dict.fromkeys(c["k_values"]) if k <= 12]
        if ks:
            res = engine.count_dense_device(dev, [0, dev.numel()], ks, min_record_len=max_k, want_freq=False)
            for k in ks:
                first = engine.first_occurrence_device(dev, k, min_record_len=max_k)
                text = engine.format_kmer_file_device(res.counts_of(0, k), first, k).cpu().numpy().tobytes()
                assert text == c["files"][str(k)].encode(), (c["name"], k)
        for k in [k for k in dict.fromkeys(c["k_values"]) if k > 14][:1]:
            keys, cnts, first, _ = engine.count_sparse_device(dev, k, min_record_len=max_k)
            order = torch.argsort(first.to(torch.int64) & 0xFFFFFFFF, stable=True)
            text = engine.format_kmer_lines_device(keys[order].contiguous(), cnts[order].contiguous(), k)
            assert text.cpu().numpy().tobytes() == c["files"][str(k)].encode(), (c["name"], k)
    # canonical rows and counts with several digits against the host formatter
    rng = np.random.default_rng(8)
    data = b">r\n" + np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 300_000)].tobytes() + b"\n>s\n" + b"A" * 5000 + b"\n"
    dev = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).cuda()
    for canonical in (False, True):
        res = engine.count_dense_device(dev, [0, dev.numel()], [3, 7], canonical=canonical, want_freq=False)
        for k in (3, 7):
            first = engine.first_occurrence_device(dev, k, min_record_len=7)
            got = engine.format_kmer_file_device(res.counts_of(0, k), first, k, canonical=canonical).cpu().numpy().tobytes()
            counts = res.counts_numpy(0, k)
            f = first.cpu().numpy().view(np.uint32)
            if canonical:
                f = np.minimum(f, f[engine.revcomp_codes(k)])
            obs = np.nonzero(counts)[0]
            obs = obs[np.argsort(f[obs], kind="stable")]
            assert got == bytes(format_kmer_lines(obs, counts[obs], k)), (canonical, k)


def test_extractor_reproduces_big_reference_outputs(tmp_path):
    """KmerExtractor on the GPU against the files the unmodified reference wrote for inputs of a few hundred
    kilobases (SHA-256 of every k{k}.txt): unwrapped lines, a 150 kb header made of base letters, tandem repeats
    (slot overflow), CRLF + N runs, thousands of short records (tail lists)."""
    import contextlib
    import hashlib
    import io
    from helpers import golden_big_cases
    from kmerml_b200.kmers.generate import KmerExtractor
    for case in golden_big_cases():
        fa = tmp_path / f"{case['name']}.fa"
        fa.write_bytes(case["fasta"])
        with contextlib.redirect_stdout(io.StringIO()):
            org = KmerExtractor(output_dir=tmp_path / "out", compress=False).extract_kmers_from_fasta(fa, case["k_values"])
        for k in case["k_values"]:
            data = (tmp_path / "out" / org / f"k{k}.txt").read_bytes()
            want = case["files"][str(k)]
            assert data.count(b"\n") == want["lines"], (case["name"], k)
            assert hashlib.sha256(data).hexdigest() == want["sha256"], (case["name"], k)
