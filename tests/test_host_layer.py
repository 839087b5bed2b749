"""Host-side drop-in layer (statistics CSVs, feature matrix, path utils, CLI argument
handling) against the fixtures produced by the unmodified reference.  No GPU."""
import contextlib
import io
import json
import os

import numpy as np
import pandas as pd
import pytest

from helpers import GOLDEN, golden_extract_cases

from kmerml_b200.kmers.statistics import KmerFeatureExtractor, features_from_digits
from kmerml_b200.ml.features import KmerFeatureBuilder
from kmerml_b200.scripts import generate_kmers_features
from kmerml_b200.utils.path_utils import ensure_directory_exists, find_files, is_valid_file

EXTRACT = {c["name"]: c for c in golden_extract_cases()}
with open(os.path.join(GOLDEN, "stats_cases.json")) as fh:
    STATS = json.load(fh)
with open(os.path.join(GOLDEN, "matrix_cases.json")) as fh:
    MATRICES = json.load(fh)


def write_kmer_files(root, organism, case):
    kdir = root / "kmers" / organism
    kdir.mkdir(parents=True)
    paths = []
    for k, text in case["files"].items():
        p = kdir / f"k{k}.txt"
        p.write_text(text)
        paths.append(p)
    return paths


@pytest.mark.parametrize("case", STATS, ids=[f"{c['name']}-{len(c['feature_set'] or [])}" for c in STATS])
def test_statistics_csv_matches_reference(case, tmp_path):
    paths = write_kmer_files(tmp_path, "GCF_900000001_1", EXTRACT[case["name"]])
    with contextlib.redirect_stdout(io.StringIO()) as out:
        res = KmerFeatureExtractor(input_paths=paths, output_dir=tmp_path / "f").extract_features(case["feature_set"])
    path = res["GCF_900000001_1"]
    if case["csv"] is None:
        assert path is None and "No features extracted" in out.getvalue()
        return
    got = path.read_text()
    if got == case["csv"]:
        return                                              # byte-identical (the usual case)
    # the reference sums the entropy terms in set-iteration (hash) order: last-ulp differences only
    a, b = pd.read_csv(io.StringIO(got)), pd.read_csv(io.StringIO(case["csv"]))
    assert list(a.columns) == list(b.columns) and a.shape == b.shape
    for col in a.columns:
        if a[col].dtype.kind == "f":
            np.testing.assert_allclose(a[col].to_numpy(), b[col].to_numpy(), rtol=1e-12, atol=0)
        else:
            assert a[col].equals(b[col]), col


@pytest.mark.parametrize("case", MATRICES, ids=[f"{'+'.join(c['cases'])}-{c['metric']}" for c in MATRICES])
def test_feature_matrix_matches_reference(case, tmp_path):
    fdir = tmp_path / "features"
    for gi, name in enumerate(case["cases"]):
        org = f"GCF_90000000{gi}_1"
        paths = write_kmer_files(tmp_path / org, org, EXTRACT[name])
        with contextlib.redirect_stdout(io.StringIO()):
            KmerFeatureExtractor(input_paths=paths, output_dir=fdir).extract_features()
    b = KmerFeatureBuilder(fdir)
    m = b.build_from_statistics_files(metric=case["metric"])
    assert [str(x) for x in m.index] == case["index"]
    assert [str(x) for x in m.columns] == case["columns"]
    np.testing.assert_allclose(m.to_numpy(dtype=np.float64), np.asarray(case["values"]), rtol=1e-12, atol=0)
    assert b.organisms == case["index"] and [str(x) for x in b.kmers] == case["columns"]
    if case["metric"] == "count":
        assert m.dtypes.map(lambda d: d.kind).eq("i").all()
        freq = b.normalize("frequency")
        np.testing.assert_allclose(freq.sum(axis=1).to_numpy(), 1.0, rtol=1e-12)


def test_leading_zero_quirk():
    """02310231 (ACGTACGT) is read as the integer 2310231 and decodes to CGTACGT; 00 -> "A"."""
    cols = features_from_digits(np.array([2310231, 0, 12]), ["gc_content", "base_counts"])
    assert list(cols["kmer"]) == ["CGTACGT", "A", "TC"]
    assert list(cols["A_count"]) == [1, 1, 0] and list(cols["C_count"]) == [2, 0, 1]


def test_builder_errors(tmp_path):
    with pytest.raises(ValueError, match="Statistics directory not set"):
        KmerFeatureBuilder().build_from_statistics_files()
    with pytest.raises(ValueError, match="No statistics files found"):
        KmerFeatureBuilder(tmp_path).build_from_statistics_files()
    assert KmerFeatureBuilder._extract_organism_id(tmp_path / "GCF_000146045_2_kmer_features.csv") == "GCF_000146045"


def test_path_utils(tmp_path):
    d = ensure_directory_exists(tmp_path / "a" / "b")
    (d / "x.fa").write_text(">x\nAC\n")
    (tmp_path / "a" / "y.fasta").write_text(">y\nAC\n")
    assert [p.name for p in find_files(tmp_path / "a", ["*.fa", "*.fasta"])] == ["y.fasta"]
    assert [p.name for p in find_files(tmp_path / "a", ["*.fa", "*.fasta"], recursive=True)] == ["x.fa", "y.fasta"]
    assert is_valid_file(d / "x.fa") and not is_valid_file(d)


def test_features_cli(tmp_path, capsys):
    assert generate_kmers_features.main(["-i", str(tmp_path), "-o", str(tmp_path / "o"), "-m", str(tmp_path / "m.json")]) == 1
    assert "No k-mer files found" in capsys.readouterr().out
    write_kmer_files(tmp_path, "GCF_1_1", EXTRACT["G0"])
    assert generate_kmers_features.main(["-i", str(tmp_path / "kmers"), "-o", str(tmp_path / "o"), "-k", "x"]) == 1
    assert generate_kmers_features.main(["-i", str(tmp_path / "kmers"), "-o", str(tmp_path / "o"), "-f", "nope",
                                         "-m", str(tmp_path / "m.json")]) == 1
    rc = generate_kmers_features.main(["-i", str(tmp_path / "kmers"), "-o", str(tmp_path / "o"), "-f", "basic",
                                       "-k", "2,8", "-m", str(tmp_path / "m.json")])
    out = capsys.readouterr().out
    assert rc == 0 and "Found 2 k-mer files" in out and "Generated 1 feature files" in out
    cols = list(pd.read_csv(tmp_path / "o" / "GCF_1_1_kmer_features.csv").columns)
    assert cols == ["kmer", "count", "k", "gc_percent", "A_count", "C_count", "G_count", "T_count"]


def test_install_as_kmerml():
    import sys
    import kmerml_b200
    saved = {k: v for k, v in sys.modules.items() if k == "kmerml" or k.startswith("kmerml.") or k == "scripts" or k.startswith("scripts.")}
    try:
        kmerml_b200.install_as_kmerml()
        from kmerml.kmers.generate import KmerExtractor                    # noqa: F401
        from kmerml.kmers.statistics import KmerFeatureExtractor as K2
        from kmerml.ml.features import KmerFeatureBuilder as B2
        from kmerml.utils.path_utils import find_files as f2
        from scripts import extract_kmers                                  # noqa: F401
        assert K2 is KmerFeatureExtractor and B2 is KmerFeatureBuilder and f2 is find_files
    finally:
        for k in [k for k in sys.modules if k == "kmerml" or k.startswith("kmerml.") or k == "scripts" or k.startswith("scripts.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_fast_csv_writer_equals_pandas(tmp_path):
    """The feature CSV is assembled from one pandas-formatted row per distinct feature combination; the text must
    be exactly what DataFrame.to_csv writes for the concatenated frames (with and without genome_size)."""
    from kmerml_b200.kmers import statistics as st
    rng = np.random.default_rng(12)
    fx = KmerFeatureExtractor(output_dir=tmp_path / "o")
    frames = []
    for k in (3, 7, 11):
        digits = rng.integers(0, 4, (4000, k))
        vals = (digits * (10 ** np.arange(k - 1, -1, -1))).sum(1).astype(np.int64)      # leading zeros vanish, as in pandas
        df = pd.DataFrame({"kmer": vals, "count": rng.integers(1, 10 ** rng.integers(1, 7), 4000)})
        frames.append(fx._extract_kmer_features(df, k, "org", st.ALL_FEATURES))
    for genome_size in (None, 12157105):
        want = pd.concat(frames, ignore_index=True)
        if genome_size:
            want["genome_size"] = genome_size
        assert st._fast_csv(frames, genome_size) == want.to_csv(index=False)
    sub = [f[["kmer", "count", "k", "gc_percent"]] for f in frames]
    assert st._fast_csv(sub, None) == pd.concat(sub, ignore_index=True).to_csv(index=False)
    only = [f[["kmer", "count", "k"]] for f in frames]
    assert st._fast_csv(only, None) == pd.concat(only, ignore_index=True).to_csv(index=False)


REFERENCE = os.environ.get("KMERML_REFERENCE", "")


@pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "kmerml"))),
                    reason="set KMERML_REFERENCE to a source tree of the original kmer-ml project")
def test_statistics_csv_against_the_live_reference(tmp_path):
    """Where a source tree of the original project is at hand (KMERML_REFERENCE): the unmodified KmerFeatureExtractor
    (child process) and the drop-in write the feature CSV for the same fresh random k-mer files; identical except for
    the last ulps of the entropy columns, which the reference sums in set-iteration (hash) order."""
    import random
    import subprocess
    import sys
    import oracle
    from helpers import fuzz_fasta
    rng = random.Random(os.getpid())
    specs = []
    for i in range(12):
        data = fuzz_fasta(rng)
        ks = sorted(rng.sample(range(1, 9), rng.randint(1, 3)))
        kdir = tmp_path / f"k{i}" / f"GCF_90000{i:04d}_1"
        kdir.mkdir(parents=True)
        wrote = False
        for k in ks:
            text = oracle.kmer_file_text(data, k, max(ks))
            (kdir / f"k{k}.txt").write_text(text)
            wrote |= bool(text)
        fs = rng.choice([None, ["gc_content", "base_counts"], ["gc_content", "base_counts", "entropy", "cpg_sites", "repeats"]])
        specs.append((i, fs, wrote))
    script = (
        "import sys, json, contextlib, io\n"
        f"sys.path.insert(0, {REFERENCE!r})\n"
        "from kmerml.kmers.statistics import KmerFeatureExtractor\n"
        "root, spec = sys.argv[1], json.loads(sys.argv[2])\n"
        "for i, fs, _ in spec:\n"
        "    with contextlib.redirect_stdout(io.StringIO()):\n"
        "        KmerFeatureExtractor(input_paths=[f'{root}/k{i}'], output_dir=f'{root}/ref{i}').extract_features(fs)\n"
    )
    subprocess.run([sys.executable, "-c", script, str(tmp_path), json.dumps(specs)], check=True, timeout=600)
    for i, fs, wrote in specs:
        with contextlib.redirect_stdout(io.StringIO()):
            KmerFeatureExtractor(input_paths=[tmp_path / f"k{i}"], output_dir=tmp_path / f"new{i}").extract_features(fs)
        name = f"GCF_90000{i:04d}_1_kmer_features.csv"
        ref_file, new_file = tmp_path / f"ref{i}" / name, tmp_path / f"new{i}" / name
        assert ref_file.exists() == new_file.exists(), i
        if not ref_file.exists():
            continue
        got, want = new_file.read_text(), ref_file.read_text()
        if got == want:
            continue
        a, b = pd.read_csv(io.StringIO(got)), pd.read_csv(io.StringIO(want))
        assert list(a.columns) == list(b.columns) and a.shape == b.shape, i
        for col in a.columns:
            if a[col].dtype.kind == "f":
                np.testing.assert_allclose(a[col].to_numpy(), b[col].to_numpy(), rtol=1e-12, atol=0)
            else:
                assert a[col].equals(b[col]), (i, col)


def test_clustering_entry_points_on_injected_distances():
    """kmerml/ml/clustering.py:6-16 are `pass` stubs in the reference; here they run on the genome x genome distance
    matrix (injected in this CPU test; the GPU produces it otherwise)."""
    from kmerml_b200.ml import clustering
    rng = np.random.default_rng(0)
    a = rng.normal(0, 0.05, (6, 8)) + np.array([1, 0, 0, 0, 0, 0, 0, 0])
    b = rng.normal(0, 0.05, (5, 8)) + np.array([0, 0, 0, 1, 0, 0, 0, 0])
    x = np.abs(np.vstack([a, b]))
    d = np.sqrt(((x[:, None, :] - x[None, :, :]) ** 2).sum(-1))
    labels, z = clustering.hierarchical_clustering(pd.DataFrame(x), n_clusters=2, distances=d)
    assert z.shape == (10, 4) and len(set(labels[:6])) == 1 and len(set(labels[6:])) == 1 and labels[0] != labels[6]
    assert clustering.hierarchical_clustering(x, distances=d)[0] is None
    km, centres = clustering.kmeans_clustering(x, n_clusters=2)
    assert centres.shape == (2, 8) and len(set(km[:6])) == 1 and km[0] != km[6]
    db = clustering.dbscan_clustering(x, eps=0.5, min_samples=3, distances=d)
    assert set(db) == {0, 1}
    with pytest.raises(ValueError):
        clustering.hierarchical_clustering(x, distances=np.zeros((3, 4)))


def test_encode_restatement_agrees_with_the_oracle():
    """tests/helpers.encode_reference (the checker of kmerml_encode) against the pinned oracle: the symbols it marks
    are exactly the windows the oracle counts at k = 1."""
    import random
    import oracle
    from helpers import encode_reference, fuzz_fasta, golden_extract_cases
    rng = random.Random(11)
    datas = [fuzz_fasta(rng) for _ in range(150)] + [c["fasta"] for c in golden_extract_cases()[:20]]
    for d in datas:
        sym = encode_reference(d)
        hist = np.bincount(sym[sym < 4], minlength=4).astype(np.uint64)
        assert np.array_equal(hist, oracle.count_dense(d, 1, 1)), d[:80]
