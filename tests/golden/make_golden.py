#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/ by running the UNMODIFIED
reference (a source tree of the original kmer-ml project, named by
KMERML_REFERENCE) under the Bio.SeqIO shim in tests/_ref.

The fixtures it writes are committed; tests read only the fixtures.

    KMERML_REFERENCE=<kmer-ml source tree> python tests/golden/make_golden.py

Outputs
  extract_cases.json  - FASTA texts + KmerExtractor outputs (k{k}.txt lines in
                        file order) + stdout lines, from
                        kmerml/kmers/generate.py:21-91
  stats_cases.json    - KmerFeatureExtractor CSV text for small k files, from
                        kmerml/kmers/statistics.py:35-147
  matrix_cases.json   - KmerFeatureBuilder matrices, from
                        kmerml/ml/features.py:28-117
  ref_timing.json     - single-core timings of the reference extractor here
  extract_dupk_cases.json - k_values holding the same k more than once (the reference counts it as
                        often, generate.py:36,49-58), same layout as extract_cases.json
  metadata_cases.json - GenomeMetadataManager._extract_genome_metadata (utils/genome_metadata.py:55-85)
                        and KmerMetadataManager._calculate_basic_stats (utils/kmer_metadata.py:59-78) on
                        the extraction cases
  extract_big_cases.json - inputs of a few 100 kb (unwrapped, long header, repeats, CRLF + N runs, many short
                        records): gzip FASTA + SHA-256 / line count of every k{k}.txt the reference wrote
"""
import base64
import contextlib
import io
import json
import os
import random
import sys
import tempfile
import time
from pathlib import Path

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent / "_ref"))      # the Bio shim
REFERENCE = os.environ.get("KMERML_REFERENCE", "")
if not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "kmerml"))):
    sys.exit("set KMERML_REFERENCE to a source tree of the original kmer-ml project")
sys.path.insert(1, REFERENCE)                      # the unmodified reference

from kmerml.kmers.generate import KmerExtractor              # noqa: E402
from kmerml.kmers.statistics import KmerFeatureExtractor     # noqa: E402
from kmerml.ml.features import KmerFeatureBuilder            # noqa: E402
from kmerml.utils.genome_metadata import GenomeMetadataManager    # noqa: E402
from kmerml.utils.kmer_metadata import KmerMetadataManager        # noqa: E402


G0 = (">chr1 test contig\nAAAAAATCGGNACGTacgtAAAAAATC\nAAAC\n>short\nACGTA\n>chr2\nACGTRACGTACGT\n")


def rand_fasta(rng, n_records, max_len, alphabet, width_choices, eol="\n", tail_newline=True,
               junk_prefix="", weird_ws=False):
    out = [junk_prefix]
    for r in range(n_records):
        out.append(f">rec{r} some description{eol}")
        length = rng.choice([0, 1, 2, 3, 5, 7, 8, 11, 12, 13, rng.randint(0, max_len), rng.randint(0, max_len)])
        seq = "".join(rng.choice(alphabet) for _ in range(length))
        width = rng.choice(width_choices)
        for i in range(0, len(seq), width):
            line = seq[i:i + width]
            if weird_ws and rng.random() < 0.2:
                line = line + rng.choice([" ", "  ", "\t", " \t ", "\x0b", "\x0c"])
            if weird_ws and rng.random() < 0.1 and len(line) > 2:
                j = rng.randint(1, len(line) - 1)
                line = line[:j] + rng.choice([" ", "\t", " \t"]) + line[j:]
            out.append(line + eol)
        if weird_ws and rng.random() < 0.3:
            out.append(eol)
    text = "".join(out)
    if not tail_newline:
        text = text.rstrip("\r\n")
    return text


def extract_cases():
    rng = random.Random(20261018)
    cases = [
        ("G0", G0, [2, 8]),
        ("G0_k1to6", G0, [1, 2, 3, 4, 5, 6]),
        ("G0_unsorted_k", G0, [8, 2, 5]),
        ("empty_file", "", [3]),
        ("only_header", ">x\n", [3]),
        ("no_header", "ACGTACGTACGT\nACGT\n", [3]),
        ("junk_then_header", "; comment\nACGTACGT\n>r1\nACGTACGTAC\n", [2, 4]),
        ("gt_midline", ">r1\nACGT>ACGTACGT\nAC>GT\n>r2\nGGGGCCCC\n", [2, 4]),
        ("crlf", ">r1 x\r\nACGTACGTAC\r\nGTAC\r\n>r2\r\nTTTTGGGGCC\r\n", [3, 5]),
        ("lone_cr", ">r1\rACGTACGTAC\rGTAC\r>r2\rTTTTGGGGCC", [3, 5]),
        ("no_trailing_newline", ">r1\nACGTACGTACGTAAC", [4, 12]),
        ("all_n", ">r1\nNNNNNNNNNNNNNNNNNNNN\n", [2, 5]),
        ("lower", ">r1\nacgtnacgtacgtacgtttgaca\n", [1, 3, 12]),
        ("exact_len", ">a\nACGTACGTACGT\n>b\nACGTACGTACG\n>c\nACGTACGTACGTA\n", [3, 12]),
        ("header_only_records", ">a\n>b\n>c\nACGTAC\n>d\n", [2]),
        ("blank_lines", ">a\n\nACGT\n\n\nACGT\n\n>b\n\n\nGGGTTTAAAC\n", [2, 8]),
        ("spaces_tabs", ">a\nAC GT AC GT\nACGT\t\nAC\tGT\nAAAA \t \n", [2, 4]),
        ("homopolymer", ">a\n" + "A" * 300 + "\n" + "A" * 123 + "\n", [1, 6, 12]),
        ("single_line_long", ">a\n" + "".join(rng.choice("ACGT") for _ in range(5000)) + "\n", [7, 12]),
    ]
    for i in range(24):
        alphabet = rng.choice(["ACGT", "ACGT", "ACGTN", "ACGTacgtNnRY-*", "ACGTacgt", "AC"])
        text = rand_fasta(
            rng,
            n_records=rng.randint(1, 8),
            max_len=rng.choice([40, 200, 1500]),
            alphabet=alphabet,
            width_choices=rng.choice([[60], [80], [70], [1, 2, 3], [5, 7, 11], [1000000]]),
            eol=rng.choice(["\n", "\n", "\r\n"]),
            tail_newline=rng.random() < 0.7,
            junk_prefix=rng.choice(["", "", "", "junk line\n", "\n\n"]),
            weird_ws=(i % 3 == 2),
        )
        ks = sorted(rng.sample(range(1, 13), rng.randint(1, 4)))
        if i % 5 == 0:
            rng.shuffle(ks)
        cases.append((f"rand{i:02d}", text, ks))
    # large-k (sparse path) cases
    for i in range(6):
        text = rand_fasta(rng, n_records=rng.randint(1, 5), max_len=600,
                          alphabet=rng.choice(["ACGT", "ACGTN", "ACGTacgtNn"]),
                          width_choices=[rng.choice([60, 80, 13])])
        ks = sorted(rng.sample(range(13, 33), 2)) + ([rng.randint(2, 12)] if i % 2 else [])
        cases.append((f"largek{i:02d}", text, ks))

    out = []
    for name, text, ks in cases:
        with tempfile.TemporaryDirectory() as td:
            fa = Path(td) / "GCF_900000001_1.fa"
            # newline="" so that the bytes on disk are exactly `text`
            with open(fa, "w", newline="") as f:
                f.write(text)
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf):
                ex = KmerExtractor(output_dir=Path(td) / "out", compress=False)
                org = ex.extract_kmers_from_fasta(fa, list(ks))
            files = {}
            for k in dict.fromkeys(ks):
                files[str(k)] = (Path(td) / "out" / org / f"k{k}.txt").read_text()
            out.append({
                "name": name,
                "fasta_b64": base64.b64encode(text.encode("latin-1")).decode(),
                "k_values": list(ks),
                "organism_id": org,
                "stdout": buf.getvalue().splitlines(),
                "files": files,
            })
    return out


def run_extract(name, text, ks):
    with tempfile.TemporaryDirectory() as td:
        fa = Path(td) / "GCF_900000001_1.fa"
        with open(fa, "w", newline="") as f:
            f.write(text)
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            ex = KmerExtractor(output_dir=Path(td) / "out", compress=False)
            org = ex.extract_kmers_from_fasta(fa, list(ks))
        files = {}
        for k in dict.fromkeys(ks):
            files[str(k)] = (Path(td) / "out" / org / f"k{k}.txt").read_text()
        return {"name": name, "fasta_b64": base64.b64encode(text.encode("latin-1")).decode(),
                "k_values": list(ks), "organism_id": org, "stdout": buf.getvalue().splitlines(), "files": files}


def dupk_cases():
    """k_values with repeated entries: `for k in k_values` (generate.py:49) runs once per entry over one dict
    per distinct k (:36), so a k listed m times is counted m times."""
    rng = random.Random(424242)
    seq = lambda n, a="ACGT": "".join(rng.choice(a) for _ in range(n))       # noqa: E731
    multi = ">r1 d\n" + "\n".join(seq(60, "ACGTN") for _ in range(12)) + "\n>tiny\nACG\n>r2\n" + seq(333, "ACGTacgt") + "\n"
    cases = [
        ("dup_22", ">r\nACGTACGT\n", [2, 2]),
        ("dup_828", G0, [8, 2, 8]),
        ("dup_333", G0, [3, 3, 3]),
        ("dup_mixed_order", multi, [5, 12, 5, 1, 12, 12]),
        ("dup_large_k", multi, [21, 4, 21]),
        ("dup_short_skip", ">a\nACGTAC\n>b\nACGTACGTACGTACGT\n", [2, 9, 2]),
    ]
    return [run_extract(*c) for c in cases]


def metadata_cases(extract):
    """Genome tallies and k-mer count summaries as the reference's metadata managers compute them."""
    out = []
    picks = [c for c in extract if c["name"] in ("G0", "G0_k1to6", "crlf", "lone_cr", "lower", "all_n", "blank_lines",
                                                 "spaces_tabs", "header_only_records", "junk_then_header", "empty_file",
                                                 "gt_midline", "rand02", "rand05", "rand11", "rand17", "rand20", "largek01")]
    for c in picks:
        text = base64.b64decode(c["fasta_b64"]).decode("latin-1")
        with tempfile.TemporaryDirectory() as td:
            fa = Path(td) / "GCF_900000001_1.fa"
            with open(fa, "w", newline="") as f:
                f.write(text)
            gm = GenomeMetadataManager(Path(td) / "meta" / "genome_metadata.json")
            g = gm._extract_genome_metadata(fa)
            genome = {key: g[key] for key in ("contigs", "total_size", "gc_content", "n_count")}
            kdir = Path(td) / "kmers" / "GCF_900000001_1"
            kdir.mkdir(parents=True)
            km = KmerMetadataManager(Path(td) / "meta" / "genome_metadata.json")
            kstats = {}
            for k, txt in c["files"].items():
                if not txt:
                    continue                 # the manager fails on an empty file (max of an empty column)
                p = kdir / f"k{k}.txt"
                p.write_text(txt)
                st = km._calculate_basic_stats(p, int(k))
                kstats[k] = {key: st[key] for key in ("k_value", "total_kmers", "unique_kmers", "max_count", "min_count",
                                                      "mean_count", "median_count", "estimated_genome_size")}
            out.append({"name": c["name"], "genome": genome, "kmers": kstats})
    return out


def many_contig_metadata_case():
    """Header lines that hold G / C / N letters and cross 2 KB boundaries (the genome-stats kernel subtracts
    header bytes per warp span): hundreds of contigs with long descriptive headers."""
    rng = random.Random(99)
    parts = []
    for i in range(400):
        parts.append(f">contig{i} GC rich N unknown scaffold NNNN GGCC len={rng.randint(1, 10 ** rng.randint(1, 9))} {'CGN' * rng.randint(0, 40)}\n")
        s = "".join(rng.choice("ACGTNacgtn") for _ in range(rng.choice([0, 1, 30, 61, 200, 2030, 2047, 2048, 2049, 5000])))
        w = rng.choice([60, 80, 1000000])
        parts.append("\n".join(s[j:j + w] for j in range(0, len(s), w)) + "\n")
    text = "".join(parts)
    import gzip
    with tempfile.TemporaryDirectory() as td:
        fa = Path(td) / "many.fa"
        with open(fa, "w", newline="") as f:
            f.write(text)
        g = GenomeMetadataManager(Path(td) / "m" / "g.json")._extract_genome_metadata(fa)
    return {"name": "many_contigs_long_headers",
            "fasta_gz_b64": base64.b64encode(gzip.compress(text.encode("latin-1"), 9, mtime=0)).decode(),
            "genome": {key: g[key] for key in ("contigs", "total_size", "gc_content", "n_count")}}


def stats_and_matrix_cases(extract):
    stats, matrices = [], []
    picks = [c for c in extract if c["name"] in ("G0", "G0_k1to6", "rand00", "rand03", "rand07", "lower", "spaces_tabs")]
    for feature_set in (None, ["gc_content", "base_counts"],
                        ["gc_content", "base_counts", "entropy", "cpg_sites", "repeats"]):
        for c in picks:
            with tempfile.TemporaryDirectory() as td:
                kdir = Path(td) / "kmers" / "GCF_900000001_1"
                kdir.mkdir(parents=True)
                paths = []
                for k, txt in c["files"].items():
                    p = kdir / f"k{k}.txt"
                    p.write_text(txt)
                    paths.append(p)
                buf = io.StringIO()
                with contextlib.redirect_stdout(buf):
                    fx = KmerFeatureExtractor(input_paths=paths, output_dir=Path(td) / "features")
                    res = fx.extract_features(required_features=feature_set)
                csv_path = res["GCF_900000001_1"]
                csv_text = csv_path.read_text() if csv_path else None
                stats.append({"name": c["name"], "feature_set": feature_set,
                              "k_order": list(c["files"].keys()), "csv": csv_text})
    # feature matrices over several organisms
    groups = [("G0", "rand00", "rand03"), ("G0_k1to6", "lower", "rand07")]
    by_name = {c["name"]: c for c in extract}
    for metric in ("count", "gc_percent"):
        for grp in groups:
            with tempfile.TemporaryDirectory() as td:
                fdir = Path(td) / "features"
                ids = []
                for gi, nm in enumerate(grp):
                    c = by_name[nm]
                    org = f"GCF_90000000{gi}_1"
                    kdir = Path(td) / "kmers" / org
                    kdir.mkdir(parents=True)
                    paths = []
                    for k, txt in c["files"].items():
                        p = kdir / f"k{k}.txt"
                        p.write_text(txt)
                        paths.append(p)
                    with contextlib.redirect_stdout(io.StringIO()):
                        KmerFeatureExtractor(input_paths=paths, output_dir=fdir).extract_features()
                    ids.append(org)
                with contextlib.redirect_stdout(io.StringIO()):
                    b = KmerFeatureBuilder(fdir)
                    m = b.build_from_statistics_files(metric=metric)
                matrices.append({
                    "cases": list(grp), "metric": metric,
                    "index": [str(x) for x in m.index], "columns": [str(x) for x in m.columns],
                    "values": [[float(v) for v in row] for row in m.to_numpy()],
                })
    return stats, matrices


def big_cases():
    """Inputs of a few hundred kilobases that cross slice boundaries of the GPU kernels in their awkward modes
    (unwrapped lines, a very long header made of base letters, tandem repeats, CRLF with N runs, thousands of
    short records).  The reference's output files are large, so only their SHA-256 and line counts are kept;
    the FASTA text travels gzip-compressed."""
    import gzip
    import hashlib
    rng = random.Random(77)
    seq = lambda n, alphabet="ACGT": "".join(rng.choice(alphabet) for _ in range(n))       # noqa: E731
    wrap = lambda s, w, eol="\n": eol.join(s[i:i + w] for i in range(0, len(s), w))           # noqa: E731
    unit = seq(171)
    short = []
    for i in range(5000):
        short.append(f">s{i}\n{seq(rng.randint(8, 70), 'ACGTACGTACGTN')}\n")
    cases = [
        ("big_unwrapped", f">chr1 one line\n{seq(260_000)}\n>chr2\n{seq(90_000)}\n", [8, 12, 21]),
        ("big_header_of_bases", f">{seq(150_000)} a header made of base letters\n{wrap(seq(120_000), 70)}\n>x\n{seq(40)}\n", [12]),
        ("big_satellite", f">sat\n{wrap(unit * 1200 + seq(60_000) + unit[:100] * 300, 80)}\n", [9, 12]),
        ("big_crlf_n_runs", ">c\r\n" + wrap(seq(100_000) + "N" * 3000 + seq(80_000, "ACGTN") + seq(20_000), 60, "\r\n") + "\r\n", [7, 11]),
        ("big_many_short_records", "".join(short), [5, 12, 17]),
    ]
    out = []
    for name, text, ks in cases:
        with tempfile.TemporaryDirectory() as td:
            fa = Path(td) / "GCF_900000001_1.fa"
            with open(fa, "w", newline="") as f:
                f.write(text)
            with contextlib.redirect_stdout(io.StringIO()):
                org = KmerExtractor(output_dir=Path(td) / "out", compress=False).extract_kmers_from_fasta(fa, list(ks))
            files = {}
            for k in ks:
                data = (Path(td) / "out" / org / f"k{k}.txt").read_bytes()
                files[str(k)] = {"sha256": hashlib.sha256(data).hexdigest(), "lines": data.count(b"\n"), "bytes": len(data)}
            out.append({"name": name, "k_values": list(ks),
                        "fasta_gz_b64": base64.b64encode(gzip.compress(text.encode("latin-1"), 9, mtime=0)).decode(),
                        "files": files})
    return out


def timing():
    rng = random.Random(0)
    seq = "".join(rng.choice("ACGT") for _ in range(200_000))
    text = ">chr\n" + "\n".join(seq[i:i + 80] for i in range(0, len(seq), 80)) + "\n"
    res = {"n_bases": len(seq), "cpu": os.cpu_count(), "rows": []}
    with tempfile.TemporaryDirectory() as td:
        fa = Path(td) / "t.fa"
        fa.write_text(text)
        for ks in ([6], [12], [8, 9, 10, 11, 12], list(range(1, 13))):
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                KmerExtractor(output_dir=Path(td) / "o", compress=False).extract_kmers_from_fasta(fa, ks)
            dt = time.perf_counter() - t0
            res["rows"].append({"k_values": ks, "seconds": dt, "mbp_per_s": len(seq) / dt / 1e6})
    return res


def main():
    ext = extract_cases()
    (HERE / "extract_cases.json").write_text(json.dumps(ext, indent=0))
    st, mx = stats_and_matrix_cases(ext)
    (HERE / "stats_cases.json").write_text(json.dumps(st, indent=0))
    (HERE / "matrix_cases.json").write_text(json.dumps(mx, indent=0))
    (HERE / "ref_timing.json").write_text(json.dumps(timing(), indent=1))
    big = big_cases()
    (HERE / "extract_big_cases.json").write_text(json.dumps(big, indent=0))
    dup = dupk_cases()
    (HERE / "extract_dupk_cases.json").write_text(json.dumps(dup, indent=0))
    meta = {"cases": metadata_cases(ext), "big": [many_contig_metadata_case()]}
    (HERE / "metadata_cases.json").write_text(json.dumps(meta, indent=0))
    print(f"{len(dup)} duplicate-k cases, {len(meta['cases'])} + {len(meta['big'])} metadata cases")
    print(f"{len(ext)} extract cases, {len(st)} stats cases, {len(mx)} matrix cases, {len(big)} big cases")


if __name__ == "__main__":
    main()
