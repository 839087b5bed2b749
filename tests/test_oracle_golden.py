"""The CPU oracle against the fixtures produced by the UNMODIFIED reference
(tests/golden/make_golden.py).  No GPU."""
import os

import numpy as np
import pytest

import oracle
from helpers import golden_dupk_cases, golden_extract_cases, golden_metadata_cases

HERE = os.path.dirname(os.path.abspath(__file__))

CASES = golden_extract_cases()


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_kmer_files_byte_identical(case):
    ml = max(case["k_values"])
    for k in dict.fromkeys(case["k_values"]):
        assert oracle.kmer_file_text(case["fasta"], k, ml) == case["files"][str(k)]


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_record_messages(case):
    """'Skipping <id>' / 'Processed <id>' lines of generate.py:45,60 follow from ids + lengths."""
    ml = max(case["k_values"])
    want = case["stdout"]
    got = []
    for rid, n in oracle.record_ids(case["fasta"]):
        if n < ml:
            got.append(f"Skipping {rid}: too short for k-mer extraction")
        else:
            got.append(f"Processed chromosome/contig: {rid}")
    assert got == want


DUPK = golden_dupk_cases()


@pytest.mark.parametrize("case", DUPK, ids=[c["name"] for c in DUPK])
def test_duplicate_k_values_count_as_often(case):
    """generate.py:36,49-58: one dict per distinct k, one counting pass per ENTRY of k_values."""
    ks = case["k_values"]
    ml = max(ks)
    for k in dict.fromkeys(ks):
        assert oracle.kmer_file_text(case["fasta"], k, ml, multiplicity=ks.count(k)) == case["files"][str(k)]


def test_metadata_managers():
    """genome_metadata.py:55-85 and kmer_metadata.py:59-78, fixtures written by the unmodified managers."""
    cases, big = golden_metadata_cases()
    assert len(cases) >= 18
    for c in cases + big:
        got = oracle.genome_stats(c["fasta"])
        for key in ("contigs", "total_size", "n_count", "gc_content"):
            assert got[key] == c["genome"][key], (c["name"], key)
    for c in cases:
        for k, want in c["kmers"].items():
            assert oracle.kmer_file_stats(c["files"][k], int(k)) == want, (c["name"], k)


def test_g0_survey_values():
    """The worked example of SURVEY.md section 4 (G0)."""
    g0 = next(c for c in CASES if c["name"] == "G0")
    c2 = oracle.count_dense(g0["fasta"], 2, 8)
    assert int(c2[oracle.kmer_to_code("AA")]) == 12
    assert int(c2[oracle.kmer_to_code("AT")]) == 2
    assert int(c2[oracle.kmer_to_code("CG")]) == 6
    c8 = oracle.count_dense(g0["fasta"], 8, 8)
    assert int(c8[oracle.kmer_to_code("ACGTACGT")]) == 2
    assert int(c8.sum()) == 17


def test_canonical_identity():
    rng = np.random.default_rng(3)
    seq = "".join("ACGT"[i] for i in rng.integers(0, 4, 500))
    data = f">r\n{seq}\n".encode()
    for k in (3, 4, 5, 6):
        fwd = oracle.count_dense(data, k)
        canon = oracle.canonical_from_forward(fwd, k)
        assert canon.sum() == fwd.sum()
        # direct canonical count with the reference's window rules
        direct = np.zeros(4 ** k, np.uint64)
        for i in range(len(seq) - k + 1):
            c = oracle.kmer_to_code(seq[i:i + k])
            direct[min(c, oracle.revcomp_code(c, k))] += 1
        assert np.array_equal(direct, canon)


def test_sparse_matches_dense():
    g0 = next(c for c in CASES if c["name"] == "rand04")
    for k in (3, 8, 12):
        counts, order = oracle.count_dense(g0["fasta"], k, 12, want_order=True)
        codes, cnts = oracle.count_sparse(g0["fasta"], k, 12)
        assert list(codes) == list(order)
        assert list(cnts) == [counts[b] for b in order]


def test_oracle_reproduces_big_reference_outputs():
    """The oracle against what the unmodified reference wrote for inputs of a few hundred kilobases (unwrapped
    lines, a long header of base letters, tandem repeats, CRLF + N runs, thousands of short records)."""
    import hashlib
    from helpers import golden_big_cases
    for case in golden_big_cases():
        ml = max(case["k_values"])
        for k in case["k_values"]:
            text = oracle.kmer_file_text(case["fasta"], k, ml).encode()
            want = case["files"][str(k)]
            assert text.count(b"\n") == want["lines"], (case["name"], k)
            assert hashlib.sha256(text).hexdigest() == want["sha256"], (case["name"], k)


REFERENCE = os.environ.get("KMERML_REFERENCE", "")


@pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "kmerml"))),
                    reason="set KMERML_REFERENCE to a source tree of the original kmer-ml project")
def test_oracle_against_the_live_reference(tmp_path):
    """Where a source tree of the original project is at hand (KMERML_REFERENCE) the UNMODIFIED reference is
    run under the Bio.SeqIO shim on fresh random FASTA files and the oracle must reproduce every k{k}.txt byte
    for byte -- the same procedure that produced tests/golden, on inputs nobody has looked at."""
    import contextlib
    import io
    import random
    import subprocess
    import sys
    from helpers import fuzz_fasta
    rng = random.Random(os.getpid())
    cases = []
    for i in range(40):
        data = fuzz_fasta(rng)
        ks = sorted(rng.sample(range(1, 13), rng.randint(1, 3))) + ([rng.randint(13, 32)] if i % 4 == 0 else [])
        (tmp_path / f"c{i}.fa").write_bytes(data)
        cases.append((i, data, ks))
    # the reference runs in a child process so that its modules never enter this interpreter
    script = (
        "import sys, json, contextlib, io\n"
        f"sys.path.insert(0, {os.path.join(HERE, '_ref')!r}); sys.path.insert(1, {REFERENCE!r})\n"
        "from kmerml.kmers.generate import KmerExtractor\n"
        "root, spec = sys.argv[1], json.loads(sys.argv[2])\n"
        "for i, ks in spec:\n"
        "    with contextlib.redirect_stdout(io.StringIO()):\n"
        "        KmerExtractor(output_dir=f'{root}/o{i}', compress=False).extract_kmers_from_fasta(f'{root}/c{i}.fa', ks)\n"
    )
    import json
    subprocess.run([sys.executable, "-c", script, str(tmp_path), json.dumps([(i, ks) for i, _, ks in cases])],
                   check=True, timeout=600)
    for i, data, ks in cases:
        for k in ks:
            want = (tmp_path / f"o{i}" / f"c{i}" / f"k{k}.txt").read_text()
            assert oracle.kmer_file_text(data, k, max(ks)) == want, (i, k, ks, data[:200])
