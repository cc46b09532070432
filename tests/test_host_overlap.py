"""CPU: the overlap-graph join logic (abyss_b200/csrc/abb_overlap.cuh -- the SAME per-item functions the CUDA kernels
call) and the product's AdjList command line and graph writers (abyss_b200/host/adjlist_main.h), run by the
single-thread harness tests/host_overlap, against the output of the unmodified reference AdjList (committed goldens,
tests/golden/make_golden_overlap.py)."""
import hashlib
import json
import os
import subprocess

import pytest

import overlap_cases as oc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("ho") / "AdjList")
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wno-unknown-pragmas", "-o", exe, os.path.join(ROOT, "tests", "host_overlap", "host_overlap.cpp")],
                   check=True, capture_output=True)
    return exe


def run_case(exe, case, tmp_path):
    fa = str(tmp_path / (case["name"] + ".fa"))
    oc.write_fasta(case, fa)
    r = subprocess.run([exe] + oc.command_args(case, fa), capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    return oc.normalise(r.stdout, exe).replace(fa.encode(), b"IN.fa")


def test_goldens(harness, tmp_path):
    want = json.load(open(os.path.join(GOLD, "overlap_cases.json")))
    cases = oc.all_cases()
    assert sorted(c["name"] for c in cases) == sorted(want)
    for c in cases:
        got = run_case(harness, c, tmp_path)
        assert len(got) == want[c["name"]]["bytes"], c["name"]
        assert hashlib.sha256(got).hexdigest() == want[c["name"]]["sha256"], c["name"]
        full = os.path.join(GOLD, "overlap_" + c["name"] + ".txt")
        if os.path.exists(full):
            assert got == open(full, "rb").read()


def test_live_against_reference(harness, tmp_path):
    # further fuzz sets against the reference's output on them (sha256 in overlap_ref_runs.json)
    want = json.load(open(os.path.join(GOLD, "overlap_ref_runs.json")))
    for c in oc.more_fuzz_cases():
        fa = str(tmp_path / "in.fa")
        oc.write_fasta(c, fa)
        b = subprocess.run([harness] + oc.command_args(c, fa), capture_output=True)
        assert b.returncode == 0, b.stderr.decode()
        assert oc.ref_run_digest(b.stdout, harness, tmp_path) == want[c["name"]], (c["name"], c["k"], c["m"], c["args"])


def test_errors(harness, tmp_path):
    fa = str(tmp_path / "n.fa")
    open(fa, "w").write(">0 12 3\nACGTNACGTACG\n>1 12 3\nACGTACGTACGA\n")
    r = subprocess.run([harness, "-k6", fa], capture_output=True, text=True)
    assert r.returncode != 0 and "nucleotide" in r.stderr  # the reference's Kmer constructor aborts on the N
    open(fa, "w").write(">0\nACGT\n")
    r = subprocess.run([harness, "-k6", fa], capture_output=True, text=True)
    assert r.returncode != 0 and "not longer than k-1" in r.stderr
    open(fa, "w").write(">a\nACGTACGTAA\n>a\nACGTACGTAC\n")
    r = subprocess.run([harness, "-k6", fa], capture_output=True, text=True)
    assert r.returncode != 0 and "duplicate ID" in r.stderr
    r = subprocess.run([harness, fa], capture_output=True, text=True)
    assert r.returncode != 0 and "missing -k,--kmer option" in r.stderr


@pytest.mark.parametrize("k,m,fmt", oc.UNITIG_RUNS)
def test_real_unitig_sets(harness, tmp_path, k, m, fmt):
    # the pipeline of bin/abyss-pe on config 1 (SURVEY.md 8d: 53 333 x 150 bp reads of a 200 kbp genome): the reference's own
    # unitig FASTA (tips, branches, blunt ends from coverage gaps) into AdjList, against the reference AdjList's output
    text, sha = oc.unitig_set_fasta(k)
    assert hashlib.sha256(text.encode()).hexdigest() == sha
    assert text.count(">") > 10
    fa = str(tmp_path / "unitigs-1.fa")
    open(fa, "w").write(text)
    b = subprocess.run([harness, f"-k{k}", f"-m{m}", fmt, fa], capture_output=True)
    assert b.returncode == 0, b.stderr.decode()
    want = json.load(open(os.path.join(GOLD, "overlap_ref_runs.json")))[f"unitigs_config1_k{k}_m{m}_{fmt[2:]}"]
    assert oc.ref_run_digest(b.stdout, harness, tmp_path) == want
    assert want["bytes"] > 0


def test_option_aliases_and_stdin(harness, tmp_path):
    # --gv = --dot, --gfa = --gfa1, -m0 = k-1, long options, several input files, contigs on standard input
    want = json.load(open(os.path.join(GOLD, "overlap_ref_runs.json")))
    for name, args, stdin in oc.alias_runs(str(tmp_path)):
        got = subprocess.run([harness] + args, input=stdin, capture_output=True, text=True)
        assert got.returncode == 0, got.stderr
        assert oc.ref_run_digest(got.stdout.encode(), harness, tmp_path) == want[name], args
