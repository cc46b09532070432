"""CPU: `abyss-bloom graph` -- the product's traversal (abyss_b200/host/bloom_graph.h) and the neighbourhood function the CUDA
kernel runs (neighbourhood(), abyss_b200/csrc/abb_graph.cuh), driven by the single-thread harness tests/host_bloom_graph on
oracle-built filters -- writes the bytes of the unmodified reference's graph on every golden; and the option errors of the
command line, which it reports before it touches a device."""
import os
import subprocess

import pytest

from bloom_graph_cases import CASES, ROOT, check_dot, harness_args, oracle_filter, write_inputs

import oracle_py

CLI = os.path.join(ROOT, "abyss_b200", "lib", "abyss-bloom")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("hbg") / "host_bloom_graph")
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wno-unknown-pragmas", "-pthread", "-o", exe,
                    os.path.join(ROOT, "tests", "host_bloom_graph", "host_bloom_graph.cpp"), os.path.join(ROOT, "oracle", "abyss_oracle.c")],
                   check=True, capture_output=True)
    return exe


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_bloom_graph(harness, tmp_path, case):
    c, d = case, str(tmp_path)
    write_inputs(c, d)
    oracle = oracle_py.load()
    for name, spec in c["filters"].items():
        assert oracle_filter(oracle, d, name, spec, c["k"]) == c["filter_sha256"][name], name
    r = subprocess.run([harness, *harness_args(c, d)], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    check_dot(c, r.stdout)


@pytest.fixture(scope="module")
def small(tmp_path_factory):
    """the g2k case's files: a rolling-hash filter (H = 3, k = 21), a counting filter, a filter with more hashes, roots"""
    c = CASES[0]
    d = str(tmp_path_factory.mktemp("bgerr"))
    write_inputs(c, d)
    oracle = oracle_py.load()
    oracle_filter(oracle, d, "main.bloom", c["filters"]["main.bloom"], c["k"])
    oracle_filter(oracle, d, "h5.bloom", dict(b="16k", H=5, l=1, reads="reads.fq"), c["k"])
    open(os.path.join(d, "count.bloom"), "wb").write(
        b"[BTLCountingBloomFilter_v1]\n\tBloomFilterSize = 64\n\tHashNum = 3\n\tKmerSize = 21\n\tBloomFilterSizeInBytes = 64\n"
        b"\tBitsPerCounter = 8\n[HeaderEnd]\n" + bytes(64))
    return d


ERRORS = [
    # -k after a command option is not a global option any more
    (["graph", "-d1", "-k21", "-R", "A" * 21, "@main.bloom"], "missing mandatory option `-k'"),
    (["graph", "-k21", "-d1", "-k21", "-R", "A" * 21, "@main.bloom"], "invalid option: `-k21'"),
    # an option with an argument that `graph' does not read
    (["graph", "-k21", "-q", "10", "-R", "A" * 21, "@main.bloom"], "invalid option: `-q10'"),
    (["graph", "-k21", "--bloom-size=1M", "-R", "A" * 21, "@main.bloom"], "invalid option: `-b1M'"),
    (["graph", "-k21", "-dx", "-R", "A" * 21, "@main.bloom"], "invalid option: `-dx'"),
    (["graph", "-k21", "-a", "nocolon", "-R", "A" * 21, "@main.bloom"], "invalid option: `-anocolon'"),
    (["graph", "-k21", "@main.bloom"], "must specify either --root or --root-fasta"),
    (["graph", "-k21", "-R", "A" * 21], "missing arguments"),
    (["graph", "-k21", "-R", "A" * 21, "@main.bloom", "@main.bloom"], "missing arguments"),
    (["graph", "-k21", "-R", "A" * 20, "@main.bloom"], "has 20 characters, -k is 21"),
    (["graph", "-k25", "-R", "A" * 25, "@main.bloom"], "holds 21-mers, -k is 25"),
    (["graph", "-k21", "-R", "A" * 21, "@count.bloom"], "is a counting Bloom filter"),
    (["graph", "-k21", "-R", "A" * 21, "-A", "x:@h5.bloom", "@main.bloom"], "has 5 hash functions, more than the 3"),
    (["graph", "-k21", "-R", "A" * 21] + ["-A", "x:@main.bloom"] * 33 + ["@main.bloom"], "at most 32 --bloom-attr filters"),
]


@pytest.mark.parametrize("args,msg", ERRORS, ids=[str(i) for i in range(len(ERRORS))])
def test_graph_option_errors(abb, small, args, msg):
    r = subprocess.run([CLI] + [a.replace("@", small + "/") for a in args], capture_output=True, text=True)
    assert r.returncode == 1, r.stderr
    assert msg in r.stderr, r.stderr
    assert r.stdout == ""
