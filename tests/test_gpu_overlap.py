"""GPU: the contig overlap graph (SURVEY.md 8f.3, AdjList/AdjList.cpp) -- the AdjList program over libabyssb200 (CUDA
hash joins, csrc/abb_overlap.cu) writes the bytes of the unmodified reference AdjList in every output format
(committed goldens of its output), through the C ABI as well, and in the
pipeline order of bin/abyss-pe: abyss-bloom-dbg -> unitig FASTA -> AdjList."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import overlap_cases as oc
from abyss_b200.synth import ReadSet

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
BIN = os.path.join(ROOT, "abyss_b200", "lib")


def run_case(exe, case, tmp_path):
    fa = str(tmp_path / (case["name"] + ".fa"))
    oc.write_fasta(case, fa)
    r = subprocess.run([exe] + oc.command_args(case, fa), capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    return oc.normalise(r.stdout, exe).replace(fa.encode(), b"IN.fa")


def test_cli_goldens(abb, tmp_path):
    exe = os.path.join(BIN, "AdjList")
    want = json.load(open(os.path.join(GOLD, "overlap_cases.json")))
    # every process start pays a CUDA context: the command line runs the tiled sets, every format on the unitig sets and a few
    # fuzz sets; the remaining fuzz sets go through the same per-item functions and writers in tests/test_host_overlap.py
    cases = [c for c in oc.all_cases() if not c["name"].startswith("fuzz") or c["name"] in ("fuzz7", "fuzz11", "fuzz23", "fuzz42")]
    for c in cases:
        got = run_case(exe, c, tmp_path)
        assert len(got) == want[c["name"]]["bytes"], c["name"]
        assert hashlib.sha256(got).hexdigest() == want[c["name"]]["sha256"], c["name"]
        full = os.path.join(GOLD, "overlap_" + c["name"] + ".txt")
        if os.path.exists(full):
            assert got == open(full, "rb").read()


def test_cli_live_against_reference(abb, tmp_path):
    # further sets against the reference's output on them (sha256 in overlap_ref_runs.json)
    exe = os.path.join(BIN, "AdjList")
    want = json.load(open(os.path.join(GOLD, "overlap_ref_runs.json")))
    for c in oc.cli_cases():
        fa = str(tmp_path / "in.fa")
        oc.write_fasta(c, fa)
        b = subprocess.run([exe] + oc.command_args(c, fa), capture_output=True)
        assert b.returncode == 0, b.stderr.decode()
        assert oc.ref_run_digest(b.stdout, exe, tmp_path) == want[c["name"]], (c["name"], c["k"], c["m"], c["args"])


def test_c_abi_edges(abb):
    # 0+ = ACGTACGTAC overlaps its own reverse complement by 4 (k = 5): the two-edge graph of AdjList's smallest example,
    # plus a 3-base overlap found only with min_overlap < k - 1
    seqs = [b"ACGTACGTAC", b"TACGTACCA", b"CCATTTTTT"]
    bases = np.frombuffer(b"".join(seqs), dtype=np.uint8).copy()
    offs = np.zeros(len(seqs) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(s) for s in seqs])
    lib = abb.load()
    h = C.c_void_p()
    abb.check(lib.abb_overlap_create(C.byref(h), 0))

    def edges(k, m, ss=0):
        e = C.POINTER(abb.OverlapEdge)()
        n = C.c_uint64()
        abb.check(lib.abb_overlap_build(h, bases.ctypes.data, offs.ctypes.data, len(seqs), k, m, ss, C.byref(e), C.byref(n)))
        return [(e[i].u, e[i].v, e[i].distance) for i in range(n.value)]

    assert edges(5, 4) == [(0, 1, -4), (1, 0, -4)]
    got = edges(5, 3)
    assert (2, 4, -3) in got and (5, 3, -3) in got  # 1+ ...CCA -> 2+ CCA...; and the complementary edge
    st = abb.OverlapStats()
    abb.check(lib.abb_overlap_get_stats(h, C.byref(st)))
    assert st.vertices == 6 and st.exact_edges == 2 and st.short_edges == len(got) - 2
    # errors: N in an end window, contig not longer than k-1
    bad = np.frombuffer(b"ACGTNACGTACG", dtype=np.uint8).copy()
    o2 = np.array([0, 12], dtype=np.uint64)
    e = C.POINTER(abb.OverlapEdge)()
    n = C.c_uint64()
    assert lib.abb_overlap_build(h, bad.ctypes.data, o2.ctypes.data, 1, 6, 0, 0, C.byref(e), C.byref(n)) == abb.ABB_EINVAL
    assert lib.abb_overlap_build(h, bad.ctypes.data, o2.ctypes.data, 1, 14, 0, 0, C.byref(e), C.byref(n)) == abb.ABB_EINVAL
    abb.check(lib.abb_overlap_destroy(h))


def test_pipeline_unitigs_to_graph(abb, tmp_path):
    # bin/abyss-pe:577: the unitig FASTA of abyss-bloom-dbg goes straight into AdjList
    c = {c["name"]: c for c in json.load(open(os.path.join(GOLD, "e2e_cases.json")))}["e2e_g20k_k32"]
    rs = ReadSet.from_coverage(c["seed"], c["genome"], c["cov"], c["L"], c["err"])
    fq = str(tmp_path / "reads.fq")
    rs.write_fastq(fq)
    fa = str(tmp_path / "unitigs-1.fa")
    r = subprocess.run([os.path.join(BIN, "abyss-bloom-dbg"), f"-k{c['k']}", f"--kc={c['kc']}", f"-b{c['b']}", f"-H{c['H']}", "-o", fa, fq],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([os.path.join(BIN, "AdjList"), f"-k{c['k']}", "-m0", "--dot", fa], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    assert r.stdout == open(os.path.join(GOLD, "overlap_unitigs_k32_dot.txt"), "rb").read()
