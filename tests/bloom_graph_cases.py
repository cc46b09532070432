"""The `abyss-bloom graph` goldens (tests/golden/bloom_graph_cases.json, written by tests/golden/make_golden_bloom_graph.py from
the unmodified reference) and what the CPU and GPU tests share: the input files of a case, the rolling-hash filters rebuilt by
the C oracle (checked against the reference's sha256), and the command line of the CPU harness."""
import gzip
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLD)
from make_golden_bloom_graph import graph_args, read_seqs, write_inputs  # noqa: E402,F401

CASES = json.load(open(os.path.join(GOLD, "bloom_graph_cases.json")))


def si_bytes(s: str) -> int:
    mult = {"k": 1 << 10, "M": 1 << 20, "G": 1 << 30}
    return int(float(s[:-1]) * mult[s[-1]]) if s[-1] in mult else int(s)


def bit_bloom_bytes(raw: bytes, size_bits: int, H: int, k: int) -> bytes:
    """BloomFilter::writeHeader + the array (what `abyss-bloom build -t rolling-hash` writes; abyss_b200/host/bloom_file.h)"""
    head = (f"[BTLBloomFilter_v1]\n\tnEntry = 0\n\tdFPR = 0.0000000000000000\n\tEntry = 0\n\tBloomFilterSizeInBytes = {len(raw)}\n"
            f"\tBloomFilterSize = {size_bits}\n\tHashNum = {H}\n\tKmerSize = {k}\n[HeaderEnd]\n")
    return head.encode() + raw


def oracle_filter(oracle, d: str, name: str, spec: dict, k: int) -> str:
    """the filter `build -t rolling-hash -b B -H H -l L` makes of spec["reads"], built by the C oracle into d/name; returns its
    sha256.  The reads of these cases are plain upper-case ACGT, so the reader passes them through unchanged."""
    bits = si_bytes(spec["b"]) * 8 // spec["l"]
    bits += -bits % 64
    levels = np.zeros(bits // 8 * spec["l"], dtype=np.uint8)
    lines = open(os.path.join(d, spec["reads"])).read().split("\n")
    seqs = [lines[i] for i in range(1, len(lines), 4)]
    oracle.casc_load(levels, bits, spec["l"], seqs, k, spec["H"])
    data = bit_bloom_bytes(levels[(spec["l"] - 1) * (bits // 8):].tobytes(), bits, spec["H"], k)
    open(os.path.join(d, name), "wb").write(data)
    return hashlib.sha256(data).hexdigest()


def harness_args(c: dict, d: str) -> list:
    """the CPU harness's command line (K DEPTH BLOOM, then -R / -f / -a / -A pairs) for the graph command line of a case"""
    args = graph_args(c, d)
    depth, out, a, i = c["k"], [], args[1:-1], 0
    while i < len(a):
        x = a[i]
        if x.startswith("-d"):
            depth, i = (int(a[i + 1]), i + 2) if x == "-d" else (int(x[2:]), i + 1)
        elif x.startswith("--bloom-attr="):
            out += ["-A", x.split("=", 1)[1]]
            i += 1
        else:
            out += ["-a" if x == "--node-attr" else x, a[i + 1]]
            i += 2
    return [str(c["k"]), str(depth), args[-1]] + out


def check_dot(c: dict, data: bytes) -> None:
    assert len(data) == c["bytes"] and data.count(b"\n") == c["lines"], (len(data), data.count(b"\n"))
    assert hashlib.sha256(data).hexdigest() == c["sha256"]
    full = os.path.join(GOLD, c["name"] + ".dot.gz")
    if os.path.exists(full):
        assert data == gzip.open(full, "rb").read()
