"""GPU: `abyss-bloom graph` over libabyssb200 -- the filter `abyss-bloom build -t rolling-hash` writes and the GraphViz graph
are the bytes of the unmodified reference (tests/golden/bloom_graph_cases.json); abb_neighbours (k_neighbours) agrees with
the C oracle on random, lower-case, N-containing and palindromic k-mers, and rejects what it cannot answer.  (The command
line's option errors come before any device call; tests/test_host_bloom_graph.py runs them.)"""
import ctypes as C
import hashlib
import os
import random
import subprocess

import numpy as np
import pytest

from bloom_graph_cases import CASES, ROOT, check_dot, graph_args, write_inputs

pytestmark = pytest.mark.gpu
CLI = os.path.join(ROOT, "abyss_b200", "lib", "abyss-bloom")


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_graph_cli(abb, tmp_path, case):
    c, d = case, str(tmp_path)
    write_inputs(c, d)
    for name, spec in c["filters"].items():
        r = subprocess.run([CLI, "build", f"-k{c['k']}", "-t", "rolling-hash", f"-b{spec['b']}", f"-H{spec['H']}", f"-l{spec['l']}",
                            os.path.join(d, name), os.path.join(d, spec["reads"])], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert hashlib.sha256(open(os.path.join(d, name), "rb").read()).hexdigest() == c["filter_sha256"][name], name
    r = subprocess.run([CLI, "graph", *graph_args(c, d)], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    check_dot(c, r.stdout)


def _oracle():
    import oracle_py
    L = oracle_py.load().lib
    L.abo_base_hash.restype = None
    L.abo_base_hash.argtypes = [C.c_char_p, C.c_uint, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    for fn in (L.abo_roll_right, L.abo_roll_left):
        fn.restype = None
        fn.argtypes = [C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_uint, C.c_ubyte, C.c_ubyte]
    return L


def _expected(L, kmer: bytes, k: int, filters):
    """(hashes[9], mask, attr[9]) by the C oracle: NTC64 of the k-mer, rolled right / left to each neighbour, getHashes with
    the graph's H and k, BloomFilter::contains of each filter over its own size and H"""
    fh, rh = C.c_uint64(), C.c_uint64()
    L.abo_base_hash(kmer, k, C.byref(fh), C.byref(rh))
    pairs = [(fh.value, rh.value)]
    for roll, out in ((L.abo_roll_right, kmer[0]), (L.abo_roll_left, kmer[-1])):
        for b in b"ACGT":
            f, r = C.c_uint64(fh.value), C.c_uint64(rh.value)
            roll(C.byref(f), C.byref(r), k, out, b)
            pairs.append((f.value, r.value))
    hashes = [min(f, r) for f, r in pairs]
    Hg = filters[0][2]
    mask, attr = 0, [0] * 9
    for v, h in enumerate(hashes):
        hv = (C.c_uint64 * Hg)(*([h] + [L.abo_extra_hash(h, k, i) for i in range(1, Hg)]))
        for j, (bits, mbits, H) in enumerate(filters):
            if L.abo_bf_contains(bits.ctypes.data, mbits, hv, H):
                if j == 0:
                    mask |= 1 << v
                else:
                    attr[v] |= 1 << (j - 1)
    return hashes, mask, attr


@pytest.mark.parametrize("k", [21, 32, 64, 96])
def test_neighbours_vs_oracle(abb, oracle, k):
    L = _oracle()
    rnd = random.Random(k)
    genome = "".join(rnd.choice("ACGT") for _ in range(3000))
    reads = [genome[i:i + 150] for i in range(0, 2850, 25)]
    # graph: H = 4, dense enough that neighbours are often present; attributes: H = 4, 2 and 1 over other sizes
    specs = [(1 << 16, 4), (1 << 15, 4), (24000, 2), (1 << 13, 1)]
    filters, handles = [], []
    for mbits, H in specs:
        bits = np.zeros(mbits // 8, dtype=np.uint8)
        oracle.bf_load(bits, reads[: len(reads) // (1 + len(filters))], k, H)
        f = abb.Filter.bits(mbits, H, k)
        f.upload(bits)
        filters.append((bits, mbits, H))
        handles.append(f)
    kmers = [genome[p:p + k] for p in rnd.sample(range(3000 - k), 60)]                # present, mostly
    kmers += ["".join(rnd.choice("ACGT") for _ in range(k)) for _ in range(20)]        # random
    kmers += [s.lower() for s in kmers[:10]] + [s[:3].lower() + s[3:] for s in kmers[10:20]]  # lower case
    kmers += [s[:k // 2] + "N" + s[k // 2 + 1:] for s in kmers[20:30]] + ["N" * k]    # with N
    half = genome[100:100 + k // 2]
    pal = half + half[::-1].translate(str.maketrans("ACGT", "TGCA"))
    kmers += [pal[:k]] if k % 2 == 0 else [pal[: k // 2] + "A" + pal[k // 2:k - 1]]    # palindrome (even k)
    got = abb.neighbours(handles[0], [s.encode() for s in kmers], attrs=handles[1:])
    for s, (hashes, mask, attr) in zip(kmers, got):
        eh, em, ea = _expected(L, s.encode(), k, filters)
        assert hashes == eh, s
        assert mask == em, s
        assert attr == ea, s
    assert any(m & 1 for _, m, _ in got) and any(a[0] for _, _, a in got)
    # argument errors
    with pytest.raises(abb.AbbError) as e:
        abb.neighbours(handles[0], [kmers[0]], attrs=handles[1:] * 11)
    assert e.value.code == abb.ABB_EINVAL
    more = abb.Filter.bits(1 << 13, 5, k)
    with pytest.raises(abb.AbbError) as e:
        abb.neighbours(handles[0], [kmers[0]], attrs=[more])
    assert e.value.code == abb.ABB_EINVAL
    spaced = abb.Filter.bits(1 << 13, 2, k, mask="1" + "0" * (k - 2) + "1")
    with pytest.raises(abb.AbbError) as e:
        abb.neighbours(spaced, [kmers[0]])
    assert e.value.code == abb.ABB_EINVAL
    for f in handles + [more, spaced]:
        f.close()
