"""Goldens of `abyss-bloom graph` (Bloom/bloom.cc:983-1153): the unmodified reference builds a rolling-hash filter
(`abyss-bloom build -t rolling-hash`) from seeded reads and writes the GraphViz neighbourhood of root k-mers in it.  Per case
this records the parameters, the sha256 of every filter file and the bytes / lines / sha256 of the dot; dots under 200 KB
are committed gzipped.

    python tests/golden/make_golden_bloom_graph.py
"""
import gzip
import hashlib
import json
import os
import random
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from abyss_b200.synth import ReadSet, revcomp  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref", "abyss-bloom-ref")
G2K = dict(seed=31, genome=2000, cov=20, L=80, err=0.01)  # the read set of graph_g2k_k21
G200K = dict(seed=23, genome=200000, cov=30, L=150, err=0.005)
G5K = dict(seed=41, genome=5000, cov=15, L=150, err=0.005)


def _main(b, H, levels=1, reads="reads.fq"):
    return {"main.bloom": dict(b=b, H=H, l=levels, reads=reads)}


# fastas: name -> [first read, end read, variant]; filters: name -> build parameters; args: the graph command line after
# `-k K`, "@name" standing for the file of that name
CASES = [
    dict(name="bg_g2k_k21_attrs", reads=G2K, k=21,
         fastas={"roots3.fa": [0, 3, "edge"], "a1.fa": [40, 60, ""], "a2.fa": [100, 200, ""], "sub1.fq": [0, 150, ""],
                 "sub2.fq": [150, 400, ""]},
         filters=dict(_main("64k", 3), **{"A1.bloom": dict(b="64k", H=3, l=1, reads="sub1.fq"),
                                          "A2.bloom": dict(b="16k", H=2, l=1, reads="sub2.fq")}),
         args=["-d5", "-f", "@roots3.fa", "-a", "first:@a1.fa", "--node-attr", "second:@a2.fa", "-A", "bloomA:@A1.bloom",
               "--bloom-attr=bloomB:@A2.bloom"]),
    dict(name="bg_g2k_k21_allreads", reads=G2K, k=21, fastas={"all.fa": [0, None, ""]}, filters=_main("64k", 3),
         args=["-f", "@all.fa"]),
    dict(name="bg_g2k_k21_R_d0", reads=G2K, k=21, fastas={}, filters=_main("64k", 3), roots=True, args=["-d0"]),
    dict(name="bg_g2k_k21_R_d3", reads=G2K, k=21, fastas={}, filters=_main("64k", 3), roots=True, args=["-d", "3"]),
    dict(name="bg_g2k_k21_l2", reads=G2K, k=21, fastas={"roots5.fa": [10, 15, ""]}, filters=_main("128k", 3, levels=2),
         args=["-d10", "-f", "@roots5.fa"]),
    dict(name="bg_tandem_k24", fixture="cyc_tandem.fa.gz", k=24, fastas={"r.fa": [0, 40, ""]}, filters=_main("256k", 3),
         args=["-f", "@r.fa"]),
    dict(name="bg_tandem_k25", fixture="cyc_tandem.fa.gz", k=25, fastas={"r.fa": [0, 40, ""]}, filters=_main("256k", 3),
         args=["-f", "@r.fa"]),
    dict(name="bg_hairpin_k24", fixture="cyc_hairpin.fa.gz", k=24, fastas={"r.fa": [0, 40, ""]}, filters=_main("256k", 3),
         args=["-f", "@r.fa"]),
    dict(name="bg_hairpin_k25", fixture="cyc_hairpin.fa.gz", k=25, fastas={"r.fa": [0, 40, ""]}, filters=_main("256k", 3),
         args=["-f", "@r.fa"]),
    dict(name="bg_g5k_k64", reads=G5K, k=64, fastas={"r.fa": [0, 10, ""]}, filters=_main("256k", 3), args=["-d20", "-f", "@r.fa"]),
    dict(name="bg_g5k_k96", reads=G5K, k=96, fastas={"r.fa": [0, 10, ""]}, filters=_main("256k", 4), args=["-f", "@r.fa"]),
    dict(name="bg_g200k_k32", reads=G200K, k=32, fastas={"r200.fa": [0, 200, ""]}, filters=_main("4M", 3),
         args=["-f", "@r200.fa"]),
    dict(name="bg_g200k_k32_d3000", reads=G200K, k=32, fastas={"r200.fa": [0, 200, ""]}, filters=_main("4M", 3),
         args=["-d", "3000", "-f", "@r200.fa"]),
]


def read_seqs(c):
    """the reads of a case, as strings"""
    if "fixture" in c:
        lines = gzip.open(os.path.join(HERE, c["fixture"]), "rt").read().split("\n")
        return [x for x in lines if x and not x.startswith(">")]
    r = c["reads"]
    rs = ReadSet.from_coverage(r["seed"], r["genome"], r["cov"], r["L"], r["err"])
    return [a.tobytes().decode() for a in rs.ascii(0, rs.n)]


def _edge(seqs):
    """lower-case ends on the first read, an 'N' inside the second"""
    out = list(seqs)
    if out:
        out[0] = out[0][:6].lower() + out[0][6:-6] + out[0][-6:].lower()
    if len(out) > 1:
        out[1] = out[1][:30] + "N" + out[1][31:]
    return out


def write_inputs(c, d):
    """the read files of a case into directory d: reads.fq (all reads, what the main filter is built from) and c["fastas"]"""
    seqs = read_seqs(c)
    with open(os.path.join(d, "reads.fq"), "w") as f:
        for i, s in enumerate(seqs):
            f.write(f"@r{i}/1\n{s}\n+\n{'I' * len(s)}\n")
    for name, (lo, hi, variant) in c["fastas"].items():
        part = seqs[lo:hi]
        if variant == "edge":
            part = _edge(part)
        with open(os.path.join(d, name), "w") as f:
            for i, s in enumerate(part):
                f.write(f"@r{lo + i}/1\n{s}\n+\n{'I' * len(s)}\n" if name.endswith(".fq") else f">r{lo + i}/1\n{s}\n")
    return seqs


def graph_args(c, d):
    return [f"-k{c['k']}"] + [a.replace("@", d + "/") for a in c["args"]] + [os.path.join(d, "main.bloom")]


def root_kmers(seqs, k):
    """-R roots: upper case, the same k-mer reverse-complemented, lower case, with an N, and one the graph lacks"""
    rnd = random.Random(5)
    a = seqs[5][10:10 + k]
    return [a, revcomp(a), seqs[7][3:3 + k].lower(), seqs[9][:10] + "N" + seqs[9][11:k], seqs[11][20:20 + k],
            "".join(rnd.choice("ACGT") for _ in range(k))]


def build_filter(d, name, spec, k):
    cmd = [REF, "build", f"-k{k}", "-t", "rolling-hash", f"-b{spec['b']}", f"-H{spec['H']}", f"-l{spec['l']}",
           os.path.join(d, name), os.path.join(d, spec["reads"])]
    subprocess.run(cmd, check=True, capture_output=True)
    return hashlib.sha256(open(os.path.join(d, name), "rb").read()).hexdigest()


def main():
    tmp = "/tmp/abyss_golden_bloom_graph"
    out = []
    for c in CASES:
        d = os.path.join(tmp, c["name"])
        shutil.rmtree(d, ignore_errors=True)
        os.makedirs(d)
        seqs = write_inputs(c, d)
        if c.get("roots"):
            rs = root_kmers(seqs, c["k"])
            c = dict(c, args=c["args"] + [x for r in rs for x in ("-R", r)])
        c = dict(c, filter_sha256={n: build_filter(d, n, s, c["k"]) for n, s in c["filters"].items()})
        data = subprocess.run([REF, "graph", *graph_args(c, d)], check=True, capture_output=True).stdout
        c = dict(c, bytes=len(data), lines=data.count(b"\n"), sha256=hashlib.sha256(data).hexdigest())
        if len(data) < 200000:
            with gzip.GzipFile(os.path.join(HERE, c["name"] + ".dot.gz"), "wb", mtime=0) as f:
                f.write(data)
        out.append(c)
        print(c["name"], c["lines"], c["bytes"])
    json.dump(out, open(os.path.join(HERE, "bloom_graph_cases.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
