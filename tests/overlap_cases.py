"""Seeded contig sets for the overlap-graph (AdjList) tests: shared by the golden generator
(tests/golden/make_golden_overlap.py, runs the unmodified AdjList), the CPU emulation test and the GPU tests."""
import os
import random

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
FORMATS = ["--adj", "--dot", "--gfa1", "--gfa2", "--asqg", "--sam"]
_COMP = {"A": "T", "C": "G", "G": "C", "T": "A"}


def rc(s):
    return "".join(_COMP[c] for c in reversed(s))


def fuzz_case(seed):
    """small contig sets dense in special cases: overlaps of k-1 and fewer bases, both strands, duplicated contigs,
    palindromes, two-letter genomes (many equal ends), lower-case ends (FOLD_CASE, no masked trimming)"""
    r = random.Random(seed)
    k = r.choice([5, 8, 12, 21, 32, 64])
    alpha = "ACGT" if r.random() < 0.7 else "AC"
    genome = "".join(r.choice(alpha) for _ in range(r.randint(200, 3000)))
    contigs = []
    pos = 0
    while pos < len(genome) - k - 2:
        length = r.randint(k, k + r.randint(1, 200))
        c = genome[pos:pos + length]
        if len(c) < k:
            break
        if r.random() < 0.5:
            c = rc(c)
        if r.random() < 0.05:
            c = c.lower()[:3] + c[3:]
        contigs.append(c)
        ov = r.choice([k - 1, k - 1, k - 1, k - 2, k - 3, max(1, k - 6), 0, r.randint(0, k - 1)])
        pos += max(1, length - ov)
    if r.random() < 0.5 and contigs:
        contigs.append(contigs[r.randrange(len(contigs))])
    if r.random() < 0.5:
        h = "".join(r.choice("ACGT") for _ in range(k))
        contigs.append(h + rc(h))
    r.shuffle(contigs)
    m = r.choice([0, 2, 3, k - 1, k - 2, max(2, k - 5), 50, max(2, k // 2)])  # the reference asserts on m = 1 (chop)
    r2 = random.Random(seed + 1)
    fmt = r2.choice(FORMATS)
    ss = r2.choice([[], ["--SS"]])
    records = [(str(i), f"{len(c)} {seed * 7 % 50 + i} x", c) for i, c in enumerate(contigs)]
    return dict(name=f"fuzz{seed}", k=k, m=m, args=[fmt] + ss, records=records)


def tiled_case(seed, genome_len, k, m, n_fmt=0):
    """a random genome cut into contigs that overlap their successor by k-1 bases (most), by m..k-2 bases, or not at
    all, on random strands, shuffled -- the shape of a unitig set, at a size where the joins see real tables"""
    r = random.Random(seed)
    genome = "".join(r.choice("ACGT") for _ in range(genome_len))
    contigs = []
    pos = 0
    while pos < genome_len - 2 * k:
        length = r.randint(k + 1, 400)
        c = genome[pos:pos + length]
        contigs.append(rc(c) if r.random() < 0.5 else c)
        ov = r.choice([k - 1] * 6 + [r.randint(max(2, m), k - 2) if m < k - 1 else k - 1, 0])
        pos += max(1, len(c) - ov)
    r.shuffle(contigs)
    records = [(f"c{i}", f"{len(c)} {r.randint(0, 5000)}", c) for i, c in enumerate(contigs)]
    return dict(name=f"tiled{seed}_k{k}_m{m}", k=k, m=m, args=[FORMATS[n_fmt]], records=records)


def fasta_case(name, fasta, k, m, fmt, ss=False):
    """the unitig FASTA of an abyss-bloom-dbg golden (what bin/abyss-pe:577 feeds to AdjList)"""
    records = []
    with open(os.path.join(GOLD, fasta)) as f:
        for line in f:
            if line.startswith(">"):
                head = line[1:].rstrip("\n").split(" ", 1)
                records.append([head[0], head[1] if len(head) > 1 else "", ""])
            else:
                records[-1][2] += line.strip()
    return dict(name=name, k=k, m=m, args=[fmt] + (["--SS"] if ss else []), records=[tuple(r) for r in records])


def all_cases():
    cases = [fuzz_case(s) for s in range(60)]
    cases += [tiled_case(1, 300000, 64, 50, 0), tiled_case(2, 300000, 32, 0, 3), tiled_case(3, 200000, 96, 50, 1), tiled_case(4, 100000, 25, 10, 2)]
    for fmt in FORMATS:
        cases.append(fasta_case("unitigs_k32_" + fmt[2:], "e2e_g20k_k32.fa", 32, 0, fmt))
        cases.append(fasta_case("unitigs_k64_" + fmt[2:], "e2e_g30k_k64.fa", 64, 50, fmt, ss=fmt == "--gfa2"))
    cases.append(fasta_case("unitigs_k25_m10", "e2e_g10k_k25_small.fa", 25, 10, "--adj"))
    return cases


def more_fuzz_cases():
    """further fuzz sets; only the sha256 of the reference's output is stored (overlap_ref_runs.json)"""
    return [fuzz_case(s) for s in range(1000, 1120)]


def cli_cases():
    """the sets the GPU AdjList command line runs against the reference's output (overlap_ref_runs.json)"""
    return [fuzz_case(s) for s in range(2000, 2008)] + [tiled_case(9, 1500000, 64, 50, 0), tiled_case(10, 800000, 40, 0, 4)]


def alias_runs(tmp_path):
    """--gv = --dot, --gfa = --gfa1, -m0 = k-1, long options, several input files, contigs on standard input:
    (name, args, stdin) over two FASTA files written to tmp_path"""
    c = tiled_case(21, 20000, 31, 20)
    half = len(c["records"]) // 2
    a_fa, b_fa = os.path.join(tmp_path, "a.fa"), os.path.join(tmp_path, "b.fa")
    write_fasta(dict(c, records=c["records"][:half]), a_fa)
    write_fasta(dict(c, records=c["records"][half:]), b_fa)
    both = open(a_fa).read() + open(b_fa).read()
    return [("alias_gv", ["--kmer=31", "--min-overlap=20", "--gv", a_fa, b_fa], None), ("alias_gfa", ["-k31", "-m0", "--gfa", a_fa, b_fa], None),
            ("alias_stdin_adj", ["-k", "31", "-m", "25", "--SS", "--adj"], both), ("alias_stdin_asqg", ["-k31", "--no-SS", "--asqg", "-"], both)]


# config 1 of SURVEY.md 8d (53 333 x 150 bp reads of a 200 kbp genome) through the reference's abyss-bloom-dbg -kK --kc=2 -b64M -H4 -j1:
# unitig sets with tips, branches and blunt ends from coverage gaps, stored as genome coordinates (unitigs_config1.json.gz)
UNITIG_SET_READS = (1, 200000, 53333, 150, 0.005)  # ReadSet(seed, genome length, reads, read length, error rate)
UNITIG_RUNS = [(32, 0, "--adj"), (32, 20, "--dot"), (48, 30, "--gfa1"), (64, 50, "--gfa2"), (96, 50, "--sam"), (40, 25, "--asqg")]


def unitig_set_genome():
    import numpy as np
    from abyss_b200.synth import ReadSet
    rs = ReadSet(*UNITIG_SET_READS)
    return np.frombuffer(b"ACGT", dtype=np.uint8)[rs.genome].tobytes().decode()


def unitig_set_fasta(k):
    """the reference's unitig FASTA at k, rebuilt from unitigs_config1.json.gz: a record is [header, pos, length] (a genome
    substring; pos < 0: the reverse complement of the one at -pos-1) or [header, sequence] (a unitig that holds read errors)"""
    import gzip
    import json
    sets = json.load(gzip.open(os.path.join(GOLD, "unitigs_config1.json.gz"), "rt"))
    g = unitig_set_genome()
    out = []
    for rec in sets[str(k)]["records"]:
        if len(rec) == 2:
            seq = rec[1]
        elif rec[1] >= 0:
            seq = g[rec[1]:rec[1] + rec[2]]
        else:
            seq = rc(g[-rec[1] - 1:-rec[1] - 1 + rec[2]])
        out.append(f">{rec[0]}\n{seq}\n")
    return "".join(out), sets[str(k)]["sha256"]


def write_fasta(case, path):
    with open(path, "w") as f:
        for name, comment, seq in case["records"]:
            f.write(f">{name} {comment}\n{seq}\n" if comment else f">{name}\n{seq}\n")


def command_args(case, fasta_path):
    return [f"-k{case['k']}", f"-m{case['m']}"] + case["args"] + [fasta_path]


def normalise(out: bytes, exe: str) -> bytes:
    """the SAM header quotes the command line: make it independent of where the binary lives"""
    return out.replace(exe.encode(), b"AdjList")


def ref_run_digest(out: bytes, exe: str, tmp_dir) -> dict:
    """sha256 and length of an output as overlap_ref_runs.json stores the reference's: independent of where the binary and the
    input files live"""
    import hashlib
    data = normalise(out, exe).replace(str(tmp_dir).encode(), b"TMP")
    return dict(sha256=hashlib.sha256(data).hexdigest(), bytes=len(data))
