"""CPU: the CLI's read ingestion (abyss_b200/host/reads.h).  BatchStream -- pieces of the file parsed by worker threads
while the GPU works on the previous batch -- must deliver exactly the records of the serial SeqReader
(DataLayer/FastaReader.cpp:130-421 semantics), in order, in batches of the requested size, wherever the piece
boundaries fall: quality lines that start with '@', '+' or '>', multi-line FASTA, Casava headers, CRLF, a last line
without newline, comment-led files (parsed serially), several files, compressed input."""
import gzip
import hashlib
import json
import os
import random
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("rd") / "host_reader")
    subprocess.run(["g++", "-std=c++17", "-O2", "-pthread", "-Wall", "-o", out, os.path.join(ROOT, "tests", "host_reader", "host_reader.cpp")],
                   check=True, capture_output=True)
    return out


def run(exe, *args, env=None):
    r = subprocess.run([exe, *map(str, args)], capture_output=True, text=True, env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stderr
    return r.stdout, [int(l.split()[2]) for l in r.stderr.splitlines() if l.startswith("# batch")]


def fastq(n, seed, crlf=False, casava=False):
    rng = random.Random(seed)
    nl = "\r\n" if crlf else "\n"
    out = []
    for i in range(n):
        L = rng.randint(1, 180)
        seq = "".join(rng.choice("ACGTNacgt") for _ in range(L))
        # qualities over the whole printable range: lines starting with '@', '+', '>' and '#' all occur
        q = "".join(chr(rng.randint(33, 74)) for _ in range(L))
        if i % 7 == 0:
            q = rng.choice("@+>#") + q[1:]
        head = f"@r{i}" + (f" {1 + i % 2}:{'Y' if i % 5 == 0 else 'N'}:0:ACGT" if casava else f"/{1 + i % 2} extra words")
        out.append(f"{head}{nl}{seq}{nl}+{nl}{q}{nl}")
    return "".join(out)


def fasta(n, seed):
    rng = random.Random(seed)
    out = []
    for i in range(n):
        out.append(f">c{i} len\n")
        for _ in range(rng.randint(1, 5)):
            out.append("".join(rng.choice("ACGTacgtN") for _ in range(rng.randint(1, 70))) + "\n")
    return "".join(out)


@pytest.mark.parametrize("mapped", [True, False])  # regular files parsed in place from a memory mapping / read through a buffer
@pytest.mark.parametrize("piece", [64, 1000, 1 << 16])
@pytest.mark.parametrize("threads", [1, 3])
def test_stream_equals_serial(exe, tmp_path, piece, threads, mapped):
    files = {}
    files["a.fq"] = fastq(3000, 1)
    files["b.fq"] = fastq(1500, 2, crlf=True, casava=True)
    files["c.fa"] = fasta(800, 3)
    files["d.fq"] = fastq(5, 4)[:-1]                      # last line without '\n'
    files["e.fq"] = "# comment first\n" + fastq(50, 5)    # not a plain FASTQ start: serial path
    files["f.fa"] = ""                                    # empty file
    paths = []
    for name, text in files.items():
        p = tmp_path / name
        p.write_text(text, newline="")
        paths.append(str(p))
    gz = tmp_path / "g.fq.gz"
    with gzip.open(gz, "wt", newline="") as f:
        f.write(fastq(700, 6))
    paths.append(str(gz))
    want, _ = run(exe, "serial", *paths)
    assert want.count("\n") > 5000
    got, batches = run(exe, "stream", threads, 997, piece, *paths, env=None if mapped else {"ABB_NO_MMAP": "1"})
    assert got == want
    assert all(b == 997 for b in batches[:-1]) and 0 < batches[-1] <= 997 and sum(batches) == want.count("\n")


def test_stream_quality_options(exe, tmp_path):
    p = tmp_path / "q.fq"
    p.write_text(fastq(2000, 9, casava=True))
    for env in ({"READER_Q": "20"}, {"READER_MASKQ": "15"}, {"READER_NO_CHASTITY": "1"}):
        want, _ = run(exe, "serial", p, env=env)
        got, _ = run(exe, "stream", 4, 300, 777, p, env=env)
        assert got == want


def write_files(d, files, gz_text=None):
    paths = []
    for name, text in files.items():
        p = os.path.join(d, name)
        with open(p, "w", newline="") as f:
            f.write(text)
        paths.append(p)
    if gz_text is not None:
        p = os.path.join(d, "g.fq.gz")
        with gzip.open(p, "wt", newline="") as f:
            f.write(gz_text)
        paths.append(p)
    return paths


def reference_reader_inputs(d):
    """ids (Casava suffix), chastity filter, masked-end trimming, case folding, multi-line FASTA, CRLF, gz"""
    return write_files(d, {"a.fq": fastq(2000, 11), "b.fq": fastq(1000, 12, crlf=True, casava=True), "c.fa": fasta(500, 13)}, fastq(300, 14))


def golden_digest(text):
    return dict(sha256=hashlib.sha256(text.encode()).hexdigest(), lines=text.count("\n"))


def test_reader_equals_reference_reader(exe, tmp_path, golden_dir):
    # the output of the UNMODIFIED reference reader (DataLayer/FastaReader.cpp through oracle/_ref/ref_arith reads dump) on the
    # same files (tests/golden/make_golden_reader.py)
    want = json.load(open(os.path.join(golden_dir, "reader_cases.json")))["fastq_fasta_gz"]
    got, _ = run(exe, "stream", 3, 500, 4096, *reference_reader_inputs(tmp_path))
    assert golden_digest(got) == want


def test_long_records(exe, tmp_path):
    # a FASTA record longer than the reader's 8 MB buffer and than any piece, on one line and folded
    rng = random.Random(21)
    big = "".join(rng.choice("ACGT") for _ in range(1 << 16)) * 160          # 10.5 Mbp
    p = tmp_path / "big.fa"
    p.write_text(">one line\n" + big + "\n>folded\n" + "\n".join(big[i:i + 70] for i in range(0, 3_000_000, 70)) + "\n>tail\nACGT\n")
    want, _ = run(exe, "serial", p)
    lines = want.split("\n")
    assert [l.split("\t")[0] for l in lines[:3]] == ["one", "folded", "tail"]
    assert len(lines[0]) == 4 + len(big) and len(lines[1]) == 7 + 3_000_060 and lines[2] == "tail\tACGT"
    got, batches = run(exe, "stream", 2, 2, 1 << 20, p)
    assert got == want and batches == [2, 1]


def test_default_batch_size_with_long_record(exe, tmp_path):
    # the CLIs' default --batch-reads (4 000 000) with a multi-Mbp record: the batch buffers are sized as a hint with a
    # ceiling (the first version asked for 1.05 * 4e6 * 5 Mbp and died with std::bad_alloc)
    rng = random.Random(5)
    genome = "".join(rng.choice("ACGT") for _ in range(1 << 16)) * 80       # 5.2 Mbp
    p = tmp_path / "genome.fa"
    p.write_text(">chr1\n" + genome + "\n>chr2\n" + genome[:1000] + "\n")
    want, _ = run(exe, "serial", p)
    got, batches = run(exe, "stream", 2, 4_000_000, 1 << 24, p)
    assert got == want and sum(batches) == 2


def test_compressed_input_and_quoting(exe, tmp_path):
    import gzip
    # a file name with a single quote and a space goes through popen's shell unharmed
    d = tmp_path / "it's a dir"
    d.mkdir()
    p = d / "r.fa.gz"
    with gzip.open(p, "wt") as f:
        f.write(">a\nACGTACGT\n>b\nTTTT\n")
    got, _ = run(exe, "serial", p)
    assert got == "a\tACGTACGT\nb\tTTTT\n"
    # a decompressor that fails is an error, not an empty input
    bad = d / "broken.fa.gz"
    bad.write_bytes(b"this is not gzip")
    r = subprocess.run([exe, "serial", str(bad)], capture_output=True, text=True)
    assert r.returncode != 0 and "decompressor" in r.stderr


def _rand_seq(rng, n, alphabet="ACGT"):
    return "".join(rng.choice(alphabet) for _ in range(n))


def sam_text(n, seed):
    """SAM with a header, every flag combination the reader looks at (FPAIRED/FREAD1/FREAD2, FREVERSE, FSECONDARY, FQCFAIL),
    `*` sequences and qualities, lower-case bases, optional fields"""
    rng = random.Random(seed)
    out = ["@HD\tVN:1.0\tSO:unsorted", "@SQ\tSN:chr1\tLN:100000", "@PG\tID:bwa\tVN:0.7"]
    for i in range(n):
        flags = rng.choice([0, 1, 0x41, 0x81, 0x51, 0x91, 0x10, 0x100, 0x141, 0x200, 0x241, 0x4, 0x45])
        L = rng.randint(20, 120)
        s = _rand_seq(rng, L, "ACGTNacgt" if rng.random() < 0.2 else "ACGT")
        q = "".join(chr(rng.randint(33, 73)) for _ in range(L))
        r = rng.random()
        if r < 0.05:
            s, q = "*", "*"
        elif r < 0.15:
            q = "*"
        extra = "\tNM:i:0\tBX:Z:ACGT-1" if rng.random() < 0.3 else ""
        out.append(f"read{i}\t{flags}\tchr1\t{rng.randint(1, 9999)}\t60\t{L}M\t=\t{rng.randint(1, 9999)}\t0\t{s}\t{q}{extra}")
    return "\n".join(out) + "\n"


def qseq_text(n, seed, export=False):
    """qseq (11 fields) or export (22 fields): machine, run, lane, tile, x, y, index, read number, bases ('.' = no call),
    qualities (offset 64), ..., filter"""
    rng = random.Random(seed)
    out = []
    for i in range(n):
        L = rng.randint(20, 100)
        s = _rand_seq(rng, L, "ACGT.")
        q = "".join(chr(rng.randint(64, 104)) for _ in range(L))
        f = ["M1", str(rng.randint(1, 9)), str(rng.randint(1, 8)), str(rng.randint(1, 99)), str(i), str(rng.randint(0, 999)),
             rng.choice(["0", "ACGTAC", ""]), rng.choice(["1", "2", "3"]), s, q]
        chaste = rng.choice(["1", "0"] if not export else ["Y", "N"])
        if export:
            f += ["chr1", "", "123", "F", "100", "20", "0", "", "", "", "N"]
        f.append(chaste)
        assert len(f) == (22 if export else 11)
        out.append("\t".join(f))
    return "\n".join(out) + "\n"


def format_inputs(d):
    return write_files(d, {"a.sam": sam_text(800, 21), "b_qseq.txt": qseq_text(600, 22), "c_export.txt": qseq_text(400, 23, export=True),
                           "d.fq": fastq(500, 24, casava=True), "e.fa": fasta(200, 25)})


READER_OPTS = [{}, {"Q": "20"}, {"MASKQ": "15"}, {"NO_CHASTITY": "1"}, {"Q": "10", "QOFF": "64"}, {"MASKQ": "12", "QOFF": "33"}, {"NO_TRIM_MASKED": "1"}]


def opts_key(opts):
    return ",".join(f"{k}={v}" for k, v in opts.items()) or "default"


@pytest.mark.parametrize("opts", READER_OPTS)
def test_sam_qseq_export_equal_reference_reader(exe, tmp_path, golden_dir, opts):
    # the record formats of DataLayer/FastaReader.cpp:270-352 next to FASTQ, with the reader options of the command line
    # (-q, -Q, --illumina-quality / --standard-quality, --no-chastity, --no-trim-masked), against the output of the UNMODIFIED
    # reference reader on the same files with the same options (tests/golden/make_golden_reader.py)
    want = json.load(open(os.path.join(golden_dir, "reader_cases.json")))["formats"][opts_key(opts)]
    paths = format_inputs(tmp_path)
    env = {"READER_" + k: v for k, v in opts.items()}
    serial, _ = run(exe, "serial", *paths, env=env)
    assert golden_digest(serial) == want
    got, _ = run(exe, "stream", 3, 250, 4096, *paths, env=env)
    assert got == serial
    got, _ = run(exe, "stream", 3, 250, 4096, *paths, env=dict(env, ABB_NO_MMAP="1"))
    assert got == serial
    assert want["lines"] > 1500


@pytest.mark.parametrize("mapped", [True, False])
def test_error_line_number_in_a_later_piece(exe, tmp_path, mapped):
    # a broken record far into the file: the message names the line of the file (FastaReader::die, FastaReader.cpp:52-58) although
    # the piece that holds it was parsed on its own (mapped pieces count the lines before them only when a message is printed)
    lines = fastq(400, 31).split("\n")
    bad = 4 * 300 + 2          # the '+' line of record 300 (0-based line index)
    assert lines[bad] == "+"
    lines[bad] = "-"
    p = tmp_path / "bad.fq"
    p.write_text("\n".join(lines))
    env = dict(os.environ, **({} if mapped else {"ABB_NO_MMAP": "1"}))
    r = subprocess.run([exe, "stream", "3", "100", "2000", str(p)], capture_output=True, text=True, env=env)
    assert r.returncode != 0
    assert f"bad.fq:{bad}: error: expected `+' and saw `-'" in r.stderr, r.stderr
    r = subprocess.run([exe, "serial", str(p)], capture_output=True, text=True)
    assert f"bad.fq:{bad}: error: expected `+' and saw `-'" in r.stderr, r.stderr
