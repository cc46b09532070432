"""Goldens of the overlap-graph stage: the unmodified reference AdjList (oracle/_ref/AdjList-ref, built by
`make -C oracle ref`) run on the seeded contig sets of tests/overlap_cases.py.  Writes overlap_cases.json
(sha256 of the output of every case), the complete output of three cases, overlap_ref_runs.json (sha256 of the
output of further fuzz sets, of the sets the GPU command line runs, of the option-alias runs and of the config-1
unitig sets) and unitigs_config1.json.gz (those unitig sets of the reference's abyss-bloom-dbg, as genome coordinates).

    python tests/golden/make_golden_overlap.py
"""
import gzip
import hashlib
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)
import overlap_cases as oc  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref", "AdjList-ref")
DBG_REF = os.path.join(ROOT, "oracle", "_ref", "abyss-bloom-dbg-ref")
FULL = {"unitigs_k64_adj", "unitigs_k32_dot", "fuzz7"}


def unitig_sets(tmp):
    """the reference's unitig FASTA of config 1 at every k of oc.UNITIG_RUNS: each record as [header, pos, length] when its
    sequence is a substring of the genome (pos < 0: of its reverse complement, at -pos-1), else [header, sequence]"""
    from abyss_b200.synth import ReadSet
    fq = os.path.join(tmp, "config1.fq")
    ReadSet(*oc.UNITIG_SET_READS).write_fastq(fq)
    g = oc.unitig_set_genome()
    g_rc = oc.rc(g)
    sets = {}
    for k in sorted({k for k, _, _ in oc.UNITIG_RUNS}):
        fa = os.path.join(tmp, f"unitigs-k{k}.fa")
        subprocess.run(["bash", "-c", f"ulimit -s 65536; {DBG_REF} -k{k} --kc=2 -b64M -H4 -j1 {fq} > {fa} 2>/dev/null"], check=True)
        text = open(fa).read()
        records = []
        for head, seq in zip(text.splitlines()[0::2], text.splitlines()[1::2]):
            assert head.startswith(">") and not seq.startswith(">")
            p = g.find(seq)
            if p >= 0:
                records.append([head[1:], p, len(seq)])
                continue
            p = g_rc.find(seq)  # seq = rc(g[q:q+len]) with q = len(g) - p - len
            records.append([head[1:], -(len(g) - p - len(seq)) - 1, len(seq)] if p >= 0 else [head[1:], seq])
        sets[str(k)] = dict(sha256=hashlib.sha256(text.encode()).hexdigest(), records=records)
    with gzip.GzipFile(os.path.join(HERE, "unitigs_config1.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(sets, separators=(",", ":")).encode())
    for k in sets:
        assert oc.unitig_set_fasta(int(k)) == (open(os.path.join(tmp, f"unitigs-k{k}.fa")).read(), sets[k]["sha256"])


def ref_runs(tmp):
    out = {}

    def run(name, args, stdin=None):
        r = subprocess.run([REF] + args, input=stdin, capture_output=True, check=True, text=stdin is not None)
        out[name] = oc.ref_run_digest(r.stdout.encode() if stdin is not None else r.stdout, REF, tmp)

    for c in oc.more_fuzz_cases() + oc.cli_cases():
        fa = os.path.join(tmp, "in.fa")
        oc.write_fasta(c, fa)
        run(c["name"], oc.command_args(c, fa))
    for name, args, stdin in oc.alias_runs(tmp):
        run(name, args, stdin)
    for k, m, fmt in oc.UNITIG_RUNS:
        fa = os.path.join(tmp, "unitigs-1.fa")
        open(fa, "w").write(oc.unitig_set_fasta(k)[0])
        run(f"unitigs_config1_k{k}_m{m}_{fmt[2:]}", [f"-k{k}", f"-m{m}", fmt, fa])
    with open(os.path.join(HERE, "overlap_ref_runs.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)


def main():
    tmp = "/tmp/abyss_golden_overlap"
    os.makedirs(tmp, exist_ok=True)
    out = {}
    for c in oc.all_cases():
        fa = os.path.join(tmp, c["name"] + ".fa")
        oc.write_fasta(c, fa)
        r = subprocess.run([REF] + oc.command_args(c, fa), capture_output=True, check=True)
        data = oc.normalise(r.stdout, REF).replace(fa.encode(), b"IN.fa")
        out[c["name"]] = dict(sha256=hashlib.sha256(data).hexdigest(), bytes=len(data), contigs=len(c["records"]))
        if c["name"] in FULL:
            with open(os.path.join(HERE, "overlap_" + c["name"] + ".txt"), "wb") as f:
                f.write(data)
    with open(os.path.join(HERE, "overlap_cases.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print(len(out), "cases")
    unitig_sets(tmp)
    ref_runs(tmp)


if __name__ == "__main__":
    main()
