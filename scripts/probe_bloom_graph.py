"""Measure `abyss-bloom graph` on a rolling-hash filter far larger than L2: build a >= 1 GiB filter from reads of the bench
genome with `abyss-bloom build -t rolling-hash`, run `graph` with many read roots at the default depth and with a few roots
at a depth that exhausts their component, and, where oracle/_ref/abyss-bloom-ref exists, the reference on the same inputs
(with a time cap) to check that the outputs are byte-identical.  Needs a CUDA device; writes profiles/r03_bloom_graph.json
(or --out).

    python scripts/probe_bloom_graph.py [--reads 4000000] [--bloom 1G] [--out FILE]

Per run: wall time; time inside the neighbour queries (abb_neighbours: copies + k_neighbours, host clock, `-v`); GPU time
of k_neighbours alone (torch.profiler over a replay of the same levels through capi.neighbours); the rest = host time
(reading roots, root set, search bookkeeping, formatting); vertices expanded per second; levels and k_neighbours launches.
"""
import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CLI = os.path.join(ROOT, "abyss_b200", "lib", "abyss-bloom")
REF = os.path.join(ROOT, "oracle", "_ref", "abyss-bloom-ref")
SEED, GENOME, L, ERR, K, H = 2, 187_500_000, 150, 0.005, 32, 3  # the bench genome (bench.py)


def levels_of(dot: bytes):
    """the search levels, in queue order, from the vertex lines of a graph: level d = the vertices printed with depth=d"""
    lv = {}
    for m in re.finditer(rb"^\t([^ \n]+) \[depth=(\d+)", dot, re.M):
        lv.setdefault(int(m.group(2)), []).append(m.group(1))
    return [lv[d] for d in sorted(lv)]


def kernel_ms(bloom: str, levels) -> float:
    """GPU time of k_neighbours over the levels of one run, from torch.profiler (CUDA activities)"""
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile
    from abyss_b200 import capi
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    head = open(bloom, "rb").read(4096)
    hdr = dict(re.findall(rb"\t(\w+) = (\S+)", head[:head.index(b"[HeaderEnd]")]))
    off = head.index(b"[HeaderEnd]\n") + len(b"[HeaderEnd]\n")
    raw = np.fromfile(bloom, dtype=np.uint8, offset=off)
    f = capi.Filter.bits(int(hdr[b"BloomFilterSize"]), int(hdr[b"HashNum"]), int(hdr[b"KmerSize"]))
    f.upload(raw)
    del raw
    capi.neighbours(f, levels[0][:1])  # warm-up: module load
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for lv in levels:
            capi.neighbours(f, lv)
        torch.cuda.synchronize()
    f.close()
    return sum(e.device_time_total for e in prof.key_averages() if "k_neighbours" in e.key) / 1000.0


def run_graph(exe, args, out_path, cap=None):
    t0 = time.perf_counter()
    with open(out_path, "wb") as o:
        try:
            r = subprocess.run([exe, "graph", "-v", *args], stdout=o, stderr=subprocess.PIPE, timeout=cap)
        except subprocess.TimeoutExpired:
            return None, None
    wall = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError(f"{exe} graph failed: {r.stderr.decode()[-2000:]}")
    return wall, r.stderr.decode()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=4_000_000)
    ap.add_argument("--bloom", default="1G")
    ap.add_argument("--roots", type=int, default=10_000)
    ap.add_argument("--deep-roots", type=int, default=10)
    ap.add_argument("--deep-depth", type=int, default=1_000_000)
    ap.add_argument("--ref-cap", type=float, default=300.0, help="seconds the reference may take per run")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_bloom_graph.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("probe_bloom_graph: no CUDA device -- nothing measured")
    from abyss_b200 import build
    from abyss_b200.synth import ReadSet, write_fastq_fast
    build.build()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": gpu, "workload": f"{a.reads} x {L} bp reads of the bench genome ({GENOME} bp, err {ERR}, seed {SEED}), "
                                   f"k={K}, `abyss-bloom build -t rolling-hash -b{a.bloom} -H{H}`", "runs": []}
    with tempfile.TemporaryDirectory() as d:
        rs = ReadSet(SEED, GENOME, a.reads, L, ERR, paired=True)
        fq = os.path.join(d, "reads.fq")
        write_fastq_fast(rs, fq, 0, a.reads)
        bloom = os.path.join(d, "g.bloom")
        t0 = time.perf_counter()
        subprocess.run([CLI, "build", f"-k{K}", "-t", "rolling-hash", f"-b{a.bloom}", f"-H{H}", bloom, fq], check=True)
        res["build_seconds"] = round(time.perf_counter() - t0, 3)
        res["filter_bytes"] = os.path.getsize(bloom)
        os.remove(fq)
        for name, n_roots, extra in (("roots_default_depth", a.roots, []), ("roots_exhaust", a.deep_roots, ["-d", str(a.deep_depth)])):
            fa = os.path.join(d, name + ".fa")
            rs.write_fastq(fa, 0, n_roots, fasta=True)
            args = [f"-k{K}", *extra, "-f", fa, bloom]
            out = os.path.join(d, name + ".dot")
            wall, err = run_graph(CLI, args, out)
            dot = open(out, "rb").read()
            m = re.search(r"Expanded (\d+) vertices in (\d+) levels", err)
            nb = float(re.search(r"Neighbour queries: ([0-9.e+-]+) s", err).group(1))
            lv = levels_of(dot)
            r = {"name": name, "roots_reads": n_roots, "args": " ".join(extra) or "default depth (k)", "lines": dot.count(b"\n"),
                 "bytes": len(dot), "sha256": hashlib.sha256(dot).hexdigest(), "wall_s": round(wall, 3),
                 "neighbour_query_s": round(nb, 3), "host_other_s": round(wall - nb, 3),
                 "vertices": int(m.group(1)), "levels": int(m.group(2)), "k_neighbours_launches": int(m.group(2)),
                 "vertices_per_s": round(int(m.group(1)) / wall)}
            r["k_neighbours_gpu_ms"] = round(kernel_ms(bloom, lv), 3)
            del dot, lv
            if os.path.exists(REF):
                ref_out = os.path.join(d, name + ".ref.dot")
                rwall, _ = run_graph(REF, args, ref_out, cap=a.ref_cap)
                if rwall is None:
                    r["reference"] = f"not measured: exceeded the {a.ref_cap:.0f} s cap"
                else:
                    same = hashlib.sha256(open(ref_out, "rb").read()).hexdigest() == r["sha256"]
                    r["reference"] = {"wall_s": round(rwall, 3), "identical_output": same, "speedup": round(rwall / wall, 2)}
                os.remove(ref_out)
            else:
                r["reference"] = "not measured: oracle/_ref/abyss-bloom-ref not built"
            os.remove(out)
            res["runs"].append(r)
            print(json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
