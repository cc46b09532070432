#!/usr/bin/env python
"""bench.py -- the abyss-bloom-dbg hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--reads R] [--dump-outputs DIR]

One "step" = one complete pass of the hot path over the synthetic read set:
    pass 1  ntHash of every k-mer of every read + ordered counting-Bloom insert
    pass 2  classify reads, Bloom-backed unitig extension, ordered replay -> unitig FASTA
on the workload BASELINE.json's metric is quoted on (configs[1]): 50 M x 150 bp synthetic
paired reads (187.5 Mbp uniform-random genome, 40x, 0.5 % substitutions), k=64, kc=3, H=4,
-b 8 GiB (7 635 497 472 one-byte counters + 954 437 184 B assembled-k-mer bit filter), 1 x B200.
k-mers/s = (sum over reads of len-k+1) / step time, counted once per input k-mer.

`value`  : reads resident in HBM when the timed region starts (abb_*_dev entry points).
`e2e`    : same job through the host-buffer C-ABI calls (abb_insert_reads[_sharded], then
           abb_assembler_process_reads_dev on the copy that insert left on the device): pinned host reads are
           copied to the device inside the timed region (once: the copy stays resident for pass 2), the unitigs and
           per-read codes come back to the host.  Both arms, and every N, must give the same FASTA (`fasta_md5`,
           checked here: a mismatch between the e2e and the device-resident arm, or between ranks, fails the run).
`roofline`: the Bloom-insert kernel (k_insert_windows, the persistent window kernel): algorithmic bytes (64*H B of
           32-byte sectors per inserted k-mer + L/(L-k+1) B of read bases, SURVEY.md section 8d) x the slots its timed
           launches applied / their summed CUDA-event time, against the measured HBM copy bandwidth in
           MEASURED_PEAKS.json.  `insert_phase` is the same over the whole insert phase (hash + insert + drains).
`cpu_baseline`: the UNMODIFIED reference (oracle/_ref/abyss-bloom-dbg-ref, built by oracle/Makefile) with all host
           threads on a bounded sample (the first S reads of the workload).  Reported: the as-run rate (`value`), the
           start-up cost that depends on -b only (`fixed_s`, 1-read input: zero-filling 8 GiB of filters,
           contigEndKmers.rehash(2^28), bloom-dbg.h:993), the marginal rate, and -- from profiles/r02_ref_full_run.json --
           the one FULL 50 M-read run measured on this pool: 626 s with 128 threads = 6.9 M k-mers/s, unitig set
           identical to this implementation's.  The sample flatters the reference (3x coverage: its extension stage,
           85 % of the full job's time, hardly runs); see reference_measurement.
`--impl reference` times that reference binary as the step (bounded sample per step).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K, KC, H, L = 64, 3, 4, 150
BLOOM_BYTES = 8 << 30
N_READS = 50_000_000
GENOME = 187_500_000
ERR = 0.005
SEED = 2
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "abyss-bloom-dbg-ref")
ALG_BYTES_PER_KMER = 64 * H + L / (L - K + 1)  # SURVEY.md section 8(d): 257.7 B
# dram__bytes_read.sum + dram__bytes_write.sum of one k_insert_windows launch (ncu --set full; profiles/README.md), per
# k-mer slot applied; None until a capture of this round's kernel exists
NCU_TRAFFIC_PER_SLOT = 766.6  # 52.93 GB read + 13.76 GB written by the launch that applied 87.0 M slots (profiles/r02_k_insert_windows_final_raw.csv)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def pass2_rooflines(phases_ms, solid_reads, bases_assembled, peak, world=1):
    """HBM rooflines of the two pass-2 kernels that probe the 7.6 GB filter at random (SURVEY.md section 8d: 32-byte sectors).
    k_classify: a solid read costs (L-k+1) * H sectors for the solid test plus 2 * 5 * 4 * H for the two depth-5 blunt-end
    look-aheads (reads that fail early are counted as zero: a lower bound); the phase also holds the re-hash of the reads.
    k_make_tiles: every graph vertex lies on 4 tiles (2 orientations x 2 directions) and a tile step probes the 8 neighbours
    with H functions (8 * H sectors).  Both stages are divided over the ranks at N > 1."""
    out = []
    try:
        per_solid = (L - K + 1) * H * 32 + 2 * 5 * 4 * H * 32
        specs = (("k_classify (solid test + blunt-end look-ahead per read; phase incl. the re-hash of the reads)", "classify",
                  solid_reads * per_solid / world, f"solid_reads x ({L - K + 1} x H + 40 x H) x 32 B"),
                 ("k_make_tiles (marker-to-marker walks: 8 neighbours x H probes per vertex step)", "tiles",
                  4 * bases_assembled * 8 * H * 32 / world, "4 x graph vertices x 8 x H x 32 B"))
        for name, phase, nbytes, formula in specs:
            ms = float(phases_ms.get(phase, 0.0))
            if ms <= 0 or nbytes <= 0:
                continue
            achieved = nbytes / (ms * 1e-3) / 1e9
            out.append({"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                        "alg_bytes": nbytes, "alg_bytes_formula": formula, "phase_ms": ms})
    except Exception as e:  # never let a derived figure break the bench line
        out.append({"error": repr(e)})
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.samples, self.stop_flag, self.index = [], False, index
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop_flag = True
        self.t.join(timeout=3)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(float(s[0])) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples if len(s) > 2 + i)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(float(self.samples[0][1])), "reasons": reasons}


def write_sample_fastq(rs, n, path):
    """first n reads of the workload as FASTQ; generated on the GPU when there is one (the numpy generator needs ~8 us/read)"""
    from abyss_b200.synth import write_fastq_fast
    ascii_fn = None
    try:
        import torch
        if torch.cuda.is_available():
            from abyss_b200.synth_torch import TorchReadSet
            trs = TorchReadSet(rs, torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0"))))
            ascii_fn = lambda lo, hi: trs.ascii(lo, hi).cpu().numpy()
    except Exception:
        ascii_fn = None
    write_fastq_fast(rs, path, 0, n, ascii_fn=ascii_fn)


def run_reference(fq, threads, out_fa):
    """abyss-bloom-dbg (unmodified reference) wall time on fq with `threads` OpenMP threads"""
    cmd = f"ulimit -s 65536; exec {REF_BIN} -k{K} --kc={KC} -b{BLOOM_BYTES} -H{H} -j{threads} {fq} > {out_fa}"
    t0 = time.perf_counter()
    r = subprocess.run(["bash", "-c", cmd], capture_output=True, text=True)
    dt = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError("reference run failed: " + r.stderr[-500:])
    return dt


def reference_measurement(sample, cores, n_runs, warmup=0):
    """The reference on a BOUNDED sample of the workload: its first `sample` reads (same genome, same k / kc / H / -b),
    plus the start-up cost that depends on -b only (1-read input).  No bounded sample is faithful to the full job: this
    one has ~3x coverage, so almost nothing is solid and the reference's extension stage -- 85 % of its 626 s on the full
    job -- hardly runs (the sample flatters the reference: 14 M k-mers/s as-run against 6.9 M on the full job); a job of
    the same SHAPE (2 M reads at 40x of a 7.5 Mbp genome) is the other way round: 195 s = 0.9 M k-mers/s, because 12
    unitigs give the reference's per-read extension no parallelism.  The full run is recorded in
    profiles/r02_ref_full_run.json and copied into the line."""
    from abyss_b200.synth import ReadSet
    rs = ReadSet(SEED, GENOME, N_READS, L, ERR, paired=True)
    tmp = tempfile.mkdtemp(prefix="abyss_ref_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    fq1, fq = os.path.join(tmp, "one.fq"), os.path.join(tmp, "sample.fq")
    write_sample_fastq(rs, 1, fq1)
    write_sample_fastq(rs, sample, fq)
    out = os.path.join(tmp, "ref.fa")
    fixed = min(run_reference(fq1, cores, out) for _ in range(2))
    times = []
    for i in range(warmup + n_runs):
        dt = run_reference(fq, cores, out)
        if i >= warmup:
            times.append(dt)
    for f in (fq1, fq, out):
        os.remove(f)
    os.rmdir(tmp)
    t = sum(times) / len(times)
    kmers = sample * (L - K + 1)
    m = {"t": t, "fixed_s": fixed, "as_run": kmers / t, "marginal": kmers / max(t - fixed, 1e-3), "kmers": kmers}
    full = os.path.join(ROOT, "profiles", "r02_ref_full_run.json")
    if os.path.exists(full):  # one full 50 M-read run of the reference, measured once on this pool (scripts/ref_full_run.py)
        fr = json.load(open(full))["reference"]
        m["full_run"] = {"wall_s": fr["wall_s"], "kmers_per_s": fr["kmers_per_s"], "cmd": fr["cmd"], "source": "profiles/r02_ref_full_run.json"}
    return m


def cpu_baseline_dict(m, cores, sample):
    d = {"value": m["as_run"], "unit": "k-mers/s", "cores": cores, "kind": "reference",
         "marginal_value": m["marginal"], "fixed_s": m["fixed_s"], "sample_s": m["t"],
         "sample": f"first {sample} reads of the workload, abyss-bloom-dbg -j{cores} (unmodified reference), files on tmpfs; "
                   f"{m['t']:.1f} s per run of which {m['fixed_s']:.1f} s do not depend on the reads (1-read run, same -b: zero-filling "
                   "the filters, contigEndKmers.rehash(2^28)); the sample has ~3x coverage, so the reference's extension stage "
                   "(most of its time on the full job) hardly runs: see full_job_measured"}
    if "full_run" in m:
        d["full_job_measured"] = m["full_run"]
    return d


def reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation on this box's host cores"""
    if rank != 0:
        return
    from abyss_b200.synth import ReadSet
    cores = os.cpu_count() or 1
    if not os.path.exists(REF_BIN):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/abyss-bloom-dbg-ref not built (make -C oracle ref)"}))
        return
    # bounded: the whole call stays within a few minutes whatever --steps / --warmup say
    runs = args.warmup + args.steps
    sample = args.ref_reads if args.ref_reads else (8_000_000 if runs <= 4 else 4_000_000 if runs <= 8 else 2_000_000)
    m = reference_measurement(sample, cores, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "k-mers/sec (Bloom insert + unitig extend)", "value": m["as_run"], "unit": "k-mers/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * m["t"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args, extra={"sample_reads": sample}),
        "cpu_baseline": cpu_baseline_dict(m, cores, sample),
        "e2e": {"value": m["as_run"], "unit": "k-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def insert_sharded(world):
    """the library's policy (abb_insert_reads_sharded_dev): below ABB_SHARD_MIN_WORLD ranks (default 4) every rank runs the whole
    insert itself -- the position-sharded insert only beats one GPU from 4 ranks on -- and only pass 2 is divided"""
    return world > 1 and world >= max(2, int(os.environ.get("ABB_SHARD_MIN_WORLD", "4")))


def parallelism(world):
    if world == 1:
        return "1 GPU"
    p2 = ("pass 2: read classification, candidate scans and tile production sharded over the ranks (all-gather / exchange), "
          "walks and file-order replay replicated")
    if insert_sharded(world):
        return (f"pass 1: counters sharded by position range over {world} GPUs, one ncclAllReduce(min) per file-order window, "
                f"all-gather of the shards (exact: same counters as 1 GPU); {p2}")
    return f"pass 1: replicated on each of the {world} GPUs (no communication; the sharded insert is used from 4 GPUs on); {p2}"


def workload_config(args, extra=None):
    c = {"workload": f"{args.reads} x {L} bp synthetic paired reads, {GENOME} bp random genome, err {ERR}, k={K} kc={KC} H={H} -b 8GiB "
                     "(BASELINE.json configs[1])",
         "reads": args.reads, "read_len": L, "k": K, "kc": KC, "num_hashes": H, "bloom_bytes": BLOOM_BYTES,
         "l2_policy": "inputs (7.5 GB reads) and filters (8.6 GB) far exceed the 126 MB L2; no flush needed",
         "parallelism": parallelism(args.gpus)}
    if extra:
        c.update(extra)
    return c


def dump_outputs(out_dir, asm, filt, read_codes):
    """--dump-outputs: what a caller of the timed path receives from its last step, as DIR/<name>.npy, so that two builds can
    be compared output for output: the unitig records in output order (seed read, length, coverage), the unitig bases
    concatenated in output order (A=0 C=1 G=2 T=3), the per-read result codes (capi.READ_CODES) and the counting filter's
    counters.  An array longer than its cap is replaced by the entries at sorted positions drawn from
    np.random.default_rng(SEED).integers(0, length, cap), so the sample depends on the array's length only; the caps keep
    the directory under 64 MB."""
    import ctypes
    import numpy as np

    def sample(a, cap, dtype):
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(SEED).integers(0, a.size, cap))]
        return a.astype(dtype)

    contigs, n, seqs = asm._last
    recs = np.array([(contigs[i].seed_read, contigs[i].length, contigs[i].coverage) for i in range(n)], dtype=np.float64).reshape(n, 3)
    base = ctypes.cast(seqs, ctypes.c_void_p).value
    bases = np.frombuffer(b"".join(ctypes.string_at(base + contigs[i].seq_offset, contigs[i].length) for i in range(n)), dtype=np.uint8)
    lut = np.full(256, 255, dtype=np.uint8)
    lut[np.frombuffer(b"ACGT", dtype=np.uint8)] = np.arange(4, dtype=np.uint8)
    arrays = {"unitig_seed_read": sample(recs[:, 0], 1 << 20, np.float64), "unitig_length": sample(recs[:, 1], 1 << 20, np.float64),
              "unitig_coverage": sample(recs[:, 2], 1 << 20, np.float64), "unitig_bases": sample(lut[bases], 1 << 22, np.float32),
              "read_codes": sample(read_codes, 1 << 20, np.float32), "counters": sample(filt.download(), 1 << 22, np.float32)}
    assert sum(a.nbytes for a in arrays.values()) <= 64_000_000
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=N_READS, help="number of reads of the workload (default: the BASELINE config)")
    ap.add_argument("--ref-reads", type=int, default=0, help="bounded CPU sample (reads); 0 = sized from --steps")
    ap.add_argument("--window", type=int, default=0, help="ordered-insert window in k-mer slots (0 = library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from abyss_b200 import build as abb_build
    if rank == 0:
        abb_build.build()
    from abyss_b200 import capi
    from abyss_b200.synth import ReadSet
    from abyss_b200.synth_torch import TorchReadSet

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    capi.load()
    dev = torch.device("cuda", local_rank)

    # ---- synthetic reads, generated on the device
    rs = ReadSet(SEED, GENOME, args.reads, L, ERR, paired=True)
    trs = TorchReadSet(rs, dev)
    bases = torch.empty(rs.n * L, dtype=torch.uint8, device=dev)
    step_reads = 1 << 21
    for s in range(0, rs.n, step_reads):
        e = min(rs.n, s + step_reads)
        bases[s * L:e * L] = trs.ascii(s, e).reshape(-1)
    offs = torch.arange(rs.n + 1, dtype=torch.int64, device=dev) * L
    del trs
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    n_kmers_expected = rs.n * (L - K + 1)
    counters = capi.counters_for_budget(BLOOM_BYTES)

    filt = capi.Filter.counting(counters, H, K, KC, device=local_rank)
    filt.set_profiling(True)
    if args.window:
        filt.set_window(args.window)
    ext = torch.cuda.ExternalStream(filt.stream(), device=dev)

    # N > 1: the NCCL communicator lives behind the C ABI; torch.distributed only ships its id and the timings
    comm = None
    if world > 1:
        def bcast(b):
            box = [b]
            dist.broadcast_object_list(box, src=0)
            return box[0]
        comm = capi.Comm(rank, world, local_rank, bcast)
    asm = capi.Assembler(filt)  # one handle for all steps: device buffers are allocated once, state is reset per step
    asm.raw_results = True      # the unitig sequences are copied to the host by the library; no Python string per unitig

    if world > 1:
        asm.set_comm(comm)      # classification, candidate scans and tile production are sharded inside the library

    def pass2(d_bases, d_offs):
        return asm.process_reads_dev(d_bases, d_offs, rs.n)

    def one_step(host=None):
        """returns (n_kmers, contigs, assembler stats, insert stats, counters)"""
        filt.clear()
        filt.stats(reset=True)
        asm.reset()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(ext)
        if host is None:
            if world > 1:
                nk = filt.insert_reads_sharded_dev(comm, bases.data_ptr(), offs.data_ptr(), rs.n)
            else:
                nk = filt.insert_reads_dev(bases.data_ptr(), offs.data_ptr(), rs.n, bases.numel())
            p1.record(ext)
            contigs = pass2(bases.data_ptr(), offs.data_ptr())
        else:
            nk = filt.insert_reads_sharded(comm, host) if world > 1 else filt.insert_reads(host)
            p1.record(ext)
            d_b, d_o, n_res = filt.resident_reads()  # the copy pass 1 made stays on the device for pass 2
            assert n_res == rs.n
            contigs = pass2(d_b, d_o)
        torch.cuda.synchronize()
        ast, ist, cnt = asm.stats(), filt.stats(), asm.counters()
        ist.ms_pass1 = p0.elapsed_time(p1)
        return nk, contigs, ast, ist, cnt

    def timed(n_steps, host=None):
        res = []
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(n_steps):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ev0.record(ext)
            out = one_step(host)
            ev1.record(ext)
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1)
            if world > 1:
                t = torch.tensor([ms], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            res.append((ms, out))
        return res

    for _ in range(args.warmup):
        timed(1)
    with ClockSampler(local_rank) as clk:
        runs = timed(args.steps)
    ms_step = sum(r[0] for r in runs) / len(runs)
    nk, contigs, ast, ist, cnt = runs[-1][1]
    assert nk == n_kmers_expected, (nk, n_kmers_expected)
    total_kmers = nk  # one job, counted once (strong scaling)
    value = total_kmers / (ms_step * 1e-3)
    digest = asm.last_digests(rs.read_id)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, asm, filt, asm.read_results())

    # ---- e2e through host buffers
    e2e = None
    if not args.no_e2e:
        hb = torch.empty(bases.numel(), dtype=torch.uint8, pin_memory=True)
        hb.copy_(bases)
        ho_t = torch.empty(offs.numel(), dtype=torch.int64, pin_memory=True)  # both input arrays in pinned host memory
        ho_t.copy_(offs)
        ho = ho_t.numpy().view(np.uint64)
        host = (hb.numpy(), ho)
        timed(1, host)
        eruns = timed(max(1, min(args.steps, 3)), host)
        ems = sum(r[0] for r in eruns) / len(eruns)
        econt = eruns[-1][1][1]
        edigest = asm.last_digests(rs.read_id)
        assert edigest == digest, ("e2e output differs from the device-resident arm", edigest, digest)
        d2h = sum(c[1] for c in econt) + 24 * len(econt) + rs.n  # unitig bases + records + per-read codes
        e2e = {"value": total_kmers / (ems * 1e-3), "unit": "k-mers/s", "ms_per_step": ems,
               "h2d_bytes_per_step": int(hb.numel()) + int(ho.nbytes), "d2h_bytes_per_step": int(d2h),
               "note": "per rank" if world > 1 else "", "fasta_md5": edigest["fasta_md5"],
               "pass1_ms": float(eruns[-1][1][3].ms_pass1)}
        del hb
    if world > 1:  # every rank must have produced the same FASTA
        box = [None] * world
        dist.all_gather_object(box, digest)
        assert all(d == box[0] for d in box), ("ranks disagree on the output", box)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peak, peak_src = peaks()
    launch_ms = ist.ms_commit / max(1, ist.commit_launches)
    slots_per_launch = ist.commit_slots / max(1, ist.commit_launches)
    # sharded insert: each rank moves 1/N of the counter sectors of every slot it evaluates; replicated insert: all of them
    sharded = insert_sharded(world)
    alg_per_slot = (64 * H) / (world if sharded else 1) + L / (L - K + 1)
    achieved = alg_per_slot * slots_per_launch / (launch_ms * 1e-3) / 1e9 if launch_ms > 0 else 0.0
    phase_ms = ist.ms_pass1
    phase_achieved = alg_per_slot * nk / (phase_ms * 1e-3) / 1e9
    kernel = "k_insert_windows (persistent ordered counting-Bloom min-increment)" if not sharded else \
        "k_sh_gather + ncclAllReduce(min) + k_sh_apply (one file-order window, counters sharded by position)"
    roofline = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": NCU_TRAFFIC_PER_SLOT * slots_per_launch if NCU_TRAFFIC_PER_SLOT else None,
                "peak_source": peak_src, "alg_bytes_per_kmer": alg_per_slot, "launches": int(ist.commit_launches),
                "slots_per_launch": slots_per_launch, "avg_launch_ms": launch_ms, "share_of_step": ist.ms_commit / ms_step,
                "insert_phase": {"ms": phase_ms, "achieved": phase_achieved, "frac": phase_achieved / peak,
                                 "what": "hash + ordered insert + drains" + (" + all-gather of the shards" if sharded else "")}}

    cpu = None
    if not args.no_cpu_baseline and os.path.exists(REF_BIN) and world == 1:
        cores = os.cpu_count() or 1
        sample = args.ref_reads or 4_000_000
        cpu = cpu_baseline_dict(reference_measurement(min(sample, rs.n), cores, 1), cores, min(sample, rs.n))

    line = {
        "metric": "k-mers/sec (Bloom insert + unitig extend)", "value": value, "unit": "k-mers/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args), "clocks": clk.summary(), "e2e": e2e,
        "gpu_launches": int(ist.launches + ast.launches), "roofline": roofline,
        "roofline_pass2": pass2_rooflines({"classify": ast.ms_classify, "tiles": ast.ms_tiles}, int(cnt.solid_reads), int(cnt.bases_assembled),
                                          peak, world),
        "cpu_baseline": cpu,
        "phases_ms": {"hash": ist.ms_hash, "insert": ist.ms_insert, "classify": ast.ms_classify, "visited": ast.ms_visited,
                      "tiles": ast.ms_tiles, "extend": ast.ms_extend, "extend_walk": ast.ms_walk, "extend_stage": ast.ms_stage,
                      "extend_repeat_check": ast.ms_repeat, "replay": ast.ms_replay, "pass2_wall": ast.ms_total,
                      "candidate_list_host": ast.ms_cand},
        "pass1_ms": ist.ms_pass1, "insert_kmers_per_s": nk / (ist.ms_pass1 * 1e-3),
        "extend_kmers_per_s": nk / ((ast.ms_classify + ast.ms_tiles + ast.ms_visited + ast.ms_extend + ast.ms_replay) * 1e-3),
        "unitigs": int(cnt.contig_id), "bases_assembled": int(cnt.bases_assembled),
        "fasta_md5": digest["fasta_md5"], "unitig_multiset_md5": digest["unitig_multiset_md5"],
        "drains": int(ist.drains), "drained_slots": int(ist.drained_slots),
        "speculation": {"rounds": int(ast.rounds), "speculated": int(ast.speculated_reads), "wasted": int(ast.wasted_reads),
                        "markers": int(ast.markers), "tiles": int(ast.tiles), "serial_fallbacks": int(ast.serial_fallbacks)},
        "deferred_inserts": int(ist.deferred),
    }
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
