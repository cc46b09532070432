"""ctypes binding of libabyssb200.so (the C ABI in include/abyss_b200.h).

This is the stub a maintainer of a Python harness would write; the C++ CLI links the same
library directly.  There is deliberately no fallback: if the CUDA library is missing the
import raises, and if no GPU is present every compute call fails with ABB_ENODEV.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libabyssb200.so")

ABB_OK, ABB_EINVAL, ABB_ENODEV, ABB_ECUDA, ABB_ENOMEM, ABB_ESTATE = 0, -1, -2, -3, -4, -5
COUNTING, BIT, CASCADING = 0, 1, 2


class AbbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libabyssb200 error {code}: {msg}")
        self.code = code


class InsertStats(C.Structure):
    _fields_ = [("kmers", C.c_uint64), ("slots", C.c_uint64), ("windows", C.c_uint64),
                ("deferred", C.c_uint64), ("launches", C.c_uint64),
                ("ms_hash", C.c_float), ("ms_insert", C.c_float), ("ms_commit", C.c_float),
                ("commit_launches", C.c_uint64), ("commit_slots", C.c_uint64), ("drains", C.c_uint64),
                ("drained_slots", C.c_uint64)]


class Contig(C.Structure):
    _fields_ = [("seed_read", C.c_uint64), ("seq_offset", C.c_uint64),
                ("length", C.c_uint32), ("coverage", C.c_uint32)]


class AssemblyParams(C.Structure):
    _fields_ = [("trim", C.c_uint), ("verbose", C.c_uint), ("read_log", C.c_uint), ("reserved", C.c_uint)]


class TraceRow(C.Structure):
    _fields_ = [("contig_id", C.c_uint64), ("seed_read", C.c_uint64), ("length", C.c_uint32), ("seed_pos", C.c_uint32),
                ("left_n", C.c_uint32), ("right_n", C.c_uint32), ("left_code", C.c_uint8), ("right_code", C.c_uint8),
                ("redundant", C.c_uint8), ("pad", C.c_uint8)]


class AssemblyStats(C.Structure):
    _fields_ = [("rounds", C.c_uint64), ("speculated_reads", C.c_uint64), ("wasted_reads", C.c_uint64),
                ("candidates", C.c_uint64), ("contigs_tried", C.c_uint64), ("launches", C.c_uint64),
                ("ms_classify", C.c_float), ("ms_visited", C.c_float), ("ms_extend", C.c_float), ("ms_replay", C.c_float),
                ("ms_tiles", C.c_float), ("ms_walk", C.c_float), ("ms_stage", C.c_float), ("ms_repeat", C.c_float), ("ms_total", C.c_float), ("ms_cand", C.c_float), ("markers", C.c_uint64), ("tiles", C.c_uint64), ("serial_fallbacks", C.c_uint64)]


class AssemblyCounters(C.Structure):
    _fields_ = [("solid_reads", C.c_uint64), ("visited_reads", C.c_uint64),
                ("reads_processed", C.c_uint64), ("bases_assembled", C.c_uint64),
                ("contig_id", C.c_uint64)]


class SuccInfo(C.Structure):
    _fields_ = [("hash", C.c_uint64 * 4), ("mask", C.c_uint8), ("pad", C.c_uint8 * 7)]


class Neighbourhood(C.Structure):
    _fields_ = [("hash", C.c_uint64 * 9), ("attr", C.c_uint32 * 9), ("mask", C.c_uint16), ("pad", C.c_uint8 * 2)]


class OverlapEdge(C.Structure):
    _fields_ = [("u", C.c_uint32), ("v", C.c_uint32), ("distance", C.c_int32)]


class OverlapStats(C.Structure):
    _fields_ = [("vertices", C.c_uint64), ("exact_edges", C.c_uint64), ("short_edges", C.c_uint64), ("blunt_vertices", C.c_uint64),
                ("launches", C.c_uint64)]


_u64p = C.POINTER(C.c_uint64)
_u8p = C.POINTER(C.c_uint8)
_vp = C.c_void_p

# name -> (restype, argtypes); every symbol declared in include/abyss_b200.h
SIGNATURES = {
    "abb_version": (C.c_int, []),
    "abb_last_error": (C.c_char_p, []),
    "abb_device_count": (C.c_int, []),
    "abb_filter_create": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_uint64, C.c_uint, C.c_uint, C.c_uint, C.c_char_p, C.c_int]),
    "abb_filter_destroy": (C.c_int, [_vp]),
    "abb_filter_kmer_size": (C.c_uint, [_vp]),
    "abb_filter_hash_num": (C.c_uint, [_vp]),
    "abb_filter_size": (C.c_uint64, [_vp]),
    "abb_filter_size_in_bytes": (C.c_uint64, [_vp]),
    "abb_filter_threshold": (C.c_uint, [_vp]),
    "abb_filter_levels": (C.c_uint, [_vp]),
    "abb_filter_set_threshold": (C.c_int, [_vp, C.c_uint]),
    "abb_insert_reads": (C.c_int, [_vp, _vp, _vp, C.c_uint64, _u64p]),
    "abb_insert_reads_dev": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.c_uint64, _u64p]),
    "abb_insert_hashes": (C.c_int, [_vp, _vp, C.c_uint64]),
    "abb_contains_hashes": (C.c_int, [_vp, _vp, C.c_uint64, _vp]),
    "abb_mincount_hashes": (C.c_int, [_vp, _vp, C.c_uint64, _vp]),
    "abb_hash_reads": (C.c_int, [C.c_uint, C.c_char_p, _vp, _vp, C.c_uint64, _vp, _vp, _u64p, C.c_int]),
    "abb_hash_reads_dev": (C.c_int, [_vp, _vp, _vp, C.c_uint64, _vp, _vp, C.c_uint64, _u64p]),
    "abb_insert_h0_dev": (C.c_int, [_vp, _vp, C.c_uint64]),
    "abb_comm_unique_id": (C.c_int, [_vp]),
    "abb_comm_create": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_int, _vp, C.c_int]),
    "abb_comm_destroy": (C.c_int, [_vp]),
    "abb_comm_rank": (C.c_int, [_vp]),
    "abb_comm_world": (C.c_int, [_vp]),
    "abb_insert_reads_sharded_dev": (C.c_int, [_vp, _vp, _vp, _vp, C.c_uint64, C.c_int, _u64p]),
    "abb_insert_reads_sharded": (C.c_int, [_vp, _vp, _vp, _vp, C.c_uint64, C.c_int, _u64p]),
    "abb_filter_resident_reads": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), _u64p]),
    "abb_filter_allgather": (C.c_int, [_vp, _vp]),
    "abb_comm_allgather_bytes": (C.c_int, [_vp, _vp, C.c_uint64, _vp]),
    "abb_comm_allreduce_max_u8": (C.c_int, [_vp, _vp, C.c_uint64, _vp]),
    "abb_comm_exchange_bytes": (C.c_int, [_vp, _vp, C.c_uint64, _vp, _u64p, _u64p, _vp]),
    "abb_filter_device_ptr": (_vp, [_vp, C.c_int]),
    "abb_filter_download": (C.c_int, [_vp, C.c_int, _vp, C.c_uint64]),
    "abb_filter_upload": (C.c_int, [_vp, C.c_int, _vp, C.c_uint64]),
    "abb_filter_clear": (C.c_int, [_vp]),
    "abb_filter_popcount": (C.c_int, [_vp, _u64p, _u64p]),
    "abb_assembler_create": (C.c_int, [C.POINTER(_vp), _vp, C.POINTER(AssemblyParams)]),
    "abb_assembler_destroy": (C.c_int, [_vp]),
    "abb_assembler_process_reads": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.POINTER(C.POINTER(Contig)), _u64p, C.POINTER(C.c_char_p)]),
    "abb_assembler_process_reads_dev": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.POINTER(C.POINTER(Contig)), _u64p, C.POINTER(C.c_char_p)]),
    "abb_assembler_stats": (C.c_int, [_vp, C.POINTER(AssemblyStats)]),
    "abb_assembler_reset": (C.c_int, [_vp]),
    "abb_assembler_classify_dev": (C.c_int, [_vp, _vp, _vp, C.c_uint64, _vp]),
    "abb_assembler_set_codes": (C.c_int, [_vp, _vp, C.c_uint64]),
    "abb_assembler_counters": (C.c_int, [_vp, C.POINTER(AssemblyCounters)]),
    "abb_assembler_set_counters": (C.c_int, [_vp, C.POINTER(AssemblyCounters)]),
    "abb_assembler_read_results": (C.c_int, [_vp, C.POINTER(_u8p), _u64p]),
    "abb_assembler_set_comm": (C.c_int, [_vp, _vp]),
    "abb_assembler_trace": (C.c_int, [_vp, C.POINTER(C.POINTER(TraceRow)), _u64p]),
    "abb_assembler_assembled_filter": (_vp, [_vp]),
    "abb_filter_insert_stats": (C.c_int, [_vp, C.POINTER(InsertStats), C.c_int]),
    "abb_filter_set_window": (C.c_int, [_vp, C.c_uint64]),
    "abb_filter_set_profiling": (C.c_int, [_vp, C.c_int]),
    "abb_filter_stream": (_vp, [_vp]),
    "abb_contains_reads": (C.c_int, [_vp, _vp, _vp, C.c_uint64, _vp, _vp, C.c_uint64, _u64p]),
    "abb_successors": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint, _vp, _vp, _vp]),
    "abb_neighbours": (C.c_int, [_vp, _vp, C.c_uint, _vp, C.c_uint64, _vp]),
    "abb_overlap_create": (C.c_int, [C.POINTER(_vp), C.c_int]),
    "abb_overlap_destroy": (C.c_int, [_vp]),
    "abb_overlap_build": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.c_uint, C.c_uint, C.c_int, C.POINTER(C.POINTER(OverlapEdge)), _u64p]),
    "abb_overlap_get_stats": (C.c_int, [_vp, C.POINTER(OverlapStats)]),
}

_lib = None


def load(path: str | None = None) -> C.CDLL:
    """Load the CUDA library; raises (no fallback) when it has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise ImportError(f"{p} not found: build it with `python -m abyss_b200.build` "
                          "(libabyssb200 is CUDA-only, there is no CPU fallback)")
    lib = C.CDLL(p)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != ABB_OK:
        raise AbbError(rc, load().abb_last_error().decode(errors="replace"))


def pack_reads(seqs) -> tuple[np.ndarray, np.ndarray]:
    """list of str/bytes -> (bases uint8[], offsets uint64[n+1])"""
    bs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    offs = np.zeros(len(bs) + 1, dtype=np.uint64)
    if bs:
        offs[1:] = np.cumsum([len(b) for b in bs], dtype=np.uint64)
    bases = np.frombuffer(b"".join(bs), dtype=np.uint8).copy() if bs else np.zeros(0, dtype=np.uint8)
    return bases, offs


def fixed_length_reads(ascii_2d: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """(n, L) uint8 array of ASCII bases -> (bases, offsets) without copying per read"""
    n, L = ascii_2d.shape
    return np.ascontiguousarray(ascii_2d).reshape(-1), (np.arange(n + 1, dtype=np.uint64) * np.uint64(L))


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(_vp)


def hash_reads(k: int, seqs_or_arrays, mask: str = "", device: int = 0):
    """RollingHashIterator over a batch: returns (h0[slots], valid[slots], slot_offsets[n+1])."""
    lib = load()
    bases, offs = seqs_or_arrays if isinstance(seqs_or_arrays, tuple) else pack_reads(seqs_or_arrays)
    lens = np.diff(offs).astype(np.int64)
    counts = np.maximum(lens - k + 1, 0).astype(np.uint64)
    slot_offs = np.zeros(len(counts) + 1, dtype=np.uint64)
    slot_offs[1:] = np.cumsum(counts, dtype=np.uint64)
    total = int(slot_offs[-1])
    h0 = np.zeros(total, dtype=np.uint64)
    valid = np.zeros(total, dtype=np.uint8)
    n_slots = C.c_uint64(0)
    check(lib.abb_hash_reads(k, mask.encode(), _ptr(bases), _ptr(offs), len(offs) - 1, _ptr(h0), _ptr(valid),
                             C.byref(n_slots), device))
    assert n_slots.value == total, (n_slots.value, total)
    return h0, valid, slot_offs


class Comm:
    """the NCCL communicator behind the C ABI (one per process / GPU).  `bcast` ships rank 0's 128-byte id to the
    other ranks: a callable (bytes | None) -> bytes, e.g. torch.distributed.broadcast_object_list."""

    def __init__(self, rank: int, world: int, device: int, bcast):
        self._lib = load()
        self._h = _vp()
        ident = np.zeros(128, dtype=np.uint8)
        if rank == 0:
            check(self._lib.abb_comm_unique_id(_ptr(ident)))
        ident = np.frombuffer(bcast(ident.tobytes() if rank == 0 else None), dtype=np.uint8).copy()
        check(self._lib.abb_comm_create(C.byref(self._h), rank, world, _ptr(ident), device))
        self.rank, self.world = rank, world

    @property
    def handle(self):
        return self._h

    def allgather_bytes(self, d_buf_ptr: int, bytes_per_rank: int, stream: int = 0):
        check(self._lib.abb_comm_allgather_bytes(self._h, _vp(d_buf_ptr), bytes_per_rank, _vp(stream)))

    def allreduce_max_u8(self, d_buf_ptr: int, n: int, stream: int = 0):
        check(self._lib.abb_comm_allreduce_max_u8(self._h, _vp(d_buf_ptr), n, _vp(stream)))

    def close(self):
        if self._h:
            self._lib.abb_comm_destroy(self._h)
            self._h = _vp()


class Filter:
    """Host mirror of the reference's Bloom filter classes over a device-resident array.

    kind COUNTING  ~ CountingBloomFilter<uint8_t>(size, H, k, threshold)  (CountingBloomFilter.hpp:31-50)
    kind BIT       ~ BloomFilter(size_bits, H, k)                          (BloomFilter.hpp:64-74)
    kind CASCADING ~ HashAgnosticCascadingBloom(size_bits, H, levels, k)   (HashAgnosticCascadingBloom.h:43-55)
    """

    def __init__(self, kind: int, size: int, num_hashes: int, k: int, arg: int = 0, mask: str = "", device: int = 0):
        self._lib = load()
        self._h = _vp()
        check(self._lib.abb_filter_create(C.byref(self._h), kind, size, num_hashes, k, arg, mask.encode(), device))
        self.kind = kind

    @classmethod
    def counting(cls, counters, num_hashes, k, threshold=0, mask="", device=0):
        return cls(COUNTING, counters, num_hashes, k, threshold, mask, device)

    @classmethod
    def bits(cls, size_bits, num_hashes, k, mask="", device=0):
        return cls(BIT, size_bits, num_hashes, k, 0, mask, device)

    @classmethod
    def cascading(cls, size_bits, num_hashes, levels, k, mask="", device=0):
        return cls(CASCADING, size_bits, num_hashes, k, levels, mask, device)

    # -- reference getters
    def getKmerSize(self): return self._lib.abb_filter_kmer_size(self._h)
    def getHashNum(self): return self._lib.abb_filter_hash_num(self._h)
    def size(self): return self._lib.abb_filter_size(self._h)
    def sizeInBytes(self): return self._lib.abb_filter_size_in_bytes(self._h)
    def threshold(self): return self._lib.abb_filter_threshold(self._h)
    def levels(self): return self._lib.abb_filter_levels(self._h)
    def set_threshold(self, t): check(self._lib.abb_filter_set_threshold(self._h, t))
    def set_window(self, w): check(self._lib.abb_filter_set_window(self._h, w))
    def set_profiling(self, on=True): check(self._lib.abb_filter_set_profiling(self._h, int(on)))
    def stream(self) -> int: return self._lib.abb_filter_stream(self._h) or 0

    @property
    def handle(self):
        return self._h

    def close(self):
        if self._h:
            self._lib.abb_filter_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- pass 1
    def insert_reads(self, seqs_or_arrays) -> int:
        bases, offs = seqs_or_arrays if isinstance(seqs_or_arrays, tuple) else pack_reads(seqs_or_arrays)
        n = C.c_uint64(0)
        check(self._lib.abb_insert_reads(self._h, _ptr(bases), _ptr(offs), len(offs) - 1, C.byref(n)))
        return n.value

    def insert_reads_dev(self, d_bases_ptr: int, d_offs_ptr: int, n_reads: int, n_bases: int) -> int:
        n = C.c_uint64(0)
        check(self._lib.abb_insert_reads_dev(self._h, _vp(d_bases_ptr), _vp(d_offs_ptr), n_reads, n_bases, C.byref(n)))
        return n.value

    # -- multi-GPU building blocks
    def hash_reads_dev(self, d_bases_ptr, d_offs_ptr, n_reads, d_h0_ptr=0, d_valid_ptr=0, capacity=0) -> int:
        n = C.c_uint64(0)
        check(self._lib.abb_hash_reads_dev(self._h, _vp(d_bases_ptr), _vp(d_offs_ptr), n_reads, _vp(d_h0_ptr), _vp(d_valid_ptr), capacity,
                                           C.byref(n)))
        return n.value

    def insert_reads_sharded_dev(self, comm: "Comm", d_bases_ptr: int, d_offs_ptr: int, n_reads: int, finalize: bool = True) -> int:
        """exact multi-GPU insert: EVERY rank passes all reads; counters sharded by position range (abb_shard.cuh)"""
        n = C.c_uint64(0)
        check(self._lib.abb_insert_reads_sharded_dev(self._h, comm.handle, _vp(d_bases_ptr), _vp(d_offs_ptr), n_reads, int(finalize),
                                                     C.byref(n)))
        return n.value

    def insert_reads_sharded(self, comm: "Comm", seqs_or_arrays, finalize: bool = True) -> int:
        bases, offs = seqs_or_arrays if isinstance(seqs_or_arrays, tuple) else pack_reads(seqs_or_arrays)
        n = C.c_uint64(0)
        check(self._lib.abb_insert_reads_sharded(self._h, comm.handle, _ptr(bases), _ptr(offs), len(offs) - 1, int(finalize), C.byref(n)))
        return n.value

    def resident_reads(self) -> tuple[int, int, int]:
        """(device bases pointer, device offsets pointer, n_reads) of the last host-buffer insert"""
        b, o, n = _vp(), _vp(), C.c_uint64(0)
        check(self._lib.abb_filter_resident_reads(self._h, C.byref(b), C.byref(o), C.byref(n)))
        return b.value or 0, o.value or 0, n.value

    def allgather(self, comm: "Comm"):
        check(self._lib.abb_filter_allgather(self._h, comm.handle))

    def insert_h0_dev(self, d_h0_ptr: int, n: int):
        check(self._lib.abb_insert_h0_dev(self._h, _vp(d_h0_ptr), n))

    def device_ptr(self, level: int = -1) -> int:
        return self._lib.abb_filter_device_ptr(self._h, level) or 0

    # -- literal hash interface
    def _hashes(self, hashes):
        h = np.ascontiguousarray(hashes, dtype=np.uint64).reshape(-1, self.getHashNum())
        return h, h.shape[0]

    def insert(self, hashes):
        h, n = self._hashes(hashes)
        check(self._lib.abb_insert_hashes(self._h, _ptr(h), n))

    def contains(self, hashes) -> np.ndarray:
        h, n = self._hashes(hashes)
        out = np.zeros(n, dtype=np.uint8)
        check(self._lib.abb_contains_hashes(self._h, _ptr(h), n, _ptr(out)))
        return out.astype(bool)

    def minCount(self, hashes) -> np.ndarray:
        h, n = self._hashes(hashes)
        out = np.zeros(n, dtype=np.uint8)
        check(self._lib.abb_mincount_hashes(self._h, _ptr(h), n, _ptr(out)))
        return out

    # -- raw array
    def download(self, level: int = -1) -> np.ndarray:
        out = np.empty(self.sizeInBytes(), dtype=np.uint8)
        check(self._lib.abb_filter_download(self._h, level, _ptr(out), out.size))
        return out

    def upload(self, data: np.ndarray, level: int = -1):
        d = np.ascontiguousarray(data, dtype=np.uint8)
        check(self._lib.abb_filter_upload(self._h, level, _ptr(d), d.size))

    def clear(self):
        check(self._lib.abb_filter_clear(self._h))

    def popcounts(self) -> tuple[int, int]:
        a, b = C.c_uint64(0), C.c_uint64(0)
        check(self._lib.abb_filter_popcount(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def popCount(self): return self.popcounts()[0]
    def filtered_popcount(self): return self.popcounts()[1]
    def FPR(self): return (self.popCount() / self.size()) ** self.getHashNum()
    def filtered_FPR(self): return (self.filtered_popcount() / self.size()) ** self.getHashNum()

    def stats(self, reset: bool = False) -> InsertStats:
        st = InsertStats()
        check(self._lib.abb_filter_insert_stats(self._h, C.byref(st), int(reset)))
        return st


READ_CODES = ["SHORTER_THAN_K", "NON_ACGT", "BLUNT_END", "NOT_SOLID", "ALL_KMERS_VISITED", "GENERATED_CONTIGS", "CANDIDATE"]


class Assembler:
    """BloomDBG::assemble (bloom-dbg.h:900-1089) over a device-resident counting filter.

    Feed batches of reads in file order with process_reads(); each call returns the unitigs the
    reference would have printed while processing exactly those reads, in the same order."""

    def __init__(self, solid: Filter, trim: int | None = None, read_log: bool = False, verbose: int = 0):
        self._lib = load()
        self._solid = solid  # keep alive
        self._h = _vp()
        self.raw_results = False
        p = AssemblyParams(0xFFFFFFFF if trim is None else trim, verbose, int(read_log), 0)
        check(self._lib.abb_assembler_create(C.byref(self._h), solid.handle, C.byref(p)))

    def close(self):
        if self._h:
            self._lib.abb_assembler_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def process_reads(self, seqs_or_arrays):
        """returns list of (seed_read_index, sequence str, coverage)"""
        bases, offs = seqs_or_arrays if isinstance(seqs_or_arrays, tuple) else pack_reads(seqs_or_arrays)
        return self._run(self._lib.abb_assembler_process_reads, _ptr(bases), _ptr(offs), len(offs) - 1)

    def process_reads_dev(self, d_bases_ptr: int, d_offs_ptr: int, n_reads: int):
        return self._run(self._lib.abb_assembler_process_reads_dev, _vp(d_bases_ptr), _vp(d_offs_ptr), n_reads)

    def reset(self):
        check(self._lib.abb_assembler_reset(self._h))

    def set_comm(self, comm):
        """multi-GPU pass 2: shard classification, candidate scans and tile production over the ranks of `comm`"""
        self._comm = comm
        check(self._lib.abb_assembler_set_comm(self._h, comm.handle if comm is not None else None))

    def classify_dev(self, d_bases_ptr: int, d_offs_ptr: int, n_reads: int, d_codes_ptr: int):
        check(self._lib.abb_assembler_classify_dev(self._h, _vp(d_bases_ptr), _vp(d_offs_ptr), n_reads, _vp(d_codes_ptr)))

    def set_codes(self, d_codes_ptr: int, n_reads: int):
        check(self._lib.abb_assembler_set_codes(self._h, _vp(d_codes_ptr), n_reads))

    def stats(self) -> AssemblyStats:
        st = AssemblyStats()
        check(self._lib.abb_assembler_stats(self._h, C.byref(st)))
        return st

    def _run(self, fn, bases_p, offs_p, n_reads):
        contigs = C.POINTER(Contig)()
        n = C.c_uint64(0)
        seqs = C.c_char_p()
        check(fn(self._h, bases_p, offs_p, n_reads, C.byref(contigs), C.byref(n), C.byref(seqs)))
        self.last_n_contigs = n.value
        self._last = (contigs, n.value, seqs)
        if self.raw_results:  # (seed_read, length, coverage) only; sequences stay in the library buffer
            return [(contigs[i].seed_read, contigs[i].length, contigs[i].coverage) for i in range(n.value)]
        out = []
        if n.value:
            base = C.cast(seqs, C.c_void_p).value
            for i in range(n.value):
                c = contigs[i]
                out.append((c.seed_read, C.string_at(base + c.seq_offset, c.length).decode(), c.coverage))
        return out

    def last_digests(self, read_id, first_id: int = 0) -> dict:
        """md5 of the FASTA the CLI would print for the last batch (`>ID LEN COV read:READID`, bloom-dbg.h:455-487) and an
        order/strand independent md5 over the canonical unitig sequences; read straight from the library buffers"""
        import hashlib
        contigs, n, seqs = self._last
        fasta, canon = hashlib.md5(), []
        comp = bytes.maketrans(b"ACGT", b"TGCA")
        base = C.cast(seqs, C.c_void_p).value
        for i in range(n):
            c = contigs[i]
            s = C.string_at(base + c.seq_offset, c.length)
            fasta.update(f">{first_id + i} {c.length} {c.coverage} read:{read_id(c.seed_read)}\n".encode())
            fasta.update(s)
            fasta.update(b"\n")
            rc = s.translate(comp)[::-1]
            canon.append(hashlib.md5(min(s, rc)).digest())
        return {"fasta_md5": fasta.hexdigest(), "unitig_multiset_md5": hashlib.md5(b"".join(sorted(canon))).hexdigest(), "unitigs": n}

    def read_results(self) -> np.ndarray:
        codes = _u8p()
        n = C.c_uint64(0)
        check(self._lib.abb_assembler_read_results(self._h, C.byref(codes), C.byref(n)))
        return np.ctypeslib.as_array(codes, shape=(n.value,)).copy() if n.value else np.zeros(0, dtype=np.uint8)

    def counters(self) -> AssemblyCounters:
        c = AssemblyCounters()
        check(self._lib.abb_assembler_counters(self._h, C.byref(c)))
        return c


def counters_for_budget(bloom_size_bytes: int) -> int:
    """bloom-dbg.cc:359-367: counters = roundUpToMultiple(round(B / 1.125), 64)"""
    r = int(bloom_size_bytes / 1.125 + 0.5)
    return r if r % 64 == 0 else r + 64 - r % 64


def kmer_pair_seed(k: int, K: int) -> str:
    """-K: two k-mers of size K at the ends of a k-bit seed (SpacedSeed::kmerPair, BloomDBG/SpacedSeed.h:30-37)"""
    if K > k // 2:
        raise ValueError("value of `-K' must be <= k/2")
    return "1" * K + "0" * (k - 2 * K) + "1" * K


def qr_seed_pair(k: int, length: int) -> str:
    """--qr-seed: a quadratic-residue seed and its mirror image (SpacedSeed::qrSeedPair, SpacedSeed.h:55-95)"""
    if length < 11 or length > k // 2:
        raise ValueError("value of `--qr-seed' must be >= 11 and <= k/2")
    qr = ["1"] * length
    for i in range(length):
        if any(j * j % length == i for j in range(1, length)):
            qr[i] = "0"
    m = ["0"] * k
    for i, c in enumerate(qr):
        m[i] = m[k - 1 - i] = c
    return "".join(m)


def bloom_dbg(read_ids, seqs_or_arrays, k: int, kc: int = 2, num_hashes: int = 4, bloom_size: int | None = None,
              counters: int | None = None, trim: int | None = None, batch_reads: int | None = None, read_log: bool = False,
              device: int = 0, mask: str = ""):
    """abyss-bloom-dbg -k K --kc KC -H H -b B [-s MASK] (countingBloomAssembly, bloom-dbg.cc:347-386) on one GPU.
    Returns (fasta_text, read_codes)."""
    if counters is None:
        counters = counters_for_budget(bloom_size)
    bases, offs = seqs_or_arrays if isinstance(seqs_or_arrays, tuple) else pack_reads(seqs_or_arrays)
    n = len(offs) - 1
    f = Filter.counting(counters, num_hashes, k, kc, mask=mask, device=device)
    f.insert_reads((bases, offs))
    a = Assembler(f, trim, read_log)
    out, codes = [], []
    cid = 0
    step = batch_reads or n or 1
    for lo in range(0, n, step):
        hi = min(n, lo + step)
        b0, b1 = int(offs[lo]), int(offs[hi])
        sub = (bases[b0:b1], (offs[lo:hi + 1] - offs[lo]).astype(np.uint64))
        for seed, seq, cov in a.process_reads(sub):
            out.append(f">{cid} {len(seq)} {cov} read:{read_ids[seed]}\n{seq}\n")
            cid += 1
        codes.append(a.read_results())
    a.close()
    f.close()
    return "".join(out), (np.concatenate(codes) if codes else np.zeros(0, dtype=np.uint8))


def overlap_graph(seqs_or_arrays, k: int, min_overlap: int = 50, ss: bool = False, device: int = 0):
    """AdjList -k K -m M [--SS] (AdjList/AdjList.cpp:140-291) on one GPU: the edges of the contig overlap graph as a list of
    (u, v, distance) with u, v = 2 * contig + sense (ContigNode), in the order the reference's graph iterates them."""
    lib = load()
    bases, offs = seqs_or_arrays if isinstance(seqs_or_arrays, tuple) else pack_reads(seqs_or_arrays)
    h = _vp()
    check(lib.abb_overlap_create(C.byref(h), device))
    try:
        e = C.POINTER(OverlapEdge)()
        n = C.c_uint64(0)
        check(lib.abb_overlap_build(h, _ptr(bases), _ptr(offs), len(offs) - 1, k, min_overlap, int(ss), C.byref(e), C.byref(n)))
        return [(e[i].u, e[i].v, e[i].distance) for i in range(n.value)]
    finally:
        lib.abb_overlap_destroy(h)


def successors(filt: "Filter", kmers, max_chain: int = 1):
    """out-edges of graph vertices (RollingBloomDBG out_edge_iterator; abb_successors): for every k-mer a list of
    (mask, [hash_A, hash_C, hash_G, hash_T]) per chain vertex, and the canonical hash of the k-mer itself."""
    lib = load()
    ks = [s.encode() if isinstance(s, str) else bytes(s) for s in kmers]
    n = len(ks)
    info = (SuccInfo * (n * max_chain))()
    ln = (C.c_uint * n)()
    self_h = (C.c_uint64 * n)()
    check(lib.abb_successors(filt.handle, b"".join(ks), n, max_chain, info, ln, self_h))
    out = []
    for i in range(n):
        out.append(([(info[i * max_chain + s].mask, list(info[i * max_chain + s].hash)) for s in range(ln[i])], self_h[i]))
    return out


def neighbours(graph: "Filter", kmers, attrs=()):
    """the k-mer and its 8 neighbours (abb_neighbours; vertex 0 = the k-mer, 1 + b = successor with last base b, 5 + b =
    predecessor with first base b, b = A, C, G, T): for every k-mer (hashes[9], mask, attr[9]) -- canonical hashes, graph
    membership (bit v = vertex v) and attribute bits (attr[v] bit j = attrs[j] contains vertex v)."""
    lib = load()
    ks = [s.encode() if isinstance(s, str) else bytes(s) for s in kmers]
    n = len(ks)
    out = (Neighbourhood * n)()
    hs = (_vp * max(1, len(attrs)))(*[a.handle for a in attrs])
    check(lib.abb_neighbours(graph.handle, hs, len(attrs), b"".join(ks), n, out))
    return [(list(out[i].hash), out[i].mask, list(out[i].attr)) for i in range(n)]
