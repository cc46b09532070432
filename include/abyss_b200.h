/*
 * abyss_b200.h -- C ABI of libabyssb200.so: the B200 (sm_100a) implementation of the
 * abyss-bloom-dbg hot path (ntHash -> Bloom insert -> Bloom-backed unitig extension).
 *
 * The reference (bcgsc/abyss 2.3.10) has no FFI layer: its seam is the duck-typed Bloom filter
 * template parameter (BloomT / SolidKmerSetT / BF) that loadSeq, allKmersInBloom,
 * RollingBloomDBG<BF> and assemble() are templated on (SURVEY.md section 8b).  Each entry point
 * below names the reference interface it replaces (file:line under the reference tree).
 * Per-k-mer virtual calls cannot feed a GPU, so everything is batch oriented.
 *
 * Conventions: extern "C"; plain pointers and sizes; every function returns ABB_OK (0) or a
 * negative ABB_E* code and records a message retrievable with abb_last_error(); no exceptions
 * cross the boundary; one host thread per handle (streams are internal); buffers are caller
 * owned.  Where the reference would print and exit(1) (Common/IOUtil.h:14-22,
 * BloomFilter.hpp:376-379) this library returns an error instead; the CLI turns it into exit.
 * There is NO CPU fallback: without a usable CUDA device every compute call fails with
 * ABB_ENODEV.
 */
#ifndef ABYSS_B200_H
#define ABYSS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ABB_VERSION 100

enum {
	ABB_OK = 0,
	ABB_EINVAL = -1, /* bad argument (what the reference would assert / exit on) */
	ABB_ENODEV = -2, /* no CUDA device / driver */
	ABB_ECUDA = -3,  /* CUDA runtime failure, see abb_last_error() */
	ABB_ENOMEM = -4,
	ABB_ESTATE = -5  /* call not valid for this handle kind / state */
};

/* filter kinds */
enum {
	ABB_COUNTING = 0, /* CountingBloomFilter<uint8_t>, vendor/btl_bloomfilter/CountingBloomFilter.hpp:26-113 */
	ABB_BIT = 1,      /* BloomFilter, vendor/btl_bloomfilter/BloomFilter.hpp:40-432 */
	ABB_CASCADING = 2 /* HashAgnosticCascadingBloom, Bloom/HashAgnosticCascadingBloom.h:26-182 */
};

typedef struct abb_filter abb_filter;
typedef struct abb_assembler abb_assembler;

/* ---- library ---- */
int abb_version(void);
const char* abb_last_error(void);
int abb_device_count(void); /* <0 on error */

/* ---- filter lifecycle --------------------------------------------------------------------
 * size: number of counters (ABB_COUNTING; CountingBloomFilter ctor :31-50 pads to a multiple of
 *       8) or number of bits per level (ABB_BIT / ABB_CASCADING; must be a multiple of 8,
 *       BloomFilter.hpp:374-379).
 * arg:  count threshold (ABB_COUNTING, `--kc`), ignored (ABB_BIT), number of levels (ABB_CASCADING).
 * mask: spaced seed ("" or NULL = none; MaskedKmer::setMask, BloomDBG/MaskedKmer.h:38-55).
 */
int abb_filter_create(abb_filter** out, int kind, uint64_t size, unsigned num_hashes, unsigned k,
                      unsigned arg, const char* mask, int device);
int abb_filter_destroy(abb_filter* f);
/* getters: getKmerSize/getHashNum/size/sizeInBytes/threshold (CountingBloomFilter.hpp:75-80) */
unsigned abb_filter_kmer_size(const abb_filter* f);
unsigned abb_filter_hash_num(const abb_filter* f);
uint64_t abb_filter_size(const abb_filter* f);
uint64_t abb_filter_size_in_bytes(const abb_filter* f); /* bytes of ONE level */
unsigned abb_filter_threshold(const abb_filter* f);
unsigned abb_filter_levels(const abb_filter* f);
int abb_filter_set_threshold(abb_filter* f, unsigned threshold);

/* ---- pass 1: loadSeq / loadFile (BloomDBG/BloomIO.h:32-41,50-94) --------------------------
 * Hash every k-mer of every read (RollingHashIterator semantics: upper-cased, windows touching a
 * non-ACGT base skipped) and insert it, with results IDENTICAL to inserting read by read, k-mer
 * by k-mer in the given order on one thread (the reference at -j1).
 * bases: concatenated read characters; offsets[n_reads+1]: start of each read in bases.
 * n_kmers_out (optional): number of k-mers inserted.
 * The _dev variant takes device-resident buffers (no host<->device copy inside the call). */
int abb_insert_reads(abb_filter* f, const char* bases, const uint64_t* offsets, uint64_t n_reads,
                     uint64_t* n_kmers_out);
int abb_insert_reads_dev(abb_filter* f, const char* d_bases, const uint64_t* d_offsets,
                         uint64_t n_reads, uint64_t n_bases, uint64_t* n_kmers_out);

/* ---- the literal `const uint64_t hashes[]` interface (for parity tests) --------------------
 * hashes: n * num_hashes values, k-mer major -- exactly what RollingHashIterator::operator*
 * yields (BloomDBG/RollingHashIterator.h:147-151).  insert (CountingBloomFilter.hpp:199-204,
 * BloomFilter.hpp:186-195, HashAgnosticCascadingBloom.h:124-133) is applied in array order. */
int abb_insert_hashes(abb_filter* f, const uint64_t* hashes, uint64_t n);
int abb_contains_hashes(abb_filter* f, const uint64_t* hashes, uint64_t n, uint8_t* out);  /* contains(): :185-196 */
int abb_mincount_hashes(abb_filter* f, const uint64_t* hashes, uint64_t n, uint8_t* out);  /* minCount(): :54-64 */

/* ---- hashing only (RollingHashIterator + RollingHash::getHashes) ---------------------------
 * For each read r and window position p < max(0, len_r - k + 1), slot = slot_offsets[r] + p where
 * slot_offsets is the exclusive prefix sum of the per-read window counts.  out_h0[slot] is the
 * canonical (masked) ntHash, out_valid[slot] is 1 if the reference iterator would yield it.
 * Returns the total number of slots through n_slots_out. */
int abb_hash_reads(unsigned k, const char* mask, const char* bases, const uint64_t* offsets,
                   uint64_t n_reads, uint64_t* out_h0, uint8_t* out_valid, uint64_t* n_slots_out,
                   int device);

/* ---- multi-GPU building blocks (SURVEY.md section 8e: hash-range sharding) ------------------
 * abb_hash_reads_dev: K1 only, device in / device out (d_h0, d_valid hold `capacity` slots).
 * abb_insert_h0_dev:  ordered insert of n canonical hashes (device resident, all valid), in array
 *                     order -- what a rank does with the k-mers it owns after the all-to-all.
 * abb_filter_device_ptr: the raw device array of a level, for the NCCL union (all-reduce max /
 *                     or) issued by the caller; synchronises the filter's stream first. */
int abb_hash_reads_dev(abb_filter* f, const char* d_bases, const uint64_t* d_offsets, uint64_t n_reads,
                       uint64_t* d_h0, uint8_t* d_valid, uint64_t capacity, uint64_t* n_slots_out);
int abb_insert_h0_dev(abb_filter* f, const uint64_t* d_h0, uint64_t n);

/* ---- multi-GPU exact insert (SURVEY.md section 8e; Bloom/bloom.cc:556-580 `-w M/N` windows are the precedent) -----
 * One process (or host thread) per GPU.  The counter array is sharded by POSITION RANGE: rank r owns counters
 * [r*chunk, (r+1)*chunk), chunk = ceil(size / world) rounded up to 16.  All ranks walk the same file-order windows
 * of all reads, touch only the counters they own, and exchange one ncclAllReduce(min, uint8) per window (partial
 * minima + veto flags); the result is the sequential -j1 counter array, bit for bit, for every world size
 * (abb_shard.cuh).  The NCCL communicator lives behind the C ABI; NCCL is dlopen()ed (libnccl.so.2), so a host
 * that never calls abb_comm_* does not need it.
 * abb_comm_unique_id: rank 0 creates the 128-byte NCCL id, the caller ships it to the other ranks (MPI, TCP, a
 *                     file, torch.distributed ...).
 * abb_comm_create:    ncclCommInitRank on `device`.
 * abb_insert_reads_sharded_dev: EVERY rank passes the same reads (device resident).  finalize != 0 all-gathers the
 *                     shards afterwards so that each rank holds the whole filter (what the extension stage needs);
 *                     with finalize == 0 only the own range of f is meaningful until abb_filter_allgather.
 * abb_comm_allgather_bytes / abb_comm_allreduce_max_u8: the collectives pass 2 needs (read codes, tile stores). */
typedef struct abb_comm abb_comm;
int abb_comm_unique_id(uint8_t id_out[128]);
int abb_comm_create(abb_comm** out, int rank, int world, const uint8_t id[128], int device);
int abb_comm_destroy(abb_comm* c);
int abb_comm_rank(const abb_comm* c);
int abb_comm_world(const abb_comm* c);
int abb_insert_reads_sharded_dev(abb_filter* f, abb_comm* c, const char* d_bases, const uint64_t* d_offsets, uint64_t n_reads,
                                 int finalize, uint64_t* n_kmers_out);
int abb_insert_reads_sharded(abb_filter* f, abb_comm* c, const char* bases, const uint64_t* offsets, uint64_t n_reads, int finalize,
                             uint64_t* n_kmers_out); /* host buffers: copies the batch to the device first */
int abb_filter_allgather(abb_filter* f, abb_comm* c);
/* the device copy of the batch the last host-buffer insert (abb_insert_reads / abb_insert_reads_sharded) made: a host
 * that inserts all reads in one batch hands these to abb_assembler_process_reads_dev instead of copying the reads a
 * second time for pass 2 (the reference reads its input files twice, BloomDBG/bloom-dbg.h:1011-1046) */
int abb_filter_resident_reads(abb_filter* f, const char** d_bases, const uint64_t** d_offsets, uint64_t* n_reads);
/* d_buf holds world * bytes_per_rank bytes, this rank's part already in place at rank * bytes_per_rank */
int abb_comm_allgather_bytes(abb_comm* c, void* d_buf, uint64_t bytes_per_rank, void* cuda_stream);
int abb_comm_allreduce_max_u8(abb_comm* c, void* d_buf, uint64_t n, void* cuda_stream);
/* all-gather of unequal parts: this rank's send_bytes go to every other rank; rank r's recv_bytes[r] bytes land at
 * d_recv_base + recv_offsets[r] (grouped ncclSend / ncclRecv; entries for the own rank are ignored) */
int abb_comm_exchange_bytes(abb_comm* c, const void* d_send, uint64_t send_bytes, void* d_recv_base, const uint64_t* recv_offsets,
                            const uint64_t* recv_bytes, void* cuda_stream);

void* abb_filter_device_ptr(abb_filter* f, int level);

/* ---- raw array <-> host (operator<< / loadFilter: CountingBloomFilter.hpp:262-379,
 * BloomFilter.hpp:98-163,288-294; for ABB_CASCADING `level` selects the level, -1 = last,
 * which is the only one the reference serialises, HashAgnosticCascadingBloom.h:143-150) */
int abb_filter_download(abb_filter* f, int level, uint8_t* host, uint64_t nbytes);
int abb_filter_upload(abb_filter* f, int level, const uint8_t* host, uint64_t nbytes);
int abb_filter_clear(abb_filter* f);

/* ---- statistics: popCount / filtered_popcount (CountingBloomFilter.hpp:219-244), getPop
 * (BloomFilter.hpp:313-320).  FPR = pow(pop/size, H) is left to the caller. */
int abb_filter_popcount(abb_filter* f, uint64_t* nonzero, uint64_t* at_or_above_threshold);

/* ---- pass 2: BloomDBG::assemble / processRead (BloomDBG/bloom-dbg.h:783-882,900-1089) -------
 * The assembler owns the "assembled k-mers" bit filter (bloom-dbg.h:910-911: size() bits, same H,
 * same k) and the contigEndKmers table (:992-993) and consumes reads in file order, batch by
 * batch.  Output is identical to the reference at -j1.
 */
typedef struct abb_assembly_params {
	unsigned trim;      /* AssemblyParams::trim (AssemblyParams.h:67), default k */
	unsigned verbose;
	unsigned read_log;  /* 1: per-read outcome codes are exact (`--read-log`); 0: a read that fails the
	                       solid test is reported NOT_SOLID without the (more expensive) blunt-end test */
	unsigned reserved;  /* flags: bit 0 = keep the `-T` trace rows of each batch (abb_assembler_trace) */
} abb_assembly_params;

typedef struct abb_contig {
	uint64_t seed_read;   /* index (in the whole input stream) of the read that seeded it */
	uint64_t seq_offset;  /* into the sequence buffer returned alongside */
	uint32_t length;      /* bases */
	uint32_t coverage;    /* getSeqAbsoluteKmerCoverage (bloom-dbg.h:95-109) */
} abb_contig;

/* counters mirror BloomDBG/AssemblyCounters.h:15-29 */
typedef struct abb_assembly_counters {
	uint64_t solid_reads, visited_reads, reads_processed, bases_assembled, contig_id;
} abb_assembly_counters;

/* The assembler works on a counting filter and takes k, H, the threshold and the spaced seed from it.  A seed must
 * begin and end with '1' (MaskedKmer::setMask, BloomDBG/MaskedKmer.h:44-47) and be symmetric
 * (RollingBloomDBGVertex::compare asserts it, RollingBloomDBG.h:141-145); sequences may then contain 'N' where no
 * vertex of a short path writes a column (pathToSeq, bloom-dbg.h:131-158). */
int abb_assembler_create(abb_assembler** out, abb_filter* solid, const abb_assembly_params* params);
int abb_assembler_destroy(abb_assembler* a);
/* Process the next batch of reads (file order).  On return *contigs / *seqs point at library-
 * owned buffers valid until the next call on this handle. */
int abb_assembler_process_reads(abb_assembler* a, const char* bases, const uint64_t* offsets,
                                uint64_t n_reads, const abb_contig** contigs, uint64_t* n_contigs,
                                const char** seqs);
/* same with device-resident read buffers (no host<->device copy of the reads inside the call) */
int abb_assembler_process_reads_dev(abb_assembler* a, const char* d_bases, const uint64_t* d_offsets,
                                    uint64_t n_reads, const abb_contig** contigs, uint64_t* n_contigs,
                                    const char** seqs);
/* Several GPUs: the per-read classification (K3a) is a pure function of the read and the solid filter, so
 * ranks may classify disjoint slices (abb_assembler_classify_dev writes one code per read, the internal
 * RC_* values, to a device buffer), exchange the codes, and hand the complete array to the rank that
 * assembles: abb_assembler_set_codes applies to the next process_reads call only. */
int abb_assembler_classify_dev(abb_assembler* a, const char* d_bases, const uint64_t* d_offsets, uint64_t n_reads,
                               uint8_t* d_codes);
int abb_assembler_set_codes(abb_assembler* a, const uint8_t* d_codes, uint64_t n_reads);
/* Start a new assembly on the same handle (the solid filter has been refilled): clears the assembled
 * filter, the contig-end table, the tile store, counters and statistics, keeps all device buffers. */
int abb_assembler_reset(abb_assembler* a);
int abb_assembler_counters(const abb_assembler* a, abb_assembly_counters* out);
/* resume from a checkpoint (resumeFromCheckpoint, BloomDBG/Checkpoint.h:158-226): restores the counters (next contig id,
 * index of the next input read); the caller uploads the two filters with abb_filter_upload */
int abb_assembler_set_counters(abb_assembler* a, const abb_assembly_counters* in);
/* optional per-read outcome log of the last batch (ReadResult, bloom-dbg.h:256-293);
 * codes: 0 SHORTER_THAN_K, 1 NON_ACGT, 2 BLUNT_END, 3 NOT_SOLID, 4 ALL_KMERS_VISITED,
 * 5 GENERATED_CONTIGS */
int abb_assembler_read_results(const abb_assembler* a, const uint8_t** codes, uint64_t* n);
/* multi-GPU pass 2 (one process per GPU, every rank holds the whole solid filter and is fed the same batches): the
 * pure per-item stages -- read classification (K3a), the candidate scans against the assembled filter (K3b) and tile
 * production -- are split over the ranks of `comm` and all-gathered; the walks and the file-order replay run
 * replicated, so every rank returns the same unitigs.  NULL = single GPU. */
int abb_assembler_set_comm(abb_assembler* a, abb_comm* comm);
/* `-T FILE` (ContigRecord, bloom-dbg.h:186-254, written by outputContig :618-619): one row per contig that was
 * handed to outputContig while the last batch was processed, in the reference's order.  contig_id = ~0 for a
 * redundant contig ("NA"); codes: 0 AMBI_IN, 1 AMBI_OUT, 2 DEAD_END, 3 CYCLE, 4 LENGTH_LIMIT (Graph/ExtendPath.h:63-80);
 * the seed is the k-mer at seed_pos of read seed_read.  Needs abb_assembly_params.reserved bit 0. */
typedef struct abb_trace_row {
	uint64_t contig_id;
	uint64_t seed_read;
	uint32_t length;    /* bases of the contig (the reference prints an uninitialised value here for redundant contigs) */
	uint32_t seed_pos;
	uint32_t left_n, right_n;
	uint8_t left_code, right_code, redundant, pad;
} abb_trace_row;
int abb_assembler_trace(const abb_assembler* a, const abb_trace_row** rows, uint64_t* n);
/* access to the assembled-k-mer bit filter (for checkpoints / tests) */
abb_filter* abb_assembler_assembled_filter(abb_assembler* a);

typedef struct abb_assembly_stats {
	uint64_t rounds;            /* speculation rounds (K3b -> K4 -> K5) */
	uint64_t speculated_reads;  /* reads extended by K4 */
	uint64_t wasted_reads;      /* speculated reads found already assembled at replay */
	uint64_t candidates;        /* solid, non-blunt reads */
	uint64_t contigs_tried;     /* unitigs produced by K4 (before the redundancy test) */
	uint64_t launches;          /* kernels launched by the assembler */
	float ms_classify, ms_visited, ms_extend, ms_replay; /* CUDA-event time per phase */
	float ms_tiles;             /* marker enumeration + tile production */
	float ms_walk, ms_stage, ms_repeat; /* inside ms_extend: K4 kernels, unitig gather+hash, repeat check */
	float ms_total, ms_cand;    /* host wall clock of the process_reads calls / of building the candidate list */
	uint64_t markers, tiles;    /* marker vertices found / marker-to-marker tiles stored */
	uint64_t serial_fallbacks;  /* reads re-walked vertex by vertex after the repeat check */
} abb_assembly_stats;
int abb_assembler_stats(const abb_assembler* a, abb_assembly_stats* out);

/* ---- debug / auxiliary queries over reads (BloomDBG/bloom-dbg.h: writeCovTrack :1280-1334, trimSeq :399-447) ----
 * For every k-mer window of every sequence (slot numbering as in abb_hash_reads): out_valid[slot] = 1 if
 * RollingHashIterator would yield it, out_flag[slot] = contains() of the filter (counting: minCount >= threshold;
 * bit / cascading: all bits of the last level) -- one GPU pass instead of one contains() call per k-mer.
 * out_flag / out_valid hold at least the number of slots (sum over sequences of max(0, len - k + 1)). */
int abb_contains_reads(abb_filter* f, const char* bases, const uint64_t* offsets, uint64_t n_reads, uint8_t* out_flag,
                       uint8_t* out_valid, uint64_t capacity, uint64_t* n_slots_out);

/* ---- out-edges of graph vertices, for the GraphViz dump `-g` (outputGraph, BloomDBG/bloom-dbg.h:1171-1242; out_edge_iterator,
 * BloomDBG/RollingBloomDBG.h:300-360): for each of n k-mers (n * k characters, ACGT) the successors that the filter contains.
 * While a vertex has exactly one out-edge the walk continues to that successor, up to max_chain (1..128) vertices, so out holds
 * n * max_chain entries: out[i * max_chain + s] describes the s-th vertex of chain i (s = 0: k-mer i itself); out_len[i] =
 * entries filled.  mask bit b (A, C, G, T = 0..3): the successor with last base b exists; hash[b]: its canonical ntHash
 * (vertex identity).  self_hash[i]: canonical hash of k-mer i.  Not available with a spaced seed. */
typedef struct abb_succ_info {
	uint64_t hash[4];
	uint8_t mask;
	uint8_t pad[7];
} abb_succ_info;
int abb_successors(abb_filter* f, const char* kmers, uint64_t n, unsigned max_chain, abb_succ_info* out, unsigned* out_len,
                   uint64_t* self_hash);

/* ---- neighbourhoods of graph vertices, for `abyss-bloom graph` (Bloom/bloom.cc:983-1153; out_edge_iterator / in_edge_iterator,
 * BloomDBG/RollingBloomDBG.h:300-453): for each of n k-mers (n * k characters, hashed as the reference hashes any character:
 * either case, non-ACGT as ntHash's seedTab gives it) the k-mer and its 8 neighbours.  Vertex v = 0: the k-mer itself;
 * v = 1 + b: its successor (shifted left, last base b = A, C, G, T); v = 5 + b: its predecessor (shifted right, first base b).
 * hash[v]: canonical ntHash (vertex identity).  mask bit v: the graph filter contains vertex v (all bits of its last level).
 * attr[v] bit j: attribute filter attrs[j] contains vertex v, probed with the GRAPH's hash values (its k and its first
 * H_j hashes) modulo the attribute filter's own size (RollingBloomDBGVisitor.h:122-131).  Bit and cascading filters only;
 * n_attrs <= 32, each attribute filter on the graph's device with at most as many hashes as the graph; no spaced seed. */
typedef struct abb_neighbourhood {
	uint64_t hash[9];
	uint32_t attr[9];
	uint16_t mask;
	uint8_t pad[2];
} abb_neighbourhood;
int abb_neighbours(abb_filter* graph, abb_filter* const* attrs, unsigned n_attrs, const char* kmers, uint64_t n,
                   abb_neighbourhood* out);

/* ---- the next stage: contig overlap graph (AdjList/AdjList.cpp:140-291; bin/abyss-pe:577 runs it on the unitig FASTA) ----
 * Vertices are ContigNode indices (Common/ContigNode.h): 2*i = contig i as given, 2*i+1 = its reverse complement.
 * Edges u -> v: the last `overlap` bases of u equal the first `overlap` bases of v; distance = -overlap.
 *  - overlap = k-1 exactly for every such pair (buildOverlapGraph, :247-268);
 *  - min_overlap <= overlap < k-1 (longest only) between vertices that the first step left without an out-edge
 *    (addOverlapsSA, :140-201); min_overlap = 0 or > k-1 means k-1 (:386-388), i.e. only the first step.
 *  - ss != 0 (--SS): only edges between vertices of the same orientation (:159,262).
 * The edge array is ordered as the reference's graph iterates it (vertices ascending, each out-list in the order
 * AdjList adds the edges), so any of its output formats can be written from it.  It is library owned and valid
 * until the next call on the handle.  Contig ends must be nucleotides (ambiguity codes are flattened as in
 * Common/Sequence.h:50-72; 'N' is an error, the reference aborts) and contigs longer than k-1. */
typedef struct abb_overlap abb_overlap;
typedef struct abb_overlap_edge {
	uint32_t u, v;
	int32_t distance;
} abb_overlap_edge;
typedef struct abb_overlap_stats {
	uint64_t vertices, exact_edges, short_edges, blunt_vertices, launches;
} abb_overlap_stats;
int abb_overlap_create(abb_overlap** out, int device);
int abb_overlap_destroy(abb_overlap* h);
int abb_overlap_build(abb_overlap* h, const char* bases, const uint64_t* offsets, uint64_t n_contigs, unsigned k,
                      unsigned min_overlap, int ss, const abb_overlap_edge** edges, uint64_t* n_edges);
int abb_overlap_get_stats(const abb_overlap* h, abb_overlap_stats* out);

/* ---- profiling hooks used by bench.py ---------------------------------------------------- */
typedef struct abb_insert_stats {
	uint64_t kmers;           /* valid k-mers inserted */
	uint64_t slots;           /* k-mer windows hashed */
	uint64_t windows;         /* ordered windows processed */
	uint64_t deferred;        /* events that lost a reservation and went through the ordered pass */
	uint64_t launches;        /* kernels launched by this library since the last reset */
	float ms_hash, ms_insert; /* CUDA-event time on the library stream since the last reset */
	float ms_commit;          /* with profiling on: summed CUDA-event time of the timed k_window launches */
	uint64_t commit_launches; /* number of k_window launches timed */
	uint64_t commit_slots;    /* k-mer slots those launches applied */
	uint64_t drains;          /* serial drains that did work, and the slots they replayed */
	uint64_t drained_slots;
} abb_insert_stats;
int abb_filter_insert_stats(abb_filter* f, abb_insert_stats* out, int reset);
/* time launches of the Bloom-insert window kernel with CUDA events (bench.py roofline) */
int abb_filter_set_profiling(abb_filter* f, int on);
/* the cudaStream_t all work of this filter (and of an assembler created on it) is issued to */
void* abb_filter_stream(abb_filter* f);
/* tuning: ordered-window size in k-mer slots (power of two, <= 2^20); 0 = default */
int abb_filter_set_window(abb_filter* f, uint64_t window_slots);

#ifdef __cplusplus
}
#endif
#endif /* ABYSS_B200_H */
