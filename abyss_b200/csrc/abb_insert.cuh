// abb_insert.cuh -- pass-1 kernels: K1 hash_reads, K2 ordered (sequentially-consistent) insert.
//
// Replaces BloomDBG::loadSeq (BloomDBG/BloomIO.h:32-41) = RollingHashIterator
// (RollingHashIterator.h:35-97) + CountingBloomFilter<uint8_t>::incrementMin
// (vendor/btl_bloomfilter/CountingBloomFilter.hpp:138-162), BloomFilter::insert
// (BloomFilter.hpp:186-195) and HashAgnosticCascadingBloom::insert
// (Bloom/HashAgnosticCascadingBloom.h:124-133).
//
// WHY AN ORDERED INSERT.  incrementMin reads the minimum of H counters and bumps the counters
// equal to it, so the final array depends on the order in which k-mers that share a counter are
// inserted; the unitig FASTA prints sums of raw counters (bloom-dbg.h:599-603) and thresholds
// them, so "same FASTA as the reference at -j1" means "same counters as the sequential,
// file-order insert".  The cascading filter has the same property.  The scheme (round 2):
//   * k-mer windows ("slots") are numbered in file order; a batch is cut into ordered windows of
//     W slots; windows run one after another, slots inside a window run in parallel.
//   * conflict map: every slot of window w marks its H filter positions in an L2-resident map of
//     two-bit entries (entry = position mod E): "touched" / "touched again".  A slot none of whose
//     entries was touched again shares no counter with any other pending event: it commutes with
//     all of them, so it applies its min-increment at once with plain byte loads/stores.  That is
//     ~97 % of the slots and costs one L2 atomic + one L2 load per position on top of the HBM
//     accesses themselves (round 1: CAS + probe + release on an 8-byte tag per position).
//     The marks of window w+1 are written by the kernel that applies window w.
//   * carry: the slots that saw "touched again" (true sharing, or an alias in the map) are carried
//     into the next window as its OLDEST events.  Carried slots are few, so they use an exact
//     open-addressing tag table keyed by the position: reserve keeps the minimum priority
//     (= file order), a carried slot that owns all its positions applies, the others are carried
//     again.  Carried slots also mark their positions "touched again" in the next window's map, so
//     every new slot that shares a counter with them waits.  One chain link resolves per window.
//   * drain: when more than kCarryLanes slots are pending (dense filters: everything conflicts), a
//     pending slot gets old, or the call ends, one CTA sorts the pending slots by file order
//     (presence bitmap), stages the counters they touch in shared memory chunk by chunk (one HBM
//     round trip per chunk) and replays them sequentially there -- about 20 ns per slot instead of
//     a dependent HBM round trip.
// Tag entries are [epoch:4 | position:36 | priority:24]; an entry from an older epoch is free, so
// the table is cleared only once every 15 windows.
#pragma once
#include "abb_device.cuh"
#include "abb_graph.cuh"
#include <cooperative_groups.h>
#include <cuda/barrier>
#include <cuda_runtime.h>

namespace abb {
namespace cg = cooperative_groups;

constexpr unsigned kPrioBits = 28;                  // priority of a carried slot = age_off - (window start - slot) < 2^28 - 1
constexpr unsigned kMaxAgeWindows = 48;             // age_off = min(kMaxAgeWindows, 2^28 / W - 1) windows; drain at 2/3 of it
constexpr unsigned kCarryLanes = 1u << 16;          // most carried slots a window serves = drain threshold
constexpr unsigned kPosBits = 36;                   // filters up to 2^36 - 1 counters / bits
constexpr uint64_t kPrioMask = (1ULL << kPrioBits) - 1;

/** exact open-addressing table of the positions the carried slots want: entry = [position + 1 : 36 | priority : 28],
 *  0 = empty.  `mask` selects the prefix of the allocation in use (sized to the number of carried slots), so that
 *  clearing it costs almost nothing. */
struct TagTable {
	unsigned long long* e; // entries
	uint64_t mask;         // slots in use - 1 (power of two)
};

ABB_D uint64_t tag_pack(uint64_t pos, uint64_t prio) { return ((pos + 1) << kPrioBits) | prio; }
ABB_D uint64_t tag_home(uint64_t pos, const TagTable& t)
{
	// Fibonacci hashing of the position
	return ((pos * 0x9E3779B97F4A7C15ULL) >> 20) & t.mask;
}

/** record "prio wants pos" keeping the smallest priority */
ABB_D void tag_reserve(const TagTable& t, uint64_t pos, uint64_t prio)
{
	const uint64_t mine = tag_pack(pos, prio);
	const uint64_t key = mine >> kPrioBits;
	uint64_t s = tag_home(pos, t);
	for (;;) {
		unsigned long long cur = __ldcg(&t.e[s]);
		if (cur == 0) {
			cur = atomicCAS(&t.e[s], 0ULL, (unsigned long long)mine);
			if (cur == 0)
				return;
		}
		if ((cur >> kPrioBits) == key) {
			if (mine < cur)
				atomicMin(&t.e[s], (unsigned long long)mine);
			return;
		}
		s = (s + 1) & t.mask;
	}
}

/** smallest priority that reserved pos (pos must have been reserved); *where = its entry */
ABB_D uint64_t tag_owner_at(const TagTable& t, uint64_t pos, uint64_t* where)
{
	const uint64_t key = pos + 1;
	uint64_t s = tag_home(pos, t);
	for (;;) {
		unsigned long long cur = __ldcg(&t.e[s]);
		if ((cur >> kPrioBits) == key) {
			*where = s;
			return cur & kPrioMask;
		}
		s = (s + 1) & t.mask;
	}
}
ABB_D uint64_t tag_owner(const TagTable& t, uint64_t pos)
{
	uint64_t where;
	return tag_owner_at(t, pos, &where);
}
/** the owner is done with pos: younger slots may now win it (priority field := all ones) */
ABB_D void tag_release_at(const TagTable& t, uint64_t pos, uint64_t where) { __stcg(&t.e[where], (unsigned long long)tag_pack(pos, kPrioMask)); }
ABB_D void tag_release(const TagTable& t, uint64_t pos)
{
	uint64_t where;
	tag_owner_at(t, pos, &where);
	tag_release_at(t, pos, where);
}

// ------------------------------------------------------------------------------------------
// the three insert semantics, applied by exactly one thread that owns all H positions
// ------------------------------------------------------------------------------------------
struct FilterView {
	uint8_t* data;      // counters, or level-0 bits
	uint64_t level_stride; // bytes between cascading levels
	unsigned levels;
};

ABB_D bool bits_contain(const uint8_t* bits, const uint64_t* pos, unsigned H)
{
	bool all = true;
	for (unsigned i = 0; i < H; ++i)
		all &= (__ldcg(bits + (pos[i] >> 3)) >> (pos[i] & 7)) & 1;
	return all;
}
/** bit set by the owner of the *bit position*; neighbouring bits of the byte may belong to
 *  other owners, hence the atomic (BloomFilter.hpp:186-195 uses __sync_or_and_fetch too) */
ABB_D void bits_set(uint8_t* bits, const uint64_t* pos, unsigned H)
{
	for (unsigned i = 0; i < H; ++i) {
		uint64_t byte = pos[i] >> 3;
		unsigned* w = reinterpret_cast<unsigned*>(bits + (byte & ~3ULL));
		atomicOr(w, 1u << ((pos[i] & 7) + 8 * (byte & 3)));
	}
}
/** HashAgnosticCascadingBloom::insert (HashAgnosticCascadingBloom.h:124-133) */
ABB_D void apply_cascading(const FilterView& f, const uint64_t* pos, unsigned H)
{
	for (unsigned l = 0; l < f.levels; ++l) {
		uint8_t* bits = f.data + (uint64_t)l * f.level_stride;
		if (!bits_contain(bits, pos, H)) {
			bits_set(bits, pos, H);
			return;
		}
	}
}

// ------------------------------------------------------------------------------------------
// K1: hash_reads -- one warp per read, closed-form ntHash via warp prefix-XOR scans
// ------------------------------------------------------------------------------------------
constexpr int kHashWarps = 8;     // warps per CTA
constexpr int kRing = 256;        // per-warp ring of prefix values; needs k + 32 <= 256

ABB_D uint64_t shfl_up64(uint64_t v, int d)
{
	unsigned lo = __shfl_up_sync(0xffffffffu, (unsigned)v, d);
	unsigned hi = __shfl_up_sync(0xffffffffu, (unsigned)(v >> 32), d);
	return ((uint64_t)hi << 32) | lo;
}
ABB_D uint64_t shfl64(uint64_t v, int src)
{
	unsigned lo = __shfl_sync(0xffffffffu, (unsigned)v, src);
	unsigned hi = __shfl_sync(0xffffffffu, (unsigned)(v >> 32), src);
	return ((uint64_t)hi << 32) | lo;
}

/**
 * For read r and window start j, slot = slot_offs[r] + j.
 *   h0[slot]    = canonical ntHash of bases[j .. j+k)         (RollingHash.h:69-102)
 *   valid[slot] = 1 iff the window holds only A/C/G/T         (RollingHashIterator.h:46-57)
 * P_i = XOR_{t<=i} R^{-t}(seed(c_t)), Q_i = XOR_{t<=i} R^{t}(seed(comp c_t)):
 *   fwd(j) = R^{j+k-1}(P_{j+k-1} ^ P_{j-1}),  rc(j) = R^{-j}(Q_{j+k-1} ^ Q_{j-1}).
 */
/** one warp hashes the L bases at `beg`; window j goes to slot slot0 + j */
ABB_D void hash_one_read(const uint8_t* __restrict__ bases, uint64_t beg, unsigned L, uint64_t slot0, unsigned k, uint64_t* P,
                         uint64_t* Q, unsigned* B, int lane, uint64_t* __restrict__ h0_out, uint8_t* __restrict__ valid_out)
{
	uint64_t carryP = 0, carryQ = 0;
	unsigned carryB = 0;
	for (unsigned base = 0; base < L; base += 32) {
		const unsigned i = base + lane;
		unsigned code = 4;
		if (i < L)
			code = base_code(bases[beg + i]);
		uint64_t p = 0, q = 0;
		if (code < 4) {
			p = sror_n(seed_of(code), i);
			q = srol_n(seed_of(3 - code), i);
		}
		// inclusive prefix XOR across the warp
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			uint64_t up = shfl_up64(p, d), uq = shfl_up64(q, d);
			if (lane >= d) {
				p ^= up;
				q ^= uq;
			}
		}
		p ^= carryP;
		q ^= carryQ;
		const unsigned badmask = __ballot_sync(0xffffffffu, code >= 4 && i < L);
		const unsigned b = carryB + __popc(badmask & (0xffffffffu >> (31 - lane)));
		P[i & (kRing - 1)] = p;
		Q[i & (kRing - 1)] = q;
		B[i & (kRing - 1)] = b;
		carryP = shfl64(p, 31);
		carryQ = shfl64(q, 31);
		carryB += __popc(badmask);
		__syncwarp();
		if (i < L && i + 1 >= k) {
			const unsigned j = i + 1 - k; // window [j, i]
			uint64_t pj = 0, qj = 0;
			unsigned bj = 0;
			if (j > 0) {
				pj = P[(j - 1) & (kRing - 1)];
				qj = Q[(j - 1) & (kRing - 1)];
				bj = B[(j - 1) & (kRing - 1)];
			}
			const uint64_t fh = srol_n(p ^ pj, i);
			const uint64_t rh = sror_n(q ^ qj, j);
			h0_out[slot0 + j] = rh < fh ? rh : fh;
			valid_out[slot0 + j] = (b == bj) ? 1 : 0;
		}
		__syncwarp();
	}
}

static __global__ void __launch_bounds__(kHashWarps * 32)
k_hash_reads(const uint8_t* __restrict__ bases, const uint64_t* __restrict__ offs,
             const uint64_t* __restrict__ slot_offs, uint64_t slot_base, uint64_t n_reads, unsigned k,
             uint64_t* __restrict__ h0_out, uint8_t* __restrict__ valid_out)
{
	__shared__ uint64_t sP[kHashWarps][kRing];
	__shared__ uint64_t sQ[kHashWarps][kRing];
	__shared__ unsigned sB[kHashWarps][kRing];
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	for (uint64_t r = (uint64_t)blockIdx.x * kHashWarps + warp; r < n_reads; r += (uint64_t)gridDim.x * kHashWarps) {
		const uint64_t beg = offs[r];
		const unsigned L = (unsigned)(offs[r + 1] - beg);
		if (L < k)
			continue;
		hash_one_read(bases, beg, L, slot_offs[r] - slot_base, k, sP[warp], sQ[warp], sB[warp], lane, h0_out, valid_out);
	}
}

// K1 with TMA staging (sm_90+/sm_100a bulk-copy engine).  A CTA of kHashWarps warps takes blocks of kTmaReads consecutive
// reads; the bytes of a block are contiguous in the batch, so ONE cp.async.bulk (cuda::device::memcpy_async_tx -> UBLKCP)
// moves them into shared memory and signals an mbarrier; the next block is in flight while the warps hash the current one
// from shared memory (double buffer; every warp takes kTmaReads / kHashWarps reads of the block, so the two block barriers
// of a stage are paid once per 32 reads).  Blocks that do not fit a stage (long reads) and the last bytes of a batch that a
// 16-byte-aligned copy would overrun are hashed straight from global memory.
constexpr unsigned kTmaStage = 8192; // bytes per stage
constexpr unsigned kTmaReads = 32;   // reads per stage: 32 x 150 bases = 4 800 bytes

static __global__ void __launch_bounds__(kHashWarps * 32)
k_hash_reads_tma(const uint8_t* __restrict__ bases, const uint64_t* __restrict__ offs,
                 const uint64_t* __restrict__ slot_offs, uint64_t slot_base, uint64_t n_reads, unsigned k,
                 uint64_t* __restrict__ h0_out, uint8_t* __restrict__ valid_out)
{
	__shared__ uint64_t sP[kHashWarps][kRing];
	__shared__ uint64_t sQ[kHashWarps][kRing];
	__shared__ unsigned sB[kHashWarps][kRing];
	extern __shared__ __align__(128) uint8_t stage_mem[]; // 2 x kTmaStage bytes (dynamic: the rings above use 40 KB of static)
	uint8_t* const stage[2] = { stage_mem, stage_mem + kTmaStage };
	__shared__ cuda::barrier<cuda::thread_scope_block> bar[2];
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const uint64_t n_blocks = (n_reads + kTmaReads - 1) / kTmaReads;
	const uint64_t n_bases = offs[n_reads]; // a copy never reaches past the reads of this launch
	if (threadIdx.x == 0) {
		init(&bar[0], 1);
		init(&bar[1], 1);
		cuda::device::experimental::fence_proxy_async_shared_cta(); // make the barriers visible to the copy engine
	}
	__syncthreads();
	// [a0, a1): the 16-byte aligned byte range of block b, or a1 == a0 when it has to be read from global memory
	auto range = [&](uint64_t b, uint64_t* a0, uint64_t* a1) {
		const uint64_t r0 = b * kTmaReads, r1 = min(n_reads, r0 + kTmaReads);
		const uint64_t lo = offs[r0] & ~15ULL, hi = (offs[r1] + 15) & ~15ULL;
		*a0 = lo;
		*a1 = (hi - lo <= kTmaStage && hi <= n_bases) ? hi : lo;
	};
	cuda::barrier<cuda::thread_scope_block>::arrival_token tok[2];
	uint64_t b = blockIdx.x;
	int st = 0;
	uint64_t a0 = 0, a1 = 0;
	if (b < n_blocks) {
		range(b, &a0, &a1);
		if (threadIdx.x == 0 && a1 > a0) {
			cuda::device::memcpy_async_tx(stage[0], bases + a0, cuda::aligned_size_t<16>(a1 - a0), bar[0]);
			tok[0] = cuda::device::barrier_arrive_tx(bar[0], 1, a1 - a0);
		}
	}
	for (; b < n_blocks; b += gridDim.x, st ^= 1) {
		// prefetch the next block of this CTA into the other stage (its previous contents were consumed before the
		// __syncthreads at the end of the previous iteration)
		const uint64_t nb = b + gridDim.x;
		uint64_t n0 = 0, n1 = 0;
		if (nb < n_blocks) {
			range(nb, &n0, &n1);
			if (threadIdx.x == 0 && n1 > n0) {
				cuda::device::memcpy_async_tx(stage[st ^ 1], bases + n0, cuda::aligned_size_t<16>(n1 - n0), bar[st ^ 1]);
				tok[st ^ 1] = cuda::device::barrier_arrive_tx(bar[st ^ 1], 1, n1 - n0);
			}
		}
		const bool staged = a1 > a0;
		if (staged) {
			if (threadIdx.x == 0)
				bar[st].wait(std::move(tok[st])); // the bytes have landed
			__syncthreads();
		}
		const uint64_t r_end = min(n_reads, (b + 1) * (uint64_t)kTmaReads);
		for (uint64_t r = b * kTmaReads + warp; r < r_end; r += kHashWarps) {
			const uint64_t beg = offs[r];
			const unsigned L = (unsigned)(offs[r + 1] - beg);
			if (L >= k) {
				if (staged)
					hash_one_read(stage[st], beg - a0, L, slot_offs[r] - slot_base, k, sP[warp], sQ[warp], sB[warp], lane, h0_out, valid_out);
				else
					hash_one_read(bases, beg, L, slot_offs[r] - slot_base, k, sP[warp], sQ[warp], sB[warp], lane, h0_out, valid_out);
			}
		}
		__syncthreads(); // everybody is done with stage[st] before it is refilled two iterations later
		a0 = n0;
		a1 = n1;
	}
}

/** the same over explicit segments (long sequences are cut into overlapping pieces so that every
 *  warp has work): segment s = bases [seg_beg[s], +seg_len[s]), its first window is slot seg_slot[s] */
static __global__ void __launch_bounds__(kHashWarps * 32)
k_hash_segments(const uint8_t* __restrict__ bases, const uint64_t* __restrict__ seg_beg, const unsigned* __restrict__ seg_len,
                const uint64_t* __restrict__ seg_slot, uint64_t n_segs, unsigned k, uint64_t* __restrict__ h0_out,
                uint8_t* __restrict__ valid_out)
{
	__shared__ uint64_t sP[kHashWarps][kRing];
	__shared__ uint64_t sQ[kHashWarps][kRing];
	__shared__ unsigned sB[kHashWarps][kRing];
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	for (uint64_t r = (uint64_t)blockIdx.x * kHashWarps + warp; r < n_segs; r += (uint64_t)gridDim.x * kHashWarps) {
		const unsigned L = seg_len[r];
		if (L < k)
			continue;
		hash_one_read(bases, seg_beg[r], L, seg_slot[r], k, sP[warp], sQ[warp], sB[warp], lane, h0_out, valid_out);
	}
}

/** spaced-seed variant: canonical hash over the '1' positions only (maskHash, nthash.hpp:537-547;
 *  a window is bad only if a non-ACGT base sits on a '1' position, RollingHashIterator.h:58-73).
 *  One warp per read, lanes stride over windows; O(k) per window (config 4 path). */
static __global__ void __launch_bounds__(kHashWarps * 32)
k_hash_reads_masked(const uint8_t* __restrict__ bases, const uint64_t* __restrict__ offs,
                    const uint64_t* __restrict__ slot_offs, uint64_t slot_base, uint64_t n_reads, unsigned k,
                    const uint8_t* __restrict__ care /* k bytes: 1 where mask == '1' */,
                    uint64_t* __restrict__ h0_out, uint8_t* __restrict__ valid_out)
{
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	for (uint64_t r = (uint64_t)blockIdx.x * kHashWarps + warp; r < n_reads;
	     r += (uint64_t)gridDim.x * kHashWarps) {
		const uint64_t beg = offs[r];
		const unsigned L = (unsigned)(offs[r + 1] - beg);
		if (L < k)
			continue;
		const uint64_t slot0 = slot_offs[r] - slot_base;
		for (unsigned j = lane; j + k <= L; j += 32) {
			uint64_t fh = 0, rh = 0;
			bool ok = true;
			for (unsigned t = 0; t < k; ++t) {
				if (!care[t])
					continue;
				unsigned code = base_code(bases[beg + j + t]);
				if (code >= 4) {
					ok = false;
					break;
				}
				fh ^= srol_n(seed_of(code), k - 1 - t);
				rh ^= srol_n(seed_of(3 - code), t);
			}
			h0_out[slot0 + j] = rh < fh ? rh : fh;
			valid_out[slot0 + j] = ok ? 1 : 0;
		}
	}
}

/** k_hash_segments for a spaced seed (unitigs of the extension stage: 'N' can only sit on '0' positions there) */
static __global__ void __launch_bounds__(kHashWarps * 32)
k_hash_segments_masked(const uint8_t* __restrict__ bases, const uint64_t* __restrict__ seg_beg,
                       const unsigned* __restrict__ seg_len, const uint64_t* __restrict__ seg_slot, uint64_t n_segs, unsigned k,
                       const uint8_t* __restrict__ care, uint64_t* __restrict__ h0_out, uint8_t* __restrict__ valid_out)
{
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	for (uint64_t r = (uint64_t)blockIdx.x * kHashWarps + warp; r < n_segs; r += (uint64_t)gridDim.x * kHashWarps) {
		const uint64_t beg = seg_beg[r];
		const unsigned L = seg_len[r];
		if (L < k)
			continue;
		const uint64_t slot0 = seg_slot[r];
		for (unsigned j = lane; j + k <= L; j += 32) {
			uint64_t fh = 0, rh = 0;
			bool ok = true;
			for (unsigned t = 0; t < k; ++t) {
				if (!care[t])
					continue;
				unsigned code = base_code(bases[beg + j + t]);
				if (code >= 4) {
					ok = false;
					break;
				}
				fh ^= srol_n(seed_of(code), k - 1 - t);
				rh ^= srol_n(seed_of(3 - code), t);
			}
			h0_out[slot0 + j] = rh < fh ? rh : fh;
			valid_out[slot0 + j] = ok ? 1 : 0;
		}
	}
}

/** per-read window counts -> (exclusive scan done by the caller with cub-free two-pass code) */
static __global__ void k_window_counts(const uint64_t* __restrict__ offs, uint64_t n_reads, unsigned k,
                                uint64_t* __restrict__ counts)
{
	uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (r < n_reads) {
		uint64_t L = offs[r + 1] - offs[r];
		counts[r] = L >= k ? L - k + 1 : 0;
	}
}

// ------------------------------------------------------------------------------------------
// K2: ordered insert over one window of slots [w0, w0 + n)
// ------------------------------------------------------------------------------------------

/** positions of slot s: either derived from h0 (stride 1) or read from the literal
 *  H-per-k-mer array of the reference interface */
template <bool LITERAL, int MAXH>
ABB_D void slot_positions(const uint64_t* __restrict__ hashes, uint64_t s, const HashCfg& cfg, uint64_t* pos)
{
	if (LITERAL) {
#pragma unroll
		for (int i = 0; i < MAXH; ++i)
			if (i < (int)cfg.H)
				pos[i] = fastmod_u64(hashes[s * cfg.H + i], cfg.mod);
	} else {
		const uint64_t h0 = hashes[s];
#pragma unroll
		for (int i = 0; i < MAXH; ++i)
			if (i < (int)cfg.H)
				pos[i] = nth_pos(h0, cfg, i);
	}
}
/** one position of slot s */
template <bool LITERAL>
ABB_D uint64_t slot_position(const uint64_t* __restrict__ hashes, uint64_t s, const HashCfg& cfg, unsigned i)
{
	return LITERAL ? fastmod_u64(hashes[s * cfg.H + i], cfg.mod) : nth_pos(hashes[s], cfg, i);
}

/** conflict map: E two-bit entries, 16 per word, entry = position mod E (E a power of two; exact when the
 *  filter has at most E positions).  bit 0: touched by a slot of the window; bit 1: touched again (by a second
 *  slot, by a second hash of the same slot, or by a carried slot). */
struct ConflictMap {
	unsigned* w;
	uint64_t mask; // E - 1
};
ABB_D void map_mark(const ConflictMap& m, uint64_t pos)
{
	const uint64_t e = pos & m.mask;
	const unsigned sh = (unsigned)(e & 15) * 2;
	const unsigned old = atomicOr(&m.w[e >> 4], 1u << sh);
	if (((old >> sh) & 3u) == 1u)
		atomicOr(&m.w[e >> 4], 2u << sh);
}
/** the marks of all H positions of a slot: the H first atomics are independent and in flight together; only then are
 *  their return values looked at (a mark issued per position would serialise H L2 round trips per thread) */
template <int MAXH>
ABB_D void map_mark_all(const ConflictMap& m, const uint64_t* pos, unsigned H)
{
	unsigned old[MAXH];
#pragma unroll
	for (int i = 0; i < MAXH; ++i)
		if (i < (int)H) {
			const uint64_t e = pos[i] & m.mask;
			old[i] = atomicOr(&m.w[e >> 4], 1u << ((unsigned)(e & 15) * 2));
		}
#pragma unroll
	for (int i = 0; i < MAXH; ++i)
		if (i < (int)H) {
			const uint64_t e = pos[i] & m.mask;
			const unsigned sh = (unsigned)(e & 15) * 2;
			if (((old[i] >> sh) & 3u) == 1u)
				atomicOr(&m.w[e >> 4], 2u << sh);
		}
}
ABB_D void map_mark_carried(const ConflictMap& m, uint64_t pos)
{
	const uint64_t e = pos & m.mask;
	atomicOr(&m.w[e >> 4], 3u << ((unsigned)(e & 15) * 2));
}
ABB_D unsigned map_get(const ConflictMap& m, uint64_t pos)
{
	const uint64_t e = pos & m.mask;
	return (__ldcg(&m.w[e >> 4]) >> ((unsigned)(e & 15) * 2)) & 3u;
}

/** device-resident control block of the insert pipeline */
struct InsertCtl {
	unsigned n_carry[2];  // lengths of the two carry lists
	unsigned old_flag;    // a slot carried again is older than the drain age
	unsigned resume;      // first window the kernel has NOT processed (it stops early when a drain is due)
	unsigned tag_mask[2]; // prefix of each tag table that is in use (to be cleared before its next use)
	unsigned pad[2];
};

/** CountingBloomFilter::incrementMin / HashAgnosticCascadingBloom::insert by a thread that is the
 *  only pending event on all of its positions */
template <int KIND, int MAXH>
ABB_D void apply_alone(const FilterView& f, const uint64_t* pos, const unsigned* v, unsigned H)
{
	if (KIND == 0) {
		// CountingBloomFilter.hpp:138-162; "if (minVal > newVal) return" = saturated at 255
		unsigned mn = 255;
#pragma unroll
		for (int i = 0; i < MAXH; ++i)
			if (i < (int)H)
				mn = min(mn, v[i]);
		if (mn == 255)
			return;
#pragma unroll
		for (int i = 0; i < MAXH; ++i)
			if (i < (int)H && v[i] == mn)
				__stcg(f.data + pos[i], (uint8_t)(mn + 1));
	} else
		apply_cascading(f, pos, H);
}

struct InsertArgs {
	const uint64_t* hashes;
	const uint8_t* valid;   // may be NULL (all slots valid)
	uint64_t n_slots;
	unsigned window;        // W
	unsigned w_begin, n_windows;
	HashCfg cfg;
	ConflictMap map[3];     // window w reads map[w % 3], marks map[(w+1) % 3] and clears map[(w+2) % 3] (read by window w-1)
	unsigned long long* tags[2];
	unsigned tag_cap;       // entries allocated per tag table (power of two)
	FilterView f;
	unsigned age_off, drain_age;
	uint64_t* carry[2];
	InsertCtl* ctl;
	unsigned long long* stats;
	unsigned dbg; // ABB_DBG what-if switches for timing experiments (results are WRONG when set): 1 no marks, 2 no counter traffic,
	              // 4 no map clear, 8 no carried reservations, 16 no grid barriers
};

ABB_D unsigned tag_mask_for(unsigned n_carried, unsigned H, unsigned cap)
{
	unsigned want = 4096;
	while (want < 8u * n_carried * H && want < cap)
		want <<= 1;
	return min(want, cap) - 1;
}

/**
 * K2: the persistent window kernel (cooperative launch, one CTA set resident for a whole chunk of windows).
 * Window w, phase A: the carried slots (exact ownership through tags[w & 1]) and the new slots [w0, w0 + n)
 * (independent unless one of their entries in the window's map was touched again) apply or are put on the other carry
 * list; the same threads mark the slots of window w + 1 in the next map and clear the tag table and map of window w - 1.
 * Grid barrier.  Phase B: the slots just carried reserve their positions in tags[(w+1) & 1] and mark them "touched
 * again" in the next window's map.  Grid barrier.  (Three maps rotate: the one window w-1 read is cleared during phase A.)  The counter loads are issued before the map / tag
 * probes so that the HBM round trip overlaps the L2 round trip.  The kernel returns early (ctl->resume) when the
 * pending slots need the serial drain.
 */
template <int KIND, bool LITERAL, int MAXH>
__global__ void __launch_bounds__(256, 4)
k_insert_windows(const InsertArgs a)
{
	cg::grid_group grid = cg::this_grid();
	const uint64_t T = (uint64_t)gridDim.x * blockDim.x;
	const uint64_t gtid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const unsigned H = a.cfg.H;
	const uint64_t W = a.window;
	uint64_t pos[MAXH];
	unsigned v[MAXH];
	if (a.w_begin == 0) { // the marks of window 0
		const unsigned n0 = (unsigned)min((uint64_t)W, a.n_slots);
		for (uint64_t t = gtid; t < n0; t += T)
			if (!a.valid || a.valid[t]) {
				slot_positions<LITERAL, MAXH>(a.hashes, t, a.cfg, pos);
				map_mark_all<MAXH>(a.map[0], pos, H);
			}
		grid.sync();
	}
	for (unsigned w = a.w_begin; w < a.n_windows; ++w) {
		const int in = (int)(w & 1), out = 1 - in;
		const ConflictMap& mcur = a.map[w % 3];
		const ConflictMap& mnext = a.map[(w + 1) % 3];
		const ConflictMap& mold = a.map[(w + 2) % 3];
		const uint64_t w0 = (uint64_t)w * W, w1 = w0 + W;
		const unsigned n = (unsigned)min(W, a.n_slots - w0);
		const unsigned n_next = w + 1 < a.n_windows ? (unsigned)min(W, a.n_slots - w1) : 0u;
		const unsigned n_in = a.ctl->n_carry[in];
		const TagTable tcur = { a.tags[in], a.ctl->tag_mask[in] };
		const unsigned old_mask_out = a.ctl->tag_mask[out];
		// ---- phase A
		for (uint64_t id = gtid; id < (uint64_t)n_in + max(n, n_next); id += T) {
			if (id < n_in) {
				const uint64_t s = a.carry[in][id];
				const uint64_t prio = s + a.age_off - w0;
				slot_positions<LITERAL, MAXH>(a.hashes, s, a.cfg, pos);
				if (KIND == 0) {
#pragma unroll
					for (int i = 0; i < MAXH; ++i)
						if (i < (int)H)
							v[i] = __ldcg(a.f.data + pos[i]);
				}
				bool owner = true;
				uint64_t where[MAXH];
#pragma unroll
				for (int i = 0; i < MAXH; ++i)
					if (i < (int)H)
						owner &= tag_owner_at(tcur, pos[i], &where[i]) == prio;
				if (owner) {
					apply_alone<KIND, MAXH>(a.f, pos, v, H);
#pragma unroll
					for (int i = 0; i < MAXH; ++i)
						if (i < (int)H)
							tag_release_at(tcur, pos[i], where[i]);
				} else {
					a.carry[out][atomicAdd(&a.ctl->n_carry[out], 1u)] = s;
					if (w0 - s > a.drain_age)
						a.ctl->old_flag = 1;
				}
				continue;
			}
			const uint64_t t = id - n_in;
			// slot w0 + t is applied, slot w1 + t is marked for the next window.  Order of issue: both hashes, the counter
			// loads and map probes of the first, then the marks of the second (they run in the shadow of the HBM round
			// trip), then the decision and the stores.
			const bool do_apply = t < n && (!a.valid || a.valid[w0 + t]);
			const bool do_mark = t < n_next && (!a.valid || a.valid[w1 + t]);
			uint64_t pos2[MAXH];
			if (do_apply)
				slot_positions<LITERAL, MAXH>(a.hashes, w0 + t, a.cfg, pos);
			if (do_mark)
				slot_positions<LITERAL, MAXH>(a.hashes, w1 + t, a.cfg, pos2);
			unsigned again = 0;
			if (do_apply) {
				if (KIND == 0) {
#pragma unroll
					for (int i = 0; i < MAXH; ++i)
						if (i < (int)H)
							v[i] = (a.dbg & 2u) ? 255u : __ldcg(a.f.data + pos[i]);
				}
#pragma unroll
				for (int i = 0; i < MAXH; ++i)
					if (i < (int)H)
						again |= map_get(mcur, pos[i]);
			}
			if (do_mark && !(a.dbg & 1u))
				map_mark_all<MAXH>(mnext, pos2, H);
			if (do_apply) {
				if (!(again & 2u))
					apply_alone<KIND, MAXH>(a.f, pos, v, H);
				else {
					a.carry[out][atomicAdd(&a.ctl->n_carry[out], 1u)] = w0 + t;
					atomicAdd(&a.stats[0], 1ULL); // slots that did not commit in their own window
				}
			}
		}
		for (uint64_t i = gtid; i <= old_mask_out; i += T) // the tag table of window w - 1
			a.tags[out][i] = 0;
		if (!(a.dbg & 4u)) { // ... and its conflict map
			uint4* mw = reinterpret_cast<uint4*>(mold.w);
			const uint64_t words4 = (mold.mask + 1) / 64; // 16 entries per word, 4 words per uint4
			for (uint64_t i = gtid; i < words4; i += T)
				mw[i] = make_uint4(0, 0, 0, 0);
		}
		if (!(a.dbg & 16u))
			grid.sync(); // (a grid barrier orders memory itself)
		// ---- phase B
		const unsigned n_out = a.ctl->n_carry[out];
		const bool stop = n_out > kCarryLanes || a.ctl->old_flag != 0;
		const bool last = w + 1 == a.n_windows;
		const unsigned new_mask = tag_mask_for(n_out, H, a.tag_cap);
		if (!stop && !last && !(a.dbg & 8u)) {
			const TagTable tnext = { a.tags[out], new_mask };
			for (uint64_t i = gtid; i < n_out; i += T) {
				const uint64_t s = a.carry[out][i];
				slot_positions<LITERAL, MAXH>(a.hashes, s, a.cfg, pos);
				const uint64_t prio = s + a.age_off - w1;
#pragma unroll
				for (int j = 0; j < MAXH; ++j)
					if (j < (int)H) {
						tag_reserve(tnext, pos[j], prio);
						map_mark_carried(mnext, pos[j]);
					}
			}
		}
		if (gtid == 0) {
			a.ctl->n_carry[in] = 0;
			a.ctl->tag_mask[out] = (!stop && !last) ? new_mask : 0u;
			a.ctl->resume = w + 1;
		}
		if (!(a.dbg & 16u))
			grid.sync();
		if (stop)
			return;
	}
}

// ---- drain: one CTA replays the pending slots in file order on counters staged in shared memory ----
constexpr unsigned kDrainThreads = 1024;
constexpr unsigned kDrainPos = 2048;   // filter positions staged per chunk
constexpr unsigned kDrainMap = 4096;   // shared-memory map entries (load <= 0.5)

/** exclusive prefix sum of one value per thread over the CTA (kDrainThreads threads); total in *total */
ABB_D unsigned block_exclusive_scan(unsigned x, unsigned* warp_sums /* [32] shared */, unsigned* total)
{
	const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	unsigned incl = x;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) {
		unsigned y = __shfl_up_sync(0xffffffffu, incl, d);
		if (lane >= (unsigned)d)
			incl += y;
	}
	if (lane == 31)
		warp_sums[warp] = incl;
	__syncthreads();
	if (warp == 0) {
		unsigned wsum = warp_sums[lane];
		unsigned winc = wsum;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			unsigned y = __shfl_up_sync(0xffffffffu, winc, d);
			if (lane >= (unsigned)d)
				winc += y;
		}
		warp_sums[lane] = winc - wsum; // exclusive
		if (lane == 31)
			*total = winc;
	}
	__syncthreads();
	return warp_sums[warp] + incl - x;
}

/** the set bits of bw[0, words) in ascending order: out[i] = first_slot + bit index; clears the words.
 *  Called by all threads of a kDrainThreads CTA; returns the number of slots written. */
ABB_D unsigned enumerate_presence(unsigned* __restrict__ bw, unsigned words, uint64_t first_slot, uint64_t* __restrict__ out,
                                  unsigned* warp_sums, unsigned* total)
{
	const unsigned per = (words + blockDim.x - 1) / blockDim.x;
	const unsigned wb = min(words, threadIdx.x * per), we = min(words, wb + per);
	unsigned cnt = 0;
	for (unsigned wd = wb; wd < we; ++wd)
		cnt += __popc(__ldcg(&bw[wd]));
	unsigned at = block_exclusive_scan(cnt, warp_sums, total);
	for (unsigned wd = wb; wd < we; ++wd) {
		unsigned m = __ldcg(&bw[wd]);
		if (m)
			bw[wd] = 0;
		while (m) {
			const unsigned b = __ffs(m) - 1;
			m &= m - 1;
			out[at++] = first_slot + (uint64_t)wd * 32 + b;
		}
	}
	__threadfence();
	__syncthreads();
	return *total;
}

/** K2c.  Does nothing unless forced, more than min_count slots are pending or a pending slot is old.
 *  Clears ctl->n_carry[other] (the list the preceding window launch has just consumed) so that it can collect
 *  the next window's carries.  `bits` is a zeroed presence bitmap for slots [lo_slot, lo_slot + 32 * bit_words)
 *  (left zeroed), `sorted` holds as many slots as the list.  stats[2] += slots replayed. */
template <int KIND, bool LITERAL, int MAXH>
__global__ void __launch_bounds__(kDrainThreads)
k_drain(const uint64_t* __restrict__ hashes, HashCfg cfg, FilterView f, const uint64_t* __restrict__ list, InsertCtl* __restrict__ ctl,
        int which, unsigned min_count, int force, unsigned* __restrict__ bits, uint64_t lo_slot, uint64_t* __restrict__ sorted,
        unsigned long long* __restrict__ stats)
{
	__shared__ unsigned long long s_key[kDrainMap];
	__shared__ unsigned short s_val[kDrainMap]; // bit 8 = dirty
	__shared__ unsigned short s_idx[kDrainPos];
	__shared__ unsigned s_warp[32];
	__shared__ unsigned s_total;
	__shared__ unsigned long long s_lo, s_hi;
	if (threadIdx.x == 0) {
		ctl->n_carry[1 - which] = 0;
		s_lo = ~0ULL;
		s_hi = 0;
	}
	const unsigned n = ctl->n_carry[which];
	const bool go = n > 0 && (force || n > min_count || ctl->old_flag);
	__syncthreads();
	if (!go)
		return;
	// 1. file order: presence bitmap over [min slot, max slot], enumerated in order
	unsigned long long lo = ~0ULL, hi = 0;
	for (unsigned x = threadIdx.x; x < n; x += blockDim.x) {
		const unsigned long long s = list[x];
		lo = s < lo ? s : lo;
		hi = s > hi ? s : hi;
	}
	for (int d = 16; d; d >>= 1) {
		unsigned long long a = __shfl_down_sync(0xffffffffu, lo, d), b = __shfl_down_sync(0xffffffffu, hi, d);
		lo = a < lo ? a : lo;
		hi = b > hi ? b : hi;
	}
	if ((threadIdx.x & 31) == 0) {
		atomicMin(&s_lo, lo);
		atomicMax(&s_hi, hi);
	}
	__syncthreads();
	const uint64_t base = (s_lo - lo_slot) & ~31ULL; // bit index of the first word
	const unsigned words = (unsigned)(((s_hi - lo_slot) - base) / 32 + 1);
	unsigned* const bw = bits + base / 32;
	for (unsigned x = threadIdx.x; x < n; x += blockDim.x) {
		const uint64_t b = list[x] - lo_slot - base;
		atomicOr(&bw[b >> 5], 1u << (b & 31));
	}
	__threadfence();
	__syncthreads();
	enumerate_presence(bw, words, lo_slot + base, sorted, s_warp, &s_total);
	// 2. replay
	if (KIND == 0) {
		const unsigned H = cfg.H;
		const unsigned per_chunk = kDrainPos / H; // slots per chunk
		for (unsigned c0 = 0; c0 < n; c0 += per_chunk) {
			const unsigned cn = min(per_chunk, n - c0);
			for (unsigned e = threadIdx.x; e < kDrainMap; e += blockDim.x)
				s_key[e] = 0;
			__syncthreads();
			for (unsigned x = threadIdx.x; x < cn * H; x += blockDim.x) {
				const unsigned j = x / H, i = x - j * H;
				const uint64_t p = slot_position<LITERAL>(hashes, sorted[c0 + j], cfg, i);
				const unsigned long long key = p + 1;
				unsigned e = (unsigned)((p * 0x9E3779B97F4A7C15ULL) >> 52) & (kDrainMap - 1);
				for (;;) {
					const unsigned long long old = atomicCAS(&s_key[e], 0ULL, key);
					if (old == 0) {
						s_val[e] = __ldcg(f.data + p);
						break;
					}
					if (old == key)
						break;
					e = (e + 1) & (kDrainMap - 1);
				}
				s_idx[x] = (unsigned short)e;
			}
			__syncthreads();
			if (threadIdx.x == 0) {
				unsigned a[MAXH], v[MAXH];
				for (unsigned j = 0; j < cn; ++j) {
					unsigned mn = 255;
#pragma unroll
					for (int i = 0; i < MAXH; ++i)
						if (i < (int)H) {
							a[i] = s_idx[j * H + i];
							v[i] = s_val[a[i]] & 0xffu;
							mn = min(mn, v[i]);
						}
					if (mn != 255) {
#pragma unroll
						for (int i = 0; i < MAXH; ++i)
							if (i < (int)H && v[i] == mn)
								s_val[a[i]] = (unsigned short)((mn + 1) | 0x100u);
					}
				}
			}
			__syncthreads();
			for (unsigned e = threadIdx.x; e < kDrainMap; e += blockDim.x)
				if (s_key[e] && (s_val[e] & 0x100u))
					__stcg(f.data + (s_key[e] - 1), (uint8_t)(s_val[e] & 0xffu));
			__threadfence();
			__syncthreads();
		}
	} else {
		if (threadIdx.x == 0) {
			uint64_t pos[MAXH];
			for (unsigned j = 0; j < n; ++j) {
				slot_positions<LITERAL, MAXH>(hashes, sorted[j], cfg, pos);
				apply_cascading(f, pos, cfg.H);
				__threadfence();
			}
		}
		__syncthreads();
	}
	if (threadIdx.x == 0) {
		ctl->n_carry[which] = 0;
		ctl->old_flag = 0;
		atomicAdd(&stats[2], (unsigned long long)n);
		atomicAdd(&stats[1], 1ULL); // drains that did work
	}
}


/** BloomFilter::insert for every valid slot (order free: OR commutes) -- the assembled-k-mer
 *  filter and plain `abyss-bloom build` bit filters */
template <bool LITERAL, int MAXH>
__global__ void __launch_bounds__(256)
k_bits_insert(const uint64_t* __restrict__ hashes, const uint8_t* __restrict__ valid, uint64_t n,
              HashCfg cfg, uint8_t* __restrict__ bits)
{
	const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (s >= n || (valid && !valid[s]))
		return;
	uint64_t pos[MAXH];
	slot_positions<LITERAL, MAXH>(hashes, s, cfg, pos);
	bits_set(bits, pos, cfg.H);
}

/** contains()/minCount() for the literal hash interface */
template <int KIND>
__global__ void __launch_bounds__(256)
k_query(const uint64_t* __restrict__ hashes, uint64_t n, HashCfg cfg, FilterView f, unsigned threshold,
        uint8_t* __restrict__ out_contains, uint8_t* __restrict__ out_min)
{
	const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (s >= n)
		return;
	if (KIND == 0) {
		unsigned mn = 255;
		for (unsigned i = 0; i < cfg.H; ++i)
			mn = min(mn, (unsigned)__ldcg(f.data + fastmod_u64(hashes[s * cfg.H + i], cfg.mod)));
		if (out_min)
			out_min[s] = (uint8_t)mn;
		if (out_contains)
			out_contains[s] = mn >= threshold;
	} else {
		// bit filter, or last level of a cascading filter (HashAgnosticCascadingBloom.h:105-109)
		const uint8_t* bits = f.data + (uint64_t)(f.levels - 1) * f.level_stride;
		uint64_t pos[kMaxHashes];
		for (unsigned i = 0; i < cfg.H; ++i)
			pos[i] = fastmod_u64(hashes[s * cfg.H + i], cfg.mod);
		bool c = bits_contain(bits, pos, cfg.H);
		if (out_contains)
			out_contains[s] = c;
		if (out_min)
			out_min[s] = c;
	}
}

/** contains() per k-mer slot from the canonical hash h0 (the other H - 1 values follow from it, nthash.hpp:337-342);
 *  slots that RollingHashIterator would skip report 0.  Used by the coverage track / sequence trimming queries
 *  (bloom-dbg.h:399-447,1280-1334). */
template <int KIND>
__global__ void __launch_bounds__(256)
k_query_h0(const uint64_t* __restrict__ h0, const uint8_t* __restrict__ valid, uint64_t n, HashCfg cfg, FilterView f, unsigned threshold,
           uint8_t* __restrict__ out_contains)
{
	for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (uint64_t)gridDim.x * blockDim.x) {
		if (!valid[s]) {
			out_contains[s] = 0;
			continue;
		}
		const uint64_t h = h0[s];
		if (KIND == 0) {
			unsigned mn = 255;
			for (unsigned i = 0; i < cfg.H; ++i)
				mn = min(mn, (unsigned)__ldcg(f.data + nth_pos(h, cfg, i)));
			out_contains[s] = mn >= threshold;
		} else {
			const uint8_t* bits = f.data + (uint64_t)(f.levels - 1) * f.level_stride;
			bool all = true;
			for (unsigned i = 0; i < cfg.H; ++i) {
				const uint64_t p = nth_pos(h, cfg, i);
				all &= (__ldcg(bits + (p >> 3)) >> (p & 7)) & 1;
			}
			out_contains[s] = all;
		}
	}
}

/** contains() of the filter for a canonical hash (counting: minCount >= threshold; bits: last level) */
template <int KIND>
struct FilterProbe {
	HashCfg cfg;
	FilterView f;
	unsigned threshold;
	ABB_HD static unsigned ld(const uint8_t* p)
	{
#if defined(__CUDA_ARCH__)
		return __ldcg(p);
#else
		return *p;
#endif
	}
	ABB_HD bool operator()(uint64_t h0) const
	{
		bool ok = true;
		for (unsigned i = 0; i < cfg.H; ++i) { // independent loads: issued back to back
			const uint64_t p = nth_pos(h0, cfg, i);
			if (KIND == 0)
				ok &= ld(f.data + p) >= threshold;
			else
				ok &= (ld(f.data + (uint64_t)(f.levels - 1) * f.level_stride + (p >> 3)) >> (p & 7)) & 1;
		}
		return ok;
	}
};

/** out-edges of graph vertices for the GraphViz dump: one thread per start k-mer runs successors_chain (abb_graph.cuh); a
 *  search frontier is a handful of vertices and a chain is a sequence of dependent lookups, so this is latency, not
 *  bandwidth -- the 4 x H lookups of one vertex are independent and overlap */
template <int KIND>
__global__ void __launch_bounds__(128)
k_successors(const uint8_t* __restrict__ kmers, uint64_t n, unsigned k, unsigned max_chain, FilterProbe<KIND> probe,
             abb_succ_info* __restrict__ info, unsigned* __restrict__ len, uint64_t* __restrict__ self)
{
	const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (w >= n)
		return;
	len[w] = successors_chain(kmers + w * k, k, max_chain, probe, info + w * max_chain, self + w);
}

/** The bit filters k_neighbours probes: [0] the graph, [1..n) the attribute filters (last level of each).  Every filter is
 *  probed with the graph's hash values -- its multipliers (mult, from the graph's k) and its first H[j] hashes -- modulo its
 *  own size, as RollingBloomDBGVisitor::discover_vertex hands the graph vertex's getHashes() to each attribute filter. */
constexpr unsigned kNbMaxFilters = 33;
constexpr unsigned kNbWarps = 4;
struct NbFilters {
	const uint8_t* bits[kNbMaxFilters];
	FastMod mod[kNbMaxFilters];
	unsigned H[kNbMaxFilters];
	unsigned start[kNbMaxFilters + 1]; // first probe of filter j in the flat probe list: 9 * (H[0] + .. + H[j-1])
	unsigned n;
	uint64_t mult[kMaxHashes];
};

/** the probe functor of neighbourhood() inside k_neighbours: the warp splits the 9 x sum(H) probes of one k-mer over its
 *  lanes (lane = probe mod 32, as K4 lays 8 neighbours x 4 hash slots over a warp), issues four per lane before it looks at
 *  any, and ORs the misses into one word per filter in shared memory (bit v = vertex v) */
struct WarpNbProbe {
	const NbFilters* F;
	unsigned* fail; // [kNbMaxFilters] of this warp's shared memory, zero on entry
	unsigned lane;
	__device__ void operator()(const uint64_t* hash, unsigned* mask, uint32_t* attr) const
	{
		const unsigned total = F->start[F->n];
		for (unsigned base = 0; base < total; base += 4 * 32) {
			unsigned bit[4], slot[4];
#pragma unroll
			for (unsigned u = 0; u < 4; ++u) {
				const unsigned p = base + 32 * u + lane;
				slot[u] = ~0u;
				bit[u] = 1;
				if (p < total) {
					unsigned j = 0;
					while (F->start[j + 1] <= p)
						++j;
					const unsigned r = p - F->start[j], v = r / F->H[j], i = r - v * F->H[j];
					uint64_t h0 = hash[0];
#pragma unroll
					for (unsigned w = 1; w < 9; ++w)
						h0 = v == w ? hash[w] : h0;
					const uint64_t t = h0 * F->mult[i]; // nth_hash with the graph's multipliers
					const uint64_t x = i == 0 ? h0 : t ^ (t >> kMultiShift);
					const uint64_t pos = fastmod_u64(x, F->mod[j]);
					bit[u] = (__ldcg(F->bits[j] + (pos >> 3)) >> (pos & 7)) & 1;
					slot[u] = j * 16 + v;
				}
			}
#pragma unroll
			for (unsigned u = 0; u < 4; ++u)
				if (!bit[u])
					atomicOr(&fail[slot[u] >> 4], 1u << (slot[u] & 15));
		}
		__syncwarp();
		*mask = ~fail[0] & 0x1FFu;
		const unsigned nA = F->n - 1;
		const unsigned ok = lane < nA ? ~fail[1 + lane] : 0u; // lane j answers for attribute filter j
#pragma unroll
		for (unsigned v = 0; v < 9; ++v)
			attr[v] = __ballot_sync(0xffffffffu, (ok >> v) & 1);
	}
};

/** neighbourhoods of one breadth-first search level of `abyss-bloom graph`: one warp per k-mer; every lane computes the 9
 *  hashes (neighbourhood(), abb_graph.cuh), the warp probes the graph and attribute filters for all 9 vertices at once --
 *  one round trip to memory per k-mer instead of the reference's sequence of 8 x H dependent lookups */
__global__ void __launch_bounds__(32 * kNbWarps)
k_neighbours(const uint8_t* __restrict__ kmers, uint64_t n, unsigned k, const __grid_constant__ NbFilters F,
             abb_neighbourhood* __restrict__ out)
{
	__shared__ unsigned s_fail[kNbWarps][kNbMaxFilters];
	const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const uint64_t w = (uint64_t)blockIdx.x * kNbWarps + warp;
	if (w >= n)
		return;
	s_fail[warp][lane] = 0;
	if (lane == 0)
		s_fail[warp][32] = 0;
	__syncwarp();
	const WarpNbProbe probe = { &F, s_fail[warp], lane };
	abb_neighbourhood r;
	neighbourhood(kmers + w * k, k, probe, &r);
	r.pad[0] = r.pad[1] = 0;
	if (lane == 0)
		out[w] = r;
}

/** popCount / filtered_popcount (CountingBloomFilter.hpp:219-244) and getPop (BloomFilter.hpp:313-320) */
static __global__ void __launch_bounds__(256)
k_popcount(const uint8_t* __restrict__ data, uint64_t nbytes, int counting, unsigned threshold,
           unsigned long long* __restrict__ out /* [2] */)
{
	unsigned long long nz = 0, th = 0;
	const uint64_t nwords = nbytes / 16;
	const uint4* w = reinterpret_cast<const uint4*>(data);
	for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nwords;
	     i += (uint64_t)gridDim.x * blockDim.x) {
		uint4 v = w[i];
		unsigned x[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
		for (int j = 0; j < 4; ++j) {
			if (counting) {
#pragma unroll
				for (int b = 0; b < 4; ++b) {
					unsigned c = (x[j] >> (8 * b)) & 0xff;
					nz += c != 0;
					th += c >= threshold;
				}
			} else
				nz += __popc(x[j]);
		}
	}
	// tail bytes
	if (blockIdx.x == 0 && threadIdx.x == 0)
		for (uint64_t i = nwords * 16; i < nbytes; ++i) {
			unsigned c = data[i];
			if (counting) {
				nz += c != 0;
				th += c >= threshold;
			} else
				nz += __popc(c);
		}
	for (int d = 16; d; d >>= 1) {
		nz += __shfl_down_sync(0xffffffffu, nz, d);
		th += __shfl_down_sync(0xffffffffu, th, d);
	}
	if ((threadIdx.x & 31) == 0) {
		atomicAdd(&out[0], nz);
		atomicAdd(&out[1], th);
	}
}

} // namespace abb
