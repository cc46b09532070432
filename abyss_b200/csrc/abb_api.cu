// abb_api.cu -- C ABI (include/abyss_b200.h): filter lifecycle, pass-1 insert, literal-hash
// interface, raw array transfer, statistics.  Host orchestration only; the arithmetic lives in
// abb_device.cuh and the kernels in abb_insert.cuh.
#include "abb_common.h"
#include "abb_insert.cuh"
#include "abb_shard.cuh"
#include <dlfcn.h>
#include <nccl.h>
#include <cub/device/device_scan.cuh>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

namespace abb {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...)
{
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof g_err, fmt, ap);
	va_end(ap);
}

constexpr uint64_t kDefaultWindow = 1ULL << 17;
constexpr uint64_t kChunkSlots = 1ULL << 27; // h0 staging: 128 Mi slots = 1 GiB + 128 MiB flags (one persistent launch + one forced drain per chunk)

static uint64_t next_pow2(uint64_t x)
{
	uint64_t p = 1;
	while (p < x)
		p <<= 1;
	return p;
}

int select_device(int device)
{
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess || n <= 0) {
		set_error("no usable CUDA device (%s); libabyssb200 has no CPU fallback",
		          e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
		return ABB_ENODEV;
	}
	if (device < 0 || device >= n) {
		set_error("device %d out of range (0..%d)", device, n - 1);
		return ABB_EINVAL;
	}
	ABB_CUDA(cudaSetDevice(device));
	// tuning knob: ABB_L2_FETCH=32 asks L2 to fetch 32 B sectors from HBM (cudaLimitMaxL2FetchGranularity).
	// Measured on B200: no gain for the random 1-byte Bloom accesses (0.85 vs 0.90 G k-mers/s), so off by default.
	static int fetch = -1;
	if (fetch < 0) {
		const char* e = getenv("ABB_L2_FETCH");
		fetch = e ? atoi(e) : 0;
	}
	if (fetch > 0)
		cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)fetch);
	return ABB_OK;
}

static FilterView view_of(const abb_filter* f)
{
	FilterView v;
	v.data = f->d_data;
	v.level_stride = f->bytes_per_level;
	v.levels = f->levels;
	return v;
}

/** conflict-map size: 2^25 two-bit entries (8 MiB per map; the three rotating maps are pinned in L2 while the insert
 *  runs, set_l2_policy); with the default window of 2^17 slots 6.4 % of the slots see an alias and are carried (2^26
 *  halves that and measured 3 % slower: the maps compete with the counter sectors for L2).  Exact (no aliases) for
 *  filters of up to 2^25 positions.  ABB_MAP_LOG2 overrides (tuning). */
static uint64_t map_entries_for(uint64_t filter_size, unsigned lg = 25)
{
	if (const char* e = getenv("ABB_MAP_LOG2")) {
		const int v = atoi(e);
		if (v >= 10 && v <= 32)
			lg = (unsigned)v;
	}
	uint64_t want = 1ULL << lg;
	const uint64_t fit = std::max<uint64_t>(next_pow2(filter_size), 1024);
	return std::min(want, fit);
}

static unsigned age_windows_for(uint64_t window)
{
	return (unsigned)std::min<uint64_t>(kMaxAgeWindows, ((1ULL << kPrioBits) - 2) / window - 1);
}

/** make sure the ordered-insert workspace exists for the current window size and hash count */
static int ensure_workspace(abb_filter* f)
{
	const uint64_t want_entries = map_entries_for(f->size, f->map_log2 ? f->map_log2 : 25);
	if (f->d_carry && f->ws_window == f->window && f->ws_H == f->H && f->map_entries == want_entries)
		return ABB_OK;
	cudaFree(f->d_map[0]); // one allocation holds both maps (one L2 access-policy window covers them)
	for (int i = 0; i < 2; ++i) {
		cudaFree(f->d_tags2[i]);
		f->d_tags2[i] = nullptr;
	}
	f->d_map[0] = f->d_map[1] = f->d_map[2] = nullptr;
	cudaFree(f->d_carry);
	cudaFree(f->d_slotbits);
	f->d_carry = nullptr;
	f->d_slotbits = nullptr;
	f->map_entries = want_entries;
	const size_t map_bytes = std::max<size_t>(f->map_entries / 4, 256);
	// at most kCarryLanes carried slots reserve H positions each; load factor <= 1/8.  Only a prefix sized to the
	// carried slots of a window is in use (tag_mask_for)
	f->tag_slots = next_pow2(8ULL * kCarryLanes * f->H);
	ABB_CUDA(cudaMalloc((void**)&f->d_map[0], 3 * map_bytes));
	ABB_CUDA(cudaMemsetAsync(f->d_map[0], 0, 3 * map_bytes, f->stream));
	f->d_map[1] = f->d_map[0] + map_bytes / sizeof(unsigned);
	f->d_map[2] = f->d_map[1] + map_bytes / sizeof(unsigned);
	for (int i = 0; i < 2; ++i) {
		ABB_CUDA(cudaMalloc((void**)&f->d_tags2[i], f->tag_slots * sizeof(unsigned long long)));
		ABB_CUDA(cudaMemsetAsync(f->d_tags2[i], 0, f->tag_slots * sizeof(unsigned long long), f->stream));
	}
	// worst case everything defers: window slots + the carried lanes, twice, plus the drain's sorted copy
	ABB_CUDA(cudaMalloc((void**)&f->d_carry, 3 * (f->window + kCarryLanes) * sizeof(uint64_t)));
	// presence bitmap of the drain: pending slots span at most age_off + 2 windows
	f->slotbit_words = ((uint64_t)age_windows_for(f->window) + 3) * f->window / 32 + 64;
	ABB_CUDA(cudaMalloc((void**)&f->d_slotbits, f->slotbit_words * sizeof(unsigned)));
	ABB_CUDA(cudaMemsetAsync(f->d_slotbits, 0, f->slotbit_words * sizeof(unsigned), f->stream));
	f->ws_window = f->window;
	f->ws_H = f->H;
	return ABB_OK;
}

#define ABB_DISPATCH_H(H, ...)            \
	do {                                  \
		if ((H) <= 4) {                   \
			constexpr int MAXH = 4;       \
			__VA_ARGS__;                  \
		} else if ((H) <= 8) {            \
			constexpr int MAXH = 8;       \
			__VA_ARGS__;                  \
		} else {                          \
			constexpr int MAXH = 32;      \
			__VA_ARGS__;                  \
		}                                 \
	} while (0)

/** While the insert runs, the two conflict maps are pinned in L2 (persisting access-policy window on the filter's stream)
 *  and everything else -- the random counter sectors, the hashes -- is treated as streaming, so that 30-60 MB of counter
 *  lines per window cannot push the maps out (ncu, round 2: without this 57 % of the map atomics missed L2 and the kernel
 *  moved 3x the algorithmic DRAM bytes).  ABB_L2_PERSIST=0 switches it off (tuning). */
static void set_l2_policy(abb_filter* f, bool on, int n_maps = 3)
{
	static int enabled = -1;
	if (enabled < 0) {
		const char* e = getenv("ABB_L2_PERSIST");
		enabled = e ? atoi(e) : 1;
	}
	if (!enabled)
		return;
	cudaStreamAttrValue attr;
	memset(&attr, 0, sizeof attr);
	if (on) {
		int max_persist = 0, max_window = 0;
		cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, f->device);
		cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, f->device);
		const size_t bytes = (size_t)n_maps * std::max<size_t>(f->map_entries / 4, 256);
		if (max_persist <= 0 || max_window <= 0)
			return;
		cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, std::min<size_t>(bytes, (size_t)max_persist));
		attr.accessPolicyWindow.base_ptr = f->d_map[0];
		attr.accessPolicyWindow.num_bytes = std::min<size_t>(bytes, (size_t)max_window);
		attr.accessPolicyWindow.hitRatio = std::min(1.0f, (float)max_persist / (float)bytes);
		attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
		attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
	} else {
		attr.accessPolicyWindow.num_bytes = 0; // no window
		attr.accessPolicyWindow.hitProp = cudaAccessPropertyNormal;
		attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
	}
	cudaStreamSetAttribute(f->stream, cudaStreamAttributeAccessPolicyWindow, &attr);
	if (!on) { // hand the carve-out back to pass 2
		cudaCtxResetPersistingL2Cache();
		cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0);
	}
	cudaGetLastError(); // best effort: a device without the feature runs without the hint
}

/** Scope that holds the L2 policy.  Changing the persisting carve-out (cudaDeviceSetLimit, cudaCtxResetPersistingL2Cache)
 *  synchronises the whole device -- including a host-to-device copy running on another stream -- so a caller that overlaps
 *  a copy with the insert takes the hold once, before the copy starts; the per-chunk scopes inside then do nothing. */
struct PolicyHold {
	abb_filter* f;
	bool took;
	PolicyHold(abb_filter* f_, int n_maps) : f(f_), took(!f_->l2_policy_held && f_->d_map[0] != nullptr)
	{
		if (took) {
			set_l2_policy(f, true, n_maps);
			f->l2_policy_held = true;
		}
	}
	~PolicyHold()
	{
		if (took) {
			set_l2_policy(f, false);
			f->l2_policy_held = false;
		}
	}
	PolicyHold(const PolicyHold&) = delete;
	PolicyHold& operator=(const PolicyHold&) = delete;
};

/** cooperative launch of the persistent window kernel with as many CTAs as fit on the device */
template <int KIND, bool LITERAL, int MAXH>
static int launch_windows(const InsertArgs& args, int device, cudaStream_t st)
{
	static int grid_cache[64] = { 0 };
	int& grid = grid_cache[device & 63];
	if (grid == 0) {
		int per_sm = 0, sms = 0;
		ABB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_insert_windows<KIND, LITERAL, MAXH>, 256, 0));
		ABB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
		grid = std::max(1, per_sm) * sms;
	}
	void* params[] = { (void*)&args };
	ABB_CUDA(cudaLaunchCooperativeKernel((void*)k_insert_windows<KIND, LITERAL, MAXH>, dim3((unsigned)grid), dim3(256), params, 0, st));
	return ABB_OK;
}

/** ordered insert of slots [0, n_slots) of `hashes` (h0 per slot, or literal H per slot); see abb_insert.cuh */
template <bool LITERAL>
static int ordered_insert(abb_filter* f, const uint64_t* d_hashes, const uint8_t* d_valid, uint64_t n_slots)
{
	if (n_slots == 0)
		return ABB_OK;
	if (f->kind == ABB_BIT) {
		ABB_DISPATCH_H(f->H, (k_bits_insert<LITERAL, MAXH><<<blocks_for(n_slots, 256), 256, 0, f->stream>>>(
		                         d_hashes, d_valid, n_slots, f->cfg, f->d_data)));
		f->st.launches += 1;
		ABB_CUDA(cudaGetLastError());
		return ABB_OK;
	}
	ABB_CHECK(ensure_workspace(f));
	cudaStream_t st = f->stream;
	const uint64_t W = f->window;
	const uint64_t n_windows = (n_slots + W - 1) / W;
	ABB_REQUIRE(n_windows < (1ULL << 31), "too many windows in one call");
	const uint64_t cap = W + kCarryLanes;
	InsertArgs a;
	a.hashes = d_hashes;
	a.valid = d_valid;
	a.n_slots = n_slots;
	a.window = (unsigned)W;
	a.w_begin = 0;
	a.n_windows = (unsigned)n_windows;
	a.cfg = f->cfg;
	for (int i = 0; i < 3; ++i) {
		a.map[i].w = f->d_map[i];
		a.map[i].mask = f->map_entries - 1;
	}
	for (int i = 0; i < 2; ++i) {
		a.tags[i] = f->d_tags2[i];
		a.carry[i] = f->d_carry + (uint64_t)i * cap;
	}
	a.tag_cap = (unsigned)f->tag_slots;
	a.f = view_of(f);
	a.age_off = (unsigned)(age_windows_for(W) * W);
	a.drain_age = a.age_off / 3 * 2;
	a.ctl = reinterpret_cast<InsertCtl*>(f->d_ctl);
	a.stats = f->d_stats;
	a.dbg = getenv("ABB_DBG") ? (unsigned)atoi(getenv("ABB_DBG")) : 0u;
	uint64_t* sorted = f->d_carry + 2 * cap;
	// the maps, both tag tables and the control block start clean
	ABB_CUDA(cudaMemsetAsync(f->d_ctl, 0, sizeof(InsertCtl), st));
	ABB_CUDA(cudaMemsetAsync(f->d_map[0], 0, 3 * std::max<size_t>(f->map_entries / 4, 256), st));
	for (int i = 0; i < 2; ++i)
		ABB_CUDA(cudaMemsetAsync(f->d_tags2[i], 0, f->tag_slots * sizeof(unsigned long long), st));
	const bool counting = f->kind == ABB_COUNTING;
	PolicyHold policy(f, 3);
	while (a.w_begin < a.n_windows) {
		const bool timed = f->profile && f->prof_used + 2 <= f->prof_ev.size();
		if (timed)
			cudaEventRecord(f->prof_ev[f->prof_used++], st);
		ABB_DISPATCH_H(f->H, {
			if (counting)
				ABB_CHECK((launch_windows<0, LITERAL, MAXH>(a, f->device, st)));
			else
				ABB_CHECK((launch_windows<1, LITERAL, MAXH>(a, f->device, st)));
		});
		if (timed)
			cudaEventRecord(f->prof_ev[f->prof_used++], st);
		InsertCtl h;
		ABB_CUDA(cudaMemcpyAsync(&h, f->d_ctl, sizeof h, cudaMemcpyDeviceToHost, st));
		ABB_CUDA(cudaStreamSynchronize(st));
		ABB_REQUIRE(h.resume > a.w_begin && h.resume <= a.n_windows, "insert kernel made no progress (window %u of %u)", h.resume, a.n_windows);
		if (timed)
			f->prof_slots += std::min<uint64_t>(n_slots, (uint64_t)h.resume * W) - (uint64_t)a.w_begin * W;
		// the list the last processed window wrote: drained when the kernel stopped for it, and at the end of the call
		const int which = 1 - (int)((h.resume - 1) & 1);
		const uint64_t w0 = (uint64_t)(h.resume - 1) * W;
		const uint64_t lo_slot = w0 > (uint64_t)a.age_off + W ? w0 - a.age_off - W : 0;
		ABB_DISPATCH_H(f->H, {
			if (counting)
				k_drain<0, LITERAL, MAXH><<<1, kDrainThreads, 0, st>>>(d_hashes, f->cfg, a.f, a.carry[which], a.ctl, which, 0, 1, f->d_slotbits, lo_slot,
				                                                      sorted, f->d_stats);
			else
				k_drain<1, LITERAL, MAXH><<<1, kDrainThreads, 0, st>>>(d_hashes, f->cfg, a.f, a.carry[which], a.ctl, which, 0, 1, f->d_slotbits, lo_slot,
				                                                      sorted, f->d_stats);
		});
		f->st.launches += 2;
		f->st.windows += h.resume - a.w_begin;
		a.w_begin = h.resume;
	}
	ABB_CUDA(cudaGetLastError());
	if (f->profile && f->prof_used) { // fold the timed k_insert_windows launches into the statistics
		ABB_CUDA(cudaStreamSynchronize(st));
		for (size_t i = 0; i + 1 < f->prof_used; i += 2) {
			float ms = 0;
			cudaEventElapsedTime(&ms, f->prof_ev[i], f->prof_ev[i + 1]);
			f->st.ms_commit += ms;
			f->st.commit_launches += 1;
		}
		f->st.commit_slots += f->prof_slots;
		f->prof_used = 0;
		f->prof_slots = 0;
	}
	return ABB_OK;
}

/** single thread: cut reads into chunks of about `cap` slots (at least one read per chunk) */
__global__ void k_chunk_bounds(const uint64_t* __restrict__ slot_offs, uint64_t n_reads, uint64_t cap,
                               uint64_t* __restrict__ bounds, unsigned max_chunks, unsigned* __restrict__ n_chunks)
{
	uint64_t r = 0;
	unsigned c = 0;
	bounds[0] = 0;
	while (r < n_reads && c + 1 < max_chunks) {
		const uint64_t limit = slot_offs[r] + cap;
		// largest r1 in (r, n_reads] with slot_offs[r1] <= limit, but at least r + 1
		uint64_t lo = r + 1, hi = n_reads;
		while (lo < hi) {
			uint64_t mid = lo + (hi - lo + 1) / 2;
			if (slot_offs[mid] <= limit)
				lo = mid;
			else
				hi = mid - 1;
		}
		r = lo;
		bounds[++c] = r;
	}
	if (r < n_reads)
		bounds[++c] = n_reads;
	*n_chunks = c;
}

/** count valid flags (k-mers actually inserted) */
__global__ void __launch_bounds__(256)
k_count_valid(const uint8_t* __restrict__ valid, uint64_t n, unsigned long long* __restrict__ out)
{
	unsigned long long c = 0;
	for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
		c += valid[i];
	for (int d = 16; d; d >>= 1)
		c += __shfl_down_sync(0xffffffffu, c, d);
	if ((threadIdx.x & 31) == 0 && c)
		atomicAdd(out, c);
}

/** K1 launcher for reads [r0, r1): h0/valid index = slot_offs[r] + j - slot_base */
int launch_hash(abb_filter* f, unsigned k, const uint8_t* d_care, const uint8_t* d_bases,
                       const uint64_t* d_offs, const uint64_t* d_slot_offs, uint64_t r0, uint64_t r1,
                       uint64_t slot_base, uint64_t* d_h0, uint8_t* d_valid, cudaStream_t stream, uint64_t* launches)
{
	(void)f;
	const uint64_t n = r1 - r0;
	if (n == 0)
		return ABB_OK;
	int sms = 148, dev = 0;
	cudaGetDevice(&dev);
	cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
	const unsigned grid = (unsigned)std::min<uint64_t>((n + kHashWarps - 1) / kHashWarps, (uint64_t)sms * 32);
	// ABB_TMA=0: K1 without the bulk-copy staging (tuning / fallback).  The opt-in to 56 KB of shared memory is a per-device
	// attribute of the kernel: a process that drives several GPUs (abyss-bloom-dbg --devices) sets it on each of them.
	static int tma_env = -1;
	static int tma_dev[64] = { 0 }; // 0 = not tried on this device, 1 = usable, -1 = not usable
	if (tma_env < 0) {
		const char* e = getenv("ABB_TMA");
		tma_env = e ? atoi(e) : 1;
	}
	int& tma_here = tma_dev[dev & 63];
	if (tma_env && tma_here == 0)
		tma_here = cudaFuncSetAttribute(k_hash_reads_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * kTmaStage) == cudaSuccess ? 1 : -1;
	const bool tma = tma_env && tma_here == 1;
	if (d_care)
		k_hash_reads_masked<<<grid, kHashWarps * 32, 0, stream>>>(d_bases, d_offs + r0, d_slot_offs + r0, slot_base, n, k, d_care,
		                                                          d_h0, d_valid);
	else if (tma && (reinterpret_cast<uintptr_t>(d_bases) & 15) == 0) {
		// read blocks staged into shared memory by the bulk-copy engine (cp.async.bulk), double buffered
		const unsigned g = (unsigned)std::min<uint64_t>((n + kTmaReads - 1) / kTmaReads, (uint64_t)sms * 4);
		k_hash_reads_tma<<<g, kHashWarps * 32, 2 * kTmaStage, stream>>>(d_bases, d_offs + r0, d_slot_offs + r0, slot_base, n, k, d_h0, d_valid);
	} else
		k_hash_reads<<<grid, kHashWarps * 32, 0, stream>>>(d_bases, d_offs + r0, d_slot_offs + r0, slot_base, n, k, d_h0, d_valid);
	if (launches)
		*launches += 1;
	ABB_CUDA(cudaGetLastError());
	return ABB_OK;
}

/** K1 over explicit (possibly overlapping) segments, see k_hash_segments */
int launch_hash_segments(unsigned k, const uint8_t* d_care, const uint8_t* d_bases, const uint64_t* d_seg_beg,
                         const unsigned* d_seg_len, const uint64_t* d_seg_slot, uint64_t n_segs, uint64_t* d_h0, uint8_t* d_valid,
                         cudaStream_t stream)
{
	if (n_segs == 0)
		return ABB_OK;
	int sms = 148, dev = 0;
	cudaGetDevice(&dev);
	cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
	const unsigned grid = (unsigned)std::min<uint64_t>((n_segs + kHashWarps - 1) / kHashWarps, (uint64_t)sms * 32);
	if (d_care)
		k_hash_segments_masked<<<grid, kHashWarps * 32, 0, stream>>>(d_bases, d_seg_beg, d_seg_len, d_seg_slot, n_segs, k, d_care,
		                                                             d_h0, d_valid);
	else
		k_hash_segments<<<grid, kHashWarps * 32, 0, stream>>>(d_bases, d_seg_beg, d_seg_len, d_seg_slot, n_segs, k, d_h0, d_valid);
	ABB_CUDA(cudaGetLastError());
	return ABB_OK;
}

/** slot_offs[0..n_reads] = exclusive prefix sum of per-read window counts; returns the total */
int compute_slot_offsets(unsigned k, const uint64_t* d_offs, uint64_t n_reads, DevBuf<uint64_t>& slot_offs,
                                DevBuf<uint8_t>& tmp, cudaStream_t stream, uint64_t* total, uint64_t* launches)
{
	ABB_CHECK(slot_offs.reserve(n_reads + 1));
	ABB_CUDA(cudaMemsetAsync(slot_offs.p + n_reads, 0, sizeof(uint64_t), stream));
	if (n_reads) {
		k_window_counts<<<blocks_for(n_reads, 256), 256, 0, stream>>>(d_offs, n_reads, k, slot_offs.p);
		ABB_CUDA(cudaGetLastError());
	}
	size_t bytes = 0;
	ABB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, slot_offs.p, slot_offs.p, n_reads + 1, stream));
	ABB_CHECK(tmp.reserve(bytes));
	ABB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, bytes, slot_offs.p, slot_offs.p, n_reads + 1, stream));
	ABB_CUDA(cudaMemcpyAsync(total, slot_offs.p + n_reads, sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
	ABB_CUDA(cudaStreamSynchronize(stream));
	if (launches)
		*launches += 3;
	return ABB_OK;
}

static int sharded_ordered_insert(abb_filter* f, abb_comm* c, const uint64_t* d_h0, const uint8_t* d_valid, uint64_t n_slots);

/** a host-to-device copy of the bases that is still in flight, in pieces of `piece` bytes on f->copy_stream
 *  (f->copy_ev[i] fires when bytes [i * piece, (i + 1) * piece) have landed); h_offs are the caller's offsets */
struct PendingCopy {
	const uint64_t* h_offs = nullptr;
	uint64_t piece = 0;
	size_t n_pieces = 0;
	size_t waited = 0; // pieces the filter's stream already waits for
};

/** make the filter's stream wait until bases [0, end) are on the device */
static int wait_bases(abb_filter* f, PendingCopy* pc, uint64_t end)
{
	if (!pc || end == 0)
		return ABB_OK;
	const size_t need = std::min<size_t>(pc->n_pieces, (size_t)((end + pc->piece - 1) / pc->piece));
	if (need > pc->waited) {
		ABB_CUDA(cudaStreamWaitEvent(f->stream, f->copy_ev[need - 1], 0)); // pieces complete in order
		pc->waited = need;
	}
	return ABB_OK;
}

static int insert_reads_dev(abb_filter* f, const uint8_t* d_bases, const uint64_t* d_offs, uint64_t n_reads,
                            uint64_t* n_kmers_out, abb_comm* comm = nullptr, PendingCopy* pc = nullptr)
{
	uint64_t total = 0;
	ABB_CHECK(compute_slot_offsets(f->k, d_offs, n_reads, f->slot_offs, f->scan_tmp, f->stream, &total, &f->st.launches));
	if (n_kmers_out)
		*n_kmers_out = 0;
	if (total == 0)
		return ABB_OK;

	// chunk the reads so that the h0 staging buffer stays bounded
	std::vector<uint64_t> bounds;
	if (total <= kChunkSlots) {
		bounds = { 0, n_reads };
	} else {
		const unsigned max_chunks = (unsigned)(total / kChunkSlots + 3) * 2;
		// a member buffer: a cudaMalloc / cudaFree per call would synchronise the device, i.e. wait for the host-to-device copy
		// that abb_insert_reads runs next to this insert
		DevBuf<uint64_t>& d_bounds = f->bounds;
		ABB_CHECK(d_bounds.reserve(max_chunks + 2));
		k_chunk_bounds<<<1, 1, 0, f->stream>>>(f->slot_offs.p, n_reads, kChunkSlots, d_bounds.p, max_chunks,
		                                      (unsigned*)(d_bounds.p + max_chunks + 1));
		f->st.launches += 1;
		std::vector<uint64_t> h(max_chunks + 2);
		ABB_CUDA(cudaMemcpyAsync(h.data(), d_bounds.p, (max_chunks + 2) * sizeof(uint64_t), cudaMemcpyDeviceToHost, f->stream));
		ABB_CUDA(cudaStreamSynchronize(f->stream));
		unsigned nc = (unsigned)(h[max_chunks + 1] & 0xffffffffu);
		bounds.assign(h.begin(), h.begin() + nc + 1);
	}
	// per-chunk slot ranges need slot_offs at the chunk boundaries
	std::vector<uint64_t> slot_at(bounds.size());
	for (size_t i = 0; i < bounds.size(); ++i)
		ABB_CUDA(cudaMemcpyAsync(&slot_at[i], f->slot_offs.p + bounds[i], sizeof(uint64_t), cudaMemcpyDeviceToHost, f->stream));
	ABB_CUDA(cudaStreamSynchronize(f->stream));

	ABB_CUDA(cudaMemsetAsync(f->d_stats + 3, 0, sizeof(unsigned long long), f->stream));
	for (size_t c = 0; c + 1 < bounds.size(); ++c) {
		const uint64_t r0 = bounds[c], r1 = bounds[c + 1];
		const uint64_t slots = slot_at[c + 1] - slot_at[c];
		if (slots == 0)
			continue;
		ABB_CHECK(f->h0.reserve(slots));
		ABB_CHECK(f->valid.reserve(slots));
		if (pc)
			ABB_CHECK(wait_bases(f, pc, pc->h_offs[r1]));
		ABB_CUDA(cudaEventRecord(f->ev0, f->stream));
		ABB_CHECK(launch_hash(f, f->k, f->d_care, d_bases, d_offs, f->slot_offs.p, r0, r1, slot_at[c], f->h0.p, f->valid.p,
		                      f->stream, &f->st.launches));
		k_count_valid<<<std::min<unsigned>(blocks_for(slots, 256), 148 * 8), 256, 0, f->stream>>>(f->valid.p, slots, f->d_stats + 3);
		f->st.launches += 1;
		ABB_CUDA(cudaEventRecord(f->ev1, f->stream));
		if (comm)
			ABB_CHECK(sharded_ordered_insert(f, comm, f->h0.p, f->valid.p, slots));
		else
			ABB_CHECK(ordered_insert<false>(f, f->h0.p, f->valid.p, slots));
		cudaEvent_t ev2 = f->ev0; // reuse: record end of insert after reading the hash time
		ABB_CUDA(cudaEventSynchronize(f->ev1));
		float ms = 0;
		ABB_CUDA(cudaEventElapsedTime(&ms, f->ev0, f->ev1));
		f->st.ms_hash += ms;
		ABB_CUDA(cudaEventRecord(ev2, f->stream));
		ABB_CUDA(cudaEventSynchronize(ev2));
		ABB_CUDA(cudaEventElapsedTime(&ms, f->ev1, ev2));
		f->st.ms_insert += ms;
		f->st.slots += slots;
	}
	unsigned long long nk = 0;
	ABB_CUDA(cudaMemcpyAsync(&nk, f->d_stats + 3, sizeof nk, cudaMemcpyDeviceToHost, f->stream));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	f->st.kmers += nk;
	if (n_kmers_out)
		*n_kmers_out = nk;
	return ABB_OK;
}

// =============================================================================================
// multi-GPU: NCCL behind the C ABI (dlopen, no link-time dependency) and the sharded ordered insert
// =============================================================================================
struct NcclApi {
	void* h = nullptr;
	ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
	ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
	ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
	ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*GroupStart)() = nullptr;
	ncclResult_t (*GroupEnd)() = nullptr;
	const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

static int load_nccl()
{
	if (g_nccl.h)
		return ABB_OK;
	const char* names[] = { getenv("ABB_NCCL_LIB"), "libnccl.so.2", "libnccl.so" };
	void* h = nullptr;
	for (const char* n : names)
		if (n && *n && (h = dlopen(n, RTLD_NOW | RTLD_GLOBAL)))
			break;
	if (!h) {
		set_error("cannot load NCCL (libnccl.so.2): %s", dlerror());
		return ABB_ENODEV;
	}
#define ABB_NCCL_SYM(field, name)                                        \
	do {                                                                 \
		*(void**)(&g_nccl.field) = dlsym(h, name);                       \
		if (!g_nccl.field) {                                             \
			set_error("NCCL library lacks %s", name);                    \
			return ABB_ENODEV;                                           \
		}                                                                \
	} while (0)
	ABB_NCCL_SYM(GetUniqueId, "ncclGetUniqueId");
	ABB_NCCL_SYM(CommInitRank, "ncclCommInitRank");
	ABB_NCCL_SYM(CommDestroy, "ncclCommDestroy");
	ABB_NCCL_SYM(AllReduce, "ncclAllReduce");
	ABB_NCCL_SYM(AllGather, "ncclAllGather");
	ABB_NCCL_SYM(Send, "ncclSend");
	ABB_NCCL_SYM(Recv, "ncclRecv");
	ABB_NCCL_SYM(GroupStart, "ncclGroupStart");
	ABB_NCCL_SYM(GroupEnd, "ncclGroupEnd");
	ABB_NCCL_SYM(GetErrorString, "ncclGetErrorString");
#undef ABB_NCCL_SYM
	g_nccl.h = h;
	return ABB_OK;
}

#define ABB_NCCL(call)                                                                                   \
	do {                                                                                                 \
		ncclResult_t r__ = (call);                                                                       \
		if (r__ != ncclSuccess) {                                                                        \
			abb::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, g_nccl.GetErrorString(r__)); \
			return ABB_ECUDA;                                                                            \
		}                                                                                                \
	} while (0)

} // namespace abb

struct abb_comm {
	ncclComm_t comm = nullptr;
	int rank = 0, world = 1, device = 0;
};

namespace abb {

static uint64_t shard_chunk(uint64_t size, unsigned world) { return ((size + world - 1) / world + 15) & ~15ULL; }

/** the window of the sharded pipeline: per-rank conflict-map load like the single-GPU window */
static uint64_t sharded_window(const abb_filter* f, unsigned world)
{
	uint64_t w = 2 * f->window * world; // 2^18 slots per rank: the per-rank conflict-map load of the single-GPU window, twice
	if (const char* e = getenv("ABB_SHARD_WINDOW"))
		w = strtoull(e, nullptr, 10);
	return std::min<uint64_t>(std::max<uint64_t>(w, 32), 1ULL << 21);
}

static int sharded_ordered_insert(abb_filter* f, abb_comm* c, const uint64_t* d_h0, const uint8_t* d_valid, uint64_t n_slots)
{
	if (n_slots == 0)
		return ABB_OK;
	const uint64_t user_window = f->window;
	f->window = sharded_window(f, (unsigned)c->world);
	f->map_log2 = 27; // each rank marks window * H / world positions: 2^20 at the default window
	int rc = ensure_workspace(f);
	const uint64_t W = f->window;
	f->window = user_window;
	f->map_log2 = 0;
	ABB_CHECK(rc);
	// carried slots served per step: the tag table holds only own positions, so world times the single-GPU number fit
	const unsigned max_lanes = (unsigned)std::min<uint64_t>((uint64_t)kCarryLanes * (unsigned)c->world, W / 2 + kCarryLanes);
	ABB_CHECK(f->sh_buf.reserve(2 * (W + (uint64_t)max_lanes) + 64));
	cudaStream_t st = f->stream;
	const uint64_t n_windows = (n_slots + W - 1) / W;
	const unsigned age_off = (unsigned)(age_windows_for(W) * W);
	const unsigned drain_age = age_off / 3 * 2;
	const uint64_t cap = 3 * (W + kCarryLanes) / 2; // two lists in the allocation of three (no drain list is needed here)
	uint64_t* carry[2] = { f->d_carry, f->d_carry + cap };
	ShardCtl* ctl = reinterpret_cast<ShardCtl*>(f->d_ctl);
	unsigned* d_nout = f->d_ctl + 4; // [n_out]; the ctl block has 8 words
	const size_t map_bytes = std::max<size_t>(f->map_entries / 4, 256);
	ConflictMap maps[2] = { { f->d_map[0], f->map_entries - 1 }, { f->d_map[1], f->map_entries - 1 } };
	const uint64_t chunk = shard_chunk(f->size, (unsigned)c->world);
	Shard sh;
	sh.lo = std::min<uint64_t>(f->size, (uint64_t)c->rank * chunk);
	sh.hi = std::min<uint64_t>(f->size, sh.lo + chunk);
	{
		ShardCtl init;
		init.n_pending = 0;
		init.pad = 0;
		init.lo_pending = ~0ULL;
		ABB_CUDA(cudaMemcpyAsync(ctl, &init, sizeof init, cudaMemcpyHostToDevice, st));
		ABB_CUDA(cudaMemsetAsync(d_nout, 0, 4 * sizeof(unsigned), st));
	}
	ABB_CUDA(cudaMemsetAsync(f->d_map[0], 0, 3 * map_bytes, st)); // the maps start clean
	unsigned n_in = 0; // host copy of the carry length (identical on every rank)
	uint64_t oldest = 0;
	int in = 0, p = 0;
	uint8_t* buf = f->sh_buf.p;
	// one step of the pipeline: the oldest carried slots + the n new slots of [w0, w0 + n); marks [w1, w1 + n_next)
	auto step = [&](uint64_t w0, unsigned n, uint64_t w1, unsigned n_next) -> int {
		const unsigned lanes_c = std::min<unsigned>(n_in, max_lanes);
		// the tag table prefix this step uses (a rank reserves only the positions it owns: 1/world of them), cleared first
		uint64_t tslots = 4096;
		while (tslots < 8ULL * lanes_c * f->H / (unsigned)c->world + 4096 && tslots < f->tag_slots)
			tslots <<= 1;
		const TagTable tab = { f->d_tags2[0], std::min<uint64_t>(tslots, f->tag_slots) - 1 };
		if (lanes_c)
			ABB_CUDA(cudaMemsetAsync(tab.e, 0, (tab.mask + 1) * sizeof(unsigned long long), st));
		const unsigned lanes = lanes_c + n;
		const uint64_t lo_slot = w0 > (uint64_t)age_off + W ? w0 - age_off - W : 0;
		uint8_t* pm = buf;
		uint8_t* ok = buf + lanes;
		const bool timed = f->profile && n && (f->st.windows % f->prof_stride) == 0 && f->prof_used + 2 <= f->prof_ev.size();
		ABB_DISPATCH_H(f->H, {
			if (lanes_c)
				k_sh_mark_carry<false, MAXH><<<blocks_for(lanes_c, 256), 256, 0, st>>>(d_h0, carry[in], lanes_c, w0, f->cfg, tab, age_off, maps[p], sh);
			if (timed)
				cudaEventRecord(f->prof_ev[f->prof_used++], st);
			k_sh_gather<false, MAXH><<<blocks_for((uint64_t)lanes_c + std::max(n, n_next), 256), 256, 0, st>>>(
			    d_h0, d_valid, w0, n, w1, n_next, f->cfg, maps[p], maps[1 - p], tab, f->d_data, age_off, carry[in], lanes_c, sh, pm, ok);
		});
		if (lanes) {
			ABB_NCCL(g_nccl.AllReduce(buf, buf, 2 * (size_t)lanes, ncclUint8, ncclMin, c->comm, st));
			ABB_DISPATCH_H(f->H, (k_sh_apply<false, MAXH><<<blocks_for((uint64_t)n_in + n, 256), 256, 0, st>>>(
			                         d_h0, d_valid, w0, n, f->cfg, tab, f->d_data, carry[in], n_in, lanes_c, sh, pm, ok, f->d_slotbits, lo_slot, ctl,
			                         f->d_stats)));
			if (timed) {
				cudaEventRecord(f->prof_ev[f->prof_used++], st);
				f->prof_slots += n;
			}
			k_sh_compact<<<1, kDrainThreads, 0, st>>>(f->d_slotbits, lo_slot, w0 + std::max<uint64_t>(n, 1), carry[1 - in], ctl, d_nout);
			unsigned h_n = 0;
			ABB_CUDA(cudaMemcpyAsync(&h_n, d_nout, sizeof h_n, cudaMemcpyDeviceToHost, st));
			if (h_n || true) // the oldest pending slot bounds the priorities
				ABB_CUDA(cudaMemcpyAsync(&oldest, carry[1 - in], sizeof oldest, cudaMemcpyDeviceToHost, st));
			ABB_CUDA(cudaStreamSynchronize(st));
			n_in = h_n;
			in = 1 - in;
			f->st.launches += 4;
		} else {
			if (timed)
				f->prof_used--; // nothing was applied
			f->st.launches += 1;
		}
		return ABB_OK;
	};
	// everything pending is retired by steps without new slots (the oldest kCarryLanes take part in each)
	auto drain = [&](uint64_t w0, unsigned until) -> int {
		while (n_in > until) {
			ABB_CHECK(step(w0, 0, w0, 0));
			f->sh_drains += 1;
		}
		return ABB_OK;
	};
	f->prof_stride = f->prof_ev.empty() ? 1 : std::max<uint64_t>(1, (2 * n_windows + f->prof_ev.size() - 1) / f->prof_ev.size());
	PolicyHold policy(f, 2); // this path alternates between the first two maps
	ABB_CHECK(step(0, 0, 0, (unsigned)std::min<uint64_t>(W, n_slots))); // marks of window 0
	p = 1 - p; // the marks went to maps[1 - p]
	for (uint64_t w = 0; w < n_windows; ++w) {
		const uint64_t w0 = w * W;
		const unsigned n = (unsigned)std::min<uint64_t>(W, n_slots - w0);
		const uint64_t w1 = w0 + W;
		const unsigned n_next = w + 1 < n_windows ? (unsigned)std::min<uint64_t>(W, n_slots - w1) : 0u;
		if (n_in > max_lanes)
			ABB_CHECK(drain(w0, max_lanes / 2));
		if (n_in && w0 - oldest > drain_age)
			ABB_CHECK(drain(w0, 0));
		ABB_CHECK(step(w0, n, w1, n_next));
		ABB_CUDA(cudaMemsetAsync(maps[p].w, 0, map_bytes, st));
		p = 1 - p;
		f->st.windows += 1;
	}
	ABB_CHECK(drain(n_slots, 0));
	ABB_CUDA(cudaGetLastError());
	if (f->profile && f->prof_used) {
		ABB_CUDA(cudaStreamSynchronize(st));
		for (size_t i = 0; i + 1 < f->prof_used; i += 2) {
			float ms = 0;
			cudaEventElapsedTime(&ms, f->prof_ev[i], f->prof_ev[i + 1]);
			f->st.ms_commit += ms;
			f->st.commit_launches += 1;
		}
		f->st.commit_slots += f->prof_slots;
		f->prof_used = 0;
		f->prof_slots = 0;
	}
	// leave the shared control block in the single-GPU layout
	ABB_CUDA(cudaMemsetAsync(f->d_ctl, 0, 8 * sizeof(unsigned), st));
	return ABB_OK;
}

} // namespace abb

using namespace abb;

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int abb_version(void) { return ABB_VERSION; }
const char* abb_last_error(void) { return g_err; }

int abb_device_count(void)
{
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess) {
		set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
		return ABB_ENODEV;
	}
	return n;
}

int abb_filter_create(abb_filter** out, int kind, uint64_t size, unsigned num_hashes, unsigned k, unsigned arg,
                      const char* mask, int device)
{
	ABB_REQUIRE(out != nullptr, "abb_filter_create: out is NULL");
	*out = nullptr;
	ABB_REQUIRE(kind == ABB_COUNTING || kind == ABB_BIT || kind == ABB_CASCADING, "unknown filter kind %d", kind);
	ABB_REQUIRE(num_hashes >= 1 && num_hashes <= kMaxHashes, "number of hash functions must be in 1..%u (MAX_HASHES)", kMaxHashes);
	ABB_REQUIRE(k >= 1 && k <= kMaxK, "k-mer size must be in 1..%u (MAX_KMER)", kMaxK);
	if (kind == ABB_COUNTING) {
		// CountingBloomFilter ctor pads the byte size to a multiple of 8 (CountingBloomFilter.hpp:40-49)
		if (size % 8)
			size += 8 - size % 8;
	} else {
		// BloomFilter::initSize exits on this (BloomFilter.hpp:374-379)
		ABB_REQUIRE(size % 8 == 0, "ERROR: Filter Size \"%llu\" is not a multiple of 8.", (unsigned long long)size);
	}
	ABB_REQUIRE(size >= 8, "filter size must be at least 8");
	ABB_REQUIRE(size < (1ULL << kPosBits), "filter size %llu exceeds the supported maximum 2^%u", (unsigned long long)size, kPosBits);
	unsigned levels = 1;
	if (kind == ABB_CASCADING) {
		ABB_REQUIRE(arg >= 1 && arg <= 255, "cascading filter needs 1..255 levels");
		levels = arg;
	}
	std::string m = mask ? mask : "";
	if (!m.empty()) {
		// MaskedKmer::setMask (BloomDBG/MaskedKmer.h:38-55): k long, only 0/1
		ABB_REQUIRE(m.size() == k, "spaced seed must be exactly k=%u characters long", k);
		for (char c : m)
			ABB_REQUIRE(c == '0' || c == '1', "spaced seed must contain only '0' and '1'");
		if (m.find('0') == std::string::npos)
			m.clear(); // all ones == no mask
	}
	ABB_CHECK(select_device(device));

	abb_filter* f = new (std::nothrow) abb_filter();
	if (!f) {
		set_error("out of host memory");
		return ABB_ENOMEM;
	}
	f->device = device;
	f->kind = kind;
	f->size = size;
	f->bytes_per_level = kind == ABB_COUNTING ? size : size / 8;
	f->H = num_hashes;
	f->k = k;
	f->threshold = kind == ABB_COUNTING ? arg : 0;
	f->levels = levels;
	f->mask = m;
	f->window = kDefaultWindow;
	f->cfg.H = num_hashes;
	f->cfg.k = k;
	f->cfg.mod = make_fastmod(size);
	for (unsigned i = 0; i < kMaxHashes; ++i)
		f->cfg.mult[i] = (uint64_t)i ^ ((uint64_t)k * kMultiSeed); // nthash.hpp:339
	auto fail = [&](int rc) {
		abb_filter_destroy(f);
		return rc;
	};
#define ABB_TRY(call)                                                                 \
	do {                                                                              \
		cudaError_t e__ = (call);                                                     \
		if (e__ != cudaSuccess) {                                                     \
			set_error("%s failed: %s", #call, cudaGetErrorString(e__));               \
			return fail(e__ == cudaErrorMemoryAllocation ? ABB_ENOMEM : ABB_ECUDA);   \
		}                                                                             \
	} while (0)
	ABB_TRY(cudaStreamCreateWithFlags(&f->stream, cudaStreamNonBlocking));
	ABB_TRY(cudaEventCreate(&f->ev0));
	ABB_TRY(cudaEventCreate(&f->ev1));
	// slack: the in-place all-gather of position shards rounds each shard up to 16 bytes (abb_filter_allgather)
	ABB_TRY(cudaMalloc((void**)&f->d_data, f->bytes_per_level * levels + 4096));
	ABB_TRY(cudaMemsetAsync(f->d_data, 0, f->bytes_per_level * levels, f->stream));
	ABB_TRY(cudaMalloc((void**)&f->d_ctl, 8 * sizeof(unsigned)));
	ABB_TRY(cudaMemsetAsync(f->d_ctl, 0, 8 * sizeof(unsigned), f->stream));
	ABB_TRY(cudaMalloc((void**)&f->d_stats, 8 * sizeof(unsigned long long)));
	ABB_TRY(cudaMemsetAsync(f->d_stats, 0, 8 * sizeof(unsigned long long), f->stream));
	if (!f->mask.empty()) {
		std::vector<uint8_t> care(k);
		for (unsigned i = 0; i < k; ++i)
			care[i] = f->mask[i] == '1';
		ABB_TRY(cudaMalloc((void**)&f->d_care, k));
		ABB_TRY(cudaMemcpyAsync(f->d_care, care.data(), k, cudaMemcpyHostToDevice, f->stream));
	}
	ABB_TRY(cudaStreamSynchronize(f->stream));
#undef ABB_TRY
	*out = f;
	return ABB_OK;
}

int abb_filter_destroy(abb_filter* f)
{
	if (!f)
		return ABB_OK;
	cudaSetDevice(f->device);
	if (f->stream)
		cudaStreamSynchronize(f->stream);
	cudaFree(f->d_data);
	cudaFree(f->d_care);
	cudaFree(f->d_tags2[0]);
	cudaFree(f->d_tags2[1]);
	cudaFree(f->d_map[0]); // holds both maps
	cudaFree(f->d_carry);
	cudaFree(f->d_slotbits);
	cudaFree(f->d_ctl);
	cudaFree(f->d_stats);
	f->bases.release();
	f->offs.release();
	f->slot_offs.release();
	f->h0.release();
	f->lit.release();
	f->bounds.release();
	f->gq_kmers.release();
	f->gq_info.release();
	f->gq_len.release();
	f->gq_self.release();
	f->gq_nb.release();
	f->valid.release();
	f->scan_tmp.release();
	f->out8.release();
	f->sh_buf.release();
	for (auto e : f->prof_ev)
		cudaEventDestroy(e);
	if (f->ev0)
		cudaEventDestroy(f->ev0);
	if (f->ev1)
		cudaEventDestroy(f->ev1);
	for (auto e : f->copy_ev)
		cudaEventDestroy(e);
	if (f->copy_stream) {
		cudaStreamSynchronize(f->copy_stream);
		cudaStreamDestroy(f->copy_stream);
	}
	if (f->stream)
		cudaStreamDestroy(f->stream);
	delete f;
	return ABB_OK;
}

unsigned abb_filter_kmer_size(const abb_filter* f) { return f ? f->k : 0; }
unsigned abb_filter_hash_num(const abb_filter* f) { return f ? f->H : 0; }
uint64_t abb_filter_size(const abb_filter* f) { return f ? f->size : 0; }
uint64_t abb_filter_size_in_bytes(const abb_filter* f) { return f ? f->bytes_per_level : 0; }
unsigned abb_filter_threshold(const abb_filter* f) { return f ? f->threshold : 0; }
unsigned abb_filter_levels(const abb_filter* f) { return f ? f->levels : 0; }

int abb_filter_set_threshold(abb_filter* f, unsigned threshold)
{
	ABB_REQUIRE(f, "NULL filter");
	if (f->kind != ABB_COUNTING) {
		set_error("threshold only applies to counting filters");
		return ABB_ESTATE;
	}
	f->threshold = threshold;
	return ABB_OK;
}

int abb_filter_set_profiling(abb_filter* f, int on)
{
	ABB_REQUIRE(f, "NULL filter");
	ABB_CUDA(cudaSetDevice(f->device));
	f->profile = on != 0;
	if (f->profile && f->prof_ev.empty()) {
		f->prof_ev.resize(2048);
		for (auto& e : f->prof_ev)
			ABB_CUDA(cudaEventCreate(&e));
	}
	return ABB_OK;
}

int abb_filter_set_window(abb_filter* f, uint64_t window_slots)
{
	ABB_REQUIRE(f, "NULL filter");
	if (window_slots == 0)
		window_slots = kDefaultWindow;
	ABB_REQUIRE(window_slots >= 32 && window_slots <= (1ULL << 20) - 64, "window must be in [32, 2^20 - 64]");
	ABB_CUDA(cudaSetDevice(f->device));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	f->window = window_slots;
	return ABB_OK;
}

int abb_insert_reads_dev(abb_filter* f, const char* d_bases, const uint64_t* d_offsets, uint64_t n_reads,
                         uint64_t n_bases, uint64_t* n_kmers_out)
{
	(void)n_bases;
	ABB_REQUIRE(f, "NULL filter");
	ABB_REQUIRE(n_reads == 0 || (d_bases && d_offsets), "NULL read buffers");
	ABB_CUDA(cudaSetDevice(f->device));
	return insert_reads_dev(f, (const uint8_t*)d_bases, d_offsets, n_reads, n_kmers_out);
}

int abb_insert_reads(abb_filter* f, const char* bases, const uint64_t* offsets, uint64_t n_reads, uint64_t* n_kmers_out)
{
	ABB_REQUIRE(f, "NULL filter");
	if (n_kmers_out)
		*n_kmers_out = 0;
	if (n_reads == 0)
		return ABB_OK;
	ABB_REQUIRE(bases && offsets, "NULL read buffers");
	ABB_REQUIRE(offsets[0] == 0, "offsets[0] must be 0");
	const uint64_t n_bases = offsets[n_reads];
	ABB_CUDA(cudaSetDevice(f->device));
	ABB_CHECK(f->bases.reserve(n_bases + 16));
	ABB_CHECK(f->offs.reserve(n_reads + 1));
	ABB_CUDA(cudaMemcpyAsync(f->offs.p, offsets, (n_reads + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, f->stream));
	f->resident_reads = n_reads;
	// The bases travel in pieces on a second stream; chunk c of the insert only waits for the pieces that hold its reads, so
	// the copy of the rest hides behind the hashing and inserting of the earlier chunks (with pinned host memory; a pageable
	// buffer makes cudaMemcpyAsync synchronous and the order is simply copy, then insert).  ABB_H2D_OVERLAP=0: one copy up front.
	static int overlap = -1;
	if (overlap < 0) {
		const char* e = getenv("ABB_H2D_OVERLAP");
		overlap = e ? atoi(e) : 1;
	}
	constexpr uint64_t kPiece = 256ULL << 20;
	if (!overlap || n_bases <= kPiece) {
		ABB_CUDA(cudaMemcpyAsync(f->bases.p, bases, n_bases, cudaMemcpyHostToDevice, f->stream));
		return insert_reads_dev(f, f->bases.p, f->offs.p, n_reads, n_kmers_out);
	}
	if (!f->copy_stream)
		ABB_CUDA(cudaStreamCreateWithFlags(&f->copy_stream, cudaStreamNonBlocking));
	if (f->kind != ABB_BIT)
		ABB_CHECK(ensure_workspace(f)); // the maps exist before the policy that pins them is set
	PolicyHold policy(f, 3); // before the copy starts: setting it later would wait for the whole copy (see PolicyHold)
	PendingCopy pc;
	pc.h_offs = offsets;
	pc.piece = kPiece;
	pc.n_pieces = (size_t)((n_bases + kPiece - 1) / kPiece);
	while (f->copy_ev.size() < pc.n_pieces) {
		cudaEvent_t ev;
		ABB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
		f->copy_ev.push_back(ev);
	}
	// the destination may still be read by work queued on the filter's stream (pass 2 of a previous job)
	ABB_CUDA(cudaEventRecord(f->ev0, f->stream));
	ABB_CUDA(cudaStreamWaitEvent(f->copy_stream, f->ev0, 0));
	for (size_t i = 0; i < pc.n_pieces; ++i) {
		const uint64_t b0 = (uint64_t)i * kPiece, b1 = std::min<uint64_t>(n_bases, b0 + kPiece);
		ABB_CUDA(cudaMemcpyAsync(f->bases.p + b0, bases + b0, b1 - b0, cudaMemcpyHostToDevice, f->copy_stream));
		ABB_CUDA(cudaEventRecord(f->copy_ev[i], f->copy_stream));
	}
	const int rc = insert_reads_dev(f, f->bases.p, f->offs.p, n_reads, n_kmers_out, nullptr, &pc);
	// The last chunk waited for the last piece, so normally everything has landed; after an early return (no k-mers, an
	// error) the copy may still be running, and the caller owns the host buffer again once this call returns.
	ABB_CUDA(cudaStreamSynchronize(f->copy_stream));
	return rc;
}

/** true: the counters are sharded over the ranks; false: every rank runs the whole insert (see abb_insert_reads_sharded_dev) */
static bool shard_policy(int world)
{
	static int min_world = -1;
	if (min_world < 0) {
		const char* e = getenv("ABB_SHARD_MIN_WORLD");
		min_world = e ? std::max(2, atoi(e)) : 4;
	}
	return world > 1 && world >= min_world;
}

int abb_insert_reads_sharded(abb_filter* f, abb_comm* c, const char* bases, const uint64_t* offsets, uint64_t n_reads, int finalize,
                             uint64_t* n_kmers_out)
{
	ABB_REQUIRE(f && c, "NULL argument");
	if (!shard_policy(c->world)) { // replicated insert: the single-GPU host path, with its copy hidden behind the insert
		ABB_REQUIRE(f->kind == ABB_COUNTING, "the sharded insert is implemented for counting filters");
		ABB_REQUIRE(f->device == c->device, "filter and communicator live on different devices");
		f->replicated_insert = true;
		(void)finalize; // nothing to all-gather: every rank holds the whole filter
		return abb_insert_reads(f, bases, offsets, n_reads, n_kmers_out);
	}
	if (n_kmers_out)
		*n_kmers_out = 0;
	ABB_REQUIRE(n_reads == 0 || (bases && offsets), "NULL read buffers");
	ABB_REQUIRE(n_reads == 0 || offsets[0] == 0, "offsets[0] must be 0");
	ABB_CUDA(cudaSetDevice(f->device));
	if (n_reads) {
		const uint64_t n_bases = offsets[n_reads];
		ABB_CHECK(f->bases.reserve(n_bases + 16));
		ABB_CHECK(f->offs.reserve(n_reads + 1));
		ABB_CUDA(cudaMemcpyAsync(f->bases.p, bases, n_bases, cudaMemcpyHostToDevice, f->stream));
		ABB_CUDA(cudaMemcpyAsync(f->offs.p, offsets, (n_reads + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, f->stream));
	}
	f->resident_reads = n_reads;
	return abb_insert_reads_sharded_dev(f, c, (const char*)f->bases.p, f->offs.p, n_reads, finalize, n_kmers_out);
}

int abb_filter_resident_reads(abb_filter* f, const char** d_bases, const uint64_t** d_offsets, uint64_t* n_reads)
{
	ABB_REQUIRE(f && d_bases && d_offsets && n_reads, "NULL argument");
	*d_bases = (const char*)f->bases.p;
	*d_offsets = f->offs.p;
	*n_reads = f->resident_reads;
	return ABB_OK;
}

int abb_insert_hashes(abb_filter* f, const uint64_t* hashes, uint64_t n)
{
	ABB_REQUIRE(f, "NULL filter");
	if (n == 0)
		return ABB_OK;
	ABB_REQUIRE(hashes, "NULL hashes");
	ABB_CUDA(cudaSetDevice(f->device));
	ABB_CHECK(f->lit.reserve(n * f->H));
	ABB_CUDA(cudaMemcpyAsync(f->lit.p, hashes, n * f->H * sizeof(uint64_t), cudaMemcpyHostToDevice, f->stream));
	ABB_CHECK(ordered_insert<true>(f, f->lit.p, nullptr, n));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	f->st.kmers += n;
	return ABB_OK;
}

int abb_insert_h0_dev(abb_filter* f, const uint64_t* d_h0, uint64_t n)
{
	ABB_REQUIRE(f, "NULL filter");
	if (n == 0)
		return ABB_OK;
	ABB_REQUIRE(d_h0, "NULL hashes");
	ABB_CUDA(cudaSetDevice(f->device));
	ABB_CHECK(ordered_insert<false>(f, d_h0, nullptr, n));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	f->st.kmers += n;
	f->st.slots += n;
	return ABB_OK;
}

int abb_hash_reads_dev(abb_filter* f, const char* d_bases, const uint64_t* d_offsets, uint64_t n_reads, uint64_t* d_h0,
                       uint8_t* d_valid, uint64_t capacity, uint64_t* n_slots_out)
{
	ABB_REQUIRE(f, "NULL filter");
	if (n_slots_out)
		*n_slots_out = 0;
	if (n_reads == 0)
		return ABB_OK;
	ABB_REQUIRE(d_bases && d_offsets, "NULL read buffers");
	ABB_CUDA(cudaSetDevice(f->device));
	uint64_t total = 0;
	ABB_CHECK(compute_slot_offsets(f->k, d_offsets, n_reads, f->slot_offs, f->scan_tmp, f->stream, &total, &f->st.launches));
	if (n_slots_out)
		*n_slots_out = total;
	if (total == 0 || !d_h0 || !d_valid)
		return ABB_OK;
	ABB_REQUIRE(capacity >= total, "output buffers hold %llu slots, %llu needed", (unsigned long long)capacity, (unsigned long long)total);
	ABB_CHECK(launch_hash(f, f->k, f->d_care, (const uint8_t*)d_bases, d_offsets, f->slot_offs.p, 0, n_reads, 0, d_h0, d_valid, f->stream,
	                      &f->st.launches));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	return ABB_OK;
}

int abb_comm_unique_id(uint8_t id_out[128])
{
	ABB_REQUIRE(id_out, "NULL id buffer");
	ABB_CHECK(load_nccl());
	static_assert(sizeof(ncclUniqueId) == 128, "NCCL unique id size");
	ncclUniqueId id;
	ABB_NCCL(g_nccl.GetUniqueId(&id));
	memcpy(id_out, &id, sizeof id);
	return ABB_OK;
}

int abb_comm_create(abb_comm** out, int rank, int world, const uint8_t id[128], int device)
{
	ABB_REQUIRE(out && id, "NULL argument");
	*out = nullptr;
	ABB_REQUIRE(world >= 1 && world <= 64 && rank >= 0 && rank < world, "rank %d / world %d out of range", rank, world);
	ABB_CHECK(load_nccl());
	ABB_CHECK(select_device(device));
	abb_comm* c = new (std::nothrow) abb_comm();
	if (!c) {
		set_error("out of host memory");
		return ABB_ENOMEM;
	}
	c->rank = rank;
	c->world = world;
	c->device = device;
	ncclUniqueId nid;
	memcpy(&nid, id, sizeof nid);
	ncclResult_t r = g_nccl.CommInitRank(&c->comm, world, nid, rank);
	if (r != ncclSuccess) {
		set_error("ncclCommInitRank failed: %s", g_nccl.GetErrorString(r));
		delete c;
		return ABB_ECUDA;
	}
	*out = c;
	return ABB_OK;
}

int abb_comm_destroy(abb_comm* c)
{
	if (!c)
		return ABB_OK;
	cudaSetDevice(c->device);
	if (c->comm && g_nccl.CommDestroy)
		g_nccl.CommDestroy(c->comm);
	delete c;
	return ABB_OK;
}

int abb_comm_rank(const abb_comm* c) { return c ? c->rank : 0; }
int abb_comm_world(const abb_comm* c) { return c ? c->world : 1; }

int abb_filter_allgather(abb_filter* f, abb_comm* c)
{
	ABB_REQUIRE(f && c, "NULL argument");
	ABB_REQUIRE(f->levels == 1, "only single-level filters are sharded");
	ABB_CUDA(cudaSetDevice(f->device));
	if (c->world == 1 || f->replicated_insert)
		return ABB_OK;
	const uint64_t chunk = shard_chunk(f->bytes_per_level, (unsigned)c->world);
	ABB_REQUIRE(chunk * c->world <= f->bytes_per_level + 4096, "too many ranks for the all-gather slack");
	ABB_NCCL(g_nccl.AllGather(f->d_data + (uint64_t)c->rank * chunk, f->d_data, chunk, ncclUint8, c->comm, f->stream));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	return ABB_OK;
}

int abb_comm_allgather_bytes(abb_comm* c, void* d_buf, uint64_t bytes_per_rank, void* cuda_stream)
{
	ABB_REQUIRE(c && (d_buf || bytes_per_rank == 0), "NULL argument");
	if (c->world == 1 || bytes_per_rank == 0)
		return ABB_OK;
	ABB_CUDA(cudaSetDevice(c->device));
	ABB_NCCL(g_nccl.AllGather((const uint8_t*)d_buf + (uint64_t)c->rank * bytes_per_rank, d_buf, bytes_per_rank, ncclUint8, c->comm,
	                          (cudaStream_t)cuda_stream));
	return ABB_OK;
}

int abb_comm_exchange_bytes(abb_comm* c, const void* d_send, uint64_t send_bytes, void* d_recv_base, const uint64_t* recv_offsets,
                            const uint64_t* recv_bytes, void* cuda_stream)
{
	ABB_REQUIRE(c && recv_offsets && recv_bytes, "NULL argument");
	if (c->world == 1)
		return ABB_OK;
	ABB_CUDA(cudaSetDevice(c->device));
	cudaStream_t st = (cudaStream_t)cuda_stream;
	ABB_NCCL(g_nccl.GroupStart());
	for (int r = 0; r < c->world; ++r) {
		if (r == c->rank)
			continue;
		if (send_bytes)
			ABB_NCCL(g_nccl.Send(d_send, send_bytes, ncclUint8, r, c->comm, st));
		if (recv_bytes[r])
			ABB_NCCL(g_nccl.Recv((uint8_t*)d_recv_base + recv_offsets[r], recv_bytes[r], ncclUint8, r, c->comm, st));
	}
	ABB_NCCL(g_nccl.GroupEnd());
	return ABB_OK;
}

int abb_comm_allreduce_max_u8(abb_comm* c, void* d_buf, uint64_t n, void* cuda_stream)
{
	ABB_REQUIRE(c && (d_buf || n == 0), "NULL argument");
	if (c->world == 1 || n == 0)
		return ABB_OK;
	ABB_CUDA(cudaSetDevice(c->device));
	ABB_NCCL(g_nccl.AllReduce(d_buf, d_buf, n, ncclUint8, ncclMax, c->comm, (cudaStream_t)cuda_stream));
	return ABB_OK;
}

int abb_insert_reads_sharded_dev(abb_filter* f, abb_comm* c, const char* d_bases, const uint64_t* d_offsets, uint64_t n_reads,
                                 int finalize, uint64_t* n_kmers_out)
{
	ABB_REQUIRE(f && c, "NULL argument");
	ABB_REQUIRE(f->kind == ABB_COUNTING, "the sharded insert is implemented for counting filters");
	ABB_REQUIRE(n_reads == 0 || (d_bases && d_offsets), "NULL read buffers");
	ABB_REQUIRE(f->device == c->device, "filter and communicator live on different devices");
	ABB_CUDA(cudaSetDevice(f->device));
	// Policy: the position-sharded insert divides the counter traffic by the world size but every rank still evaluates every
	// lane and pays a collective per window; measured on B200 it beats one GPU only from 4 ranks on (pass 1 of the bench job:
	// 2.17 s on 1 GPU, 2.81 s sharded over 2, 1.78 s over 4).  Below ABB_SHARD_MIN_WORLD ranks (default 4) every rank
	// therefore runs the whole insert itself -- same bytes, no communication -- and only pass 2 is divided.
	const bool shard = shard_policy(c->world);
	f->replicated_insert = !shard;
	ABB_CHECK(insert_reads_dev(f, (const uint8_t*)d_bases, d_offsets, n_reads, n_kmers_out, shard ? c : nullptr));
	if (finalize)
		ABB_CHECK(abb_filter_allgather(f, c));
	return ABB_OK;
}

void* abb_filter_device_ptr(abb_filter* f, int level)
{
	if (!f)
		return nullptr;
	if (level < 0)
		level = (int)f->levels - 1;
	if ((unsigned)level >= f->levels)
		return nullptr;
	cudaSetDevice(f->device);
	cudaStreamSynchronize(f->stream);
	return f->d_data + (uint64_t)level * f->bytes_per_level;
}

static int query_hashes(abb_filter* f, const uint64_t* hashes, uint64_t n, uint8_t* out, bool want_min)
{
	ABB_REQUIRE(f, "NULL filter");
	if (n == 0)
		return ABB_OK;
	ABB_REQUIRE(hashes && out, "NULL buffer");
	ABB_CUDA(cudaSetDevice(f->device));
	ABB_CHECK(f->lit.reserve(n * f->H));
	ABB_CHECK(f->out8.reserve(n));
	ABB_CUDA(cudaMemcpyAsync(f->lit.p, hashes, n * f->H * sizeof(uint64_t), cudaMemcpyHostToDevice, f->stream));
	const FilterView fv = view_of(f);
	if (f->kind == ABB_COUNTING)
		k_query<0><<<blocks_for(n, 256), 256, 0, f->stream>>>(f->lit.p, n, f->cfg, fv, f->threshold, want_min ? nullptr : f->out8.p,
		                                                       want_min ? f->out8.p : nullptr);
	else
		k_query<1><<<blocks_for(n, 256), 256, 0, f->stream>>>(f->lit.p, n, f->cfg, fv, 0, want_min ? nullptr : f->out8.p,
		                                                       want_min ? f->out8.p : nullptr);
	f->st.launches += 1;
	ABB_CUDA(cudaGetLastError());
	ABB_CUDA(cudaMemcpyAsync(out, f->out8.p, n, cudaMemcpyDeviceToHost, f->stream));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	return ABB_OK;
}

int abb_contains_hashes(abb_filter* f, const uint64_t* hashes, uint64_t n, uint8_t* out) { return query_hashes(f, hashes, n, out, false); }
int abb_mincount_hashes(abb_filter* f, const uint64_t* hashes, uint64_t n, uint8_t* out) { return query_hashes(f, hashes, n, out, true); }

int abb_contains_reads(abb_filter* f, const char* bases, const uint64_t* offsets, uint64_t n_reads, uint8_t* out_flag, uint8_t* out_valid,
                       uint64_t capacity, uint64_t* n_slots_out)
{
	ABB_REQUIRE(f, "NULL filter");
	if (n_slots_out)
		*n_slots_out = 0;
	if (n_reads == 0)
		return ABB_OK;
	ABB_REQUIRE(bases && offsets, "NULL read buffers");
	ABB_REQUIRE(offsets[0] == 0, "offsets[0] must be 0");
	ABB_CUDA(cudaSetDevice(f->device));
	const uint64_t n_bases = offsets[n_reads];
	// own staging buffers: the batch a previous insert left resident (abb_filter_resident_reads) stays valid
	DevBuf<uint8_t> d_bases;
	DevBuf<uint64_t> d_offs;
	auto done = [&](int rc) {
		d_bases.release();
		d_offs.release();
		return rc;
	};
	int rc = d_bases.reserve(n_bases + 16);
	if (rc == ABB_OK)
		rc = d_offs.reserve(n_reads + 1);
	if (rc != ABB_OK)
		return done(rc);
	auto run = [&]() -> int {
		ABB_CUDA(cudaMemcpyAsync(d_bases.p, bases, n_bases, cudaMemcpyHostToDevice, f->stream));
		ABB_CUDA(cudaMemcpyAsync(d_offs.p, offsets, (n_reads + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, f->stream));
		uint64_t total = 0;
		ABB_CHECK(compute_slot_offsets(f->k, d_offs.p, n_reads, f->slot_offs, f->scan_tmp, f->stream, &total, &f->st.launches));
		if (n_slots_out)
			*n_slots_out = total;
		if (total == 0 || (!out_flag && !out_valid))
			return ABB_OK;
		ABB_REQUIRE(capacity >= total, "output buffers hold %llu slots, %llu needed", (unsigned long long)capacity, (unsigned long long)total);
		ABB_CHECK(f->h0.reserve(total));
		ABB_CHECK(f->valid.reserve(total));
		ABB_CHECK(f->out8.reserve(total));
		ABB_CHECK(launch_hash(f, f->k, f->d_care, d_bases.p, d_offs.p, f->slot_offs.p, 0, n_reads, 0, f->h0.p, f->valid.p, f->stream, &f->st.launches));
		const FilterView fv = view_of(f);
		const unsigned grid = std::min<unsigned>(blocks_for(total, 256), 148 * 16);
		if (f->kind == ABB_COUNTING)
			k_query_h0<0><<<grid, 256, 0, f->stream>>>(f->h0.p, f->valid.p, total, f->cfg, fv, f->threshold, f->out8.p);
		else
			k_query_h0<1><<<grid, 256, 0, f->stream>>>(f->h0.p, f->valid.p, total, f->cfg, fv, 0, f->out8.p);
		f->st.launches += 1;
		ABB_CUDA(cudaGetLastError());
		if (out_flag)
			ABB_CUDA(cudaMemcpyAsync(out_flag, f->out8.p, total, cudaMemcpyDeviceToHost, f->stream));
		if (out_valid)
			ABB_CUDA(cudaMemcpyAsync(out_valid, f->valid.p, total, cudaMemcpyDeviceToHost, f->stream));
		ABB_CUDA(cudaStreamSynchronize(f->stream));
		return ABB_OK;
	};
	rc = run();
	cudaStreamSynchronize(f->stream);
	return done(rc);
}

int abb_successors(abb_filter* f, const char* kmers, uint64_t n, unsigned max_chain, abb_succ_info* out, unsigned* out_len, uint64_t* self_hash)
{
	ABB_REQUIRE(f, "NULL filter");
	if (n == 0)
		return ABB_OK;
	ABB_REQUIRE(kmers && out && out_len && self_hash, "NULL buffer");
	ABB_REQUIRE(max_chain >= 1 && max_chain <= 128, "max_chain must be in 1..128");
	ABB_REQUIRE(f->mask.empty(), "graph neighbourhood queries are not available with a spaced seed");
	ABB_REQUIRE(f->H <= 64, "too many hash functions");
	ABB_CUDA(cudaSetDevice(f->device));
	DevBuf<uint8_t>& d_k = f->gq_kmers;
	DevBuf<abb_succ_info>& d_info = f->gq_info;
	DevBuf<unsigned>& d_len = f->gq_len;
	DevBuf<uint64_t>& d_self = f->gq_self;
	auto run = [&]() -> int {
		ABB_CHECK(d_k.reserve(n * f->k));
		ABB_CHECK(d_info.reserve(n * max_chain));
		ABB_CHECK(d_len.reserve(n));
		ABB_CHECK(d_self.reserve(n));
		ABB_CUDA(cudaMemcpyAsync(d_k.p, kmers, n * f->k, cudaMemcpyHostToDevice, f->stream));
		ABB_CUDA(cudaMemsetAsync(d_info.p, 0, n * max_chain * sizeof(abb_succ_info), f->stream));
		const FilterView fv = view_of(f);
		if (f->kind == ABB_COUNTING) {
			const FilterProbe<0> probe = { f->cfg, fv, f->threshold };
			k_successors<0><<<blocks_for(n, 128), 128, 0, f->stream>>>(d_k.p, n, f->k, max_chain, probe, d_info.p, d_len.p, d_self.p);
		} else {
			const FilterProbe<1> probe = { f->cfg, fv, 0 };
			k_successors<1><<<blocks_for(n, 128), 128, 0, f->stream>>>(d_k.p, n, f->k, max_chain, probe, d_info.p, d_len.p, d_self.p);
		}
		f->st.launches += 1;
		ABB_CUDA(cudaGetLastError());
		ABB_CUDA(cudaMemcpyAsync(out, d_info.p, n * max_chain * sizeof(abb_succ_info), cudaMemcpyDeviceToHost, f->stream));
		ABB_CUDA(cudaMemcpyAsync(out_len, d_len.p, n * sizeof(unsigned), cudaMemcpyDeviceToHost, f->stream));
		ABB_CUDA(cudaMemcpyAsync(self_hash, d_self.p, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, f->stream));
		ABB_CUDA(cudaStreamSynchronize(f->stream));
		return ABB_OK;
	};
	const int rc = run();
	cudaStreamSynchronize(f->stream);
	return rc;
}

int abb_neighbours(abb_filter* graph, abb_filter* const* attrs, unsigned n_attrs, const char* kmers, uint64_t n, abb_neighbourhood* out)
{
	abb_filter* const f = graph;
	ABB_REQUIRE(f, "NULL filter");
	ABB_REQUIRE(n_attrs <= 32, "at most 32 attribute filters, %u given", n_attrs);
	ABB_REQUIRE(n_attrs == 0 || attrs, "NULL attribute filter list");
	ABB_REQUIRE(f->mask.empty(), "graph neighbourhood queries are not available with a spaced seed");
	ABB_REQUIRE(f->kind != ABB_COUNTING, "the graph of `abyss-bloom graph' is a bit or cascading filter, not a counting filter");
	NbFilters F = {};
	auto add = [&](const abb_filter* a, unsigned j) {
		F.bits[j] = a->d_data + (uint64_t)(a->levels - 1) * a->bytes_per_level; // the last level: what the reference serialises
		F.mod[j] = a->cfg.mod;
		F.H[j] = a->H;
		F.start[j + 1] = F.start[j] + 9 * a->H;
	};
	add(f, 0);
	for (unsigned j = 0; j < n_attrs; ++j) {
		const abb_filter* a = attrs[j];
		ABB_REQUIRE(a, "NULL attribute filter %u", j);
		ABB_REQUIRE(a->kind != ABB_COUNTING, "attribute filter %u is a counting filter", j);
		ABB_REQUIRE(a->device == f->device, "attribute filter %u is on device %d, the graph on %d", j, a->device, f->device);
		ABB_REQUIRE(a->H <= f->H, "attribute filter %u has %u hash functions, more than the graph's %u (it is probed with the graph's hash values)",
		            j, a->H, f->H);
		add(a, 1 + j);
	}
	F.n = 1 + n_attrs;
	for (unsigned i = 0; i < kMaxHashes; ++i)
		F.mult[i] = f->cfg.mult[i];
	if (n == 0)
		return ABB_OK;
	ABB_REQUIRE(kmers && out, "NULL buffer");
	ABB_CUDA(cudaSetDevice(f->device));
	DevBuf<uint8_t>& d_k = f->gq_kmers;
	DevBuf<abb_neighbourhood>& d_nb = f->gq_nb;
	auto run = [&]() -> int {
		ABB_CHECK(d_k.reserve(n * f->k));
		ABB_CHECK(d_nb.reserve(n));
		ABB_CUDA(cudaMemcpyAsync(d_k.p, kmers, n * f->k, cudaMemcpyHostToDevice, f->stream));
		k_neighbours<<<blocks_for(n, kNbWarps), 32 * kNbWarps, 0, f->stream>>>(d_k.p, n, f->k, F, d_nb.p);
		f->st.launches += 1;
		ABB_CUDA(cudaGetLastError());
		ABB_CUDA(cudaMemcpyAsync(out, d_nb.p, n * sizeof(abb_neighbourhood), cudaMemcpyDeviceToHost, f->stream));
		ABB_CUDA(cudaStreamSynchronize(f->stream));
		return ABB_OK;
	};
	const int rc = run();
	cudaStreamSynchronize(f->stream);
	return rc;
}

int abb_hash_reads(unsigned k, const char* mask, const char* bases, const uint64_t* offsets, uint64_t n_reads,
                   uint64_t* out_h0, uint8_t* out_valid, uint64_t* n_slots_out, int device)
{
	ABB_REQUIRE(k >= 1 && k <= kMaxK, "k-mer size must be in 1..%u", kMaxK);
	if (n_slots_out)
		*n_slots_out = 0;
	if (n_reads == 0)
		return ABB_OK;
	ABB_REQUIRE(bases && offsets, "NULL read buffers");
	ABB_CHECK(select_device(device));
	std::string m = mask ? mask : "";
	if (!m.empty()) {
		ABB_REQUIRE(m.size() == k, "spaced seed must be exactly k=%u characters long", k);
		if (m.find('0') == std::string::npos)
			m.clear();
	}
	const uint64_t n_bases = offsets[n_reads];
	DevBuf<uint8_t> d_bases, d_valid, tmp, d_care;
	DevBuf<uint64_t> d_offs, d_slot, d_h0;
	int rc = ABB_OK;
	auto cleanup = [&]() {
		d_bases.release(); d_valid.release(); tmp.release(); d_care.release();
		d_offs.release(); d_slot.release(); d_h0.release();
	};
#define ABB_TRYRC(expr) do { rc = (expr); if (rc != ABB_OK) { cleanup(); return rc; } } while (0)
	auto cu = [&](cudaError_t e, const char* what) {
		if (e != cudaSuccess) { set_error("%s: %s", what, cudaGetErrorString(e)); return (int)ABB_ECUDA; }
		return (int)ABB_OK;
	};
	ABB_TRYRC(d_bases.reserve(n_bases + 16));
	ABB_TRYRC(d_offs.reserve(n_reads + 1));
	ABB_TRYRC(cu(cudaMemcpy(d_bases.p, bases, n_bases, cudaMemcpyHostToDevice), "H2D bases"));
	ABB_TRYRC(cu(cudaMemcpy(d_offs.p, offsets, (n_reads + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice), "H2D offsets"));
	if (!m.empty()) {
		std::vector<uint8_t> care(k);
		for (unsigned i = 0; i < k; ++i)
			care[i] = m[i] == '1';
		ABB_TRYRC(d_care.reserve(k));
		ABB_TRYRC(cu(cudaMemcpy(d_care.p, care.data(), k, cudaMemcpyHostToDevice), "H2D mask"));
	}
	uint64_t total = 0;
	ABB_TRYRC(compute_slot_offsets(k, d_offs.p, n_reads, d_slot, tmp, 0, &total, nullptr));
	if (n_slots_out)
		*n_slots_out = total;
	if (total && out_h0 && out_valid) {
		ABB_TRYRC(d_h0.reserve(total));
		ABB_TRYRC(d_valid.reserve(total));
		ABB_TRYRC(launch_hash(nullptr, k, m.empty() ? nullptr : d_care.p, d_bases.p, d_offs.p, d_slot.p, 0, n_reads, 0, d_h0.p,
		                      d_valid.p, 0, nullptr));
		ABB_TRYRC(cu(cudaMemcpy(out_h0, d_h0.p, total * sizeof(uint64_t), cudaMemcpyDeviceToHost), "D2H h0"));
		ABB_TRYRC(cu(cudaMemcpy(out_valid, d_valid.p, total, cudaMemcpyDeviceToHost), "D2H valid"));
	}
#undef ABB_TRYRC
	cleanup();
	return ABB_OK;
}

static int level_ptr(abb_filter* f, int level, uint64_t nbytes, uint8_t** p)
{
	ABB_REQUIRE(f, "NULL filter");
	if (level < 0)
		level = (int)f->levels - 1;
	ABB_REQUIRE((unsigned)level < f->levels, "level %d out of range", level);
	ABB_REQUIRE(nbytes == f->bytes_per_level, "buffer is %llu bytes, the filter level is %llu", (unsigned long long)nbytes,
	            (unsigned long long)f->bytes_per_level);
	*p = f->d_data + (uint64_t)level * f->bytes_per_level;
	return ABB_OK;
}

int abb_filter_download(abb_filter* f, int level, uint8_t* host, uint64_t nbytes)
{
	uint8_t* p = nullptr;
	ABB_CHECK(level_ptr(f, level, nbytes, &p));
	ABB_REQUIRE(host, "NULL buffer");
	ABB_CUDA(cudaSetDevice(f->device));
	ABB_CUDA(cudaMemcpyAsync(host, p, nbytes, cudaMemcpyDeviceToHost, f->stream));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	return ABB_OK;
}

int abb_filter_upload(abb_filter* f, int level, const uint8_t* host, uint64_t nbytes)
{
	uint8_t* p = nullptr;
	ABB_CHECK(level_ptr(f, level, nbytes, &p));
	ABB_REQUIRE(host, "NULL buffer");
	ABB_CUDA(cudaSetDevice(f->device));
	ABB_CUDA(cudaMemcpyAsync(p, host, nbytes, cudaMemcpyHostToDevice, f->stream));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	return ABB_OK;
}

int abb_filter_clear(abb_filter* f)
{
	ABB_REQUIRE(f, "NULL filter");
	ABB_CUDA(cudaSetDevice(f->device));
	ABB_CUDA(cudaMemsetAsync(f->d_data, 0, f->bytes_per_level * f->levels, f->stream));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	return ABB_OK;
}

int abb_filter_popcount(abb_filter* f, uint64_t* nonzero, uint64_t* at_or_above_threshold)
{
	ABB_REQUIRE(f, "NULL filter");
	ABB_CUDA(cudaSetDevice(f->device));
	ABB_CUDA(cudaMemsetAsync(f->d_stats + 4, 0, 2 * sizeof(unsigned long long), f->stream));
	// bit / cascading: population of the LAST level (the one contains() consults)
	const uint8_t* p = f->d_data + (uint64_t)(f->levels - 1) * f->bytes_per_level;
	k_popcount<<<148 * 8, 256, 0, f->stream>>>(p, f->bytes_per_level, f->kind == ABB_COUNTING, f->threshold, f->d_stats + 4);
	f->st.launches += 1;
	ABB_CUDA(cudaGetLastError());
	unsigned long long h[2] = { 0, 0 };
	ABB_CUDA(cudaMemcpyAsync(h, f->d_stats + 4, sizeof h, cudaMemcpyDeviceToHost, f->stream));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	if (nonzero)
		*nonzero = h[0];
	if (at_or_above_threshold)
		*at_or_above_threshold = f->kind == ABB_COUNTING ? h[1] : h[0];
	return ABB_OK;
}

void* abb_filter_stream(abb_filter* f) { return f ? (void*)f->stream : nullptr; }

int abb_filter_insert_stats(abb_filter* f, abb_insert_stats* out, int reset)
{
	ABB_REQUIRE(f, "NULL filter");
	ABB_CUDA(cudaSetDevice(f->device));
	unsigned long long h[3] = { 0, 0, 0 };
	ABB_CUDA(cudaMemcpyAsync(h, f->d_stats, sizeof h, cudaMemcpyDeviceToHost, f->stream));
	ABB_CUDA(cudaStreamSynchronize(f->stream));
	f->st.deferred = h[0];
	f->st.drains = h[1] + f->sh_drains;
	f->st.drained_slots = h[2];
	if (out)
		*out = f->st;
	if (reset) {
		f->sh_drains = 0;
		f->st = abb_insert_stats{};
		ABB_CUDA(cudaMemsetAsync(f->d_stats, 0, 3 * sizeof(unsigned long long), f->stream));
	}
	return ABB_OK;
}

} // extern "C"
