// abb_common.h -- host-side plumbing shared by the C-ABI translation units.
#pragma once
#include "../../include/abyss_b200.h"
#include "abb_device.cuh"
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdio>
#include <string>
#include <vector>

namespace abb {

void set_error(const char* fmt, ...);

#define ABB_CUDA(call)                                                                             \
	do {                                                                                           \
		cudaError_t e__ = (call);                                                                  \
		if (e__ != cudaSuccess) {                                                                  \
			abb::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
			return (e__ == cudaErrorMemoryAllocation) ? ABB_ENOMEM                                 \
			       : (e__ == cudaErrorNoDevice || e__ == cudaErrorInsufficientDriver) ? ABB_ENODEV \
			                                                                          : ABB_ECUDA; \
		}                                                                                          \
	} while (0)

#define ABB_CHECK(expr)            \
	do {                           \
		int rc__ = (expr);         \
		if (rc__ != ABB_OK)        \
			return rc__;           \
	} while (0)

#define ABB_REQUIRE(cond, ...)         \
	do {                               \
		if (!(cond)) {                 \
			abb::set_error(__VA_ARGS__); \
			return ABB_EINVAL;         \
		}                              \
	} while (0)

/** growable device buffer */
template <typename T>
struct DevBuf {
	T* p = nullptr;
	size_t cap = 0;
	int reserve(size_t n)
	{
		if (n <= cap)
			return ABB_OK;
		if (p)
			cudaFree(p);
		p = nullptr;
		cap = 0;
		size_t want = n + n / 8 + 256;
		ABB_CUDA(cudaMalloc((void**)&p, want * sizeof(T)));
		cap = want;
		return ABB_OK;
	}
	void release()
	{
		if (p)
			cudaFree(p);
		p = nullptr;
		cap = 0;
	}
};

inline unsigned blocks_for(uint64_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

// host helpers implemented in abb_api.cu, shared with abb_assemble.cu
int select_device(int device);
/** slot_offs[0..n_reads] = exclusive prefix sum of per-read k-mer window counts; *total = sum */
int compute_slot_offsets(unsigned k, const uint64_t* d_offs, uint64_t n_reads, DevBuf<uint64_t>& slot_offs,
                         DevBuf<uint8_t>& tmp, cudaStream_t stream, uint64_t* total, uint64_t* launches);

} // namespace abb

struct abb_filter;
namespace abb {
/** K1 for reads [r0, r1): h0/valid index = slot_offs[r] + j - slot_base */
int launch_hash(abb_filter* f, unsigned k, const uint8_t* d_care, const uint8_t* d_bases, const uint64_t* d_offs,
                const uint64_t* d_slot_offs, uint64_t r0, uint64_t r1, uint64_t slot_base, uint64_t* d_h0, uint8_t* d_valid,
                cudaStream_t stream, uint64_t* launches);
int launch_hash_segments(unsigned k, const uint8_t* d_care, const uint8_t* d_bases, const uint64_t* d_seg_beg, const unsigned* d_seg_len,
                         const uint64_t* d_seg_slot, uint64_t n_segs, uint64_t* d_h0, uint8_t* d_valid, cudaStream_t stream);
}

/** The filter handle (opaque in the C ABI). */
struct abb_filter {
	int device = 0;
	int kind = ABB_COUNTING;
	uint64_t size = 0;            // counters, or bits per level
	uint64_t bytes_per_level = 0; // bytes of one level
	unsigned H = 0, k = 0, threshold = 0, levels = 1;
	std::string mask;
	uint8_t* d_care = nullptr; // k bytes (mask == '1'), only with a spaced seed
	uint8_t* d_data = nullptr;
	abb::HashCfg cfg;
	cudaStream_t stream = nullptr;
	cudaEvent_t ev0 = nullptr, ev1 = nullptr;
	// host-buffer insert: the bases travel in pieces on their own stream while earlier chunks are hashed and inserted
	cudaStream_t copy_stream = nullptr;
	std::vector<cudaEvent_t> copy_ev; // copy_ev[i]: piece i has landed

	// ordered-insert workspace (abb_insert.cuh K2)
	uint64_t window = 0;      // slots per window
	uint64_t ws_window = 0;   // window the workspace below was sized for
	unsigned ws_H = 0;
	uint64_t map_entries = 0; // two-bit entries per conflict map (power of two)
	unsigned map_log2 = 0;    // 0 = default size
	unsigned* d_map[3] = { nullptr, nullptr, nullptr }; // one allocation
	unsigned long long* d_tags2[2] = { nullptr, nullptr }; // tag tables of the carried slots (alternating windows)
	uint64_t tag_slots = 0;
	uint64_t* d_carry = nullptr;    // two carry lists and the drain's sorted list, (window + kCarryLanes) slots each
	unsigned* d_slotbits = nullptr; // presence bitmap of the drain
	uint64_t slotbit_words = 0;
	unsigned* d_ctl = nullptr;             // abb::InsertCtl
	unsigned long long* d_stats = nullptr; // [0] deferred [1] drains [2] slots replayed by drains [3..4] popcount scratch

	// per-call buffers (bases/offs keep the device copy of the last host batch: abb_filter_resident_reads)
	uint64_t resident_reads = 0;
	bool l2_policy_held = false;    // an enclosing scope already pinned the conflict maps in L2 (abb_api.cu PolicyHold)
	bool replicated_insert = false; // the last "sharded" insert ran replicated (small worlds): nothing to all-gather
	abb::DevBuf<uint8_t> bases;
	abb::DevBuf<uint64_t> offs, slot_offs, h0, lit, bounds;
	abb::DevBuf<uint8_t> valid, scan_tmp, out8, sh_buf;
	// abb_successors staging (a graph dump issues thousands of small queries: no allocation per call)
	abb::DevBuf<uint8_t> gq_kmers;
	abb::DevBuf<abb_succ_info> gq_info;
	abb::DevBuf<unsigned> gq_len;
	abb::DevBuf<uint64_t> gq_self;
	abb::DevBuf<abb_neighbourhood> gq_nb; // abb_neighbours results (the k-mers go through gq_kmers)

	// statistics
	abb_insert_stats st = {};
	bool profile = false; // time the k_window launches with CUDA events (every prof_stride-th window)
	uint64_t prof_stride = 1, prof_slots = 0, sh_drains = 0;
	std::vector<cudaEvent_t> prof_ev;
	size_t prof_used = 0;
};
