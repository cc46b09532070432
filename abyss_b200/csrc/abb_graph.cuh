// abb_graph.cuh -- out-edges of de Bruijn graph vertices for the GraphViz dump `-g` (outputGraph, BloomDBG/bloom-dbg.h:1171-1242),
// and the neighbourhoods `abyss-bloom graph` expands (Bloom/bloom.cc:983-1153).
// Shared by the CUDA kernels k_successors / k_neighbours (abb_insert.cuh) and the CPU test harnesses (tests/host_graph,
// tests/host_bloom_graph).
#pragma once
#include "../../include/abyss_b200.h"
#include "abb_device.cuh"

namespace abb {

/** RollingBloomDBG::out_edge_iterator (BloomDBG/RollingBloomDBG.h:300-360): shift the k-mer left, try A, C, G, T as the last base,
 *  keep those the filter contains (`probe(canonical hash)`).  While a vertex has exactly one out-edge the walk moves on to that
 *  successor, up to max_chain (<= 128) vertices: unbranched paths -- nearly all of a genome's graph -- cost one query per
 *  max_chain vertices instead of one per vertex.  out[s] = out-edges of the s-th vertex of the chain (s = 0: the k-mer itself):
 *  mask bit b = the successor with base b exists, hash[b] = its canonical hash (vertex identity: RollingBloomDBGVertex compares
 *  canonical k-mers).  *self = canonical hash of the start k-mer.  Returns the number of vertices expanded. */
template <typename Probe>
ABB_HD unsigned successors_chain(const uint8_t* km, unsigned k, unsigned max_chain, const Probe& probe, abb_succ_info* out, uint64_t* self)
{
	const RollTab rt = make_rolltab(k);
	HashPair h = { 0, 0 }; // NTC64 from scratch (nthash.hpp:268-272)
	for (unsigned t = 0; t < k; ++t) {
		const unsigned c = base_code(km[t]) & 3u;
		h.fh = srol1(h.fh) ^ seed_of(c);
		h.rh ^= srol_n(seed_of(3 - c), t);
	}
	*self = h.canonical();
	unsigned appended[8] = { 0, 0, 0, 0, 0, 0, 0, 0 }; // bases appended so far, 2 bits each
	unsigned s = 0;
	while (s < max_chain) {
		// the base that leaves on this shift: from the start k-mer while it lasts, then from the appended bases
		const unsigned first = s < k ? base_code(km[s]) & 3u : (appended[(s - k) >> 4] >> (2 * ((s - k) & 15))) & 3u;
		unsigned mask = 0;
		for (unsigned b = 0; b < 4; ++b) {
			const uint64_t h0 = roll_right(h, rt, first, b).canonical();
			out[s].hash[b] = h0;
			if (probe(h0))
				mask |= 1u << b;
		}
		out[s].mask = (uint8_t)mask;
		++s;
		if ((mask & (mask - 1)) != 0 || mask == 0 || s == max_chain)
			break;
		unsigned nb = 0;
		while (!((mask >> nb) & 1))
			++nb;
		h = roll_right(h, rt, first, nb);
		appended[(s - 1) >> 4] |= nb << (2 * ((s - 1) & 15));
	}
	return s;
}

/** The two ntHash seeds of any character (nthash.hpp:29-64): seedTab[c] on the forward strand and, for the complement,
 *  seedTab[c & cpOff] with cpOff = 7.  A, C, G, T of either case get their own seeds and U counts as T; 'N' and the other
 *  characters hash as 0 forward, while on the reverse strand their low three bits pick the seed.  A `-R` root of
 *  `abyss-bloom graph` is hashed as given, without case folding or validation, so this is what its bytes decide. */
ABB_HD uint64_t rc_seed(unsigned char c) { return seed_of((0x14002434u >> (4 * (c & 7u))) & 0xFu); }
ABB_HD uint64_t fwd_seed(unsigned char c)
{
	if (c < 8)
		return rc_seed(c); // seedTab[0..7] is the cpOff row
	return seed_of((c & 0xDFu) == 'U' ? 3u : base_code(c));
}

/** A k-mer and its 8 neighbours, the vertices the reference's undirected breadth-first search looks at when it expands a
 *  vertex (Graph/BreadthFirstSearch.h:139-154): out_edge_iterator shifts left and tries A, C, G, T as the last base,
 *  in_edge_iterator shifts right and tries them as the first base (BloomDBG/RollingBloomDBG.h:300-453).  hash[0] = the
 *  canonical hash of the k-mer, hash[1 + b] of its successor with last base b, hash[5 + b] of its predecessor with first base b.
 *  The leaving base may be any character, so the rolls are written out with its two seeds (roll_right / roll_left with the
 *  seeds of a code; nthash.hpp:242-257,282-297).  probe(hash, &mask, attr) fills the graph membership mask (bit v = vertex v)
 *  and the per-vertex attribute bits. */
template <typename Probe>
ABB_HD void neighbourhood(const uint8_t* km, unsigned k, const Probe& probe, abb_neighbourhood* out)
{
	HashPair h = { 0, 0 }; // NTF64 / NTR64 from scratch (nthash.hpp:220-239)
	for (unsigned t = 0; t < k; ++t) {
		h.fh = srol1(h.fh) ^ fwd_seed(km[t]);
		h.rh ^= srol_n(rc_seed(km[t]), t);
	}
	const RollTab rt = make_rolltab(k);
	const uint64_t firstF = srol_n(fwd_seed(km[0]), k), firstR = rc_seed(km[0]);      // leaves on a shift left
	const uint64_t lastF = fwd_seed(km[k - 1]), lastR = srol_n(rc_seed(km[k - 1]), k); // leaves on a shift right
	uint64_t hash[9];
	hash[0] = h.canonical();
#pragma unroll
	for (unsigned b = 0; b < 4; ++b) {
		const HashPair o = { srol1(h.fh) ^ seed_of(b) ^ firstF, sror1(h.rh ^ rt.rk[3 - b] ^ firstR) };
		const HashPair i = { sror1(h.fh ^ rt.rk[b] ^ lastF), srol1(h.rh) ^ seed_of(3 - b) ^ lastR };
		hash[1 + b] = o.canonical();
		hash[5 + b] = i.canonical();
	}
	unsigned mask = 0;
	probe(hash, &mask, out->attr);
	out->mask = (uint16_t)mask;
#pragma unroll
	for (unsigned v = 0; v < 9; ++v)
		out->hash[v] = hash[v];
}

} // namespace abb
