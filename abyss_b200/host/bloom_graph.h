// bloom_graph.h -- `abyss-bloom graph`: the GraphViz neighbourhood of root k-mers in the de Bruijn graph of a rolling-hash
// Bloom filter (Bloom/bloom.cc:983-1153, visitor Bloom/RollingBloomDBGVisitor.h, search Graph/BreadthFirstSearch.h:100-173
// with undirected = true).  The reference's order on the host, the Bloom lookups behind functors: abyss_bloom.cc passes the
// C ABI (abb_hash_reads, abb_contains_reads, abb_neighbours: CUDA), the CPU test harness (tests/host_bloom_graph) an
// emulation built on the same device functions.
//
// Kept apart from graph_dump.h (`abyss-bloom-dbg -g`): that search walks directed edges from trimmed reads, has no depth
// and caches unbranched chains; this one walks both edge directions from a root set, level by level, to a depth.
#pragma once
#include "../../include/abyss_b200.h"
#include "reads.h"
#include <iostream>
#include <unordered_set>

namespace host {

struct BloomGraphOpts {
	unsigned k = 0;
	unsigned depth = 0;
	int verbose = 0;
	std::vector<std::string> roots;                               // -R, as given (neither case-folded nor checked)
	std::vector<std::string> rootFastas;                          // -f
	std::vector<std::pair<std::string, std::string>> fastaAttrs;  // -a STR:FASTA
	std::vector<std::string> bloomAttrs;                          // -A STR (the filters themselves sit behind the query)
};

/** A root vertex: the string it was first inserted with and its canonical ntHash.  The reference keeps its roots in a
 *  std::unordered_set<RollingBloomDBGVertex> whose hasher is the canonical hash (RollingBloomDBG.h:163-172) and whose
 *  equality is canonical k-mer identity; a libstdc++ unordered_set iterates in an order fixed by the hash codes, the
 *  insertion sequence and the prime rehash policy, so a set with the same hasher filled in the same sequence iterates
 *  in the same order.  Equal canonical hashes stand for equal canonical k-mers (a collision has probability 2^-64). */
struct GraphRoot {
	std::string kmer;
	uint64_t h0;
};
struct GraphRootHash {
	size_t operator()(const GraphRoot& r) const { return (size_t)r.h0; }
};
struct GraphRootEq {
	bool operator()(const GraphRoot& a, const GraphRoot& b) const { return a.h0 == b.h0; }
};

/** for_each_batch(path, fn): fn(const ReadBatch&) for each batch of the FASTA at path (FastaReader(FOLD_CASE) options);
 *  hash_reads(bases, offsets, n, h0, valid): abb_hash_reads; contains_reads(bases, offsets, n, flag, capacity): graph
 *  membership of every window (abb_contains_reads); neighbours(kmers, n, out): abb_neighbours with the -A filters in option order. */
template <typename BatchesFn, typename HashFn, typename ContainsFn, typename NbFn>
void bloom_graph(const BloomGraphOpts& o, BatchesFn for_each_batch, HashFn hash_reads, ContainsFn contains_reads, NbFn neighbours,
                 std::ostream& os)
{
	static const char BASES[] = "ACGT";
	const unsigned k = o.k;
	std::vector<uint64_t> h0;
	std::vector<uint8_t> valid, flag;
	// the hash and validity of every window of a batch, slots numbered as abb_hash_reads numbers them
	auto hash_batch = [&](const ReadBatch& b) {
		uint64_t slots = 0;
		for (size_t i = 0; i < b.size(); ++i) {
			const uint64_t L = b.offsets[i + 1] - b.offsets[i];
			slots += L >= k ? L - k + 1 : 0;
		}
		h0.resize(slots + 1);
		valid.resize(slots + 1);
		hash_reads(b.bases.data(), b.offsets.data(), b.size(), h0.data(), valid.data());
		return slots;
	};

	// -a: the k-mers of each FASTA (bloom.cc:1068-1097; only the vertices the search discovers are looked up, all of which
	// the graph contains, so the reference's vertex_exists filter on these sets changes nothing)
	std::vector<std::unordered_set<uint64_t>> fastaSets(o.fastaAttrs.size());
	for (size_t a = 0; a < o.fastaAttrs.size(); ++a) {
		if (o.verbose)
			std::cerr << "Loading k-mers from `" << o.fastaAttrs[a].second << "', to be annotated with '" << o.fastaAttrs[a].first << "'\n";
		size_t count = 0;
		for_each_batch(o.fastaAttrs[a].second, [&](const ReadBatch& b) {
			const uint64_t slots = hash_batch(b);
			for (uint64_t s = 0; s < slots; ++s)
				if (valid[s]) {
					fastaSets[a].insert(h0[s]);
					++count;
				}
		});
		if (o.verbose)
			std::cerr << "Loaded " << count << " k-mers in total\n";
	}

	// the root set, filled in the reference's sequence (bloom.cc:1116-1140): -R in option order, then every k-mer of every -f
	std::unordered_set<GraphRoot, GraphRootHash, GraphRootEq> roots;
	std::vector<abb_neighbourhood> nb;
	std::string kbuf;
	if (!o.roots.empty()) {
		kbuf.clear();
		for (const std::string& r : o.roots)
			kbuf += r;
		nb.resize(o.roots.size());
		neighbours(kbuf.data(), o.roots.size(), nb.data());
		for (size_t i = 0; i < o.roots.size(); ++i)
			if (nb[i].mask & 1u)
				roots.insert(GraphRoot{ o.roots[i], nb[i].hash[0] });
	}
	for (const std::string& path : o.rootFastas)
		for_each_batch(path, [&](const ReadBatch& b) {
			const uint64_t slots = hash_batch(b);
			flag.resize(slots + 1);
			contains_reads(b.bases.data(), b.offsets.data(), b.size(), flag.data(), (uint64_t)flag.size());
			uint64_t s = 0;
			for (size_t i = 0; i < b.size(); ++i) {
				const uint64_t L = b.offsets[i + 1] - b.offsets[i];
				for (uint64_t p = 0; p + k <= L; ++p, ++s)
					if (valid[s] && flag[s])
						roots.insert(GraphRoot{ std::string(b.bases.data() + b.offsets[i] + p, k), h0[s] });
			}
		});

	// breadth-first search (breadthFirstSearchImpl, undirected).  The queue is FIFO and every vertex is one deeper than the
	// vertex that discovered it, so it holds the search levels one after another: the neighbourhoods of a whole level are
	// one query, and the level is then expanded in queue order on the host, where the colours live.
	std::string out;
	out.reserve(1 << 20);
	auto flush = [&](bool force) {
		if (force || out.size() >= (1u << 20)) {
			os.write(out.data(), (std::streamsize)out.size());
			out.clear();
		}
	};
	auto vertex_line = [&](const std::string& s, unsigned depth, uint64_t h, uint32_t bloomBits) { // discover_vertex
		out += '\t';
		out += s;
		out += " [depth=";
		out += std::to_string(depth);
		for (size_t a = 0; a < fastaSets.size(); ++a)
			if (fastaSets[a].count(h)) {
				out += ',';
				out += o.fastaAttrs[a].first;
			}
		for (size_t a = 0; a < o.bloomAttrs.size(); ++a)
			if ((bloomBits >> a) & 1u) {
				out += ',';
				out += o.bloomAttrs[a];
			}
		out += "];\n";
		flush(false);
	};
	auto edge_line = [&](const std::string& u, const std::string& v) {
		out += '\t';
		out += u;
		out += " -> ";
		out += v;
		out += ";\n";
	};

	out += "digraph  {\n";
	std::unordered_set<uint64_t> seen; // the colour map: white = absent (a seen vertex is one level deeper than its discoverer)
	std::vector<std::string> frontier, next;
	frontier.reserve(roots.size());
	for (const GraphRoot& r : roots) {
		frontier.push_back(r.kmer);
		seen.insert(r.h0);
	}
	uint64_t levels = 0, vertices = 0;
	for (unsigned depth = 0; !frontier.empty(); ++depth) {
		kbuf.clear();
		for (const std::string& u : frontier)
			kbuf += u;
		nb.resize(frontier.size());
		neighbours(kbuf.data(), frontier.size(), nb.data());
		++levels;
		vertices += frontier.size();
		if (depth == 0)
			for (size_t i = 0; i < frontier.size(); ++i)
				vertex_line(frontier[i], 0, nb[i].hash[0], nb[i].attr[0]);
		next.clear();
		for (size_t i = 0; i < frontier.size(); ++i) { // examine_vertex u
			const std::string& u = frontier[i];
			const abb_neighbourhood& r = nb[i];
			for (unsigned b = 0; b < 4; ++b) { // out-edges (u, v): forward, printed whenever they are followed
				if (!((r.mask >> (1 + b)) & 1u))
					continue;
				const uint64_t h = r.hash[1 + b];
				std::string v = u.substr(1) + BASES[b];
				if (!seen.count(h)) { // tree_edge
					if (depth >= o.depth)
						continue; // BFS_SKIP_ELEMENT: stays white
					seen.insert(h);
					edge_line(u, v);
					vertex_line(v, depth + 1, h, r.attr[1 + b]);
					next.push_back(std::move(v));
				} else { // non_tree_edge
					edge_line(u, v);
					flush(false);
				}
			}
			for (unsigned b = 0; b < 4; ++b) { // in-edges (v, u): printed only where v is u itself (a self-loop)
				if (!((r.mask >> (5 + b)) & 1u))
					continue;
				const uint64_t h = r.hash[5 + b];
				std::string v = BASES[b] + u.substr(0, k - 1);
				if (!seen.count(h)) {
					if (depth >= o.depth)
						continue;
					seen.insert(h);
					vertex_line(v, depth + 1, h, r.attr[5 + b]);
					next.push_back(std::move(v));
				} else if (h == r.hash[0]) {
					edge_line(v, u);
					flush(false);
				}
			}
		}
		frontier.swap(next);
	}
	out += "}\n";
	flush(true);
	if (o.verbose)
		std::cerr << "Expanded " << vertices << " vertices in " << levels << " levels\n";
}

} // namespace host
