// tests/host_bloom_graph/host_bloom_graph.cpp -- TEST INFRASTRUCTURE ONLY (never linked into libabyssb200).
//
// CPU emulation of `abyss-bloom graph`: the product's traversal (abyss_b200/host/bloom_graph.h) with the GPU queries replaced
// by single-thread loops over the SAME device function (neighbourhood() of csrc/abb_graph.cuh, the hash helpers of
// abb_device.cuh) on filter files read with abyss_b200/host/bloom_file.h; windows of reads are hashed by the C oracle.
// Output is compared with the unmodified reference's graph.
//
//   host_bloom_graph K DEPTH BLOOM [-R KMER | -f FASTA | -a STR:FASTA | -A STR:BLOOM]... > graph.dot
#include "../../abyss_b200/csrc/abb_graph.cuh"
#include "../../abyss_b200/host/bloom_file.h"
#include "../../abyss_b200/host/bloom_graph.h"
extern "C" {
#include "../../oracle/abyss_oracle.h"
}

using namespace abb;

struct BitFilter {
	std::vector<uint8_t> bits;
	FastMod mod;
	unsigned H;
	bool has(uint64_t h0, const HashCfg& cfg) const // cfg: the graph's multipliers
	{
		for (unsigned i = 0; i < H; ++i) {
			const uint64_t p = fastmod_u64(nth_hash(h0, cfg, i), mod);
			if (!((bits[p >> 3] >> (p & 7)) & 1))
				return false;
		}
		return true;
	}
};

static BitFilter load(const std::string& path, unsigned* k)
{
	host::BloomHeader h;
	BitFilter f;
	host::read_bit_bloom(path, h, f.bits);
	f.mod = make_fastmod(h.size);
	f.H = h.hashNum;
	if (k)
		*k = h.kmerSize;
	return f;
}

int main(int argc, char** argv)
{
	if (argc < 4) {
		fprintf(stderr, "usage: host_bloom_graph K DEPTH BLOOM [-R KMER | -f FASTA | -a STR:FASTA | -A STR:BLOOM]...\n");
		return 2;
	}
	host::BloomGraphOpts o;
	o.k = atoi(argv[1]);
	o.depth = (unsigned)strtoul(argv[2], nullptr, 10);
	unsigned fk = 0;
	const BitFilter graph = load(argv[3], &fk);
	if (fk != o.k) {
		fprintf(stderr, "filter k %u != %u\n", fk, o.k);
		return 2;
	}
	std::vector<BitFilter> attrs;
	for (int i = 4; i + 1 < argc; i += 2) {
		const std::string opt = argv[i], arg = argv[i + 1];
		const size_t colon = arg.find(':');
		if (opt == "-R")
			o.roots.push_back(arg);
		else if (opt == "-f")
			o.rootFastas.push_back(arg);
		else if (opt == "-a")
			o.fastaAttrs.emplace_back(arg.substr(0, colon), arg.substr(colon + 1));
		else if (opt == "-A") {
			o.bloomAttrs.push_back(arg.substr(0, colon));
			attrs.push_back(load(arg.substr(colon + 1), nullptr));
		}
	}
	const unsigned k = o.k;
	HashCfg cfg;
	cfg.H = graph.H;
	cfg.k = k;
	cfg.mod = graph.mod;
	for (unsigned i = 0; i < kMaxHashes; ++i)
		cfg.mult[i] = (uint64_t)i ^ ((uint64_t)k * kMultiSeed);
	auto probe = [&](const uint64_t* hash, unsigned* mask, uint32_t* attr) {
		*mask = 0;
		for (unsigned v = 0; v < 9; ++v) {
			if (graph.has(hash[v], cfg))
				*mask |= 1u << v;
			attr[v] = 0;
			for (size_t j = 0; j < attrs.size(); ++j)
				if (attrs[j].has(hash[v], cfg))
					attr[v] |= 1u << j;
		}
	};
	auto windows = [&](const char* bases, const uint64_t* offsets, uint64_t n, auto fn) { // fn(slot, h0) for the valid windows
		uint64_t s = 0;
		std::vector<uint64_t> h;
		std::vector<uint32_t> pos;
		for (uint64_t r = 0; r < n; ++r) {
			const uint64_t L = offsets[r + 1] - offsets[r];
			const uint64_t w = L >= k ? L - k + 1 : 0;
			h.resize(w + 1);
			pos.resize(w + 1);
			const size_t nv = w ? abo_hash_seq(bases + offsets[r], L, k, 1, nullptr, h.data(), pos.data()) : 0;
			for (size_t i = 0; i < nv; ++i)
				fn(s + pos[i], h[i]);
			s += w;
		}
		return s;
	};
	host::ReadOpts ropt;
	host::bloom_graph(
	    o,
	    [&](const std::string& path, auto fn) {
		    host::BatchStream stream({ path }, ropt, 500, 2);
		    while (const host::ReadBatch* b = stream.next())
			    fn(*b);
	    },
	    [&](const char* bases, const uint64_t* offsets, uint64_t n, uint64_t* h0, uint8_t* valid) {
		    const uint64_t slots = windows(bases, offsets, n, [&](uint64_t, uint64_t) {});
		    std::fill(valid, valid + slots, 0);
		    windows(bases, offsets, n, [&](uint64_t s, uint64_t h) {
			    valid[s] = 1;
			    h0[s] = h;
		    });
	    },
	    [&](const char* bases, const uint64_t* offsets, uint64_t n, uint8_t* flag, uint64_t) {
		    const uint64_t slots = windows(bases, offsets, n, [&](uint64_t, uint64_t) {});
		    std::fill(flag, flag + slots, 0);
		    windows(bases, offsets, n, [&](uint64_t s, uint64_t h) { flag[s] = graph.has(h, cfg); });
	    },
	    [&](const char* kmers, uint64_t n, abb_neighbourhood* out) {
		    for (uint64_t i = 0; i < n; ++i)
			    neighbourhood((const uint8_t*)kmers + i * k, k, probe, out + i);
	    },
	    std::cout);
	return 0;
}
