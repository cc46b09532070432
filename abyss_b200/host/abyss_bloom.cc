// abyss-bloom (B200) -- the `build` command of the reference's abyss-bloom for the ntHash filter
// family (Bloom/bloom.cc:584-622,625-800): `-t counting` (CountingBloomFilter<uint8_t>, the
// filter abyss-bloom-dbg loads with -i) and `-t rolling-hash [-l LEVELS]`
// (HashAgnosticCascadingBloom, last level serialised); and the `graph` command on the filter
// `-t rolling-hash` writes (bloom.cc:983-1153): the GraphViz neighbourhood of root k-mers, with
// the neighbour lookups of each search level in one CUDA launch (bloom_graph.h).  The Konnector
// filter family (`-t konnector`, city hash) and union/intersect/compare/kmers/trim, which work
// on it, are out of scope (SURVEY.md section 2).  Output files are byte-compatible with the
// reference's.
//
//   abyss-bloom build [-v] -k K [-b SIZE] [-H N] [-l LEVELS] [-t counting|rolling-hash] OUT.bloom READS...
//   abyss-bloom graph [-v] -k K [-d N] [-R KMER]... [-f FASTA]... [-a STR:FASTA]... [-A STR:BLOOM]... BLOOM
#include "../../include/abyss_b200.h"
#include "bloom_file.h"
#include "bloom_graph.h"
#include "reads.h"
#include <getopt.h>
#include <cmath>
#include <iomanip>

#define PROGRAM "abyss-bloom"
using namespace host;

static void check(int rc, const char* what)
{
	if (rc != ABB_OK) {
		std::cerr << PROGRAM ": " << what << ": " << abb_last_error() << "\n";
		exit(EXIT_FAILURE);
	}
}
static void usage()
{
	std::cerr << "Usage: " PROGRAM " build [-v] -k K [-b SIZE] [-H N] [-l LEVELS] [-t counting|rolling-hash] <OUTPUT_BLOOM_FILE> <READS_FILE_1> [READS_FILE_2]...\n"
	             "       " PROGRAM " graph [-v] -k K [-d N] [-R KMER]... [-f FASTA]... [-a STR:FASTA]... [-A STR:BLOOM]... <BLOOM_FILE>\n"
	             "Try `" PROGRAM " --help' for more information.\n";
	exit(EXIT_FAILURE);
}

[[noreturn]] static void die_with_usage_error()
{
	std::cerr << "Try `" PROGRAM " --help' for more information.\n";
	exit(EXIT_FAILURE);
}

// `graph' parses the reference's whole option table in two passes (bloom.cc:242-287,297-344,989-1034): the global options
// -k and -v up to the first other option, then the command's own.  A command option that takes an argument but means nothing
// to `graph' (-b, -H, -q, ..., and -k after a command option) is "invalid", because the argument is never read.
static const char kGraphShortopts[] = "a:A:b:B:d:f:h:H:j:k:l:L:m:n:q:rR:vt:w:";
enum { OPT_HELP = 1, OPT_VERSION, OPT_BED, OPT_FASTA, OPT_RAW };
static int g_chastity = 1, g_trimMasked = 1, g_qualityOffset = 0;
static const struct option kGraphLongopts[] = {
	{ "bloom-size", required_argument, NULL, 'b' }, { "bloom-type", required_argument, NULL, 't' },
	{ "buffer-size", required_argument, NULL, 'B' }, { "depth", required_argument, NULL, 'd' },
	{ "hash-seed", required_argument, NULL, 'h' }, { "num-hashes", required_argument, NULL, 'H' },
	{ "threads", required_argument, NULL, 'j' }, { "kmer", required_argument, NULL, 'k' },
	{ "levels", required_argument, NULL, 'l' }, { "init-level", required_argument, NULL, 'L' },
	{ "chastity", no_argument, &g_chastity, 1 }, { "no-chastity", no_argument, &g_chastity, 0 },
	{ "trim-masked", no_argument, &g_trimMasked, 1 }, { "no-trim-masked", no_argument, &g_trimMasked, 0 },
	{ "num-locks", required_argument, NULL, 'n' }, { "trim-quality", required_argument, NULL, 'q' },
	{ "standard-quality", no_argument, &g_qualityOffset, 33 }, { "illumina-quality", no_argument, &g_qualityOffset, 64 },
	{ "fasta-attr", required_argument, NULL, 'a' }, { "node-attr", required_argument, NULL, 'a' },
	{ "bloom-attr", required_argument, NULL, 'A' }, { "verbose", no_argument, NULL, 'v' },
	{ "help", no_argument, NULL, OPT_HELP }, { "version", no_argument, NULL, OPT_VERSION },
	{ "window", required_argument, NULL, 'w' }, { "method", required_argument, NULL, 'm' },
	{ "inverse", required_argument, NULL, 'r' }, { "root", required_argument, NULL, 'R' },
	{ "root-fasta", required_argument, NULL, 'f' }, { "bed", no_argument, NULL, OPT_BED },
	{ "fasta", no_argument, NULL, OPT_FASTA }, { "raw", no_argument, NULL, OPT_RAW },
	{ NULL, 0, NULL, 0 }
};

/** `istringstream(arg) >> token` read the whole argument: one whitespace-free word, leading blanks allowed */
static bool whole_word(const char* arg, std::string* word)
{
	const char* p = arg;
	while (*p && isspace((unsigned char)*p))
		++p;
	const char* e = p;
	while (*e && !isspace((unsigned char)*e))
		++e;
	if (e == p || *e)
		return false;
	word->assign(p, e);
	return true;
}
/** `istringstream(arg) >> unsigned integer` read the whole argument (a '-' sign wraps around, as num_get does) */
static bool whole_uint(const char* arg, uint64_t* v)
{
	std::string w;
	if (!whole_word(arg, &w))
		return false;
	size_t i = (w[0] == '+' || w[0] == '-') ? 1 : 0;
	if (i == w.size() || w.find_first_not_of("0123456789", i) != std::string::npos)
		return false;
	errno = 0;
	const uint64_t x = strtoull(w.c_str() + i, nullptr, 10);
	if (errno == ERANGE)
		return false;
	*v = w[0] == '-' ? (uint64_t)0 - x : x;
	return true;
}
[[noreturn]] static void invalid_option(int c, const char* arg)
{
	std::cerr << PROGRAM ": invalid option: `-" << (char)c << arg << "'\n";
	exit(EXIT_FAILURE);
}

static void load_bit_filter(const std::string& path, BloomHeader& h, std::vector<uint8_t>& raw, const char* what)
{
	std::ifstream probe(path, std::ios::binary);
	if (!probe) {
		std::cerr << PROGRAM ": `" << path << "': cannot open\n";
		exit(EXIT_FAILURE);
	}
	std::string magic;
	std::getline(probe, magic);
	if (magic == "[BTLCountingBloomFilter_v1]") {
		std::cerr << PROGRAM ": `" << path << "' is a counting Bloom filter; " << what
		          << " must be a filter written by `" PROGRAM " build -t rolling-hash'\n";
		exit(EXIT_FAILURE);
	}
	read_bit_bloom(path, h, raw);
}

/** `abyss-bloom graph` (bloom.cc:983-1153) */
static int graph(int argc, char** argv)
{
	unsigned k = 0;
	int verbose = 0;
	optind = 2;
	for (int c, prev = optind; (c = getopt_long(argc, argv, kGraphShortopts, kGraphLongopts, NULL)) != -1; prev = optind) { // parseGlobalOpts
		if (c == '?')
			die_with_usage_error();
		if (c == 'k') {
			uint64_t v = 0;
			if (!whole_uint(optarg, &v))
				invalid_option(c, optarg);
			k = (unsigned)v;
		} else if (c == 'v')
			++verbose;
		else if (c == OPT_HELP || c == OPT_VERSION)
			usage();
		else {
			optind = prev; // the first command option: the command parses from here
			break;
		}
	}
	if (k == 0) {
		std::cerr << PROGRAM ": missing mandatory option `-k'\n";
		die_with_usage_error();
	}
	host::BloomGraphOpts o;
	o.k = k;
	o.verbose = verbose;
	uint64_t depth = k; // the default depth is k
	std::vector<std::string> bloomAttrPaths;
	for (int c; (c = getopt_long(argc, argv, kGraphShortopts, kGraphLongopts, NULL)) != -1;) {
		bool ok = optarg == NULL; // an argument nobody reads is invalid
		std::string w;
		switch (c) {
		case '?': die_with_usage_error();
		case 'a':
		case 'A':
			if ((ok = whole_word(optarg, &w) && w.find(':') != std::string::npos)) {
				const size_t pos = w.find(':');
				if (c == 'a')
					o.fastaAttrs.emplace_back(w.substr(0, pos), w.substr(pos + 1));
				else {
					o.bloomAttrs.push_back(w.substr(0, pos));
					bloomAttrPaths.push_back(w.substr(pos + 1));
				}
			}
			break;
		case 'd': ok = whole_uint(optarg, &depth); break;
		case 'f':
			if ((ok = whole_word(optarg, &w)))
				o.rootFastas.push_back(w);
			break;
		case 'R':
			if ((ok = whole_word(optarg, &w)))
				o.roots.push_back(w);
			break;
		}
		if (!ok)
			invalid_option(c, optarg);
	}
	o.depth = (unsigned)depth;
	if (o.roots.empty() && o.rootFastas.empty()) {
		std::cerr << PROGRAM ": must specify either --root or --root-fasta\n";
		die_with_usage_error();
	}
	if (argc - optind != 1) {
		std::cerr << PROGRAM ": missing arguments\n";
		die_with_usage_error();
	}
	const std::string bloomPath = argv[optind];
	// where the reference asserts or reads past its arrays, stop with a message instead
	for (const std::string& r : o.roots)
		if (r.size() != k) {
			std::cerr << PROGRAM ": root k-mer `" << r << "' has " << r.size() << " characters, -k is " << k << "\n";
			exit(EXIT_FAILURE);
		}
	if (bloomAttrPaths.size() > 32) {
		std::cerr << PROGRAM ": at most 32 --bloom-attr filters are supported, " << bloomAttrPaths.size() << " given\n";
		exit(EXIT_FAILURE);
	}
	if (verbose)
		std::cerr << "Loading main Bloom filter from `" << bloomPath << "'...\n";
	BloomHeader h;
	std::vector<uint8_t> raw;
	load_bit_filter(bloomPath, h, raw, "the graph");
	if (h.kmerSize != k) {
		std::cerr << PROGRAM ": `" << bloomPath << "' holds " << h.kmerSize << "-mers, -k is " << k << "\n";
		exit(EXIT_FAILURE);
	}
	std::vector<BloomHeader> attrHeaders(bloomAttrPaths.size());
	std::vector<std::vector<uint8_t>> attrRaw(bloomAttrPaths.size());
	for (size_t j = 0; j < bloomAttrPaths.size(); ++j) {
		if (verbose)
			std::cerr << "Loading Bloom filter from `" << bloomAttrPaths[j] << "', to be annotated with '" << o.bloomAttrs[j] << "'\n";
		load_bit_filter(bloomAttrPaths[j], attrHeaders[j], attrRaw[j], "a --bloom-attr filter");
		if (attrHeaders[j].hashNum > h.hashNum) {
			std::cerr << PROGRAM ": `" << bloomAttrPaths[j] << "' has " << attrHeaders[j].hashNum << " hash functions, more than the "
			          << h.hashNum << " of the graph's filter, whose hash values it is probed with\n";
			exit(EXIT_FAILURE);
		}
	}
	abb_filter* g = nullptr;
	check(abb_filter_create(&g, ABB_BIT, h.size, h.hashNum, h.kmerSize, 0, "", 0), "filter");
	check(abb_filter_upload(g, 0, raw.data(), raw.size()), "upload");
	std::vector<abb_filter*> attrs;
	for (size_t j = 0; j < bloomAttrPaths.size(); ++j) {
		const BloomHeader& ah = attrHeaders[j];
		abb_filter* a = nullptr;
		check(abb_filter_create(&a, ABB_BIT, ah.size, ah.hashNum, ah.kmerSize, 0, "", 0), "filter");
		check(abb_filter_upload(a, 0, attrRaw[j].data(), attrRaw[j].size()), "upload");
		std::vector<uint8_t>().swap(attrRaw[j]);
		attrs.push_back(a);
	}
	std::vector<uint8_t>().swap(raw);
	host::ReadOpts ropt;
	ropt.chastityFilter = g_chastity;
	ropt.trimMasked = g_trimMasked;
	ropt.qualityOffset = g_qualityOffset;
	double nbSeconds = 0;
	host::bloom_graph(
	    o,
	    [&](const std::string& path, auto fn) {
		    host::BatchStream stream({ path }, ropt, 1u << 20);
		    while (const host::ReadBatch* b = stream.next())
			    fn(*b);
	    },
	    [&](const char* bases, const uint64_t* offsets, uint64_t n, uint64_t* h0, uint8_t* valid) {
		    check(abb_hash_reads(k, "", bases, offsets, n, h0, valid, nullptr, 0), "hash");
	    },
	    [&](const char* bases, const uint64_t* offsets, uint64_t n, uint8_t* flag, uint64_t cap) {
		    check(abb_contains_reads(g, bases, offsets, n, flag, nullptr, cap, nullptr), "contains");
	    },
	    [&](const char* kmers, uint64_t n, abb_neighbourhood* out) {
		    const auto t0 = std::chrono::steady_clock::now();
		    check(abb_neighbours(g, attrs.data(), (unsigned)attrs.size(), kmers, n, out), "neighbours");
		    nbSeconds += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
	    },
	    std::cout);
	std::cout.flush();
	if (verbose)
		std::cerr << "Neighbour queries: " << std::setprecision(6) << nbSeconds << " s\n";
	for (abb_filter* a : attrs)
		abb_filter_destroy(a);
	abb_filter_destroy(g);
	if (!std::cout) {
		std::cerr << PROGRAM ": error writing the graph\n";
		return EXIT_FAILURE;
	}
	return EXIT_SUCCESS;
}

/** `abyss-bloom info FILE`: printBloomStats (Bloom/bloom.cc:433-441,823-846) for the two ntHash-family file formats.
 *  (The reference's `info` reads the Konnector format only; the filters of this path are the BTL ones, so this command
 *  prints the same three lines for them, with the population counted on the GPU.) */
static int info(int argc, char** argv)
{
	int device = 0;
	std::string path;
	for (int i = 2; i < argc; ++i) {
		const std::string a = argv[i];
		if (a.rfind("--device=", 0) == 0)
			device = atoi(a.c_str() + 9);
		else if (a == "-v" || a == "--verbose")
			;
		else
			path = a;
	}
	if (path.empty()) {
		std::cerr << PROGRAM ": missing arguments\n";
		usage();
	}
	std::ifstream probe(path, std::ios::binary);
	std::string magic;
	std::getline(probe, magic);
	probe.close();
	BloomHeader h;
	std::vector<uint8_t> raw;
	abb_filter* f = nullptr;
	if (magic == "[BTLCountingBloomFilter_v1]") {
		read_counting_bloom(path, h, raw);
		check(abb_filter_create(&f, ABB_COUNTING, h.size, h.hashNum, h.kmerSize, 1, "", device), "filter");
	} else {
		read_bit_bloom(path, h, raw);
		check(abb_filter_create(&f, ABB_BIT, h.size, h.hashNum, h.kmerSize, 0, "", device), "filter");
	}
	check(abb_filter_upload(f, 0, raw.data(), raw.size()), "upload");
	uint64_t nz = 0;
	check(abb_filter_popcount(f, &nz, nullptr), "popcount");
	std::cerr << "Bloom size (bits): " << h.size << "\n"
	          << "Bloom popcount (bits): " << nz << "\n"
	          << "Bloom filter FPR: " << std::setprecision(3) << 100 * std::pow((double)nz / (double)h.size, (double)h.hashNum) << "%\n";
	abb_filter_destroy(f);
	return EXIT_SUCCESS;
}

int main(int argc, char** argv)
{
	if (argc >= 2 && std::string(argv[1]) == "info")
		return info(argc, argv);
	if (argc >= 2 && std::string(argv[1]) == "graph")
		return graph(argc, argv);
	if (argc < 2 || std::string(argv[1]) != "build") {
		std::cerr << PROGRAM ": only the `build' (-t counting | rolling-hash), `graph' and `info' commands are implemented on the B200\n";
		usage();
	}
	uint64_t bloomSize = 500ULL << 20; // [500M]
	unsigned k = 0, numHashes = 1, levels = 1, threads = 1;
	int verbose = 0, device = 0;
	uint64_t batchReads = 4000000;
	std::string type = "konnector";
	ReadOpts ropt;
	static int chastity = 1, trimMasked = 1, qualityOffset = 0; // 0 = the format's own offset
	static const struct option longopts[] = {
		{ "bloom-size", required_argument, NULL, 'b' }, { "kmer", required_argument, NULL, 'k' },
		{ "num-hashes", required_argument, NULL, 'H' }, { "levels", required_argument, NULL, 'l' },
		{ "bloom-type", required_argument, NULL, 't' }, { "threads", required_argument, NULL, 'j' },
		{ "trim-quality", required_argument, NULL, 'q' }, { "verbose", no_argument, NULL, 'v' },
		{ "chastity", no_argument, &chastity, 1 }, { "no-chastity", no_argument, &chastity, 0 },
		{ "trim-masked", no_argument, &trimMasked, 1 }, { "no-trim-masked", no_argument, &trimMasked, 0 },
		{ "standard-quality", no_argument, &qualityOffset, 33 }, { "illumina-quality", no_argument, &qualityOffset, 64 },
		{ "device", required_argument, NULL, 1000 }, { "batch-reads", required_argument, NULL, 1001 },
		{ NULL, 0, NULL, 0 }
	};
	optind = 2;
	for (int c; (c = getopt_long(argc, argv, "b:B:h:H:j:k:l:n:q:t:vw:", longopts, NULL)) != -1;) {
		switch (c) {
		case '?': usage(); break;
		case 'b':
			if (!si_to_bytes(optarg, &bloomSize)) {
				std::cerr << PROGRAM ": invalid option: `-b" << optarg << "'\n";
				exit(EXIT_FAILURE);
			}
			break;
		case 'k': k = (unsigned)atoi(optarg); break;
		case 'H': numHashes = (unsigned)atoi(optarg); break;
		case 'l': levels = (unsigned)atoi(optarg); break;
		case 'j': threads = (unsigned)atoi(optarg); break;
		case 'q': ropt.qualityThreshold = atoi(optarg); break;
		case 't': type = optarg; break;
		case 'v': ++verbose; break;
		case 1000: device = atoi(optarg); break;
		case 1001: batchReads = strtoull(optarg, nullptr, 10); break;
		case 'B': case 'h': case 'n': break; // I/O buffer, city-hash seed, lock count: no effect here
		case 'w':
			std::cerr << PROGRAM ": -w (Bloom windows) only applies to `-t konnector' filters\n";
			exit(EXIT_FAILURE);
		}
	}
	ropt.chastityFilter = chastity;
	ropt.trimMasked = trimMasked;
	ropt.qualityOffset = qualityOffset;
	if (k == 0) {
		std::cerr << PROGRAM ": missing mandatory option `-k'\n";
		usage();
	}
	if (type != "counting" && type != "rolling-hash") {
		std::cerr << PROGRAM ": `-t " << type << "' is not available on the B200: use 'rolling-hash' or 'counting'\n";
		usage();
	}
	if (argc - optind < 2) {
		std::cerr << PROGRAM ": missing arguments\n";
		usage();
	}
	const std::string outputPath = argv[optind++];
	std::vector<std::string> files(argv + optind, argv + argc);

	abb_filter* f = nullptr;
	uint64_t levelBits = 0;
	if (type == "counting") {
		if (levels != 1)
			std::cerr << PROGRAM ": warning: -l option has no effect when using `-t counting'\n";
		/* buildCountingBloom (bloom.cc:604-622): CountingBloomFilter<uint8_t>(bytes, H, k, 0) */
		check(abb_filter_create(&f, ABB_COUNTING, bloomSize, numHashes, k, 0, "", device), "filter");
	} else {
		/* buildRollingHashBloom (bloom.cc:584-601): level size = roundUpToMultiple(bits / levels, 64) */
		levelBits = bloomSize * 8 / levels;
		if (levelBits % 64)
			levelBits += 64 - levelBits % 64;
		check(abb_filter_create(&f, ABB_CASCADING, levelBits, numHashes, k, levels, "", device), "filter");
	}
	uint64_t readCount = 0;
	{
		host::BatchStream stream(files, ropt, batchReads, threads > 1 ? threads : 0, verbose != 0);
		while (const ReadBatch* batch = stream.next()) {
			check(abb_insert_reads(f, batch->bases.data(), batch->offsets.data(), batch->size(), nullptr), "insert");
			readCount += batch->size();
			if (verbose)
				std::cerr << "Loaded " << readCount << " reads into Bloom filter\n";
		}
	}
	if (verbose) {
		uint64_t nz = 0, th = 0;
		check(abb_filter_popcount(f, &nz, &th), "popcount");
		std::cerr << "Bloom size: " << abb_filter_size(f) << "\nBloom popcount: " << nz << "\nBloom filter FPR: " << std::setprecision(3)
		          << 100 * std::pow((double)nz / (double)abb_filter_size(f), (double)numHashes) << "%\n"
		          << "Writing bloom filter to `" << outputPath << "'...\n";
	}
	std::vector<uint8_t> raw(abb_filter_size_in_bytes(f));
	check(abb_filter_download(f, -1, raw.data(), raw.size()), "download");
	std::ofstream out(outputPath, std::ios::binary);
	if (!out) {
		std::cerr << "error: `" << outputPath << "': cannot open for writing\n";
		exit(EXIT_FAILURE);
	}
	if (type == "counting") {
		BloomHeader h;
		h.size = abb_filter_size(f);
		h.sizeInBytes = abb_filter_size_in_bytes(f);
		h.hashNum = numHashes;
		h.kmerSize = k;
		write_counting_bloom(out, h, raw);
	} else
		write_bit_bloom(out, levelBits, numHashes, k, raw);
	out.flush();
	if (!out) {
		std::cerr << "error: `" << outputPath << "': write failed\n";
		exit(EXIT_FAILURE);
	}
	abb_filter_destroy(f);
	return EXIT_SUCCESS;
}
