// Host front-end (see vorbis_parse.h). Reference behaviour cited per function; paths relative to the reference root.
#include "vorbis_parse.h"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <exception>
#include <map>
#include <new>

namespace pov {

// ---------------------------------------------------------------------------------------------------------------
// bit reader
// ---------------------------------------------------------------------------------------------------------------
inline uint64_t BitCursor::window() const {
	const uint64_t byte = pos >> 3;
	const uint64_t total = nbits >> 3;
	uint64_t w = 0;
	if(byte + 8 <= total) memcpy(&w, data + byte, 8);                 // little-endian host (x86-64 / aarch64)
	else for(uint64_t i = byte, k = 0; i < total && k < 8; ++i, ++k) w |= (uint64_t) data[i] << (8 * k);
	return w >> (pos & 7);
}
inline uint32_t BitCursor::get(int n) {
	if(n <= 0) return 0;
	const uint64_t w = window();
	if(pos + (uint64_t) n > nbits) overrun = true;                    // zero bits beyond the end (Utils.hpp:389-392)
	pos += (uint64_t) n;
	return (uint32_t) (w & ((n >= 32) ? 0xFFFFFFFFull : ((1ull << n) - 1)));
}

static int ilog(uint32_t v) { int r = 0; while(v) { ++r; v >>= 1; } return r; }    // Utils.hpp:47-56 highest_bit

struct Fail {
	ParseError& e;
	bool operator()(const char* fmt, ...) const {
		char buf[400];
		va_list ap;
		va_start(ap, fmt);
		vsnprintf(buf, sizeof buf, fmt, ap);
		va_end(ap);
		e.failed = true;
		e.msg = buf;
		return false;
	}
};
#define REQUIRE(cond, ...) do { if(!(cond)) return fail(__VA_ARGS__); } while(0)

// ---------------------------------------------------------------------------------------------------------------
// Ogg page CRC (polynomial 0x04c11db7, MSB first, init 0) — src/Utils.cpp:13-30 / src/crctable.h compute the same
// ---------------------------------------------------------------------------------------------------------------
static uint32_t g_crc[8][256];
static bool g_crc_ready = false;
static void crc_init() {
	for(uint32_t i = 0; i < 256; ++i) {
		uint32_t r = i << 24;
		for(int k = 0; k < 8; ++k) r = (r & 0x80000000u) ? (r << 1) ^ 0x04c11db7u : (r << 1);
		g_crc[0][i] = r;
	}
	for(uint32_t i = 0; i < 256; ++i)
		for(int t = 1; t < 8; ++t) g_crc[t][i] = g_crc[0][g_crc[t - 1][i] >> 24] ^ (g_crc[t - 1][i] << 8);
	g_crc_ready = true;
}
uint32_t ogg_crc(uint32_t crc, const uint8_t* p, size_t n) {
	if(!g_crc_ready) crc_init();
	while(n >= 8) {
		crc ^= ((uint32_t) p[0] << 24) | ((uint32_t) p[1] << 16) | ((uint32_t) p[2] << 8) | p[3];
		crc = g_crc[7][crc >> 24] ^ g_crc[6][(crc >> 16) & 255] ^ g_crc[5][(crc >> 8) & 255] ^ g_crc[4][crc & 255] ^
		      g_crc[3][p[4]] ^ g_crc[2][p[5]] ^ g_crc[1][p[6]] ^ g_crc[0][p[7]];
		p += 8; n -= 8;
	}
	while(n--) crc = (crc << 8) ^ g_crc[0][(crc >> 24) ^ *p++];
	return crc;
}

// ---------------------------------------------------------------------------------------------------------------
// codebooks — src/ParseOggVorbis.hpp:120-375
// ---------------------------------------------------------------------------------------------------------------
static double float32_unpack(uint32_t v) {             // Utils.hpp:194-203
	double mant = (double) (v & 0x1fffff);
	if(v & 0x80000000u) mant = -mant;
	long e = (long) ((v & 0x7fe00000u) >> 21) - 20 - 768;
	if(e > 63) e = 63;
	if(e < -63) e = -63;
	return ldexp(mant, (int) e);
}

static uint32_t pow_u32(uint32_t base, uint32_t e) {   // Utils.hpp:205-217 with BaseT = uint32_t (wraps mod 2^32)
	uint32_t r = 1;
	while(e) { if(e & 1) r *= base; base *= base; e >>= 1; }
	return r;
}

// Vorbis I 3.2.1: every entry takes the lowest-valued free codeword of its length; the tree must end up exactly
// full (hpp:151-185 rejects over- and under-specified trees, a single-entry book included).
bool build_huff_tables(const uint8_t* lengths, uint32_t n_entries, int lut_bits, HuffTables& out, std::string& why) {
	std::vector<uint8_t> lens;
	std::vector<uint32_t> nums;
	for(uint32_t i = 0; i < n_entries; ++i) if(lengths[i]) { lens.push_back(lengths[i]); nums.push_back(i); }
	uint32_t avail[33];
	memset(avail, 0, sizeof avail);
	const size_t n = lens.size();
	std::vector<uint32_t> code(n);
	size_t k = 0;
	if(n == 0) { why = "codebook: no used entries (hpp:183 underspecified)"; return false; }
	for(size_t i = 0; i < n; ++i) if(lens[i] > 32) { why = "codebook: codeword length > 32 (hpp:132)"; return false; }
	// first entry takes the all-zero codeword
	{
		const int L = lens[0];
		code[0] = 0;
		for(int i = 1; i <= L; ++i) avail[i] = 1u << (32 - i);
		k = 1;
	}
	for(; k < n; ++k) {
		int z = lens[k];
		while(z > 0 && !avail[z]) --z;
		if(z <= 0) { why = "codebook: overspecified Huffman tree (hpp:159,168)"; return false; }
		const uint32_t res = avail[z];
		avail[z] = 0;
		code[k] = res;                                   // left-aligned (MSB-first) codeword
		for(int y = lens[k]; y > z; --y) avail[y] = res + (1u << (32 - y));
	}
	for(int i = 1; i <= 32; ++i) if(avail[i] != 0) { why = "codebook: underspecified Huffman tree (hpp:183-184)"; return false; }
	// sorted table for the slow path + LUT for codes of <= lut_bits
	std::vector<size_t> order(n);
	for(size_t i = 0; i < n; ++i) order[i] = i;
	std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return code[a] < code[b]; });
	out.sorted_code.resize(n); out.sorted_entry.resize(n); out.sorted_len.resize(n);
	for(size_t i = 0; i < n; ++i) {
		out.sorted_code[i] = code[order[i]];
		out.sorted_entry[i] = nums[order[i]];
		out.sorted_len[i] = lens[order[i]];
	}
	out.lut.assign((size_t) 1 << lut_bits, 0);
	for(size_t i = 0; i < n; ++i) {
		const int L = lens[i];
		if(L > lut_bits) continue;
		// the stream delivers the codeword MSB first into the LSb-first bit order: reverse the L code bits
		uint32_t rev = 0;
		for(int b = 0; b < L; ++b) if(code[i] & (1u << (31 - b))) rev |= 1u << b;
		for(uint32_t fill = rev; fill < (1u << lut_bits); fill += 1u << L)
			out.lut[fill] = (nums[i] << 6) | (uint32_t) L;
	}
	return true;
}

static bool assign_codewords(HuffBook& book, const Fail& fail) {
	HuffTables t;
	std::string why;
	if(!build_huff_tables(book.lengths.data(), book.n_entries, HuffBook::kFastBits, t, why)) return fail("%s", why.c_str());
	book.fast = std::move(t.lut);
	book.sorted_code = std::move(t.sorted_code);
	book.sorted_entry = std::move(t.sorted_entry);
	book.sorted_len = std::move(t.sorted_len);
	return true;
}

uint32_t HuffBook::decode(BitCursor& br) const {
	const uint64_t w = br.window();
	const uint32_t f = fast[w & ((1u << kFastBits) - 1)];
	if(f & 63) {
		if(br.pos + (f & 63) > br.nbits) br.overrun = true;
		br.pos += f & 63;
		return f >> 6;
	}
	// slow path: rebuild the MSB-first codeword prefix from the next 32 stream bits and binary-search it
	uint32_t msb = 0;
	const uint32_t lo32 = (uint32_t) w;
	for(int b = 0; b < 32; ++b) if(lo32 & (1u << b)) msb |= 1u << (31 - b);
	size_t lo = 0, hi = sorted_code.size();
	while(hi - lo > 1) {
		const size_t mid = (lo + hi) / 2;
		if(sorted_code[mid] <= msb) lo = mid; else hi = mid;
	}
	const int L = sorted_len[lo];
	if(br.pos + (uint64_t) L > br.nbits) br.overrun = true;
	br.pos += (uint64_t) L;
	return sorted_entry[lo];
}

static bool parse_codebook(BitCursor& br, HuffBook& book, const Fail& fail) {
	REQUIRE(br.get(24) == 0x564342, "codebook: bad sync pattern (hpp:255)");
	book.dim = br.get(16);
	REQUIRE(book.dim > 0, "codebook: dimensions == 0 (hpp:257)");
	book.n_entries = br.get(24);
	REQUIRE(book.n_entries > 0, "codebook: entries == 0 (hpp:259)");
	book.lengths.assign(book.n_entries, 0);
	const bool ordered = br.get(1);
	if(!ordered) {
		const bool sparse = br.get(1);
		// every entry costs at least one bit (sparse flag) or five (length): a packet too short for them is truncated,
		// whatever the 24-bit entry count claims
		REQUIRE((uint64_t) book.n_entries * (sparse ? 1u : 5u) <= br.nbits - std::min(br.nbits, br.pos), "codebook: truncated (hpp:327)");
		for(uint32_t i = 0; i < book.n_entries; ++i) {
			if(sparse && !br.get(1)) continue;
			book.lengths[i] = (uint8_t) (br.get(5) + 1);
		}
		REQUIRE(!br.overrun, "codebook: truncated (hpp:327)");
	} else {
		uint32_t len = br.get(5) + 1, cur = 0;
		while(cur < book.n_entries) {
			const uint32_t number = br.get(ilog(book.n_entries - cur));
			REQUIRE(cur + number <= book.n_entries, "codebook: ordered lengths overflow (hpp:290)");
			REQUIRE(len <= 32, "codebook: codeword length > 32 (hpp:132)");
			for(uint32_t i = cur; i < cur + number; ++i) book.lengths[i] = (uint8_t) len;
			cur += number;
			++len;
			REQUIRE(!br.overrun, "codebook: truncated (hpp:327)");
		}
	}
	if(!assign_codewords(book, fail)) return false;
	book.lookup_type = br.get(4);
	REQUIRE(book.lookup_type <= 2, "codebook: lookup type %u (hpp:299)", book.lookup_type);
	if(book.lookup_type != 0) {
		const double minimum = float32_unpack(br.get(32));
		const double delta = float32_unpack(br.get(32));
		const int value_bits = (int) br.get(4) + 1;
		const bool sequence_p = br.get(1);
		// The expanded table holds n_entries * dim floats. The reference computes that product (and, for lookup type 2, the
		// multiplicand count) in 32 bits; here both are 64-bit, and a table beyond kMaxVqValues floats is refused as
		// unsupported instead of being allocated (a crafted 117-byte header can ask for 275 GB).
		constexpr uint64_t kMaxVqValues = 1ull << 24;
		const uint64_t table_values = (uint64_t) book.n_entries * book.dim;
		REQUIRE(table_values <= kMaxVqValues, "codebook: VQ table of %llu values exceeds this build's limit of %llu",
		        (unsigned long long) table_values, (unsigned long long) kMaxVqValues);
		uint64_t n_values;
		if(book.lookup_type == 1) {          // lookup1_values (hpp:314-316), 32-bit wrap-around included
			uint32_t nv = 0;
			while(pow_u32(nv + 1, book.dim) <= book.n_entries) ++nv;
			n_values = nv;
		} else {
			n_values = table_values;
		}
		REQUIRE(n_values * (uint64_t) value_bits <= br.nbits - std::min(br.nbits, br.pos), "codebook: truncated multiplicands (hpp:327)");
		std::vector<uint32_t> mult((size_t) n_values);
		for(size_t i = 0; i < (size_t) n_values; ++i) mult[i] = br.get(value_bits);
		// hpp:212-245: double arithmetic, each element rounded to float; `last` re-reads the rounded value
		book.vq.assign((size_t) table_values, 0.f);
		if(book.lookup_type == 1) {
			REQUIRE(n_values > 0, "codebook: no lookup values");
			for(uint32_t e = 0; e < book.n_entries; ++e) {
				double last = 0;
				uint32_t div = 1;
				for(uint32_t d = 0; d < book.dim; ++d) {
					const uint32_t off = (div ? e / div : 0) % (uint32_t) n_values;
					const float v = (float) (mult[off] * delta + minimum + last);
					book.vq[(size_t) e * book.dim + d] = v;
					if(sequence_p) last = v;
					div *= (uint32_t) n_values;
				}
			}
		} else {
			size_t off = 0;
			for(uint32_t e = 0; e < book.n_entries; ++e) {
				double last = 0;
				for(uint32_t d = 0; d < book.dim; ++d, ++off) {
					const float v = (float) (mult[off] * delta + minimum + last);
					book.vq[off] = v;
					if(sequence_p) last = v;
				}
			}
		}
	}
	REQUIRE(!br.overrun, "codebook: truncated (hpp:327)");
	return true;
}

// ---------------------------------------------------------------------------------------------------------------
// floors, residues, mappings, modes — hpp:377-471, 622-663, 765-835
// ---------------------------------------------------------------------------------------------------------------
static bool parse_floor(BitCursor& br, Floor1Setup& f, uint32_t n_books, const Fail& fail) {
	f.type = br.get(16);
	if(f.type == 0) {                                   // hpp:385-398: parsed, never decodable (hpp:402)
		br.get(8); br.get(16); br.get(16); br.get(6); br.get(8);
		const int nb = (int) br.get(4) + 1;
		for(int i = 0; i < nb; ++i) REQUIRE(br.get(8) < n_books, "floor0: book out of range (hpp:395)");
		return true;
	}
	REQUIRE(f.type == 1, "invalid floor type %u (hpp:606)", f.type);
	const int parts = (int) br.get(5);
	int maxc = -1;
	f.partition_class.resize(parts);
	for(int i = 0; i < parts; ++i) { f.partition_class[i] = (uint8_t) br.get(4); maxc = std::max(maxc, (int) f.partition_class[i]); }
	f.classes.resize(maxc + 1);
	for(auto& c : f.classes) {
		c.dim = br.get(3) + 1;
		c.subclass_bits = br.get(2);
		c.masterbook = c.subclass_bits ? br.get(8) : 0;
		if(c.subclass_bits) REQUIRE(c.masterbook < n_books, "floor1: masterbook out of range");
		for(int k = 0; k < (1 << c.subclass_bits); ++k) {
			c.books[k] = (int32_t) br.get(8) - 1;
			REQUIRE(c.books[k] < (int32_t) n_books, "floor1: subclass book out of range");
		}
	}
	f.multiplier = br.get(2) + 1;
	f.rangebits = br.get(4);
	f.xs.clear();
	f.xs.push_back(0);
	f.xs.push_back((uint16_t) (1u << f.rangebits));
	for(uint8_t pc : f.partition_class)
		for(uint32_t j = 0; j < f.classes[pc].dim; ++j) f.xs.push_back((uint16_t) br.get((int) f.rangebits));
	REQUIRE(f.xs.size() <= POV_MAX_POSTS, "floor1: too many posts");
	return true;
}

static bool parse_residue(BitCursor& br, ResidueSetup& r, const Fail& fail) {
	r.type = br.get(16);
	REQUIRE(r.type <= 2, "residue type %u (hpp:634)", r.type);
	r.begin = br.get(24);
	r.end = br.get(24);
	REQUIRE(r.begin <= r.end, "residue begin > end (hpp:638)");
	r.partition_size = br.get(24) + 1;
	r.n_class = br.get(6) + 1;
	r.classbook = br.get(8);
	uint32_t cascade[POV_MAX_CLASSES];
	for(uint32_t i = 0; i < r.n_class; ++i) {
		const uint32_t low = br.get(3);
		const uint32_t high = br.get(1) ? br.get(5) : 0;
		cascade[i] = high * 8 + low;
	}
	memset(r.books, POV_NO_BOOK, sizeof r.books);
	for(uint32_t i = 0; i < r.n_class; ++i)
		for(int j = 0; j < 8; ++j)
			if(cascade[i] & (1u << j)) r.books[i * 8 + j] = (uint8_t) br.get(8);
	return true;
}

static bool parse_mapping(BitCursor& br, MappingSetup& m, uint32_t channels, uint32_t n_floors, uint32_t n_residues, const Fail& fail) {
	REQUIRE(br.get(16) == 0, "mapping type != 0 (hpp:777)");
	m.n_submaps = br.get(1) ? br.get(4) + 1 : 1;
	if(br.get(1)) {
		const uint32_t steps = br.get(8) + 1;
		const int bits = ilog(channels - 1);
		REQUIRE(bits > 0, "mapping: coupling on a mono stream (Utils.hpp:347 assert)");
		for(uint32_t i = 0; i < steps; ++i) {
			const uint32_t mg = br.get(bits), an = br.get(bits);
			REQUIRE(mg != an && mg < channels && an < channels, "mapping: invalid coupling (hpp:788-790)");
			m.mag.push_back((uint8_t) mg);
			m.ang.push_back((uint8_t) an);
		}
	}
	REQUIRE(br.get(2) == 0, "mapping: reserved bits set (hpp:793)");
	m.mux.assign(channels, 0);
	if(m.n_submaps > 1)
		for(auto& x : m.mux) { x = (uint8_t) br.get(4); REQUIRE(x < m.n_submaps, "mapping: mux out of range (hpp:799)"); }
	m.submap_floor.resize(m.n_submaps);
	m.submap_residue.resize(m.n_submaps);
	for(uint32_t i = 0; i < m.n_submaps; ++i) {
		br.get(8);                                       // time configuration placeholder, discarded (hpp:805)
		m.submap_floor[i] = (uint8_t) br.get(8);
		REQUIRE(m.submap_floor[i] < n_floors, "mapping: floor out of range (hpp:807)");
		m.submap_residue[i] = (uint8_t) br.get(8);
		REQUIRE(m.submap_residue[i] < n_residues, "mapping: residue out of range (hpp:809)");
	}
	return true;
}

// hpp:897-963
static bool parse_setup_packet(const uint8_t* p, size_t len, VorbisSetup& s, const Fail& fail) {
	REQUIRE(len >= 16 && p[0] == 5 && memcmp(p + 1, "vorbis", 6) == 0, "setup header: bad packet type/signature (hpp:1344-1347)");
	BitCursor br;
	br.reset(p + 7, len - 7);
	const uint32_t nbooks = br.get(8) + 1;
	s.books.resize(nbooks);
	for(auto& b : s.books) if(!parse_codebook(br, b, fail)) return false;
	const uint32_t ntime = br.get(6) + 1;
	for(uint32_t i = 0; i < ntime; ++i) REQUIRE(br.get(16) == 0, "setup: time-domain transform != 0 (hpp:917)");
	REQUIRE(!br.overrun, "setup: truncated (hpp:918)");
	s.floors.resize(br.get(6) + 1);
	for(auto& f : s.floors) if(!parse_floor(br, f, nbooks, fail)) return false;
	REQUIRE(!br.overrun, "setup: truncated (hpp:927)");
	s.residues.resize(br.get(6) + 1);
	for(auto& r : s.residues) if(!parse_residue(br, r, fail)) return false;
	REQUIRE(!br.overrun, "setup: truncated (hpp:936)");
	s.mappings.resize(br.get(6) + 1);
	for(auto& m : s.mappings) if(!parse_mapping(br, m, s.channels, (uint32_t) s.floors.size(), (uint32_t) s.residues.size(), fail)) return false;
	REQUIRE(!br.overrun, "setup: truncated (hpp:945)");
	s.modes.resize(br.get(6) + 1);
	for(auto& m : s.modes) {
		m.blockflag = (uint8_t) br.get(1);
		REQUIRE(br.get(16) == 0, "mode: window type != 0 (hpp:828)");
		REQUIRE(br.get(16) == 0, "mode: transform type != 0 (hpp:830)");
		m.mapping = (uint8_t) br.get(8);
		REQUIRE(m.mapping < s.mappings.size(), "mode: mapping out of range (hpp:832)");
	}
	REQUIRE(!br.overrun, "setup: truncated (hpp:954)");
	REQUIRE(br.get(1) == 1, "setup: framing bit not set (hpp:957)");
	REQUIRE(!br.overrun, "setup: truncated (hpp:958)");
	// hpp:960-961 + 1351: the rest of the last byte must be zero padding and the packet must end there
	REQUIRE(br.nbits - br.pos < 8, "setup: trailing data after the framing bit (hpp:961)");
	REQUIRE(br.get((int) (br.nbits - br.pos)) == 0, "setup: non-zero padding (hpp:960)");
	uint32_t maxe = 0;
	for(auto& b : s.books) maxe = std::max(maxe, b.n_entries);
	s.entry_bits = maxe > 65536 ? 32 : 16;
	// What the residue walk below relies on, checked once per setup instead of once per packet. The reference checks the
	// classbook at decode time (hpp:700) and indexes the VQ books unchecked (hpp:727); for a VQ dimension that does not
	// divide the partition size its type-1 loop (hpp:744-752) writes past the partition, its type-0 loop (hpp:736-742) leaves
	// bins untouched: neither is decodable audio, so such a setup is refused here.
	for(size_t ri = 0; ri < s.residues.size(); ++ri) {
		const ResidueSetup& r = s.residues[ri];
		REQUIRE(r.classbook < nbooks, "residue %zu: classbook %u out of range (hpp:700)", ri, r.classbook);
		for(uint32_t i = 0; i < r.n_class * 8; ++i) {
			const uint32_t bk = r.books[i];
			if(bk == POV_NO_BOOK) continue;
			REQUIRE(bk < nbooks, "residue %zu: VQ book %u out of range (hpp:727)", ri, bk);
			REQUIRE(r.partition_size % s.books[bk].dim == 0, "residue %zu: VQ dimension %u does not divide the partition size %u (unsupported)",
			        ri, s.books[bk].dim, r.partition_size);
		}
	}
	return true;
}

// ---------------------------------------------------------------------------------------------------------------
// audio packet -> descriptors: hpp:1128-1211 (mode/window, floor Y reads, residue classification + cascade walk)
// and the emit bookkeeping of VorbisStreamDecodeState (hpp:1019-1059, 1061-1067)
// ---------------------------------------------------------------------------------------------------------------
// The walk is Vorbis I 8.6.2 as the reference implements it (hpp:697-760): 8 passes over the partitions, a classification
// word every cb.dim partitions in pass 0, then per partition and channel the vectors of the (class, pass) book.
// One deliberate difference: the reference advances `partition_count` INSIDE its channel loop (hpp:755), which is the
// spec's order only when a submap has one channel (always true for residue type 2, and for mono streams); with several
// channels of type 0/1 it skips partitions and can index past the vector. Here — and in the device kernels — the count
// advances once per partition, as the spec says (DESIGN.md "Deliberate divergences"). The hot loop keeps the bit position in
// a register, decodes through the 10-bit first-level tables in place and writes the entry numbers straight into a
// per-thread scratch array sized for the worst case (every partition coded in every pass with one-dimensional vectors).
static bool decode_residue_submap(BitCursor& br, const VorbisSetup& s, const ResidueSetup& r, uint32_t nch, const uint8_t* used,
                                  uint32_t vlen, std::vector<uint8_t>& payload, const Fail& fail) {
	// header: n_entries (patched at the end), cls[nch][parts], entries
	const uint32_t lb = std::min(r.begin, vlen), le = std::min(r.end, vlen);
	const uint32_t parts = (le - lb) / r.partition_size;
	const size_t head = payload.size();
	const size_t cls_bytes = ((size_t) nch * parts + 3) & ~(size_t) 3;
	payload.resize(head + 4 + cls_bytes, 0);
	const size_t cls_at = head + 4;
	if(le == lb) return true;                            // hpp:704-705: nothing to read, no bits consumed
	REQUIRE(r.classbook < s.books.size(), "residue: classbook out of range (hpp:700)");
	const HuffBook& cb = s.books[r.classbook];
	const uint32_t cw = cb.dim;
	const uint32_t row = parts + cw;                     // classification row of one channel (a last word may overhang)
	static thread_local std::vector<uint8_t> cls_buf;
	static thread_local std::vector<uint32_t> ent_buf;
	if(cls_buf.size() < (size_t) nch * row) cls_buf.resize((size_t) nch * row);
	const size_t worst = (size_t) 8 * parts * nch * r.partition_size;
	if(ent_buf.size() < worst) ent_buf.resize(worst);
	uint8_t* cls = cls_buf.data();
	memset(cls, 0, (size_t) nch * row);
	uint32_t* out = ent_buf.data();
	// (class, pass) -> book, vectors per partition; resolved once per call (<= 64 * 8 slots, a few used)
	const HuffBook* vbook[POV_MAX_CLASSES * 8];
	uint32_t vcount[POV_MAX_CLASSES * 8];
	for(uint32_t i = 0; i < r.n_class * 8; ++i) {
		const uint32_t book = r.books[i];
		vbook[i] = nullptr; vcount[i] = 0;
		if(book == POV_NO_BOOK || book >= s.books.size()) continue;      // out of range: reported when (if) it is used
		vbook[i] = &s.books[book];
		vcount[i] = r.partition_size / vbook[i]->dim;                    // dim | partition_size checked at setup conversion
	}
	const uint8_t* const data = br.data;
	const uint64_t nbits = br.nbits, safe_end = nbits >= 64 ? nbits - 63 : 0;     // pos < safe_end: 8 readable bytes at the cursor
	uint64_t pos = br.pos;
	constexpr uint32_t kMask = (1u << HuffBook::kFastBits) - 1;
	for(uint32_t pass = 0; pass < 8; ++pass) {
		uint32_t pc = 0;
		while(pc < parts) {
			if(pass == 0) {
				for(uint32_t j = 0; j < nch; ++j) {
					if(!used[j]) continue;
					br.pos = pos;
					uint32_t t = cb.decode(br);
					pos = br.pos;
					for(uint32_t i = cw; i > 0; --i) { cls[(size_t) j * row + i - 1 + pc] = (uint8_t) (t % r.n_class); t /= r.n_class; }
				}
			}
			for(uint32_t i = 0; i < cw && pc < parts; ++i, ++pc) {
				for(uint32_t j = 0; j < nch; ++j) {
					if(!used[j]) continue;
					const uint32_t slot = (uint32_t) cls[(size_t) j * row + pc] * 8 + pass;
					const uint32_t book = r.books[slot];
					if(book == POV_NO_BOOK) continue;
					REQUIRE(vbook[slot] != nullptr, "residue: VQ book out of range");
					const HuffBook& vb = *vbook[slot];
					REQUIRE(vb.lookup_type != 0 || vcount[slot] == 0, "residue: invalid VQ entry (hpp:369-370,739,748)");
					const uint32_t* fast = vb.fast.data();
					for(uint32_t k = vcount[slot]; k > 0; --k) {
						uint32_t e;
						uint32_t f = 0;
						if(pos < safe_end) {                         // one unaligned load
							uint64_t w;
							memcpy(&w, data + (pos >> 3), 8);
							f = fast[(uint32_t) (w >> (pos & 7)) & kMask];
						}
						if(f & 63) { pos += f & 63; e = f >> 6; }
						else {                                        // long codeword or the tail of the packet
							br.pos = pos;
							e = vb.decode(br);
							pos = br.pos;
							REQUIRE(e < vb.n_entries, "residue: invalid VQ entry (hpp:369-370,739,748)");
						}
						*out++ = e;
					}
				}
			}
		}
	}
	br.pos = pos;
	if(pos > nbits) br.overrun = true;
	for(uint32_t j = 0; j < nch; ++j) memcpy(&payload[cls_at + (size_t) j * parts], &cls[(size_t) j * row], parts);
	const uint32_t ne = (uint32_t) (out - ent_buf.data());
	memcpy(&payload[head], &ne, 4);
	const size_t at = payload.size();
	if(s.entry_bits == 16) {
		payload.resize(at + (((size_t) ne * 2 + 3) & ~(size_t) 3), 0);
		uint16_t* o = (uint16_t*) &payload[at];
		for(uint32_t i = 0; i < ne; ++i) o[i] = (uint16_t) ent_buf[i];
	} else {
		payload.resize(at + (size_t) ne * 4);
		memcpy(&payload[at], ent_buf.data(), (size_t) ne * 4);
	}
	return true;
}

// The host walk of one audio packet (floor Y lists and residue entry numbers) into st.ys / st.payload. *status: the POV_PKT_*
// word the device walk (k_packet_decode) reports for the same failure, 0 when none does.
static bool walk_audio_packet(StreamWork& st, BitCursor& br, const MappingSetup& mp, uint32_t half, pov_packet& pk, uint32_t* status,
                              const Fail& fail) {
	const VorbisSetup& s = st.setup;
	const uint32_t C = s.channels;
	// 4.3.2 floor curve decode (hpp:478-518): Y values only, the curve itself is rendered on the GPU
	uint32_t used = 0;
	for(uint32_t c = 0; c < C; ++c) {
		const Floor1Setup& f = s.floors[mp.submap_floor[mp.mux[c]]];
		REQUIRE(f.type == 1, "floor0 decode is not implemented by the reference (hpp:402)");
		if(br.get(1) == 0) continue;                     // hpp:478-481: unused
		used |= 1u << c;
		static const uint32_t ranges[4] = {256, 128, 86, 64};
		const int ybits = ilog(ranges[f.multiplier - 1] - 1);
		const size_t at = st.ys.size();
		st.ys.push_back((uint16_t) br.get(ybits));
		st.ys.push_back((uint16_t) br.get(ybits));
		for(uint8_t pc : f.partition_class) {
			const FloorClass& cl = f.classes[pc];
			const uint32_t csub = (1u << cl.subclass_bits) - 1;
			uint32_t cval = cl.subclass_bits ? s.books[cl.masterbook].decode(br) : 0;
			for(uint32_t i = 0; i < cl.dim; ++i) {
				const int32_t book = cl.books[cval & csub];
				cval >>= cl.subclass_bits;
				const uint32_t y = book >= 0 ? s.books[book].decode(br) : 0;
				REQUIRE(y <= 0xFFFF, "floor1: coded Y value %u exceeds this build's 16-bit Y arena", y);
				st.ys.push_back((uint16_t) y);
			}
		}
		REQUIRE(st.ys.size() - at == f.xs.size(), "floor1: Y/X count mismatch (hpp:519)");
	}
	pk.floor_used = (uint16_t) used;
	// 4.3.3 nonzero propagate (hpp:1174-1180)
	uint32_t prop = used;
	for(size_t k = 0; k < mp.mag.size(); ++k)
		if(((prop >> mp.mag[k]) | (prop >> mp.ang[k])) & 1) prop |= (1u << mp.mag[k]) | (1u << mp.ang[k]);
	// 4.3.4 residue decode (hpp:1182-1209)
	for(uint32_t sm = 0; sm < mp.n_submaps; ++sm) {
		uint8_t ch_used[POV_MAX_CHANNELS];
		uint32_t nch = 0;
		for(uint32_t c = 0; c < C; ++c) if(mp.mux[c] == sm) ch_used[nch++] = (prop >> c) & 1;
		const ResidueSetup& r = s.residues[mp.submap_residue[sm]];
		if(nch == 0) {
			// hpp:680 CHECK(num_channel > 0): a submap without channels is fatal in the reference
			return fail("residue: submap %u has no channels (hpp:680)", sm);
		}
		const uint8_t one = 1;                           // type 2, hpp:688: always decoded, whatever the floors said
		const bool ok = r.type == 2 ? decode_residue_submap(br, s, r, 1, &one, nch * half, st.payload, fail)
		                            : decode_residue_submap(br, s, r, nch, ch_used, half, st.payload, fail);
		if(!ok) { *status = POV_PKT_VQ_ENTRY; return false; }
	}
	return true;
}

// A packet whose walk failed, as silence: no floor used, and per submap the residue payload of a packet in which no channel is
// used (entry count 0, every classification 0), the bytes decode_residue_submap writes for it.
static void silence_audio_packet(StreamWork& st, const MappingSetup& mp, uint32_t half, pov_packet& pk) {
	const VorbisSetup& s = st.setup;
	pk.floor_used = 0;
	for(uint32_t sm = 0; sm < mp.n_submaps; ++sm) {
		uint32_t nch = 0;
		for(uint32_t c = 0; c < s.channels; ++c) nch += mp.mux[c] == sm;
		const ResidueSetup& r = s.residues[mp.submap_residue[sm]];
		const uint32_t vch = r.type == 2 ? 1 : nch, vlen = r.type == 2 ? nch * half : half;
		const uint32_t parts = (std::min(r.end, vlen) - std::min(r.begin, vlen)) / r.partition_size;
		st.payload.resize(st.payload.size() + 4 + (((size_t) vch * parts + 3) & ~(size_t) 3), 0);
	}
}

static bool decode_audio_packet(StreamWork& st, const uint8_t* p, size_t len, int64_t expected_end, const Fail& fail, const ParseOptions& opt) {
	const VorbisSetup& s = st.setup;
	BitCursor br;
	br.reset(p, len);
	st.abs_total_pos.push_back(st.total_pos);
	st.expected_end.push_back(expected_end);
	REQUIRE(br.get(1) == 0, "audio packet: packet type bit set (hpp:1142)");
	const uint32_t mode_idx = br.get(ilog((uint32_t) s.modes.size() - 1));
	REQUIRE(mode_idx < s.modes.size(), "audio packet: mode %u out of range (hpp:1147)", mode_idx);
	const ModeSetup& mode = s.modes[mode_idx];
	const MappingSetup& mp = s.mappings[mode.mapping];
	uint32_t wflags = 0;
	if(mode.blockflag) { wflags = br.get(1); wflags |= br.get(1) << 1; }          // hpp:1150-1153
	const uint32_t n = s.blocksize[mode.blockflag ? 1 : 0], half = n / 2;

	pov_packet pk;
	memset(&pk, 0, sizeof pk);
	pk.mode = (uint8_t) mode_idx;
	pk.window_flags = (uint8_t) wflags;
	pk.ys_off = st.ys.size();
	pk.spec_off = st.payload.size();
	if(st.raw) {
		// the device walks the packet from here (POV_INPUT_PACKETS): hand over the bytes, zero padded to a multiple of 4.
		// The checks the host walk would have made on the way (floor0, hpp:402; empty submap, hpp:680) depend on the setup
		// only and are made once, by setup_supports_device_entropy(), before a stream is decoded this way.
		REQUIRE(len <= 0xFFFFFFFFull, "audio packet too large");
		pk.packet_bytes = (uint32_t) len;
		st.payload.insert(st.payload.end(), p, p + len);
		st.payload.resize((st.payload.size() + 3) & ~(size_t) 3, 0);
	} else if(st.walk_bad != UINT32_MAX) {
		silence_audio_packet(st, mp, half, pk);          // (cut_damage: after the stream's first failed walk)
	} else {
		uint32_t status = 0;
		if(!walk_audio_packet(st, br, mp, half, pk, &status, fail)) {
			if(!opt.cut_damage) return false;
			st.walk_bad = (uint32_t) st.packets.size(); st.walk_status = status; st.walk_msg = fail.e.msg;
			fail.e.failed = false; fail.e.msg.clear();
			st.ys.resize(pk.ys_off); st.payload.resize(pk.spec_off);
			silence_audio_packet(st, mp, half, pk);
		}
	}
	// emit bookkeeping (hpp:1061-1067, 1019-1059)
	st.prev_n = st.cur_n;
	st.cur_n = n;
	uint64_t frames = st.prev_n ? st.prev_n / 4 + st.cur_n / 4 : 0;
	if(expected_end >= 0) {
		REQUIRE(st.total_pos <= (uint64_t) expected_end, "granule position behind the decoded position (hpp:1029)");
		REQUIRE(st.total_pos + frames >= (uint64_t) expected_end, "granule position beyond the decodable frames (hpp:1041)");
		frames = (uint64_t) expected_end - st.total_pos;
	}
	pk.emit_frames = (uint32_t) frames;
	pk.pcm_off = st.frames;
	st.frames += frames;
	st.total_pos += frames;
	st.packets.push_back(pk);
	return true;
}

// ---------------------------------------------------------------------------------------------------------------
// Ogg pages + packet dispatch — hpp:51-102, 1283-1340, 1385-1485
// ---------------------------------------------------------------------------------------------------------------
static uint32_t rd32(const uint8_t* p) { return (uint32_t) p[0] | ((uint32_t) p[1] << 8) | ((uint32_t) p[2] << 16) | ((uint32_t) p[3] << 24); }

static bool parse_id_packet(const uint8_t* p, size_t len, VorbisSetup& s, const Fail& fail) {
	REQUIRE(len >= 16 && p[0] == 1 && memcmp(p + 1, "vorbis", 6) == 0, "id header: bad packet type/signature (hpp:1285-1288)");
	REQUIRE(len - 7 == 23, "id header: wrong size (hpp:1289)");
	const uint8_t* h = p + 7;
	REQUIRE(h[22] == 1, "id header: framing flag (hpp:1292)");
	REQUIRE(rd32(h) == 0, "id header: vorbis_version != 0 (hpp:1293)");
	s.channels = h[4];
	// the reference takes any uint8_t channel count (hpp:107); this build's descriptors carry per-channel bit masks and
	// fixed [POV_MAX_CHANNELS] arrays, so more channels are refused here, before any audio packet is walked
	REQUIRE(s.channels >= 1 && s.channels <= POV_MAX_CHANNELS, "id header: %u channels (this build supports 1..%u)", s.channels, POV_MAX_CHANNELS);
	s.sample_rate = rd32(h + 5);
	s.blocksize[0] = 1u << (h[21] & 15);
	s.blocksize[1] = 1u << (h[21] >> 4);
	REQUIRE(s.blocksize[0] >= 64 && s.blocksize[0] <= 8192 && s.blocksize[1] >= 64 && s.blocksize[1] <= 8192, "id header: blocksize out of range (hpp:1295-1296)");
	REQUIRE(s.blocksize[0] <= s.blocksize[1], "id header: blocksize_0 > blocksize_1 (hpp:1298)");
	return true;
}

static bool check_comment_packet(const uint8_t* p, size_t len, const Fail& fail) {       // hpp:1303-1340
	REQUIRE(len >= 16 && p[0] == 3 && memcmp(p + 1, "vorbis", 6) == 0, "comment header: bad packet type/signature (hpp:1308-1311)");
	size_t off = 7;
	REQUIRE(off + 4 <= len, "comment header truncated (hpp:1313)");
	const uint32_t vendor = rd32(p + off); off += 4;
	REQUIRE(off + vendor <= len, "comment header truncated (hpp:1317)");
	off += vendor;
	REQUIRE(off + 4 <= len, "comment header truncated (hpp:1320)");
	const uint32_t count = rd32(p + off);
	REQUIRE(off + (uint64_t) count * 4 < len, "comment header truncated (hpp:1323)");
	off += 4;
	for(uint32_t i = 0; i < count; ++i) {
		REQUIRE(off + 4 <= len, "comment header truncated (hpp:1327)");
		const uint32_t l = rd32(p + off); off += 4;
		REQUIRE(off + l <= len, "comment header truncated (hpp:1331)");
		off += l;
	}
	REQUIRE(off + 1 == len && p[off] == 1, "comment header: framing (hpp:1336-1337)");
	return true;
}

// The state of the stream an audio packet is being decoded into, from before the packet: what cut_damage rolls back to.
struct PacketMark {
	size_t stream = SIZE_MAX;                            // SIZE_MAX: no audio packet is being decoded
	size_t ys = 0, payload = 0, positions = 0;
	uint32_t prev_n = 0, cur_n = 0, walk_bad = UINT32_MAX;
};

static bool parse_ogg_file_checked(const uint8_t* data, size_t len, std::vector<StreamWork>& streams, ParseError& err, const ParseOptions& opt,
                                   PacketMark& mark);
// Never throws: an allocation failure (or any other exception) while parsing hostile input is a parse error like the rest.
bool parse_ogg_file(const uint8_t* data, size_t len, std::vector<StreamWork>& streams, ParseError& err, const ParseOptions& opt) {
	try {
		PacketMark m;
		if(parse_ogg_file_checked(data, len, streams, err, opt, m)) return true;
		if(!opt.cut_damage) return false;
		if(m.stream != SIZE_MAX) {                       // the failing packet leaves no trace: its stream is a strict parse's of the prefix
			StreamWork& st = streams[m.stream];
			st.ys.resize(m.ys); st.payload.resize(m.payload);
			st.abs_total_pos.resize(m.positions); st.expected_end.resize(m.positions);
			st.prev_n = m.prev_n; st.cur_n = m.cur_n;
			if(m.walk_bad == UINT32_MAX) { st.walk_bad = UINT32_MAX; st.walk_status = 0; st.walk_msg.clear(); }
		}
		for(StreamWork& st : streams) st.pending.clear();
		err.cut = true;
		return true;
	} catch(const std::bad_alloc&) {
		err.failed = true; err.msg = "out of memory while parsing (sizes in the stream beyond what this machine can hold)";
	} catch(const std::exception& e) {
		err.failed = true; err.msg = std::string("internal error while parsing: ") + e.what();
	} catch(...) {
		err.failed = true; err.msg = "internal error while parsing";
	}
	return false;
}

static bool parse_ogg_file_checked(const uint8_t* data, size_t len, std::vector<StreamWork>& streams, ParseError& err, const ParseOptions& opt,
                                   PacketMark& mark) {
	Fail fail{err};
	std::map<uint32_t, size_t> live;                     // serial -> index into streams (erased at EOS, hpp:1480)
	size_t pos = 0;
	while(len - pos >= 27) {                             // hpp:69-74: a short tail is plain EOF
		const uint8_t* h = data + pos;
		REQUIRE(memcmp(h, "OggS", 4) == 0, "page: capture pattern (hpp:77)");
		REQUIRE(h[4] == 0, "page: stream structure version (hpp:78)");
		const uint8_t flags = h[5];
		int64_t granule;
		memcpy(&granule, h + 6, 8);
		const uint32_t serial = rd32(h + 14);
		const uint32_t crc_expected = rd32(h + 22);
		const uint32_t nseg = h[26];
		REQUIRE(len - pos - 27 >= nseg, "page: truncated segment table (hpp:84)");
		const uint8_t* seg = h + 27;
		uint32_t body = 0;
		for(uint32_t i = 0; i < nseg; ++i) body += seg[i];
		const bool spans_out = nseg && seg[nseg - 1] == 255;
		if(!opt.allow_spanning) REQUIRE(!spans_out, "page: packets spanning pages are not supported (hpp:89)");
		REQUIRE(len - pos - 27 - nseg >= body, "page: truncated body (hpp:90)");
		const uint8_t* payload = seg + nseg;
		{
			uint8_t hdr[27];
			memcpy(hdr, h, 27);
			memset(hdr + 22, 0, 4);
			uint32_t crc = ogg_crc(0, hdr, 27);
			crc = ogg_crc(crc, seg, nseg);
			crc = ogg_crc(crc, payload, body);
			REQUIRE(crc == crc_expected, "page: CRC mismatch (hpp:98)");
		}
		if(flags & 2) {                                  // first page of a logical stream (hpp:1435-1438)
			REQUIRE(!live.count(serial), "page: duplicate begin-of-stream (hpp:1436)");
			live[serial] = streams.size();
			streams.emplace_back();
			streams.back().serial = serial;
		}
		REQUIRE(live.count(serial), "page: unknown stream serial (hpp:1439)");
		StreamWork& st = streams[live[serial]];
		if(opt.allow_spanning) {
			// a page either continues the packet its predecessor left open, or it does not (RFC 3533 section 6, header_type bit 0)
			REQUIRE(((flags & 1) != 0) == !st.pending.empty(), "page: continuation flag does not match the previous page of the stream");
		}
		// the granule position belongs to the last packet that ENDS on this page (hpp:1456-1459; RFC 3533: -1 if none does)
		int last_end = -1;
		for(uint32_t i = 0; i < nseg; ++i) if(seg[i] != 255) last_end = (int) i;
		size_t off = 0;
		uint32_t plen = 0;
		for(uint32_t i = 0; i < nseg; ++i) {
			plen += seg[i];
			if(seg[i] == 255) continue;
			const uint8_t* pp = payload + off;
			size_t pbytes = plen;
			if(!st.pending.empty()) {                        // the tail of a packet begun on an earlier page
				st.pending.insert(st.pending.end(), pp, pp + plen);
				pp = st.pending.data(); pbytes = st.pending.size();
			}
			const int64_t expected = ((int) i == last_end) ? granule : -1;
			if(st.packets_seen == 0) {
				if(!parse_id_packet(pp, pbytes, st.setup, fail)) return false;
				st.have_id = true;
				st.setup_key.assign((const char*) pp, pbytes);
			} else if(st.packets_seen == 1) {
				if(!check_comment_packet(pp, pbytes, fail)) return false;
				st.have_comment = true;
			} else if(st.packets_seen == 2) {
				// A corpus usually repeats a handful of setups: reuse the last one parsed by this thread when the raw
				// header bytes are identical (codebook + VQ table construction is the expensive part of a short file).
				static thread_local std::string cached_key;
				static thread_local VorbisSetup cached_setup;
				st.setup_key.append((const char*) pp, pbytes);
				if(st.setup_key == cached_key) {
					st.setup = cached_setup;
				} else {
					if(!parse_setup_packet(pp, pbytes, st.setup, fail)) return false;
					cached_key = st.setup_key;
					cached_setup = st.setup;
				}
				st.have_setup = true;
				st.raw = opt.raw_packets && setup_supports_device_entropy(st.setup);
			} else {
				mark.stream = live[serial];
				mark.ys = st.ys.size(); mark.payload = st.payload.size(); mark.positions = st.abs_total_pos.size();
				mark.prev_n = st.prev_n; mark.cur_n = st.cur_n; mark.walk_bad = st.walk_bad;
				if(!decode_audio_packet(st, pp, pbytes, expected, fail, opt)) {
					err.msg = "audio packet " + std::to_string(st.packets.size()) + ": " + err.msg;
					return false;
				}
				mark.stream = SIZE_MAX;
			}
			++st.packets_seen;
			st.pending.clear();
			off += plen;
			plen = 0;
		}
		if(plen) st.pending.insert(st.pending.end(), payload + off, payload + off + plen);      // (only with allow_spanning)
		if(flags & 4) { st.ended = true; live.erase(serial); }          // hpp:1478-1481
		pos += 27 + nseg + body;
	}
	return true;
}

// ---------------------------------------------------------------------------------------------------------------
// parsed setup -> ABI structs
// ---------------------------------------------------------------------------------------------------------------
bool setup_supports_device_entropy(const VorbisSetup& s) {
	if(s.books.size() > 255) return false;
	for(const Floor1Setup& f : s.floors)
		if(f.type != 1 || f.partition_class.size() > 31 || f.classes.size() > 16) return false;      // floor0: hpp:402
	for(const MappingSetup& m : s.mappings)
		for(uint32_t sm = 0; sm < m.n_submaps; ++sm) {
			bool any = false;
			for(uint8_t x : m.mux) any |= (x == sm);
			if(!any) return false;                                                                    // hpp:680, fatal per packet
		}
	return true;
}

bool setup_to_abi(const VorbisSetup& in, SetupAbi& out, std::string& why) {
	memset(&out.s, 0, sizeof out.s);
	if(in.channels > POV_MAX_CHANNELS) { why = "more than 8 channels"; return false; }
	out.cbs.resize(in.books.size());
	for(size_t i = 0; i < in.books.size(); ++i) {
		out.cbs[i].dim = in.books[i].dim;
		out.cbs[i].n_entries = in.books[i].n_entries;
		out.cbs[i].lookup_type = in.books[i].lookup_type;
		out.cbs[i].reserved = 0;
		out.cbs[i].vq = in.books[i].lookup_type ? in.books[i].vq.data() : nullptr;
		out.cbs[i].lengths = in.books[i].lengths.empty() ? nullptr : in.books[i].lengths.data();
	}
	out.floors.resize(in.floors.size());
	out.floor_syntax.resize(in.floors.size());
	for(size_t i = 0; i < in.floors.size(); ++i) {
		pov_floor1_syntax& fs = out.floor_syntax[i];
		memset(&fs, 0, sizeof fs);
		if(in.floors[i].type == 1 && in.floors[i].partition_class.size() <= 32 && in.floors[i].classes.size() <= 16) {
			const Floor1Setup& f = in.floors[i];
			fs.n_partitions = (uint8_t) f.partition_class.size();
			fs.n_classes = (uint8_t) f.classes.size();
			for(size_t k = 0; k < f.partition_class.size(); ++k) fs.partition_class[k] = f.partition_class[k];
			for(size_t k = 0; k < f.classes.size(); ++k) {
				fs.class_dim[k] = (uint8_t) f.classes[k].dim;
				fs.class_subclass_bits[k] = (uint8_t) f.classes[k].subclass_bits;
				fs.class_masterbook[k] = (uint8_t) f.classes[k].masterbook;
				for(int b = 0; b < 8; ++b) fs.class_books[k][b] = (b < (1 << f.classes[k].subclass_bits)) ? (int16_t) f.classes[k].books[b] : (int16_t) -1;
			}
		}
		memset(&out.floors[i], 0, sizeof(pov_floor1));
		if(in.floors[i].type != 1) {
			// floor0 cannot be decoded by the reference either (hpp:402); give the slot a harmless 2-post placeholder,
			// any packet that selects it is rejected by decode_audio_packet
			out.floors[i].n_posts = 2; out.floors[i].multiplier = 1; out.floors[i].xs[1] = 64;
			continue;
		}
		out.floors[i].n_posts = (uint16_t) in.floors[i].xs.size();
		out.floors[i].multiplier = (uint8_t) in.floors[i].multiplier;
		for(size_t k = 0; k < in.floors[i].xs.size(); ++k) out.floors[i].xs[k] = in.floors[i].xs[k];
	}
	out.residues.resize(in.residues.size());
	for(size_t i = 0; i < in.residues.size(); ++i) {
		const ResidueSetup& r = in.residues[i];
		pov_residue& o = out.residues[i];
		o.type = r.type; o.begin = r.begin; o.end = r.end; o.partition_size = r.partition_size; o.n_class = r.n_class; o.classbook = r.classbook;
		memcpy(o.books, r.books, sizeof o.books);
	}
	out.mappings.resize(in.mappings.size());
	for(size_t i = 0; i < in.mappings.size(); ++i) {
		const MappingSetup& m = in.mappings[i];
		pov_mapping& o = out.mappings[i];
		memset(&o, 0, sizeof o);
		o.n_submaps = m.n_submaps; o.n_couplings = (uint32_t) m.mag.size();
		for(size_t c = 0; c < m.mux.size(); ++c) o.mux[c] = m.mux[c];
		for(size_t k = 0; k < m.submap_floor.size(); ++k) { o.submap_floor[k] = m.submap_floor[k]; o.submap_residue[k] = m.submap_residue[k]; }
		for(size_t k = 0; k < m.mag.size(); ++k) { o.coupling_mag[k] = m.mag[k]; o.coupling_ang[k] = m.ang[k]; }
	}
	out.modes.resize(in.modes.size());
	for(size_t i = 0; i < in.modes.size(); ++i) { out.modes[i].blockflag = in.modes[i].blockflag; out.modes[i].mapping = in.modes[i].mapping; }
	pov_setup& s = out.s;
	s.abi_version = POV_ABI_VERSION;
	s.channels = in.channels; s.sample_rate = in.sample_rate;
	s.blocksize[0] = in.blocksize[0]; s.blocksize[1] = in.blocksize[1];
	s.n_codebooks = (uint32_t) out.cbs.size(); s.codebooks = out.cbs.data();
	s.n_floors = (uint32_t) out.floors.size(); s.floors = out.floors.data();
	s.n_residues = (uint32_t) out.residues.size(); s.residues = out.residues.data();
	s.n_mappings = (uint32_t) out.mappings.size(); s.mappings = out.mappings.data();
	s.n_modes = (uint32_t) out.modes.size(); s.modes = out.modes.data();
	s.floor_syntax = out.floor_syntax.data();
	return true;
}

}  // namespace pov
