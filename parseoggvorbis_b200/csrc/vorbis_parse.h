// Host front-end: Ogg framing, Vorbis header/setup parse and the per-packet entropy decode that stays sequential
// on the CPU. It turns a bitstream into the packed work descriptors of include/pov_synth.h (Y lists, residue
// classifications + VQ entry numbers, window flags, emit counts); all arithmetic on spectra happens on the GPU.
//
// Behaviour (including error conditions and end-of-packet handling) follows the reference decoder
// (src/ParseOggVorbis.hpp, src/Utils.hpp); the structure is our own: flat tables, a 64-bit window bit reader and
// LUT-driven Huffman decode instead of the reference's per-bit tree walk.
#ifndef POV_VORBIS_PARSE_H
#define POV_VORBIS_PARSE_H

#include <stdint.h>

#include <memory>
#include <string>
#include <vector>

#include "../../include/pov_synth.h"

namespace pov {

// LSb-first bit reader over one packet. Reading past the end yields zero bits and sets `overrun`
// (reference: src/Utils.hpp:338, 389-392 — "We allow to reach the end").
struct BitCursor {
	const uint8_t* data = nullptr;
	uint64_t nbits = 0;     // total bits available
	uint64_t pos = 0;       // next bit
	bool overrun = false;
	void reset(const uint8_t* p, size_t nbytes) { data = p; nbits = (uint64_t) nbytes * 8; pos = 0; overrun = false; }
	inline uint64_t window() const;          // next up-to-57 valid bits, zero filled beyond the end
	inline uint32_t get(int n);              // 0 <= n <= 32
	inline void skip(int n) { pos += (uint64_t) n; }
};

struct HuffBook {
	uint32_t dim = 0, n_entries = 0, lookup_type = 0;
	std::vector<float> vq;                   // [n_entries*dim] when lookup_type != 0 (hpp:212-245)
	std::vector<uint8_t> lengths;            // codeword length per entry, 0 = unused (hpp:126, 270-272)
	// decode tables
	static constexpr int kFastBits = 10;
	std::vector<uint32_t> fast;              // [1<<kFastBits]: (entry << 6) | len, len == 0 -> slow path
	std::vector<uint32_t> sorted_code;       // bit-reversed-free representation: left-aligned codewords, ascending
	std::vector<uint32_t> sorted_entry;
	std::vector<uint8_t>  sorted_len;
	uint32_t decode(BitCursor& br) const;    // returns entry number (hpp:347-360 semantics)
};

struct FloorClass { uint32_t dim = 0, subclass_bits = 0, masterbook = 0; int32_t books[8] = {0}; };
struct Floor1Setup {
	uint32_t type = 1;                       // 0 is parsed but cannot be decoded (hpp:402)
	std::vector<uint8_t> partition_class;
	std::vector<FloorClass> classes;
	uint32_t multiplier = 1, rangebits = 0;
	std::vector<uint16_t> xs;
};
struct ResidueSetup {
	uint32_t type = 0, begin = 0, end = 0, partition_size = 1, n_class = 1, classbook = 0;
	uint8_t books[POV_MAX_CLASSES * 8];
};
struct MappingSetup {
	uint32_t n_submaps = 1;
	std::vector<uint8_t> mux, submap_floor, submap_residue;
	std::vector<uint8_t> mag, ang;
};
struct ModeSetup { uint8_t blockflag = 0, mapping = 0; };

// The codebooks of a setup (decode tables + VQ arenas, ~0.5 MB for the stereo fixture) are immutable once the setup
// header is parsed: copies of a setup (one per decoded file of a corpus) share them.
class BookTable {
	std::shared_ptr<std::vector<HuffBook>> p_ = std::make_shared<std::vector<HuffBook>>();
public:
	void resize(size_t n) { p_ = std::make_shared<std::vector<HuffBook>>(n); }     // a fresh table, never the shared one
	size_t size() const { return p_->size(); }
	const HuffBook& operator[](size_t i) const { return (*p_)[i]; }
	HuffBook& operator[](size_t i) { return (*p_)[i]; }
	std::vector<HuffBook>::iterator begin() { return p_->begin(); }
	std::vector<HuffBook>::iterator end() { return p_->end(); }
	std::vector<HuffBook>::const_iterator begin() const { return p_->begin(); }
	std::vector<HuffBook>::const_iterator end() const { return p_->end(); }
};

struct VorbisSetup {
	uint32_t channels = 0, sample_rate = 0, blocksize[2] = {0, 0};
	BookTable books;
	std::vector<Floor1Setup> floors;
	std::vector<ResidueSetup> residues;
	std::vector<MappingSetup> mappings;
	std::vector<ModeSetup> modes;
	int entry_bits = 16;
};

// One decoded logical stream: descriptors ready for pov_batch_upload (POV_INPUT_ENTRIES layout).
struct StreamWork {
	uint32_t serial = 0;
	VorbisSetup setup;
	bool have_id = false, have_comment = false, have_setup = false, ended = false;
	std::vector<uint8_t> pending;             // allow_spanning: the bytes so far of a packet that continues on the next page
	bool raw = false;                         // the payload holds raw audio packets (POV_INPUT_PACKETS), not entry numbers
	std::string setup_key;                    // raw id + setup packet bytes: identical keys <=> identical setups
	uint32_t packets_seen = 0;
	// per audio packet
	std::vector<pov_packet> packets;          // stream index / offsets are batch-relative to THIS StreamWork
	std::vector<uint16_t> ys;
	std::vector<uint8_t> payload;
	std::vector<uint64_t> abs_total_pos;      // before the packet (dump: "abs_total_pos")
	std::vector<int64_t> expected_end;        // dump: "expected_ending_total_pos"
	// cut_damage with the host walk: the first packet whose walk failed (it and every later packet of the stream are silence,
	// see ParseOptions), the POV_PKT_* word the device walk reports for that failure (0: none matches) and the host's text
	uint32_t walk_bad = UINT32_MAX, walk_status = 0;
	std::string walk_msg;
	// overlap bookkeeping (hpp:983-988)
	uint32_t prev_n = 0, cur_n = 0;
	uint64_t total_pos = 0;
	uint64_t frames = 0;
};

// cut: the parse ran with cut_damage, found damage and stopped there; msg holds what a strict parse fails with.
struct ParseError { bool failed = false, cut = false; std::string msg; };

// raw_packets: audio packets are not entropy-decoded here; the descriptors carry the packet bytes (POV_INPUT_PACKETS:
// mode, window flags and the emit bookkeeping only need the first bits of a packet) and the device walks the rest.
// allow_spanning: packets may continue on the next page of their stream (RFC 3533 lacing value 255 at a page end +
// "continued" flag). The reference refuses such files (hpp:89) and so does the default here; real-world encoders produce
// them routinely (setup headers above 4 KB, high bit rates).
// cut_damage (POV_PARSE_CUT_DAMAGE): the first failing check of the framing, headers or an audio packet's geometry ends the
// parse of the file with success and err.cut set: every stream keeps the audio packets completed before it, the failing
// packet and everything after it are dropped. A failing host walk of an audio packet's floors and residues instead keeps the
// packet as silence (no floor used, residue payloads that decode nothing) and marks the stream (walk_bad); later packets of
// that stream are not walked and are silence too.
struct ParseOptions { bool raw_packets = false; bool allow_spanning = false; bool cut_damage = false; };

// Parses a whole Ogg file from memory (hpp:1428 full_read_from_memory). Streams appear in order of their BOS page.
// Returns false and fills err on the first failing check, like the reference's OkOrError chain (with cut_damage, see above;
// an exception is a failure in both modes).
bool parse_ogg_file(const uint8_t* data, size_t len, std::vector<StreamWork>& streams, ParseError& err, const ParseOptions& opt = ParseOptions());

// Huffman decode tables from codeword lengths (Vorbis I 3.2.1, hpp:151-185): a first-level table indexed by the next
// `lut_bits` stream bits ((entry << 6) | length, 0 = longer codeword) and the codewords sorted by their left-aligned value
// for the rest. Shared by the host decoder (HuffBook) and the device tables of pov_setup_register. False: not a full tree.
struct HuffTables {
	std::vector<uint32_t> lut, sorted_code, sorted_entry;
	std::vector<uint8_t> sorted_len;
};
bool build_huff_tables(const uint8_t* lengths, uint32_t n_entries, int lut_bits, HuffTables& out, std::string& why);

// Converts a parsed setup into the ABI structs (storage owned by `keep`).
struct SetupAbi {
	pov_setup s;
	std::vector<pov_codebook> cbs;
	std::vector<pov_floor1> floors;
	std::vector<pov_residue> residues;
	std::vector<pov_mapping> mappings;
	std::vector<pov_mode> modes;
	std::vector<pov_floor1_syntax> floor_syntax;
};
bool setup_to_abi(const VorbisSetup& in, SetupAbi& out, std::string& why_unsupported);
// Can the packets of a stream with this setup be walked on the device? (floor1 only, no empty submap, table sizes in range)
bool setup_supports_device_entropy(const VorbisSetup& s);

uint32_t ogg_crc(uint32_t crc, const uint8_t* p, size_t n);

}  // namespace pov
#endif
