// Whole-file / corpus decode: host front-end (vorbis_parse.cpp) -> descriptor batch -> C ABI -> CUDA kernels.
// Mirrors the reference's entry points ogg_vorbis_full_read_from_memory (src/ParseOggVorbis.hpp:1493,
// src/ParseOggVorbis.cpp:28-41) and OggReader::full_read_from_memory (hpp:1428): 0 = ok, non-zero = error + message.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "api_internal.h"
#include "debug_dump.h"
#include "kernels.h"
#include "resample.h"
#include "vorbis_parse.h"

using namespace pov;

// ---------------------------------------------------------------------------------------------------------------
// parsed file handle (host only; usable without a GPU, e.g. from worker processes)
// ---------------------------------------------------------------------------------------------------------------
struct pov_parsed {
	std::vector<StreamWork> streams;
	std::vector<std::unique_ptr<SetupAbi>> abi;        // one per stream
	std::vector<pov_stream> stream_rec;                // single-stream batches
};

static bool finish_stream_tables(pov_parsed& P, std::string& why) {
	P.abi.clear();
	P.stream_rec.clear();
	for(StreamWork& st : P.streams) {
		std::unique_ptr<SetupAbi> a(new SetupAbi());
		if(!st.have_setup) {
			memset(&a->s, 0, sizeof a->s);
		} else if(!setup_to_abi(st.setup, *a, why)) {
			return false;
		}
		P.abi.push_back(std::move(a));
		pov_stream rec;
		memset(&rec, 0, sizeof rec);
		rec.setup_id = 0; rec.first_packet = 0; rec.n_packets = (uint32_t) st.packets.size();
		rec.pcm_frames = st.frames; rec.pcm_base = 0;
		P.stream_rec.push_back(rec);
		for(pov_packet& pk : st.packets) pk.stream = 0;
	}
	return true;
}

extern "C" int pov_ogg_parse_memory(const uint8_t* data, size_t len, pov_parsed** out, const char** error_out) {
	return pov_ogg_parse_memory_ex(data, len, 0, out, error_out);
}

extern "C" int pov_ogg_parse_memory_ex(const uint8_t* data, size_t len, uint32_t flags, pov_parsed** out, const char** error_out) {
	static thread_local char errbuf[512];
	if(!out || (!data && len)) return POV_ERR_ARG;
	*out = nullptr;
	try {
	std::unique_ptr<pov_parsed> P(new pov_parsed());
	ParseError err;
	ParseOptions opt;
	opt.raw_packets = (flags & POV_PARSE_RAW_PACKETS) != 0;
	opt.allow_spanning = (flags & POV_PARSE_ALLOW_SPANNING) != 0;
	opt.cut_damage = (flags & POV_PARSE_CUT_DAMAGE) != 0;
	if(!parse_ogg_file(data, len, P->streams, err, opt)) {
		snprintf(errbuf, sizeof errbuf, "check failed: %s", err.msg.c_str());
		if(error_out) *error_out = errbuf;
		return POV_ERR_STREAM;
	}
	std::string why;
	if(!finish_stream_tables(*P, why)) {
		snprintf(errbuf, sizeof errbuf, "unsupported stream: %s", why.c_str());
		if(error_out) *error_out = errbuf;
		return POV_ERR_UNSUPPORTED;
	}
	*out = P.release();
	return POV_OK;
	} catch(...) {
		snprintf(errbuf, sizeof errbuf, "out of memory or internal error while building the descriptors");
		if(error_out) *error_out = errbuf;
		return POV_ERR_ARG;
	}
}

extern "C" uint32_t pov_parsed_stream_count(const pov_parsed* p) { return p ? (uint32_t) p->streams.size() : 0; }

extern "C" int pov_parsed_get(const pov_parsed* p, uint32_t stream, pov_setup* setup_out, pov_batch* batch_out) {
	if(!p || stream >= p->streams.size()) return POV_ERR_ARG;
	const StreamWork& st = p->streams[stream];
	if(setup_out) *setup_out = p->abi[stream]->s;
	if(batch_out) {
		memset(batch_out, 0, sizeof *batch_out);
		batch_out->input_kind = st.raw ? POV_INPUT_PACKETS : POV_INPUT_ENTRIES;
		batch_out->pcm_layout = POV_PCM_PLANAR;
		batch_out->n_streams = 1; batch_out->streams = &p->stream_rec[stream];
		batch_out->n_packets = (uint32_t) st.packets.size(); batch_out->packets = st.packets.data();
		batch_out->ys = st.ys.data(); batch_out->n_ys = st.ys.size();
		batch_out->payload = st.payload.data(); batch_out->payload_bytes = st.payload.size();
		batch_out->pcm_floats = st.frames * st.setup.channels;
	}
	return POV_OK;
}

extern "C" void pov_parsed_free(pov_parsed* p) { delete p; }

// ---------------------------------------------------------------------------------------------------------------
// one batch out of several parsed streams
// ---------------------------------------------------------------------------------------------------------------
struct HostBatch {
	std::vector<pov_stream> streams;
	std::vector<pov_packet> packets;
	std::vector<uint16_t> ys;
	std::vector<uint8_t> payload;
	uint64_t pcm_floats = 0;
	bool raw = false;                          // the payload holds raw audio packets (POV_INPUT_PACKETS)
	pov_batch view() const {
		pov_batch b;
		memset(&b, 0, sizeof b);
		b.input_kind = raw ? POV_INPUT_PACKETS : POV_INPUT_ENTRIES; b.pcm_layout = POV_PCM_PLANAR;
		b.n_streams = (uint32_t) streams.size(); b.streams = streams.data();
		b.n_packets = (uint32_t) packets.size(); b.packets = packets.data();
		b.ys = ys.data(); b.n_ys = ys.size();
		b.payload = payload.data(); b.payload_bytes = payload.size();
		b.pcm_floats = pcm_floats;
		return b;
	}
	void clear() { streams.clear(); packets.clear(); ys.clear(); payload.clear(); pcm_floats = 0; }
	void append(const StreamWork& st, uint32_t setup_id) {
		pov_stream rec;
		memset(&rec, 0, sizeof rec);
		rec.setup_id = setup_id; rec.first_packet = (uint32_t) packets.size(); rec.n_packets = (uint32_t) st.packets.size();
		rec.pcm_frames = st.frames; rec.pcm_base = pcm_floats;
		const uint32_t si = (uint32_t) streams.size();
		const uint64_t ybase = ys.size(), pbase = payload.size();
		for(const pov_packet& src : st.packets) {
			pov_packet pk = src;
			pk.stream = si; pk.ys_off += ybase; pk.spec_off += pbase;
			packets.push_back(pk);
		}
		ys.insert(ys.end(), st.ys.begin(), st.ys.end());
		payload.insert(payload.end(), st.payload.begin(), st.payload.end());
		pcm_floats += st.frames * st.setup.channels;
		streams.push_back(rec);
	}
};

static int register_stream_setup_slow(pov_ctx* ctx, const StreamWork& st, uint32_t* id);
static int register_stream_setup(pov_ctx* ctx, const StreamWork& st, uint32_t* id) {
	auto it = ctx->setup_by_key.find(st.setup_key);
	if(it != ctx->setup_by_key.end()) { *id = it->second; return POV_OK; }
	const int rc = register_stream_setup_slow(ctx, st, id);
	if(rc == POV_OK) ctx->setup_by_key[st.setup_key] = *id;
	return rc;
}

static int register_stream_setup_slow(pov_ctx* ctx, const StreamWork& st, uint32_t* id) {
	SetupAbi a;
	std::string why;
	if(!setup_to_abi(st.setup, a, why)) return pov_fail(ctx, POV_ERR_UNSUPPORTED, "unsupported stream: %s", why.c_str());
	return pov_setup_register(ctx, &a.s, id);
}

// Whole-file decode into a pov_decoded (T = float) or pov_decoded_s16 (T = int16_t, POV_PCM_S16 batch; never a debug dump).
template <class T, class Out>
static int decode_memory(pov_ctx* ctx, const uint8_t* data, size_t len, const char* debug_out, Out* out) {
	constexpr bool kS16 = std::is_same<T, int16_t>::value;
	if(!ctx || !out || (!data && len)) return POV_ERR_ARG;
	memset(out, 0, sizeof *out);
	std::vector<StreamWork> streams;
	ParseError err;
	// without a dump the audio packets go to the device as they are (entropy decode there); the dump writer needs the
	// host-side Y lists, so that path keeps the host walk. A file whose streams cannot all be walked on the device is parsed again.
	ParseOptions opt;
	opt.raw_packets = ctx->device_entropy && !debug_out;
	opt.allow_spanning = ctx->allow_spanning;
	for(int attempt = 0; attempt < 2; ++attempt) {
		streams.clear();
		err = ParseError();
		if(!parse_ogg_file(data, len, streams, err, opt)) return pov_fail(ctx, POV_ERR_STREAM, "check failed: %s", err.msg.c_str());
		bool mixed = false;
		for(const StreamWork& st : streams) if(st.have_setup && st.raw != opt.raw_packets) mixed = true;
		if(!mixed) break;
		opt.raw_packets = false;
	}
	// keep the streams that reached their setup header; all must agree on the channel layout to share one PCM array
	std::vector<const StreamWork*> use;
	for(const StreamWork& st : streams) if(st.have_setup) use.push_back(&st);
	if(use.empty()) return POV_OK;                      // nothing decodable: the reference also returns ok
	for(const StreamWork* st : use)
		if(st->setup.channels != use[0]->setup.channels || st->setup.sample_rate != use[0]->setup.sample_rate)
			return pov_fail(ctx, POV_ERR_UNSUPPORTED, "logical streams with different channel layouts in one file");
	if(debug_out && use.size() != 1) return pov_fail(ctx, POV_ERR_UNSUPPORTED, "debug dump needs exactly one logical stream");
	HostBatch hb;
	hb.raw = opt.raw_packets;
	for(const StreamWork* st : use) {
		uint32_t id = 0;
		int rc = register_stream_setup(ctx, *st, &id);
		if(rc) return rc;
		hb.append(*st, id);
	}
	const uint32_t C = use[0]->setup.channels;
	out->channels = C; out->sample_rate = use[0]->setup.sample_rate;
	out->audio_packets = (uint32_t) hb.packets.size();
	uint64_t frames = 0;
	for(const StreamWork* st : use) frames += st->frames;
	out->frames = frames;
	if(hb.packets.empty()) return POV_OK;

	pov_batch b = hb.view();
	if(kS16) b.pcm_layout |= POV_PCM_S16;
	pov_batch_handle* h = nullptr;
	int rc = pov_batch_upload(ctx, &b, &h);
	if(rc) return rc;
	rc = debug_out ? pov_batch_run_staged(ctx, h) : pov_batch_run(ctx, h);
	std::vector<T> arena(hb.pcm_floats);
	if(!rc) {
		if constexpr(kS16) rc = pov_batch_fetch_pcm_s16(ctx, h, arena.data(), arena.size(), 1);
		else rc = pov_batch_fetch_pcm(ctx, h, arena.data(), arena.size(), 1);
	}
	if(!rc) rc = pov_batch_status(ctx, h, nullptr, 0);
	if constexpr(!kS16) {
		if(!rc && debug_out) {
			StageHost sg;
			rc = pov_batch_fetch_stage_all(ctx, h, sg);
			std::string werr;
			if(!rc && !write_debug_dump(debug_out, *use[0], *h, 0, sg, arena.data(), werr)) rc = pov_fail(ctx, POV_ERR_ARG, "debug dump: %s", werr.c_str());
		}
	}
	pov_batch_free(ctx, h);
	if(rc) return rc;
	// planar [C][frames] across the (chained) streams
	T* pcm = (T*) malloc(sizeof(T) * std::max<uint64_t>(1, frames * C));
	if(!pcm) return pov_fail(ctx, POV_ERR_ARG, "out of memory");
	uint64_t at = 0;
	for(size_t i = 0; i < use.size(); ++i) {
		const pov_stream& rec = hb.streams[i];
		for(uint32_t c = 0; c < C; ++c)
			memcpy(pcm + (uint64_t) c * frames + at, arena.data() + rec.pcm_base + (uint64_t) c * rec.pcm_frames, sizeof(T) * rec.pcm_frames);
		at += rec.pcm_frames;
	}
	out->pcm = pcm;
	return POV_OK;
}

extern "C" int pov_ogg_vorbis_decode_memory(pov_ctx* ctx, const uint8_t* data, size_t len, const char* debug_out, pov_decoded* out) try {
	return decode_memory<float>(ctx, data, len, debug_out, out);
} POV_NOTHROW_END(ctx)

extern "C" int pov_ogg_vorbis_decode_memory_s16(pov_ctx* ctx, const uint8_t* data, size_t len, pov_decoded_s16* out) try {
	return decode_memory<int16_t>(ctx, data, len, nullptr, out);
} POV_NOTHROW_END(ctx)

extern "C" void pov_decoded_free(pov_decoded* d) {
	if(!d) return;
	free(d->pcm);
	d->pcm = nullptr;
}

extern "C" void pov_decoded_s16_free(pov_decoded_s16* d) {
	if(!d) return;
	free(d->pcm);
	d->pcm = nullptr;
}

// ---------------------------------------------------------------------------------------------------------------
// one file of a corpus: the parse of the stream table and of the corpus decode's workers
// ---------------------------------------------------------------------------------------------------------------
// Parses file k into `file` and appends the record of every stream that reaches its setup header to `info`. A framing or
// header error returns false with the corpus decode's text in `error`; with opt.cut_damage the file is cut there instead, and
// the same text goes to `damage`.
static bool parse_corpus_file(uint32_t k, const uint8_t* data, size_t len, const ParseOptions& opt, std::vector<StreamWork>& file,
                              std::vector<pov_stream_info>& info, std::string& error, std::string& damage) {
	ParseError err;
	file.clear();
	damage.clear();
	const bool ok = parse_ogg_file(data, len, file, err, opt);
	if(!ok || err.cut) (ok ? damage : error) = "file " + std::to_string(k) + ": check failed: " + err.msg;
	if(!ok) return false;
	for(const StreamWork& st : file) {
		if(!st.have_setup) continue;
		pov_stream_info r = {};
		r.file = k; r.channels = st.setup.channels; r.sample_rate = st.setup.sample_rate; r.frames = st.frames;
		info.push_back(r);
	}
	return true;
}

extern "C" int pov_corpus_streams(uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t flags, uint32_t host_threads,
                                  pov_stream_info** out, uint64_t* n_streams_out, const char** error_out) {
	static thread_local char errbuf[512];
	if(!out || !n_streams_out || (n_files && (!data || !len))) return POV_ERR_ARG;
	*out = nullptr; *n_streams_out = 0;
	try {
	if(host_threads == 0) { const uint32_t hc = std::thread::hardware_concurrency(); host_threads = hc > 1 ? hc - 1 : 1; }
	host_threads = std::max(1u, std::min(host_threads, n_files));
	std::vector<std::vector<pov_stream_info>> per_file(n_files);
	std::vector<std::string> error(n_files);
	std::atomic<uint32_t> next(0), first_error(n_files);
	ParseOptions opt;
	opt.raw_packets = true;
	opt.allow_spanning = (flags & POV_PARSE_ALLOW_SPANNING) != 0;
	opt.cut_damage = (flags & POV_PARSE_CUT_DAMAGE) != 0;
	auto worker = [&]() {
		std::vector<StreamWork> file;
		std::string damage;
		for(;;) {
			const uint32_t i = next.fetch_add(1);
			if(i >= n_files || i > first_error.load()) return;          // (files after a failed one are not needed)
			bool ok = false;
			try {
				ok = parse_corpus_file(i, data[i], len[i], opt, file, per_file[i], error[i], damage);
			} catch(...) {
				error[i] = "file " + std::to_string(i) + ": out of memory or internal error while parsing";
			}
			uint32_t f = first_error.load();                           // the lowest failing index wins
			while(!ok && i < f && !first_error.compare_exchange_weak(f, i)) {}
		}
	};
	std::vector<std::thread> pool;
	for(uint32_t t = 1; t < host_threads; ++t) pool.emplace_back(worker);
	worker();
	for(auto& t : pool) t.join();
	if(first_error.load() < n_files) {
		snprintf(errbuf, sizeof errbuf, "%s", error[first_error.load()].c_str());
		if(error_out) *error_out = errbuf;
		return POV_ERR_STREAM;
	}
	uint64_t n = 0;
	for(const auto& v : per_file) n += v.size();
	if(n) {
		pov_stream_info* p = (pov_stream_info*) malloc(n * sizeof(pov_stream_info));
		if(!p) throw std::bad_alloc();
		uint64_t at = 0;
		for(const auto& v : per_file) { memcpy(p + at, v.data(), v.size() * sizeof(pov_stream_info)); at += v.size(); }
		*out = p;
	}
	*n_streams_out = n;
	return POV_OK;
	} catch(...) {
		snprintf(errbuf, sizeof errbuf, "out of memory or internal error while building the stream table");
		if(error_out) *error_out = errbuf;
		return POV_ERR_ARG;
	}
}

extern "C" void pov_corpus_streams_free(pov_stream_info* p) { free(p); }

// ---------------------------------------------------------------------------------------------------------------
// corpus decode: `host_threads` front-end workers parse files into chunks, the calling thread feeds the GPU
// ---------------------------------------------------------------------------------------------------------------
namespace {
struct CorpusState;

// A chunk leaves its worker as one assembled batch in pinned host memory: the calling thread only turns the chunk-local
// setup numbers into registered setup ids (one map lookup per distinct setup, normally one per chunk), validates the
// descriptors and queues the copies, which then run as plain DMA.
struct Chunk {
	CorpusState* pool = nullptr;               // `buf` goes back to its pool when the chunk is destroyed
	uint32_t first_file = 0, n_files = 0;
	PinnedBuf buf;                             // streams | packets | ys | payload, each 16-byte aligned
	pov_batch view = {};                       // pointers into buf; pov_stream::setup_id = index into `setups` until patched
	pov_stream* streams = nullptr;             // writable alias of view.streams
	std::vector<StreamWork> setups;            // one representative stream (headers only) per distinct setup
	std::vector<pov_stream_info> info;         // every stream that reached its setup header, in file order (= the batch's streams)
	std::string error;
	// cut mode: per file the geometry damage text ("" if none), per stream (as `info`) the packet whose host walk failed and the
	// reason to report for it, and the index of the chunk's first stream among the call's stream-table records
	std::vector<std::string> damage;
	std::vector<uint32_t> walk_bad;
	std::vector<std::string> walk_text;
	uint64_t first_record = 0;
	Chunk(CorpusState* pool, uint32_t first_file, uint32_t n_files) : pool(pool), first_file(first_file), n_files(n_files) {}
	~Chunk();
};

// Output format of a corpus decode: float32 (sink, checksum), int16 (POV_PCM_S16: sink16, sum16), or the caller's device
// memory (dev: float32 or int16 by dev->pcm_layout; no PCM leaves the device), optionally resampled / downmixed (rs: the
// synthesis writes a float32 arena of the slot, the resample kernel the caller's memory).
struct CorpusOut {
	bool s16 = false;
	const pov_device_pcm* dev = nullptr;
	const pov_resample* rs = nullptr;
	pov_pcm_sink sink = nullptr;
	pov_pcm_sink_s16 sink16 = nullptr;
	void* user = nullptr;
	double* checksum = nullptr;
	int64_t* sum16 = nullptr;
	bool cut = false;                          // cut mode (pov_ctx_set_cut_damage): k_cut_damaged runs after the synthesis
	uint32_t pcm_layout() const { return POV_PCM_PLANAR | (s16 ? POV_PCM_S16 : 0u); }     // of the chunks' batches
	bool has_sink() const { return s16 ? sink16 != nullptr : sink != nullptr; }
	int deliver(const pov_stream_info& s, uint64_t frames, const void* planar) const {
		return s16 ? sink16(s.file, s.channels, frames, (const int16_t*) planar, user) : sink(s.file, s.channels, frames, (const float*) planar, user);
	}
};

// Where a chunk's PCM goes (place_chunk).
struct Placement {
	uint64_t arena = 0;                        // pov_batch::pcm_floats of the upload: the slot's arena, or the caller's capacity
	uint64_t values = 0;                       // samples the chunk yields
	bool into_caller = false;                  // the synthesis writes the caller's memory (pov_batch_upload_into)
	size_t host_bytes = 0;                     // host output: PCM bytes summed and copied to the slot's pinned buffer
	std::vector<ResampleDesc> rs;              // resampled output: slot arena -> caller's memory, one launch of rs_tiles blocks
	uint64_t rs_tiles = 0;
	std::vector<CutDesc> cut;                  // cut mode: every stream where the synthesis writes it, one launch of cut_tiles blocks
	uint64_t cut_tiles = 0;
};

// POV_CORPUS_TIMING=1: where the calling thread's time goes (stderr), to tell a starved consumer from a slow one, and what the
// slot streams spent in copy-in + kernels and in copy-out; =2 adds a per-chunk timeline. Both come from four events per chunk
// on the slot streams (queued, copy-in done, kernels done, copy-out done). Without the variable every call is a no-op.
struct CorpusTiming {
	enum Phase { kWait, kRetire, kUpload, kFetch, kRun };     // the calling thread's intervals (the first four: timeline columns)
	bool on = false, timeline = false;
	double t_begin = 0, t_last = 0, host[5] = {0, 0, 0, 0, 0};
	std::vector<cudaEvent_t> ev;                               // 4 per chunk
	std::vector<double> tl_host;                               // 4 per chunk, host clock: chunk taken, slot free, upload queued, all queued

	static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
	explicit CorpusTiming(uint32_t n_chunks) {
		const char* e = getenv("POV_CORPUS_TIMING");
		on = e != nullptr;
		timeline = on && atoi(e) >= 2;
		ev.assign(on ? 4 * (size_t) n_chunks : 0, nullptr);
		for(cudaEvent_t& x : ev) cudaEventCreate(&x);
		tl_host.assign(ev.size(), 0.0);
		t_begin = t_last = now();
	}
	~CorpusTiming() { for(cudaEvent_t x : ev) if(x) cudaEventDestroy(x); }
	void mark(Phase p, uint32_t ci) {                          // the calling thread ends phase p of chunk ci
		if(!on) return;
		const double t = now();
		host[p] += t - t_last;
		t_last = t;
		if(p != kRun) tl_host[4 * (size_t) ci + p] = t - t_begin;
	}
	void event(uint32_t ci, int k, cudaStream_t st) { if(on) cudaEventRecord(ev[4 * (size_t) ci + k], st); }
	void report(const std::vector<uint32_t>& chunk_first) {
		if(!on) return;
		const uint32_t n_chunks = (uint32_t) chunk_first.size() - 1;
		double copy_in_kernels = 0, copy_out = 0;              // ms, summed over the chunks
		for(uint32_t ci = 0; ci < n_chunks; ++ci) {
			float a = 0, b = 0;
			if(cudaEventElapsedTime(&a, ev[4 * ci], ev[4 * ci + 2]) == cudaSuccess && cudaEventElapsedTime(&b, ev[4 * ci + 2], ev[4 * ci + 3]) == cudaSuccess) { copy_in_kernels += a; copy_out += b; }
		}
		fprintf(stderr, "pov_decode_corpus: %u chunks in %.3f s on the calling thread: wait for parsed chunks %.3f, "
		        "setup ids + wait for the slot %.3f, validate+queue upload %.3f, launch %.3f, fetch/issue %.3f; on the streams (sum over chunks): "
		        "copy in + kernels %.3f s, copy out %.3f s\n",
		        n_chunks, now() - t_begin, host[kWait], host[kRetire], host[kUpload], host[kRun], host[kFetch], copy_in_kernels * 1e-3, copy_out * 1e-3);
		if(timeline) for(uint32_t ci = 0; ci < n_chunks; ++ci) {
			float t[4] = {-1, -1, -1, -1};
			for(int k = 0; k < 4; ++k) if(cudaEventElapsedTime(&t[k], ev[0], ev[4 * ci + k]) != cudaSuccess) t[k] = -1;
			fprintf(stderr, "chunk %3u files %4u..%4u: queued %8.3f copy-in done %8.3f kernels done %8.3f copy-out done %8.3f ms | host: taken %8.3f "
			        "slot free %8.3f upload queued %8.3f all queued %8.3f ms\n", ci, chunk_first[ci], chunk_first[ci + 1], t[0], t[1], t[2], t[3],
			        tl_host[4 * ci] * 1e3, tl_host[4 * ci + 1] * 1e3, tl_host[4 * ci + 2] * 1e3, tl_host[4 * ci + 3] * 1e3);
		}
		(void) cudaGetLastError();                              // (chunks without audio packets record no events)
	}
};

// What pov_decode_corpus keeps between calls on a context: the sibling contexts (a stream each), the batch slots with their
// pinned PCM and status buffers, the pool of pinned staging buffers the workers assemble chunks into, and the filter tables.
struct CorpusState {
	int device = 0;
	static constexpr int kSlots = 4;           // chunks in flight: while two copy their PCM out, the others compute (the copy-out,
	                                           // 4 bytes per PCM sample over PCIe, is the bound of the whole decode)
	pov_ctx* sibling[kSlots - 1] = {nullptr};
	struct Slot {
		pov_ctx* ctx = nullptr;                // slot 0: the caller's context; the others: a sibling each, so that the copies of
		                                       // one chunk never wait for another chunk's work
		void* d_sum = nullptr;                 // 8 bytes: float64 checksum, or the int64 sum of an int16 decode
		pov_batch_handle* h = nullptr;
		PinnedBuf pinned, status;              // the chunk's PCM arena (float or int16) and its status words
		PinnedBuf rs_host;                     // resampled output: the chunk's descriptors (pinned source of their upload)
		DevBuf rs_dev;
		PinnedBuf cut_host, cut_res;           // cut mode: the chunk's CutDesc (source of their upload) and CutResult (copied back)
		DevBuf cut_dev, cut_res_dev;
		cudaEvent_t done = nullptr;
		uint32_t n_packets = 0;                // status words retire() checks (0: the chunk did not reach its copy-out)
		std::unique_ptr<Chunk> in_flight;      // its pinned buffer is the source of copies that may still be running
		int submit(pov_ctx* caller, std::unique_ptr<Chunk> ck, const Placement& pl, const CorpusOut& fmt, CorpusTiming& tm, uint32_t ci);
		int retire(pov_ctx* caller, const CorpusOut& fmt, bool& stopped);
		void report_cuts(pov_ctx* caller) const;
	} slot[kSlots];
	std::mutex pmu;
	std::condition_variable pcv;
	std::vector<PinnedBuf> free_bufs;
	uint32_t n_bufs = 0, max_bufs = 0;
	struct Filter { float* taps = nullptr; uint32_t K = 0, hl = 0; };
	std::map<std::pair<uint32_t, uint32_t>, Filter> filters;   // by (L, M): polyphase tables [K][L] on the device, shared by the slots

	PinnedBuf acquire(size_t need, const std::atomic<bool>& stop) {
		PinnedBuf b;
		{
			std::unique_lock<std::mutex> lk(pmu);
			pcv.wait(lk, [&] { return !free_bufs.empty() || n_bufs < max_bufs || stop.load(); });
			if(!free_bufs.empty()) { b = free_bufs.back(); free_bufs.pop_back(); }
			else if(n_bufs < max_bufs) ++n_bufs;
			else return b;                         // stopping
		}
		if(b.reserve(need) != cudaSuccess) {
			std::lock_guard<std::mutex> lk(pmu);
			--n_bufs;                              // the buffer this call stood for no longer exists
			pcv.notify_one();
		}
		return b;
	}
	void release(PinnedBuf b) {
		if(!b.ptr) return;
		std::lock_guard<std::mutex> lk(pmu);
		free_bufs.push_back(b);
		pcv.notify_one();
	}
	~CorpusState() {
		cudaSetDevice(device);
		for(auto& sl : slot) {
			if(!sl.ctx) continue;
			cudaStreamSynchronize(sl.ctx->stream);
			sl.in_flight.reset();
			if(sl.h) pov_batch_free(sl.ctx, sl.h);
			sl.pinned.release(); sl.status.release(); sl.rs_host.release(); sl.rs_dev.release();
			sl.cut_host.release(); sl.cut_res.release(); sl.cut_dev.release(); sl.cut_res_dev.release();
			if(sl.done) cudaEventDestroy(sl.done);
			if(sl.d_sum) cudaFree(sl.d_sum);
		}
		for(auto& b : free_bufs) b.release();
		for(auto& f : filters) if(f.second.taps) cudaFree(f.second.taps);
		for(pov_ctx* sb : sibling) if(sb) pov_ctx_destroy(sb);
	}
};
Chunk::~Chunk() { if(pool) pool->release(buf); }
void corpus_state_free(void* p) { delete (CorpusState*) p; }

inline size_t align16(size_t x) { return (x + 15) & ~(size_t) 15; }

// Chunks on their way from the workers, which finish them in any order, to the calling thread, which takes them in order.
struct ChunkQueue {
	CorpusState& cs;
	const uint32_t max_ready;
	std::mutex mu;
	std::condition_variable cv_ready, cv_space;
	std::map<uint32_t, std::unique_ptr<Chunk>> ready;    // by chunk index
	uint32_t consumed = 0;                               // chunks handed to the calling thread so far (guarded by mu)
	std::atomic<bool> stop{false};
	std::vector<std::thread> pool;

	ChunkQueue(CorpusState& cs, uint32_t max_ready) : cs(cs), max_ready(max_ready) {}
	~ChunkQueue() { close(); }                           // the pool is joined on every way out (an exception included)
	// Back-pressure by chunk INDEX, not by count: the chunk the consumer is waiting for always passes, however many later
	// chunks the other workers have finished in the meantime (a count limit can fill the queue with later chunks and then
	// block the one worker that holds the chunk everybody is waiting for).
	void put(uint32_t ci, std::unique_ptr<Chunk> ck) {
		std::unique_lock<std::mutex> lk(mu);
		cv_space.wait(lk, [&] { return ci < consumed + max_ready || stop.load(); });
		ready[ci] = std::move(ck);
		cv_ready.notify_all();
	}
	std::unique_ptr<Chunk> take(uint32_t ci) {
		std::unique_lock<std::mutex> lk(mu);
		cv_ready.wait(lk, [&] { return ready.count(ci) != 0; });
		std::unique_ptr<Chunk> ck = std::move(ready[ci]);
		ready.erase(ci);
		consumed = ci + 1;
		cv_space.notify_all();
		return ck;
	}
	void close() {                                       // stops and joins the workers; chunks nobody took are dropped
		stop.store(true);
		{ std::lock_guard<std::mutex> lk(mu); cv_space.notify_all(); }
		{ std::lock_guard<std::mutex> lk(cs.pmu); cs.pcv.notify_all(); }
		for(auto& t : pool) if(t.joinable()) t.join();
		ready.clear();
	}
};
}  // namespace

static int decode_corpus(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t host_threads,
                         const CorpusOut& fmt, uint64_t* frames_out, uint64_t* total_values_out);

// Every corpus entry point starts here: whatever way the call fails, pov_corpus_report then has no report to give.
static void corpus_call_begins(pov_ctx* ctx) { if(ctx) ctx->corpus_report_ok = false; }

extern "C" int pov_decode_corpus(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len,
                                 uint32_t host_threads, uint64_t* frames_out, uint64_t* total_values_out, double* checksum_out) try {
	corpus_call_begins(ctx);
	CorpusOut fmt;
	fmt.checksum = checksum_out;
	return decode_corpus(ctx, n_files, data, len, host_threads, fmt, frames_out, total_values_out);
} POV_NOTHROW_END(ctx)

extern "C" int pov_decode_corpus_pcm(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t host_threads,
                                     pov_pcm_sink sink, void* user, uint64_t* frames_out, uint64_t* total_values_out, double* checksum_out) try {
	corpus_call_begins(ctx);
	if(!sink) return pov_fail(ctx, POV_ERR_ARG, "pov_decode_corpus_pcm: null sink");
	CorpusOut fmt;
	fmt.sink = sink; fmt.user = user; fmt.checksum = checksum_out;
	return decode_corpus(ctx, n_files, data, len, host_threads, fmt, frames_out, total_values_out);
} POV_NOTHROW_END(ctx)

extern "C" int pov_decode_corpus_s16(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t host_threads,
                                     pov_pcm_sink_s16 sink, void* user, uint64_t* frames_out, uint64_t* total_values_out, int64_t* sum_out) try {
	corpus_call_begins(ctx);
	CorpusOut fmt;
	fmt.s16 = true; fmt.sink16 = sink; fmt.user = user; fmt.sum16 = sum_out;
	return decode_corpus(ctx, n_files, data, len, host_threads, fmt, frames_out, total_values_out);
} POV_NOTHROW_END(ctx)

// Everything about the caller's regions that can be checked before a launch: pov_decode_corpus_device writes nothing otherwise.
// Stream i's region holds out_ch[i] channels of out_frames[i] frames (the table's channels and frames without resampling).
static int validate_device_pcm(pov_ctx* ctx, const pov_device_pcm* o, const uint32_t* out_ch, const uint64_t* out_frames, const char* fn) {
	if(!o) return pov_fail(ctx, POV_ERR_ARG, "%s: null output description", fn);
	if((o->pcm_layout & ~POV_PCM_S16) != POV_PCM_PLANAR) return pov_fail(ctx, POV_ERR_ARG, "%s: pcm_layout 0x%x: only POV_PCM_PLANAR, optionally | POV_PCM_S16", fn, o->pcm_layout);
	const uint32_t n = o->n_streams;
	if(n == 0) return POV_OK;
	if(!o->stream_base || !o->channel_stride || !o->file || !o->channels || !o->frames) return pov_fail(ctx, POV_ERR_ARG, "%s: null table arrays", fn);
	int rc = pov_check_pcm_dev(ctx, o->pcm_dev, pcm_elem_bytes(o->pcm_layout), fn);
	if(rc) return rc;
	if(o->capacity > SIZE_MAX / pcm_elem_bytes(o->pcm_layout)) return pov_fail(ctx, POV_ERR_ARG, "%s: capacity of %llu samples does not fit the address space", fn, (unsigned long long) o->capacity);
	std::vector<uint32_t> order(n);
	for(uint32_t i = 0; i < n; ++i) {
		const uint64_t base = o->stream_base[i], stride = o->channel_stride[i], C = out_ch[i];
		if(o->channels[i] == 0 || o->channels[i] > POV_MAX_CHANNELS) return pov_fail(ctx, POV_ERR_ARG, "%s: stream %u: %u channels", fn, i, o->channels[i]);
		if(stride < out_frames[i]) return pov_fail(ctx, POV_ERR_ARG, "%s: stream %u: channel stride %llu < %llu frames", fn, i, (unsigned long long) stride, (unsigned long long) out_frames[i]);
		if(base > o->capacity || stride > (o->capacity - base) / C)          // (subtraction form: nothing may wrap)
			return pov_fail(ctx, POV_ERR_ARG, "%s: stream %u: region [%llu, +%llu x %llu) exceeds the capacity of %llu samples", fn, i,
			                (unsigned long long) base, (unsigned long long) C, (unsigned long long) stride, (unsigned long long) o->capacity);
		order[i] = i;
	}
	std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return o->stream_base[a] < o->stream_base[b]; });
	uint64_t end = 0;                                  // end of the regions before, in base order (empty regions overlap nothing)
	uint32_t last = 0;
	for(uint32_t b : order) {
		if(o->channel_stride[b] == 0) continue;
		if(o->stream_base[b] < end) return pov_fail(ctx, POV_ERR_ARG, "%s: the regions of streams %u and %u overlap", fn, last, b);
		const uint64_t e = o->stream_base[b] + out_ch[b] * o->channel_stride[b];
		if(e > end) { end = e; last = b; }
	}
	return POV_OK;
}

extern "C" int pov_decode_corpus_device(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t host_threads,
                                        const pov_device_pcm* out, uint64_t* frames_out, uint64_t* total_values_out) try {
	corpus_call_begins(ctx);
	if(!ctx) return POV_ERR_ARG;
	cudaSetDevice(ctx->device);
	const bool tables = out && out->n_streams && out->channels && out->frames;
	const int rc = validate_device_pcm(ctx, out, tables ? out->channels : nullptr, tables ? out->frames : nullptr, "pov_decode_corpus_device");
	if(rc) return rc;
	CorpusOut fmt;
	fmt.s16 = (out->pcm_layout & POV_PCM_S16) != 0; fmt.dev = out;
	return decode_corpus(ctx, n_files, data, len, host_threads, fmt, frames_out, total_values_out);
} POV_NOTHROW_END(ctx)

// (L, M) of stream i of a resampled decode; the ratio was checked before the decode started
static void stream_ratio(const pov_resample& rs, uint32_t in_rate, uint32_t* L, uint32_t* M) {
	uint32_t hl = 0;
	if(rs.out_rate == 0) { *L = *M = 1; return; }
	resample_design(in_rate, rs.out_rate, L, M, &hl, nullptr);
}

extern "C" int pov_decode_corpus_device_resampled(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len,
                                                  uint32_t host_threads, const pov_device_pcm* out, const pov_resample* rs,
                                                  uint64_t* frames_out, uint64_t* total_values_out) try {
	corpus_call_begins(ctx);
	if(!ctx) return POV_ERR_ARG;
	cudaSetDevice(ctx->device);
	const char* fn = "pov_decode_corpus_device_resampled";
	if(!out) return pov_fail(ctx, POV_ERR_ARG, "%s: null output description", fn);
	if(!rs) return pov_fail(ctx, POV_ERR_ARG, "%s: null resample description", fn);
	if(rs->flags & ~POV_RESAMPLE_MONO) return pov_fail(ctx, POV_ERR_ARG, "%s: flags 0x%x: only POV_RESAMPLE_MONO", fn, rs->flags);
	const uint32_t n = out->n_streams;
	if(n && !rs->sample_rate) return pov_fail(ctx, POV_ERR_ARG, "%s: null sample_rate table", fn);
	const bool tables = n && out->channels && out->frames;
	std::vector<uint32_t> och(tables ? n : 0);
	std::vector<uint64_t> ofr(tables ? n : 0);
	for(uint32_t i = 0; i < n; ++i) {
		const uint32_t in = rs->sample_rate[i];
		uint32_t L = 1, M = 1, hl = 0;
		if(in == 0) return pov_fail(ctx, POV_ERR_ARG, "%s: stream %u: sample rate 0", fn, i);
		if(rs->out_rate && !resample_design(in, rs->out_rate, &L, &M, &hl, nullptr))
			return pov_fail(ctx, POV_ERR_UNSUPPORTED, "%s: stream %u: %u Hz -> %u Hz needs %u filter phases (max(L, M) for L = %u, M = %u), "
			                "past the supported %u", fn, i, in, rs->out_rate, std::max(L, M), L, M, POV_RESAMPLE_MAX_PHASES);
		if(tables) {
			och[i] = (rs->flags & POV_RESAMPLE_MONO) ? 1 : out->channels[i];
			ofr[i] = resample_frames(out->frames[i], L, M);
		}
	}
	const int rc = validate_device_pcm(ctx, out, och.data(), ofr.data(), fn);
	if(rc) return rc;
	CorpusOut fmt;
	fmt.dev = out; fmt.rs = rs;                // the slots' arenas are float32 whatever the output type
	return decode_corpus(ctx, n_files, data, len, host_threads, fmt, frames_out, total_values_out);
} POV_NOTHROW_END(ctx)

// The device table of ratio (L, M) in the kernel's order, [K][L] with K = ceil(N / L) and zeros past N; built on the calling
// thread the first time the ratio appears and kept for the context's lifetime. A copy (L = M = 1) has none.
static int resample_filter_table(pov_ctx* ctx, CorpusState& cs, uint32_t L, uint32_t M, const float** taps, uint32_t* K, uint32_t* hl) {
	*taps = nullptr; *K = 0; *hl = 0;
	if(L == 1 && M == 1) return POV_OK;
	CorpusState::Filter& f = cs.filters[std::make_pair(L, M)];
	if(!f.taps) {
		uint32_t l = 0, m = 0, h = 0;
		std::vector<float> taps_h;
		if(!resample_design(M, L, &l, &m, &h, &taps_h)) return pov_fail(ctx, POV_ERR_UNSUPPORTED, "resample ratio %u/%u past the supported phases", L, M);
		const uint32_t N = (uint32_t) taps_h.size(), k_n = (N + L - 1) / L;
		std::vector<float> poly((size_t) k_n * L, 0.0f);
		for(uint32_t k = 0; k < k_n; ++k)
			for(uint32_t p = 0; p < L && p + k * L < N; ++p) poly[(size_t) k * L + p] = taps_h[p + k * L];
		cudaError_t e = cudaMalloc((void**) &f.taps, poly.size() * sizeof(float));
		if(e == cudaSuccess) e = cudaMemcpy(f.taps, poly.data(), poly.size() * sizeof(float), cudaMemcpyHostToDevice);
		if(e != cudaSuccess) {
			if(f.taps) cudaFree(f.taps);
			f.taps = nullptr;
			return pov_fail(ctx, POV_ERR_CUDA, "resample filter table: %s", cudaGetErrorString(e));
		}
		f.K = k_n; f.hl = h;
	}
	*taps = f.taps; *K = f.K; *hl = f.hl;
	return POV_OK;
}

// chunk_first[k] = index of chunk k's first file; the last entry is n_files.
static std::vector<uint32_t> chunk_bounds(const pov_ctx* ctx, uint32_t n_files) {
	// Files per chunk: with the entropy decode on the device a chunk's kernels are latency bound (one thread walks one packet),
	// so more packets per launch cost nothing and the PCM copy-out — the PCIe bound of the whole decode — runs in long
	// transfers; with the host walk smaller chunks keep the parser threads and the device overlapped.
	uint32_t files_per_chunk = ctx->device_entropy ? 256 : 64;
	if(const char* e = getenv("POV_CORPUS_CHUNK")) files_per_chunk = std::max(1, atoi(e));
	// The first chunks are small and grow by half each (1/8 of the size, then x 1.5): every worker starts on a chunk of its own
	// at once, one worker parses a file in about twice the time the copy-out of its PCM takes, so chunk k is ready just before
	// the copy-out of chunks 0..k-1 ends and the link never waits for a parser.
	std::vector<uint32_t> chunk_first;
	uint32_t at = 0, size = std::max(1u, files_per_chunk / 8);
	while(at < n_files) {
		chunk_first.push_back(at);
		at += std::min(size, n_files - at);
		size = std::min(files_per_chunk, size + (size + 1) / 2);
	}
	chunk_first.push_back(n_files);
	return chunk_first;
}

// Creates ctx->corpus, the CorpusState, on the context's first corpus decode.
static int make_corpus_state(pov_ctx* ctx) {
	if(ctx->corpus) return POV_OK;
	std::unique_ptr<CorpusState> cs(new CorpusState());
	cs->device = ctx->device;
	const char* e = nullptr;
	cs->slot[0].ctx = ctx;
	for(int k = 1; k < CorpusState::kSlots; ++k) {
		if(pov_ctx_create(ctx->device, &cs->sibling[k - 1], &e) != POV_OK) return pov_fail(ctx, POV_ERR_CUDA, "pov_decode_corpus: %s", e ? e : "sibling context");
		cs->sibling[k - 1]->device_entropy = ctx->device_entropy;
		cs->slot[k].ctx = cs->sibling[k - 1];
	}
	for(auto& sl : cs->slot) {
		if(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming) != cudaSuccess || cudaMalloc(&sl.d_sum, 8) != cudaSuccess)
			return pov_fail(ctx, POV_ERR_CUDA, "pov_decode_corpus: cudaEventCreate / cudaMalloc failed");
	}
	ctx->corpus = cs.release();
	ctx->corpus_free = corpus_state_free;
	return POV_OK;
}

// A worker's job: parse the chunk's files into one batch, then copy it into a pinned buffer of the pool. When any stream of
// the chunk cannot be walked on the device, the whole chunk is parsed again with the host walk. Failures go to ck.error.
static void assemble_chunk(Chunk& ck, const uint8_t* const* data, const size_t* len, ParseOptions opt, uint32_t pcm_layout,
                           const std::atomic<bool>& stop, HostBatch& hb, std::vector<StreamWork>& file) {
	for(int attempt = 0; attempt < 2; ++attempt) {
		bool mixed = false;
		hb.clear(); hb.raw = opt.raw_packets;
		ck.setups.clear(); ck.info.clear(); ck.walk_bad.clear(); ck.walk_text.clear();
		ck.damage.assign(opt.cut_damage ? ck.n_files : 0, std::string());
		std::string damage;
		for(uint32_t f = ck.first_file; f < ck.first_file + ck.n_files; ++f) {
			if(!parse_corpus_file(f, data[f], len[f], opt, file, ck.info, ck.error, damage)) return;
			if(opt.cut_damage) ck.damage[f - ck.first_file] = damage;
			for(StreamWork& st : file) {
				if(!st.have_setup) continue;
				if(st.raw != opt.raw_packets) mixed = true;
				if(opt.cut_damage) {
					ck.walk_bad.push_back(st.walk_bad);
					ck.walk_text.push_back(st.walk_status ? pov_status_text(st.walk_status) : st.walk_msg);
				}
				uint32_t k = 0;
				while(k < ck.setups.size() && ck.setups[k].setup_key != st.setup_key) ++k;
				hb.append(st, k);
				if(k == ck.setups.size()) {
					st.packets.clear(); st.ys.clear(); st.payload.clear();
					ck.setups.push_back(std::move(st));
				}
			}
		}
		if(!mixed) break;
		opt.raw_packets = false;
	}
	if(hb.packets.empty()) return;
	// pageable vectors -> one pinned buffer (this copy runs on the worker, the DMA later needs no staging)
	const size_t o_st = 0, o_pk = o_st + align16(hb.streams.size() * sizeof(pov_stream)),
	             o_ys = o_pk + align16(hb.packets.size() * sizeof(pov_packet)), o_pl = o_ys + align16(hb.ys.size() * sizeof(uint16_t)),
	             need = o_pl + align16(hb.payload.size());
	ck.buf = ck.pool->acquire(need, stop);
	if(!ck.buf.ptr) { if(!stop.load()) ck.error = "pov_decode_corpus: pinned staging buffer allocation failed"; return; }
	uint8_t* q = (uint8_t*) ck.buf.ptr;
	memcpy(q + o_st, hb.streams.data(), hb.streams.size() * sizeof(pov_stream));
	memcpy(q + o_pk, hb.packets.data(), hb.packets.size() * sizeof(pov_packet));
	memcpy(q + o_ys, hb.ys.data(), hb.ys.size() * sizeof(uint16_t));
	memcpy(q + o_pl, hb.payload.data(), hb.payload.size());
	ck.view = hb.view();                       // with every pointer moved into the pinned buffer
	ck.view.pcm_layout = pcm_layout;
	ck.streams = (pov_stream*) (q + o_st);
	ck.view.streams = ck.streams; ck.view.packets = (const pov_packet*) (q + o_pk);
	ck.view.ys = (const uint16_t*) (q + o_ys); ck.view.payload = q + o_pl;
}

// Cut mode: a descriptor per stream of a chunk with audio packets, from the base and channel stride place_chunk gave its record.
static int place_cuts(const CorpusOut& fmt, const Chunk& ck, Placement& pl) {
	pl.cut.clear();
	pl.cut_tiles = 0;
	if(!fmt.cut || ck.view.n_packets == 0) return POV_OK;
	for(uint32_t i = 0; i < ck.view.n_streams; ++i) {
		const pov_stream& rec = ck.streams[i];
		CutDesc d;
		memset(&d, 0, sizeof d);
		d.base = rec.pcm_base; d.stride = rec.pcm_frames; d.frames = ck.info[i].frames;
		d.first_packet = rec.first_packet; d.n_packets = rec.n_packets; d.walk_bad = ck.walk_bad[i]; d.channels = ck.info[i].channels;
		d.tiles = std::max<uint64_t>(1, (d.frames + kCutTile - 1) / kCutTile);
		d.tile_first = pl.cut_tiles;
		pl.cut_tiles += d.channels * d.tiles;
		pl.cut.push_back(d);
	}
	return POV_OK;
}

// Where the chunk's PCM goes. Host output: packed in the slot's arena as assembled. Device output: each parsed stream is
// checked against the caller's record at its index (`next_record` counts the records over the call) and pointed at the
// caller's region (the kernels address planar PCM as pcm_base + c * pcm_frames + f, so pcm_frames is the channel stride).
// Resampled: the stream goes to the slot's arena instead, with a descriptor from there to the caller's region.
static int place_chunk(pov_ctx* ctx, CorpusState& cs, const CorpusOut& fmt, Chunk& ck, uint64_t& next_record, Placement& pl) {
	pl.arena = pl.values = ck.view.pcm_floats;
	pl.into_caller = fmt.dev && !fmt.rs;
	pl.host_bytes = fmt.dev ? 0 : pl.values * pcm_elem_bytes(fmt.pcm_layout());
	pl.rs.clear();
	pl.rs_tiles = 0;
	if(!fmt.dev) return place_cuts(fmt, ck, pl);
	const pov_device_pcm& o = *fmt.dev;
	if(pl.into_caller) pl.arena = o.capacity;
	else pl.arena = pl.values = 0;
	for(size_t i = 0; i < ck.info.size(); ++i) {
		const pov_stream_info& s = ck.info[i];
		const uint64_t k = next_record++;
		if(k >= o.n_streams)
			return pov_fail(ctx, POV_ERR_ARG, "file %u: pov_decode_corpus_device: more logical streams than the %u records of the stream table", s.file, o.n_streams);
		if(o.file[k] != s.file || o.channels[k] != s.channels || o.frames[k] != s.frames)
			return pov_fail(ctx, POV_ERR_ARG, "file %u: pov_decode_corpus_device: stream %llu is (file %u, %u channels, %llu frames), the table says "
			                "(file %u, %u channels, %llu frames)", s.file, (unsigned long long) k, s.file, s.channels,
			                (unsigned long long) s.frames, o.file[k], o.channels[k], (unsigned long long) o.frames[k]);
		if(fmt.rs && fmt.rs->sample_rate[k] != s.sample_rate)
			return pov_fail(ctx, POV_ERR_ARG, "file %u: pov_decode_corpus_device_resampled: stream %llu has a sample rate of %u Hz, the table says %u Hz",
			                s.file, (unsigned long long) k, s.sample_rate, fmt.rs->sample_rate[k]);
		pov_stream* rec = ck.view.n_packets ? &ck.streams[i] : nullptr;    // (a chunk without audio packets has no batch)
		if(!fmt.rs) {
			if(rec) { rec->pcm_base = o.stream_base[k]; rec->pcm_frames = o.channel_stride[k]; }
			continue;
		}
		// the stream's channels 4-aligned in the slot's arena (so the synthesis takes its vector stores, as into 4-aligned
		// regions of pov_decode_corpus_device), and a descriptor from there to the caller's region
		const uint64_t stride = (s.frames + 3) & ~3ull;
		if(rec) { rec->pcm_base = pl.arena; rec->pcm_frames = stride; }
		ResampleDesc d;
		memset(&d, 0, sizeof d);
		stream_ratio(*fmt.rs, s.sample_rate, &d.L, &d.M);
		d.in_base = pl.arena; d.in_stride = stride; d.in_frames = s.frames; d.in_channels = s.channels;
		d.mono = (fmt.rs->flags & POV_RESAMPLE_MONO) != 0;
		d.inv_c = 1.0f / (float) s.channels;
		d.out_channels = d.mono ? 1 : s.channels;
		d.out_base = o.stream_base[k]; d.out_stride = o.channel_stride[k]; d.out_frames = resample_frames(s.frames, d.L, d.M);
		d.tile = resample_tile(d.L, d.M);
		pl.arena += s.channels * stride;
		pl.values += d.out_channels * d.out_frames;
		if(d.out_frames) {
			const int rc = resample_filter_table(ctx, cs, d.L, d.M, &d.taps, &d.K, &d.hl);
			if(rc) return rc;
			d.tile_first = pl.rs_tiles;
			pl.rs_tiles += d.out_channels * ((d.out_frames + d.tile - 1) / d.tile);
			pl.rs.push_back(d);
		}
	}
	return place_cuts(fmt, ck, pl);
}

// Queues a placed chunk on the slot: setup ids, upload, synthesis, then the checksum or the resample kernel, the copy-outs
// and `done`. Copy-in and kernels run on the slot context's stream. The PCM copy-out forks to its copy-out stream without a
// join, so the next chunk's copy-in and kernels are not queued behind the other slots' copy-outs; the status copy joins back,
// and `done` is recorded on the copy-out stream. From the upload on, the chunk stays in the slot until retire(): its pinned
// buffer is the source of the copies.
int CorpusState::Slot::submit(pov_ctx* caller, std::unique_ptr<Chunk> ck, const Placement& pl, const CorpusOut& fmt, CorpusTiming& tm, uint32_t ci) {
	auto forward = [&](int rc) { if(ctx != caller) pov_fail(caller, rc, "%s", pov_last_error(ctx)); return rc; };
	std::vector<uint32_t> ids(ck->setups.size(), 0);
	int rc = POV_OK;
	for(size_t k = 0; k < ck->setups.size() && rc == POV_OK; ++k) rc = register_stream_setup(ctx, ck->setups[k], &ids[k]);
	if(rc) return forward(rc);
	for(uint32_t i = 0; i < ck->view.n_streams; ++i) ck->streams[i].setup_id = ids[ck->streams[i].setup_id];
	tm.mark(CorpusTiming::kRetire, ci);
	pov_batch b = ck->view;
	b.pcm_floats = pl.arena;
	tm.event(ci, 0, ctx->stream);
	rc = pl.into_caller ? pov_batch_upload_into(ctx, &b, fmt.dev->pcm_dev, &h) : pov_batch_upload(ctx, &b, &h);
	tm.event(ci, 1, ctx->stream);
	in_flight = std::move(ck);                 // from here on retire() has to wait for the stream before the buffer is reused
	n_packets = 0;
	cudaEventRecord(done, ctx->stream);
	tm.mark(CorpusTiming::kUpload, ci);
	if(!rc) rc = pov_batch_run(ctx, h);
	tm.mark(CorpusTiming::kRun, ci);
	if(rc) return forward(rc);
	const size_t status_bytes = (size_t) b.n_packets * sizeof(uint32_t), rs_bytes = pl.rs.size() * sizeof(ResampleDesc);
	const size_t cut_bytes = pl.cut.size() * sizeof(CutDesc), res_bytes = pl.cut.size() * sizeof(CutResult);
	if(pinned.reserve(pl.host_bytes) != cudaSuccess || status.reserve(status_bytes) != cudaSuccess || rs_host.reserve(rs_bytes) != cudaSuccess ||
	   cut_host.reserve(cut_bytes) != cudaSuccess || cut_res.reserve(res_bytes) != cudaSuccess)
		return pov_fail(caller, POV_ERR_CUDA, "cudaMallocHost failed");
	if(fmt.cut) {
		// before everything that reads the PCM: the stream's descriptors up through the slot's pinned buffer, then one launch
		memcpy(cut_host.ptr, pl.cut.data(), cut_bytes);
		cudaError_t e = cut_dev.reserve(cut_bytes);
		if(e == cudaSuccess) e = cut_res_dev.reserve(res_bytes);
		if(e == cudaSuccess) e = cudaMemcpyAsync(cut_dev.ptr, cut_host.ptr, cut_bytes, cudaMemcpyHostToDevice, ctx->stream);
		if(e == cudaSuccess) {
			ctx->h2d_bytes += cut_bytes;
			e = launch_cut_damaged(pov_batch_pcm_dev(h), fmt.s16, (const CutDesc*) cut_dev.ptr, (uint32_t) pl.cut.size(), pl.cut_tiles,
			                       (const uint32_t*) h->d_status.ptr, (const pov_packet*) h->d_packets.ptr, (CutResult*) cut_res_dev.ptr,
			                       ctx->stream, &ctx->launches);
		}
		if(e != cudaSuccess) return pov_fail(caller, POV_ERR_CUDA, "cut kernel: %s", cudaGetErrorString(e));
	}
	if(pl.host_bytes) {
		const cudaError_t e = pov_checksum_launch(pov_batch_pcm_dev(h), fmt.s16, pl.values, d_sum, ctx->stream, &ctx->launches);
		if(e != cudaSuccess) return pov_fail(caller, POV_ERR_CUDA, "checksum kernel: %s", cudaGetErrorString(e));
	} else if(!pl.rs.empty()) {
		// descriptors up through the slot's pinned buffer (its last copy ended when the slot retired), then one launch
		memcpy(rs_host.ptr, pl.rs.data(), rs_bytes);
		cudaError_t e = rs_dev.reserve(rs_bytes);
		if(e == cudaSuccess) e = cudaMemcpyAsync(rs_dev.ptr, rs_host.ptr, rs_bytes, cudaMemcpyHostToDevice, ctx->stream);
		if(e == cudaSuccess) {
			ctx->h2d_bytes += rs_bytes;
			e = launch_resample((const float*) pov_batch_pcm_dev(h), (const ResampleDesc*) rs_dev.ptr, (uint32_t) pl.rs.size(), pl.rs_tiles,
			                    fmt.dev->pcm_dev, (fmt.dev->pcm_layout & POV_PCM_S16) != 0, ctx->stream, &ctx->launches);
		}
		if(e != cudaSuccess) return pov_fail(caller, POV_ERR_CUDA, "resample kernel: %s", cudaGetErrorString(e));
	}
	tm.event(ci, 2, ctx->stream);
	cudaError_t e = pl.host_bytes ? pov_copy_out_async(ctx, pinned.ptr, pov_batch_pcm_dev(h), pl.host_bytes, true, false) : cudaSuccess;
	if(e == cudaSuccess && fmt.cut) e = pov_copy_out_async(ctx, cut_res.ptr, cut_res_dev.ptr, res_bytes, pl.host_bytes == 0, false);
	if(e == cudaSuccess) e = pov_copy_out_async(ctx, status.ptr, h->d_status.ptr, status_bytes, pl.host_bytes == 0 && !fmt.cut, true);
	if(e != cudaSuccess) rc = pov_fail(caller, POV_ERR_CUDA, "pov_decode_corpus: copy-out failed: %s", cudaGetErrorString(e));
	tm.event(ci, 3, ctx->out_stream);
	if(!rc && cudaEventRecord(done, ctx->out_stream) != cudaSuccess) rc = pov_fail(caller, POV_ERR_CUDA, "pov_decode_corpus: cudaEventRecord failed");
	if(!rc) n_packets = b.n_packets;
	return rc;
}

// Waits for the slot's chunk, turns its status words into the reference's error, delivers its streams and gives its pinned
// buffer back. The output edge (hpp:966-973 gotPcmData, hpp:1047-1053): every logical stream of the chunk, in file order,
// from the calling thread; the samples stay valid during the callback only (they live in this slot's pinned buffer). After
// the first failure nothing more is delivered (`stopped`: chunks in flight are only drained).
int CorpusState::Slot::retire(pov_ctx* caller, const CorpusOut& fmt, bool& stopped) {
	if(!in_flight) return POV_OK;
	int rc = POV_OK;
	if(cudaEventSynchronize(done) != cudaSuccess) rc = pov_fail(caller, POV_ERR_CUDA, "pov_decode_corpus: chunk failed on the device");
	const uint32_t* words = (const uint32_t*) status.ptr;
	if(fmt.cut) {
		if(rc == POV_OK && n_packets) report_cuts(caller);
	} else {
		for(uint32_t p = 0; p < n_packets && rc == POV_OK; ++p)
			if(words[p]) rc = pov_fail(caller, POV_ERR_STREAM, "chunk at file %u, audio packet %u: check failed: %s", in_flight->first_file, p, pov_status_text(words[p]));
	}
	if(rc == POV_OK && fmt.has_sink() && !stopped && n_packets) {
		const Chunk& ck = *in_flight;
		const size_t esz = pcm_elem_bytes(fmt.pcm_layout());
		for(uint32_t i = 0; i < ck.view.n_streams && rc == POV_OK; ++i) {
			const pov_stream& rec = ck.streams[i];
			if(rec.pcm_frames == 0) continue;                  // hpp:1045: nothing is delivered for an empty chunk
			if(fmt.deliver(ck.info[i], rec.pcm_frames, (const uint8_t*) pinned.ptr + rec.pcm_base * esz) != 0)
				rc = pov_fail(caller, POV_ERR_STREAM, "file %u: check failed: callbacks.gotPcmData(channelPcms) (hpp:1052: the sink asked to stop)", ck.info[i].file);
		}
	}
	if(rc != POV_OK) stopped = true;
	in_flight.reset();
	return rc;
}

// Cut mode: the streams k_cut_damaged found damaged, from its results, into the caller's report (decode_corpus filled it for
// undamaged streams when the chunk was taken).
void CorpusState::Slot::report_cuts(pov_ctx* caller) const {
	const Chunk& ck = *in_flight;
	const CutResult* res = (const CutResult*) cut_res.ptr;
	uint32_t in_file = 0;                                  // the stream's index among its file's records
	for(uint32_t i = 0; i < ck.view.n_streams; ++i) {
		const pov_stream_info& s = ck.info[i];
		in_file = (i && ck.info[i - 1].file == s.file) ? in_file + 1 : 0;
		const CutResult& r = res[i];
		if(r.packet == 0xFFFFFFFFu) continue;
		caller->corpus_valid[ck.first_record + i] = r.valid_frames;
		pov_file_report& f = caller->corpus_files[s.file];
		f.valid_frames -= s.frames - r.valid_frames;
		f.status = POV_ERR_STREAM;
		if(!f.message[0])
			snprintf(f.message, sizeof f.message, "file %u: stream %u: check failed: audio packet %u: %s", s.file, in_file, r.packet,
			         r.packet == ck.walk_bad[i] ? ck.walk_text[i].c_str() : pov_status_text(r.status));
	}
}

static int decode_corpus(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t host_threads,
                         const CorpusOut& fmt_in, uint64_t* frames_out, uint64_t* total_values_out) {
	if(!ctx || (n_files && (!data || !len))) return POV_ERR_ARG;
	CorpusOut fmt = fmt_in;
	fmt.cut = ctx->cut_damage;
	cudaSetDevice(ctx->device);
	// automatic: every core but one — the calling thread validates, queues and retires chunks and must not be time-sliced
	// against the parsers (measured on 16 cores: 15 workers 6.8e9 samples/s and stable, 16 workers 2.6-3.7e9)
	if(host_threads == 0) { const uint32_t hc = std::thread::hardware_concurrency(); host_threads = hc > 1 ? hc - 1 : 1; }
	const std::vector<uint32_t> chunk_first = chunk_bounds(ctx, n_files);
	const uint32_t n_chunks = (uint32_t) chunk_first.size() - 1;
	const uint32_t max_ready = std::max<uint32_t>(4, 2 * host_threads);
	int rc = make_corpus_state(ctx);
	if(rc) return rc;
	CorpusState& cs = *(CorpusState*) ctx->corpus;
	cs.max_bufs = std::max(cs.max_bufs, max_ready + host_threads + CorpusState::kSlots + 1);       // queued + being filled + in flight + one spare
	for(auto& sl : cs.slot)
		if(cudaMemsetAsync(sl.d_sum, 0, 8, sl.ctx->stream) != cudaSuccess) return pov_fail(ctx, POV_ERR_CUDA, "pov_decode_corpus: cudaMemset failed");
	if(fmt.dev) {
		// device output: no PCM write may start before the work the caller has queued on its stream (e.g. a fill of the tensor)
		cudaEvent_t ev = nullptr;
		cudaError_t e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
		if(e == cudaSuccess) e = cudaEventRecord(ev, (cudaStream_t) fmt.dev->cuda_stream);
		for(auto& sl : cs.slot) if(e == cudaSuccess) e = cudaStreamWaitEvent(sl.ctx->stream, ev, 0);
		if(ev) cudaEventDestroy(ev);
		if(e != cudaSuccess) return pov_fail(ctx, POV_ERR_CUDA, "pov_decode_corpus_device: ordering after the caller's stream: %s", cudaGetErrorString(e));
	}

	ParseOptions opt;
	opt.raw_packets = ctx->device_entropy;
	opt.allow_spanning = ctx->allow_spanning;
	opt.cut_damage = fmt.cut;
	ctx->corpus_files.assign(n_files, pov_file_report());
	ctx->corpus_valid.clear();
	std::atomic<uint32_t> next_chunk(0);
	ChunkQueue queue(cs, max_ready);           // (declared after what the workers use: its destructor joins them)
	auto worker = [&]() {
		cudaSetDevice(ctx->device);
		HostBatch hb;
		std::vector<StreamWork> file;
		for(;;) {
			const uint32_t ci = next_chunk.fetch_add(1);
			if(ci >= n_chunks || queue.stop.load()) return;
			std::unique_ptr<Chunk> ck(new Chunk(&cs, chunk_first[ci], chunk_first[ci + 1] - chunk_first[ci]));
			try {                  // a worker never lets an exception escape its thread: the chunk carries the error instead
				assemble_chunk(*ck, data, len, opt, fmt.pcm_layout(), queue.stop, hb, file);
			} catch(...) {
				if(ck->error.empty()) ck->error = "chunk at file " + std::to_string(ck->first_file) + ": out of memory or internal error while assembling the batch";
			}
			queue.put(ci, std::move(ck));
		}
	};
	for(uint32_t t = 0; t < host_threads; ++t) queue.pool.emplace_back(worker);

	// kSlots batch slots: while the GPU transforms chunk i and copies its PCM and status words to pinned host memory, the
	// calling thread validates and queues the next chunks. A slot is retired (status words, sink) and reused kSlots chunks later.
	CorpusTiming tm(n_chunks);
	Placement pl;
	uint64_t total = 0, next_record = 0;       // next_record: device output, index of the next stream-table record
	bool stopped = false;
	for(uint32_t ci = 0; ci < n_chunks && rc == POV_OK; ++ci) {
		std::unique_ptr<Chunk> ck = queue.take(ci);
		tm.mark(CorpusTiming::kWait, ci);
		if(!ck->error.empty()) { rc = pov_fail(ctx, POV_ERR_STREAM, "%s", ck->error.c_str()); break; }
		if(frames_out) {
			std::fill(frames_out + ck->first_file, frames_out + ck->first_file + ck->n_files, 0);
			for(const pov_stream_info& s : ck->info) frames_out[s.file] += s.frames;
		}
		// the report as if nothing were damaged; geometry damage is known now, content damage when the chunk retires
		ck->first_record = ctx->corpus_valid.size();
		for(const pov_stream_info& s : ck->info) {
			pov_file_report& f = ctx->corpus_files[s.file];
			++f.n_streams; f.frames += s.frames; f.valid_frames += s.frames;
			ctx->corpus_valid.push_back(s.frames);
		}
		for(uint32_t k = 0; k < ck->damage.size(); ++k) {
			if(ck->damage[k].empty()) continue;
			pov_file_report& f = ctx->corpus_files[ck->first_file + k];
			f.status = POV_ERR_STREAM;
			snprintf(f.message, sizeof f.message, "%s", ck->damage[k].c_str());
		}
		rc = place_chunk(ctx, cs, fmt, *ck, next_record, pl);
		if(rc) break;
		if(ck->view.n_packets == 0) continue;
		CorpusState::Slot& sl = cs.slot[ci % CorpusState::kSlots];
		rc = sl.retire(ctx, fmt, stopped);     // the chunk that used this slot kSlots chunks ago
		if(rc) break;
		rc = sl.submit(ctx, std::move(ck), pl, fmt, tm, ci);
		total += pl.values;
		tm.mark(CorpusTiming::kFetch, ci);
	}
	for(uint32_t k = 0; k < (uint32_t) CorpusState::kSlots; ++k) {          // oldest chunk first (file order at the output edge)
		const int r2 = cs.slot[(n_chunks + k) % CorpusState::kSlots].retire(ctx, fmt, stopped);
		if(rc == POV_OK) rc = r2;
	}
	if(rc == POV_OK && fmt.dev && next_record != fmt.dev->n_streams)
		rc = pov_fail(ctx, POV_ERR_ARG, "pov_decode_corpus_device: the corpus has %llu logical streams, the stream table %u",
		              (unsigned long long) next_record, fmt.dev->n_streams);
	tm.report(chunk_first);
	queue.close();
	double h_sum = 0;
	int64_t h_sum16 = 0;
	for(auto& sl : cs.slot) {
		double part = 0;
		int64_t part16 = 0;
		if(rc == POV_OK && !fmt.dev &&
		   (cudaMemcpyAsync(fmt.s16 ? (void*) &part16 : (void*) &part, sl.d_sum, 8, cudaMemcpyDeviceToHost, sl.ctx->stream) != cudaSuccess ||
		    cudaStreamSynchronize(sl.ctx->stream) != cudaSuccess))
			rc = pov_fail(ctx, POV_ERR_CUDA, "pov_decode_corpus: checksum copy failed");
		h_sum += part;
		h_sum16 += part16;
		cudaStreamSynchronize(sl.ctx->stream);
	}
	for(pov_ctx* sb : cs.sibling) {            // the siblings' work is the caller's
		ctx->launches += sb->launches; ctx->h2d_bytes += sb->h2d_bytes; ctx->d2h_bytes += sb->d2h_bytes;
		sb->launches = sb->h2d_bytes = sb->d2h_bytes = 0;
	}
	if(total_values_out) *total_values_out = total;
	if(fmt.checksum) *fmt.checksum = h_sum;
	if(fmt.sum16) *fmt.sum16 = h_sum16;
	ctx->corpus_report_ok = rc == POV_OK;
	return rc;
}

extern "C" int pov_corpus_report(const pov_ctx* ctx, uint32_t n_files, pov_file_report* files, uint64_t n_streams, uint64_t* stream_valid_frames) {
	if(!ctx || !ctx->corpus_report_ok || (n_files && !files) || n_files != ctx->corpus_files.size() ||
	   (stream_valid_frames && n_streams != ctx->corpus_valid.size()))
		return POV_ERR_ARG;
	if(n_files) memcpy(files, ctx->corpus_files.data(), n_files * sizeof(pov_file_report));
	if(stream_valid_frames && n_streams) memcpy(stream_valid_frames, ctx->corpus_valid.data(), n_streams * sizeof(uint64_t));
	return POV_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// same shape as the reference's C entry point (hpp:1493): decode, discard the PCM, report errors as a string
// ---------------------------------------------------------------------------------------------------------------
extern "C" int pov_ogg_vorbis_full_read_from_memory(const char* data, size_t data_len, const char** error_out) {
	static thread_local char errbuf[512];
	static thread_local pov_ctx* tl_ctx = nullptr;
	if(!tl_ctx) {
		const char* e = nullptr;
		if(pov_ctx_create(0, &tl_ctx, &e) != POV_OK) {
			snprintf(errbuf, sizeof errbuf, "%s", e ? e : "pov_ctx_create failed");
			if(error_out) *error_out = errbuf;
			return 1;
		}
	}
	pov_decoded d;
	const int rc = pov_ogg_vorbis_decode_memory(tl_ctx, (const uint8_t*) data, data_len, nullptr, &d);
	pov_decoded_free(&d);
	if(rc != POV_OK) {
		snprintf(errbuf, sizeof errbuf, "%s", pov_last_error(tl_ctx));
		if(error_out) *error_out = errbuf;
		return 1;
	}
	return 0;
}
