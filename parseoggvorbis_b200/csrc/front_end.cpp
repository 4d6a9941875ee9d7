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
// stream table of a corpus (host only): the corpus workers' parse, packets discarded
// ---------------------------------------------------------------------------------------------------------------
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
	auto worker = [&]() {
		std::vector<StreamWork> file;
		ParseOptions opt;
		opt.raw_packets = true;
		opt.allow_spanning = (flags & POV_PARSE_ALLOW_SPANNING) != 0;
		for(;;) {
			const uint32_t i = next.fetch_add(1);
			if(i >= n_files || i > first_error.load()) return;          // (files after a failed one are not needed)
			try {
				ParseError err;
				file.clear();
				if(!parse_ogg_file(data[i], len[i], file, err, opt)) {
					error[i] = "file " + std::to_string(i) + ": check failed: " + err.msg;
					uint32_t f = first_error.load();
					while(i < f && !first_error.compare_exchange_weak(f, i)) {}
					continue;
				}
				for(const StreamWork& st : file) {
					if(!st.have_setup) continue;
					pov_stream_info r;
					memset(&r, 0, sizeof r);
					r.file = i; r.channels = st.setup.channels; r.sample_rate = st.setup.sample_rate; r.frames = st.frames;
					per_file[i].push_back(r);
				}
			} catch(...) {
				error[i] = "file " + std::to_string(i) + ": out of memory or internal error while parsing";
				uint32_t f = first_error.load();
				while(i < f && !first_error.compare_exchange_weak(f, i)) {}
			}
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
// float64 sum of a float arena into *(double*) d_sum, or (s16) exact int64 sum of an int16 arena into *(uint64_t*) d_sum
cudaError_t pov_checksum_launch(const void* pcm, bool s16, uint64_t n, void* d_sum, cudaStream_t st, uint64_t* launches);

namespace {
struct PinnedBuf { uint8_t* p = nullptr; size_t cap = 0; };

// A chunk leaves its worker as one assembled batch in pinned host memory: the calling thread only turns the chunk-local
// setup numbers into registered setup ids (one map lookup per distinct setup, normally one per chunk), validates the
// descriptors and queues the copies, which then run as plain DMA.
struct Chunk {
	uint32_t first_file = 0, n_files = 0;
	PinnedBuf buf;                             // streams | packets | ys | payload, each 16-byte aligned
	pov_batch view;                            // pointers into buf; pov_stream::setup_id = index into `setups` until patched
	pov_stream* streams = nullptr;             // writable alias of view.streams
	std::vector<StreamWork> setups;            // one representative stream (headers only) per distinct setup
	std::vector<uint64_t> frames;              // per file
	std::vector<uint32_t> stream_file, stream_channels;   // per stream of the batch: file index (corpus-wide), channel count
	std::vector<uint64_t> stream_frames;       // per stream of the batch
	std::vector<uint32_t> stream_rate;         // per stream of the batch: sample rate
	std::string error;
};

// What pov_decode_corpus keeps between calls on a context: the sibling context (second stream), the two batch slots with
// their device arenas and pinned PCM buffers, and the pool of pinned staging buffers the workers assemble chunks into.
struct CorpusState {
	int device = 0;
	static constexpr int kSlots = 4;           // chunks in flight: while two copy their PCM out, the others compute (the copy-out,
	                                           // 4 bytes per PCM sample over PCIe, is the bound of the whole decode)
	pov_ctx* sibling[kSlots - 1] = {nullptr};
	struct Slot {
		pov_ctx* ctx = nullptr;                // slot 0: the caller's context; slot 1: the sibling, so that the copies of one
		                                       // chunk never wait for the other chunk's work
		void* d_sum = nullptr;                 // 8 bytes: float64 checksum, or the int64 sum of an int16 decode
		pov_batch_handle* h = nullptr;
		uint8_t* pinned = nullptr; size_t pinned_cap = 0;     // the chunk's PCM arena (float or int16)
		uint32_t* status = nullptr; size_t status_cap = 0;
		cudaEvent_t done = nullptr;
		cudaEvent_t t_begin = nullptr, t_kernels = nullptr, t_end = nullptr;   // POV_CORPUS_TIMING only
		uint32_t n_packets = 0, first_file = 0;
		ResampleDesc* rs_host = nullptr; size_t rs_cap = 0;  // resampled output: the chunk's descriptors (pinned source of their upload)
		DevBuf rs_dev;
		std::unique_ptr<Chunk> in_flight;      // its pinned buffer is the source of copies that may still be running
		bool busy = false;
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
		if(b.cap < need) {
			if(b.p) cudaFreeHost(b.p);
			b.p = nullptr; b.cap = need + need / 4;
			if(cudaHostAlloc((void**) &b.p, b.cap, cudaHostAllocDefault) != cudaSuccess) {
				b.p = nullptr; b.cap = 0;
				std::lock_guard<std::mutex> lk(pmu);
				--n_bufs;                              // the buffer this call stood for no longer exists
				pcv.notify_one();
			}
		}
		return b;
	}
	void release(PinnedBuf b) {
		if(!b.p) return;
		std::lock_guard<std::mutex> lk(pmu);
		free_bufs.push_back(b);
		pcv.notify_one();
	}
	~CorpusState() {
		cudaSetDevice(device);
		for(auto& sl : slot) {
			if(!sl.ctx) continue;
			cudaStreamSynchronize(sl.ctx->stream);
			if(sl.in_flight) { if(sl.in_flight->buf.p) cudaFreeHost(sl.in_flight->buf.p); sl.in_flight.reset(); }
			if(sl.h) pov_batch_free(sl.ctx, sl.h);
			if(sl.pinned) cudaFreeHost(sl.pinned);
			if(sl.status) cudaFreeHost(sl.status);
			if(sl.rs_host) cudaFreeHost(sl.rs_host);
			sl.rs_dev.release();
			if(sl.done) cudaEventDestroy(sl.done);
			if(sl.t_begin) { cudaEventDestroy(sl.t_begin); cudaEventDestroy(sl.t_kernels); cudaEventDestroy(sl.t_end); }
			if(sl.d_sum) cudaFree(sl.d_sum);
		}
		for(auto& b : free_bufs) cudaFreeHost(b.p);
		for(auto& f : filters) if(f.second.taps) cudaFree(f.second.taps);
		for(pov_ctx* sb : sibling) if(sb) pov_ctx_destroy(sb);
	}
};
void corpus_state_free(void* p) { delete (CorpusState*) p; }

inline size_t align16(size_t x) { return (x + 15) & ~(size_t) 15; }
}  // namespace

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
};

static int decode_corpus(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t host_threads,
                         const CorpusOut& fmt, uint64_t* frames_out, uint64_t* total_values_out);

extern "C" int pov_decode_corpus(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len,
                                 uint32_t host_threads, uint64_t* frames_out, uint64_t* total_values_out, double* checksum_out) try {
	CorpusOut fmt;
	fmt.checksum = checksum_out;
	return decode_corpus(ctx, n_files, data, len, host_threads, fmt, frames_out, total_values_out);
} POV_NOTHROW_END(ctx)

extern "C" int pov_decode_corpus_pcm(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t host_threads,
                                     pov_pcm_sink sink, void* user, uint64_t* frames_out, uint64_t* total_values_out, double* checksum_out) try {
	if(!sink) return pov_fail(ctx, POV_ERR_ARG, "pov_decode_corpus_pcm: null sink");
	CorpusOut fmt;
	fmt.sink = sink; fmt.user = user; fmt.checksum = checksum_out;
	return decode_corpus(ctx, n_files, data, len, host_threads, fmt, frames_out, total_values_out);
} POV_NOTHROW_END(ctx)

extern "C" int pov_decode_corpus_s16(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t host_threads,
                                     pov_pcm_sink_s16 sink, void* user, uint64_t* frames_out, uint64_t* total_values_out, int64_t* sum_out) try {
	CorpusOut fmt;
	fmt.s16 = true; fmt.sink16 = sink; fmt.user = user; fmt.sum16 = sum_out;
	return decode_corpus(ctx, n_files, data, len, host_threads, fmt, frames_out, total_values_out);
} POV_NOTHROW_END(ctx)

int pov_check_pcm_dev(pov_ctx* ctx, const void* p, size_t align, const char* fn);      // api.cu

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

static int decode_corpus(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t host_threads,
                         const CorpusOut& fmt, uint64_t* frames_out, uint64_t* total_values_out) {
	if(!ctx || (n_files && (!data || !len))) return POV_ERR_ARG;
	const bool has_sink = fmt.s16 ? fmt.sink16 != nullptr : fmt.sink != nullptr;
	const uint32_t pcm_layout = POV_PCM_PLANAR | (fmt.s16 ? POV_PCM_S16 : 0u);
	const size_t esz = pcm_elem_bytes(pcm_layout);                      // bytes per PCM sample in the arenas and over PCIe
	cudaSetDevice(ctx->device);
	// automatic: every core but one — the calling thread validates, queues and retires chunks and must not be time-sliced
	// against the parsers (measured on 16 cores: 15 workers 6.8e9 samples/s and stable, 16 workers 2.6-3.7e9)
	if(host_threads == 0) { const uint32_t hc = std::thread::hardware_concurrency(); host_threads = hc > 1 ? hc - 1 : 1; }
	// Files per chunk: with the entropy decode on the device a chunk's kernels are latency bound (one thread walks one packet),
	// so more packets per launch cost nothing and the PCM copy-out — the PCIe bound of the whole decode — runs in long
	// transfers; with the host walk smaller chunks keep the parser threads and the device overlapped.
	uint32_t files_per_chunk = ctx->device_entropy ? 256 : 64;
	if(const char* e = getenv("POV_CORPUS_CHUNK")) files_per_chunk = std::max(1, atoi(e));
	// The first chunks are small and grow by half each (1/8 of the size, then x 1.5): every worker starts on a chunk of its own
	// at once, one worker parses a file in about twice the time the copy-out of its PCM takes, so chunk k is ready just before
	// the copy-out of chunks 0..k-1 ends and the link never waits for a parser. chunk_first[k] = index of chunk k's first file.
	std::vector<uint32_t> chunk_first;
	{
		uint32_t at = 0, size = std::max(1u, files_per_chunk / 8);
		while(at < n_files) {
			chunk_first.push_back(at);
			at += std::min(size, n_files - at);
			size = std::min(files_per_chunk, size + (size + 1) / 2);
		}
		chunk_first.push_back(n_files);
	}
	const uint32_t n_chunks = (uint32_t) chunk_first.size() - 1;
	const uint32_t max_ready = std::max<uint32_t>(4, 2 * host_threads);

	// ---- resources that outlive the call ----
	int rc = POV_OK;
	if(!ctx->corpus) {
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
	}
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
	uint64_t sibling_launches0 = 0, sibling_h2d0 = 0, sibling_d2h0 = 0;
	for(pov_ctx* sb : cs.sibling) { sibling_launches0 += sb->launches; sibling_h2d0 += sb->h2d_bytes; sibling_d2h0 += sb->d2h_bytes; }

	std::atomic<uint32_t> next_chunk(0);
	std::mutex mu;
	std::condition_variable cv_ready, cv_space;
	std::map<uint32_t, std::unique_ptr<Chunk>> ready;    // by chunk index
	uint32_t consumed = 0;                               // chunks handed to the calling thread so far (guarded by mu)
	std::atomic<bool> stop(false);

	auto worker = [&]() {
		cudaSetDevice(ctx->device);
		HostBatch hb;
		std::vector<StreamWork> file;
		for(;;) {
			const uint32_t ci = next_chunk.fetch_add(1);
			if(ci >= n_chunks || stop.load()) return;
			std::unique_ptr<Chunk> ck(new Chunk());
			memset(&ck->view, 0, sizeof ck->view);
			ck->first_file = chunk_first[ci];
			ck->n_files = chunk_first[ci + 1] - chunk_first[ci];
			ck->frames.assign(ck->n_files, 0);
			hb.clear();
			ParseOptions opt;
			opt.raw_packets = ctx->device_entropy;
			opt.allow_spanning = ctx->allow_spanning;
			try {                  // a worker never lets an exception escape its thread: the chunk carries the error instead
			for(int attempt = 0; attempt < 2; ++attempt) {       // (second round only if a stream cannot be walked on the device)
			bool mixed = false;
			hb.clear(); hb.raw = opt.raw_packets;
			ck->setups.clear(); ck->stream_file.clear(); ck->stream_channels.clear(); ck->stream_frames.clear(); ck->stream_rate.clear();
			ck->frames.assign(ck->n_files, 0);
			for(uint32_t i = 0; i < ck->n_files && ck->error.empty(); ++i) {
				ParseError err;
				file.clear();
				if(!parse_ogg_file(data[ck->first_file + i], len[ck->first_file + i], file, err, opt)) {
					ck->error = "file " + std::to_string(ck->first_file + i) + ": check failed: " + err.msg;
					break;
				}
				for(StreamWork& st : file) {
					if(!st.have_setup) continue;
					if(st.raw != opt.raw_packets) mixed = true;
					uint32_t k = 0;
					while(k < ck->setups.size() && ck->setups[k].setup_key != st.setup_key) ++k;
					hb.append(st, k);
					ck->frames[i] += st.frames;
					ck->stream_file.push_back(ck->first_file + i);
					ck->stream_channels.push_back(st.setup.channels);
					ck->stream_frames.push_back(st.frames);
					ck->stream_rate.push_back(st.setup.sample_rate);
					if(k == ck->setups.size()) {
						st.packets.clear(); st.ys.clear(); st.payload.clear();
						ck->setups.push_back(std::move(st));
					}
				}
			}
			if(!mixed || !ck->error.empty()) break;
			opt.raw_packets = false;
			}
			if(ck->error.empty() && !hb.packets.empty()) {
				// pageable vectors -> one pinned buffer (this copy runs on the worker, the DMA later needs no staging)
				const size_t o_st = 0, o_pk = o_st + align16(hb.streams.size() * sizeof(pov_stream)),
				             o_ys = o_pk + align16(hb.packets.size() * sizeof(pov_packet)), o_pl = o_ys + align16(hb.ys.size() * sizeof(uint16_t)),
				             need = o_pl + align16(hb.payload.size());
				ck->buf = cs.acquire(need, stop);
				if(!ck->buf.p) { if(!stop.load()) ck->error = "pov_decode_corpus: pinned staging buffer allocation failed"; }
				else {
					uint8_t* q = ck->buf.p;
					memcpy(q + o_st, hb.streams.data(), hb.streams.size() * sizeof(pov_stream));
					memcpy(q + o_pk, hb.packets.data(), hb.packets.size() * sizeof(pov_packet));
					memcpy(q + o_ys, hb.ys.data(), hb.ys.size() * sizeof(uint16_t));
					memcpy(q + o_pl, hb.payload.data(), hb.payload.size());
					pov_batch& b = ck->view;
					b.input_kind = hb.raw ? POV_INPUT_PACKETS : POV_INPUT_ENTRIES; b.pcm_layout = pcm_layout;
					ck->streams = (pov_stream*) (q + o_st);
					b.n_streams = (uint32_t) hb.streams.size(); b.streams = ck->streams;
					b.n_packets = (uint32_t) hb.packets.size(); b.packets = (const pov_packet*) (q + o_pk);
					b.ys = (const uint16_t*) (q + o_ys); b.n_ys = hb.ys.size();
					b.payload = q + o_pl; b.payload_bytes = hb.payload.size();
					b.pcm_floats = hb.pcm_floats;
				}
			}
			} catch(...) {
				if(ck->error.empty()) ck->error = "chunk at file " + std::to_string(ck->first_file) + ": out of memory or internal error while assembling the batch";
			}
			// Back-pressure by chunk INDEX, not by count: the chunk the consumer is waiting for always passes, however many
			// later chunks the other workers have finished in the meantime (a count limit can fill the queue with later chunks
			// and then block the one worker that holds the chunk everybody is waiting for).
			std::unique_lock<std::mutex> lk(mu);
			cv_space.wait(lk, [&] { return ci < consumed + max_ready || stop.load(); });
			ready[ci] = std::move(ck);
			cv_ready.notify_all();
		}
	};
	// the pool is joined on every way out of this function (an exception on the calling thread included)
	struct PoolJoiner {
		std::vector<std::thread> pool;
		std::atomic<bool>& stop; std::mutex& mu; std::condition_variable& cv_space; CorpusState& cs;
		~PoolJoiner() {
			stop.store(true);
			{ std::lock_guard<std::mutex> lk(mu); cv_space.notify_all(); }
			{ std::lock_guard<std::mutex> lk(cs.pmu); cs.pcv.notify_all(); }
			for(auto& t : pool) if(t.joinable()) t.join();
		}
	} joiner{{}, stop, mu, cv_space, cs};
	std::vector<std::thread>& pool = joiner.pool;
	for(uint32_t t = 0; t < host_threads; ++t) pool.emplace_back(worker);

	uint64_t total = 0;
	std::vector<ResampleDesc> rs_descs;                  // resampled output: the descriptors of the chunk being queued
	uint64_t dev_stream = 0;                             // device output: index of the next stream-table record
	double h_sum = 0;
	int64_t h_sum16 = 0;
	// Two batch slots: while the GPU transforms chunk i and copies its PCM and status words to pinned host memory, the
	// calling thread validates and queues chunk i+1. A slot is checked (status words) and reused two chunks later.
	typedef CorpusState::Slot Slot;
	const bool timing = getenv("POV_CORPUS_TIMING") != nullptr;
	double g_copy_in_kernels = 0, g_copy_out = 0;
	if(timing) for(auto& sl : cs.slot) if(!sl.t_begin) { cudaEventCreate(&sl.t_begin); cudaEventCreate(&sl.t_kernels); cudaEventCreate(&sl.t_end); }
	// POV_CORPUS_TIMING=2: also a per-chunk timeline (four events per chunk: queued, copy-in done, kernels done, copy-out done)
	const bool timeline = timing && atoi(getenv("POV_CORPUS_TIMING")) >= 2;
	std::vector<cudaEvent_t> tl(timeline ? 4 * (size_t) n_chunks : 0, nullptr);
	for(auto& e : tl) cudaEventCreate(&e);
	std::vector<double> tl_host(timeline ? 4 * (size_t) n_chunks : 0, 0.0);    // host clock: chunk taken, slot free, upload queued, all queued
	bool stopped = false;
	auto retire = [&](Slot& sl) -> int {           // wait for a slot's chunk and turn its status words into the reference's error
		if(!sl.busy) return POV_OK;
		sl.busy = false;
		const bool ok = cudaEventSynchronize(sl.done) == cudaSuccess;
		if(timing && ok && sl.n_packets) {
			float a = 0, b = 0;
			if(cudaEventElapsedTime(&a, sl.t_begin, sl.t_kernels) == cudaSuccess && cudaEventElapsedTime(&b, sl.t_kernels, sl.t_end) == cudaSuccess) { g_copy_in_kernels += a; g_copy_out += b; }
		}
		int out = POV_OK;
		if(!ok) out = pov_fail(ctx, POV_ERR_CUDA, "pov_decode_corpus: chunk failed on the device");
		for(uint32_t p = 0; p < sl.n_packets && out == POV_OK; ++p)
			if(sl.status[p]) {
				const char* what = (sl.status[p] & POV_PKT_FLOOR_PREDICTED) ? "predicted <= range (hpp:536)"
				                 : (sl.status[p] & POV_PKT_FLOOR_RANGE)     ? "floor[i] < 256 (hpp:587)"
				                                                            : "temp.size() > 0 (hpp:739,748: VQ entry out of range)";
				out = pov_fail(ctx, POV_ERR_STREAM, "chunk at file %u, audio packet %u: check failed: %s", sl.first_file, p, what);
			}
		// the output edge (hpp:966-973 gotPcmData, hpp:1047-1053): every logical stream of the chunk, in file order, from the
		// calling thread; the samples stay valid during the callback only (they live in this slot's pinned buffer)
		if(out == POV_OK && has_sink && !stopped && sl.in_flight && sl.n_packets) {
			const Chunk& ck = *sl.in_flight;
			for(uint32_t i = 0; i < ck.view.n_streams && out == POV_OK; ++i) {
				const pov_stream& rec = ck.streams[i];
				if(rec.pcm_frames == 0) continue;                  // hpp:1045: nothing is delivered for an empty chunk
				const void* planar = sl.pinned + rec.pcm_base * esz;
				if((fmt.s16 ? fmt.sink16(ck.stream_file[i], ck.stream_channels[i], rec.pcm_frames, (const int16_t*) planar, fmt.user)
				            : fmt.sink(ck.stream_file[i], ck.stream_channels[i], rec.pcm_frames, (const float*) planar, fmt.user)) != 0)
					out = pov_fail(ctx, POV_ERR_STREAM, "file %u: check failed: callbacks.gotPcmData(channelPcms) (hpp:1052: the sink asked to stop)", ck.stream_file[i]);
			}
		}
		if(out != POV_OK) stopped = true;          // after the first failure nothing more is delivered (chunks in flight are only drained)
		if(sl.in_flight) { cs.release(sl.in_flight->buf); sl.in_flight.reset(); }
		return out;
	};

	// POV_CORPUS_TIMING=1: where the calling thread's time goes (stderr), to tell a starved consumer from a slow one
	double t_wait = 0, t_retire = 0, t_upload = 0, t_run = 0, t_fetch = 0;
	auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
	const double t_begin = now();
	for(uint32_t ci = 0; ci < n_chunks && rc == POV_OK; ++ci) {
		std::unique_ptr<Chunk> ck;
		double t0 = now();
		{
			std::unique_lock<std::mutex> lk(mu);
			cv_ready.wait(lk, [&] { return ready.count(ci) != 0; });
			ck = std::move(ready[ci]);
			ready.erase(ci);
			consumed = ci + 1;
			cv_space.notify_all();
		}
		t_wait += now() - t0; t0 = now();
		if(timeline) tl_host[4 * ci] = t0 - t_begin;
		if(!ck->error.empty()) { rc = pov_fail(ctx, POV_ERR_STREAM, "%s", ck->error.c_str()); cs.release(ck->buf); break; }
		if(frames_out) for(uint32_t i = 0; i < ck->n_files; ++i) frames_out[ck->first_file + i] = ck->frames[i];
		rs_descs.clear();
		uint64_t rs_arena = 0, rs_tiles = 0, rs_values = 0;
		if(fmt.dev) {
			// each parsed stream against the caller's record at its index, then to the caller's region (the kernels address planar
			// PCM as pcm_base + c * pcm_frames + f, so pcm_frames is the channel stride)
			const pov_device_pcm& o = *fmt.dev;
			for(size_t i = 0; i < ck->stream_file.size() && rc == POV_OK; ++i, ++dev_stream) {
				const uint64_t k = dev_stream;
				if(k >= o.n_streams)
					rc = pov_fail(ctx, POV_ERR_ARG, "file %u: pov_decode_corpus_device: more logical streams than the %u records of the stream table",
					              ck->stream_file[i], o.n_streams);
				else if(o.file[k] != ck->stream_file[i] || o.channels[k] != ck->stream_channels[i] || o.frames[k] != ck->stream_frames[i])
					rc = pov_fail(ctx, POV_ERR_ARG, "file %u: pov_decode_corpus_device: stream %llu is (file %u, %u channels, %llu frames), the table says "
					              "(file %u, %u channels, %llu frames)", ck->stream_file[i], (unsigned long long) k, ck->stream_file[i], ck->stream_channels[i],
					              (unsigned long long) ck->stream_frames[i], o.file[k], o.channels[k], (unsigned long long) o.frames[k]);
				else if(fmt.rs && fmt.rs->sample_rate[k] != ck->stream_rate[i])
					rc = pov_fail(ctx, POV_ERR_ARG, "file %u: pov_decode_corpus_device_resampled: stream %llu has a sample rate of %u Hz, the table says %u Hz",
					              ck->stream_file[i], (unsigned long long) k, ck->stream_rate[i], fmt.rs->sample_rate[k]);
				else if(fmt.rs) {
					// the stream's channels 4-aligned in the slot's arena (so the synthesis takes its vector stores, as into 4-aligned
					// regions of pov_decode_corpus_device), and a descriptor from there to the caller's region
					const uint64_t fr = ck->stream_frames[i], stride = (fr + 3) & ~3ull;
					const uint32_t C = ck->stream_channels[i];
					if(ck->view.n_packets) { ck->streams[i].pcm_base = rs_arena; ck->streams[i].pcm_frames = stride; }
					ResampleDesc dsc;
					memset(&dsc, 0, sizeof dsc);
					stream_ratio(*fmt.rs, ck->stream_rate[i], &dsc.L, &dsc.M);
					dsc.in_base = rs_arena; dsc.in_stride = stride; dsc.in_frames = fr; dsc.in_channels = C;
					dsc.mono = (fmt.rs->flags & POV_RESAMPLE_MONO) != 0;
					dsc.inv_c = 1.0f / (float) C;
					dsc.out_channels = dsc.mono ? 1 : C;
					dsc.out_base = o.stream_base[k]; dsc.out_stride = o.channel_stride[k]; dsc.out_frames = resample_frames(fr, dsc.L, dsc.M);
					dsc.tile = resample_tile(dsc.L, dsc.M);
					rs_arena += C * stride;
					rs_values += dsc.out_channels * dsc.out_frames;
					if(dsc.out_frames) {
						rc = resample_filter_table(ctx, cs, dsc.L, dsc.M, &dsc.taps, &dsc.K, &dsc.hl);
						dsc.tile_first = rs_tiles;
						rs_tiles += dsc.out_channels * ((dsc.out_frames + dsc.tile - 1) / dsc.tile);
						rs_descs.push_back(dsc);
					}
				}
				else if(ck->view.n_packets) {
					ck->streams[i].pcm_base = o.stream_base[k];
					ck->streams[i].pcm_frames = o.channel_stride[k];
				}
			}
			if(rc) { cs.release(ck->buf); break; }
		}
		if(ck->view.n_packets == 0) { cs.release(ck->buf); continue; }
		Slot& sl = cs.slot[ci % CorpusState::kSlots];
		pov_ctx* cx = sl.ctx;
		std::vector<uint32_t> ids(ck->setups.size(), 0);
		for(size_t k = 0; k < ck->setups.size() && rc == POV_OK; ++k) {
			rc = register_stream_setup(cx, ck->setups[k], &ids[k]);
			if(rc && cx != ctx) pov_fail(ctx, rc, "%s", pov_last_error(cx));
		}
		if(rc) { cs.release(ck->buf); break; }
		for(uint32_t i = 0; i < ck->view.n_streams; ++i) ck->streams[i].setup_id = ids[ck->streams[i].setup_id];
		rc = retire(sl);                           // the chunk that used this slot two iterations ago
		if(rc) { cs.release(ck->buf); break; }
		t_retire += now() - t0; t0 = now();
		if(timeline) tl_host[4 * ci + 1] = t0 - t_begin;
		pov_batch b = ck->view;
		const uint64_t pcm_floats = fmt.rs ? rs_values : b.pcm_floats;    // samples the chunk yields
		if(fmt.rs) b.pcm_floats = rs_arena;
		else if(fmt.dev) b.pcm_floats = fmt.dev->capacity;
		const uint32_t n_packets = b.n_packets;
		if(timing) cudaEventRecord(sl.t_begin, cx->stream);
		if(timeline) cudaEventRecord(tl[4 * ci], cx->stream);
		rc = fmt.dev && !fmt.rs ? pov_batch_upload_into(cx, &b, fmt.dev->pcm_dev, &sl.h) : pov_batch_upload(cx, &b, &sl.h);
		if(timeline) cudaEventRecord(tl[4 * ci + 1], cx->stream);      // pinned sources: the copies are queued, the chunk stays alive until retire()
		sl.in_flight = std::move(ck);
		sl.busy = true;                            // from here on retire() has to wait for the stream before the buffer is reused
		sl.n_packets = 0;
		cudaEventRecord(sl.done, cx->stream);
		t_upload += now() - t0; t0 = now();
		if(timeline) tl_host[4 * ci + 2] = t0 - t_begin;
		if(!rc) rc = pov_batch_run(cx, sl.h);
		t_run += now() - t0; t0 = now();
		if(rc && cx != ctx) pov_fail(ctx, rc, "%s", pov_last_error(cx));
		if(!rc) {
			const size_t need = fmt.dev ? 0 : pcm_floats * esz;
			if(need > sl.pinned_cap) {
				if(sl.pinned) cudaFreeHost(sl.pinned);
				sl.pinned = nullptr;
				sl.pinned_cap = need + need / 4;
				if(cudaMallocHost((void**) &sl.pinned, sl.pinned_cap) != cudaSuccess) { sl.pinned_cap = 0; rc = pov_fail(ctx, POV_ERR_CUDA, "cudaMallocHost failed"); break; }
			}
			const size_t sneed = (size_t) n_packets * sizeof(uint32_t);
			if(sneed > sl.status_cap) {
				if(sl.status) cudaFreeHost(sl.status);
				sl.status = nullptr;
				sl.status_cap = sneed + sneed / 4;
				if(cudaMallocHost((void**) &sl.status, sl.status_cap) != cudaSuccess) { sl.status_cap = 0; rc = pov_fail(ctx, POV_ERR_CUDA, "cudaMallocHost failed"); break; }
			}
			if(!fmt.dev) {
				cudaError_t e = pov_checksum_launch(pov_batch_pcm_dev(sl.h), fmt.s16, pcm_floats, sl.d_sum, cx->stream, &cx->launches);
				if(e != cudaSuccess) { rc = pov_fail(ctx, POV_ERR_CUDA, "checksum kernel: %s", cudaGetErrorString(e)); break; }
			} else if(fmt.rs && !rs_descs.empty()) {
				// descriptors up through the slot's pinned buffer (its last copy ended when the slot retired), then one launch
				const size_t bytes = rs_descs.size() * sizeof(ResampleDesc);
				if(bytes > sl.rs_cap) {
					if(sl.rs_host) cudaFreeHost(sl.rs_host);
					sl.rs_host = nullptr;
					sl.rs_cap = bytes + bytes / 4;
					if(cudaMallocHost((void**) &sl.rs_host, sl.rs_cap) != cudaSuccess) { sl.rs_cap = 0; rc = pov_fail(ctx, POV_ERR_CUDA, "cudaMallocHost failed"); break; }
				}
				memcpy(sl.rs_host, rs_descs.data(), bytes);
				cudaError_t e = sl.rs_dev.reserve(bytes);
				if(e == cudaSuccess) e = cudaMemcpyAsync(sl.rs_dev.ptr, sl.rs_host, bytes, cudaMemcpyHostToDevice, cx->stream);
				if(e == cudaSuccess) {
					cx->h2d_bytes += bytes;
					e = launch_resample((const float*) pov_batch_pcm_dev(sl.h), (const ResampleDesc*) sl.rs_dev.ptr, (uint32_t) rs_descs.size(), rs_tiles,
					                    fmt.dev->pcm_dev, (fmt.dev->pcm_layout & POV_PCM_S16) != 0, cx->stream, &cx->launches);
				}
				if(e != cudaSuccess) { rc = pov_fail(ctx, POV_ERR_CUDA, "resample kernel: %s", cudaGetErrorString(e)); break; }
			}
			if(timing) cudaEventRecord(sl.t_kernels, cx->stream);
			if(timeline) cudaEventRecord(tl[4 * ci + 2], cx->stream);
			// delivery of the PCM (not for device output) and the status words to the host, on the slot's copy-out stream: the next
			// chunk's copy-in and kernels on cx->stream are then not queued behind the other slots' copy-outs (they only wait for this one)
			cudaError_t ce = need ? pov_copy_out_async(cx, sl.pinned, pov_batch_pcm_dev(sl.h), need, true, false) : cudaSuccess;
			if(ce == cudaSuccess) ce = pov_copy_out_async(cx, sl.status, sl.h->d_status.ptr, sneed, need == 0, true);
			if(ce != cudaSuccess) rc = pov_fail(ctx, POV_ERR_CUDA, "pov_decode_corpus: copy-out failed: %s", cudaGetErrorString(ce));
			if(timing) cudaEventRecord(sl.t_end, cx->out_stream);
			if(timeline) cudaEventRecord(tl[4 * ci + 3], cx->out_stream);
			if(!rc && cudaEventRecord(sl.done, cx->out_stream) != cudaSuccess) rc = pov_fail(ctx, POV_ERR_CUDA, "pov_decode_corpus: cudaEventRecord failed");
			if(!rc) { sl.n_packets = n_packets; sl.first_file = sl.in_flight->first_file; }
		}
		total += pcm_floats;
		t_fetch += now() - t0;
		if(timeline) tl_host[4 * ci + 3] = now() - t_begin;
	}
	for(uint32_t k = 0; k < (uint32_t) CorpusState::kSlots; ++k) {          // oldest chunk first (file order at the output edge)
		const int r2 = retire(cs.slot[(n_chunks + k) % CorpusState::kSlots]);
		if(rc == POV_OK) rc = r2;
	}
	if(rc == POV_OK && fmt.dev && dev_stream != fmt.dev->n_streams)
		rc = pov_fail(ctx, POV_ERR_ARG, "pov_decode_corpus_device: the corpus has %llu logical streams, the stream table %u",
		              (unsigned long long) dev_stream, fmt.dev->n_streams);
	if(timing)
		fprintf(stderr, "pov_decode_corpus: %u chunks in %.3f s on the calling thread: wait for parsed chunks %.3f, "
		        "setup ids + wait for the slot %.3f, validate+queue upload %.3f, launch %.3f, fetch/issue %.3f; on the streams (sum over chunks): "
		        "copy in + kernels %.3f s, copy out %.3f s\n",
		        n_chunks, now() - t_begin, t_wait, t_retire, t_upload, t_run, t_fetch, g_copy_in_kernels * 1e-3, g_copy_out * 1e-3);
	if(timeline) {
		for(uint32_t ci = 0; ci < n_chunks; ++ci) {
			float t[4] = {-1, -1, -1, -1};
			for(int k = 0; k < 4; ++k) if(cudaEventElapsedTime(&t[k], tl[0], tl[4 * ci + k]) != cudaSuccess) t[k] = -1;
			fprintf(stderr, "chunk %3u files %4u..%4u: queued %8.3f copy-in done %8.3f kernels done %8.3f copy-out done %8.3f ms | host: taken %8.3f "
			        "slot free %8.3f upload queued %8.3f all queued %8.3f ms\n", ci, chunk_first[ci], chunk_first[ci + 1], t[0], t[1], t[2], t[3],
			        tl_host[4 * ci] * 1e3, tl_host[4 * ci + 1] * 1e3, tl_host[4 * ci + 2] * 1e3, tl_host[4 * ci + 3] * 1e3);
		}
		(void) cudaGetLastError();
	}
	for(auto& e : tl) if(e) cudaEventDestroy(e);
	stop.store(true);
	{ std::lock_guard<std::mutex> lk(mu); cv_space.notify_all(); }
	{ std::lock_guard<std::mutex> lk(cs.pmu); cs.pcv.notify_all(); }
	for(auto& t : pool) t.join();
	for(auto& kv : ready) if(kv.second) cs.release(kv.second->buf);          // chunks nobody consumed (error paths)
	ready.clear();
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
	{
		uint64_t l1 = 0, a1 = 0, b1 = 0;
		for(pov_ctx* sb : cs.sibling) { l1 += sb->launches; a1 += sb->h2d_bytes; b1 += sb->d2h_bytes; }
		ctx->launches += l1 - sibling_launches0;
		ctx->h2d_bytes += a1 - sibling_h2d0;
		ctx->d2h_bytes += b1 - sibling_d2h0;
	}
	if(total_values_out) *total_values_out = total;
	if(fmt.checksum) *fmt.checksum = h_sum;
	if(fmt.sum16) *fmt.sum16 = h_sum16;
	return rc;
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
