// C-ABI implementation (include/pov_synth.h): contexts, setup registration, batch upload / run / fetch.
// Host code only; the kernels are in kernels_staged.cu and kernel_fused.cu.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include <exception>
#include <new>

#include "api_internal.h"
#include "host_tables.h"
#include "kernels.h"
#include "vorbis_parse.h"

using namespace pov;

// ---------------------------------------------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------------------------------------------
int pov_fail(pov_ctx* ctx, int code, const char* fmt, ...) {
	if(ctx) {
		va_list ap;
		va_start(ap, fmt);
		vsnprintf(ctx->err, sizeof ctx->err, fmt, ap);
		va_end(ap);
	}
	return code;
}

// Nothing may throw across the C boundary (include/pov_synth.h): every entry point that allocates is a function-try-block
// ending in this handler (std::bad_alloc from a descriptor that asks for absurd sizes, std::length_error, ...).
int pov_fail_exception(pov_ctx* ctx) {
	try { throw; }
	catch(const std::bad_alloc&) { return pov_fail(ctx, POV_ERR_ARG, "out of host memory (descriptor sizes beyond what this machine can hold)"); }
	catch(const std::exception& e) { return pov_fail(ctx, POV_ERR_ARG, "internal error: %s", e.what()); }
	catch(...) { return pov_fail(ctx, POV_ERR_ARG, "internal error: unknown exception"); }
}

#define CUDA_TRY(ctx, expr)                                                                                       \
	do {                                                                                                          \
		cudaError_t e__ = (expr);                                                                                 \
		if(e__ != cudaSuccess)                                                                                    \
			return pov_fail(ctx, POV_ERR_CUDA, "%s:%d: CUDA error: %s (%s)", __FILE__, __LINE__, cudaGetErrorString(e__), #expr); \
	} while(0)

template <class T>
static cudaError_t dev_upload(T** dptr, const T* h, size_t count, cudaStream_t st) {
	*dptr = nullptr;
	if(count == 0) return cudaSuccess;
	cudaError_t e = cudaMalloc((void**) dptr, count * sizeof(T));
	if(e != cudaSuccess) return e;
	return cudaMemcpyAsync(*dptr, h, count * sizeof(T), cudaMemcpyHostToDevice, st);
}

static bool is_pow2_in(uint32_t v, uint32_t lo, uint32_t hi) { return v >= lo && v <= hi && (v & (v - 1)) == 0; }
static uint32_t ilog2u(uint32_t v) { uint32_t r = 0; while(v > 1) { v >>= 1; ++r; } return r; }

// growable device buffer
cudaError_t DevBuf::reserve(size_t bytes) {
	if(bytes <= cap) return cudaSuccess;
	if(ptr) cudaFree(ptr);
	ptr = nullptr; cap = 0;
	size_t want = bytes + bytes / 8 + 256;
	cudaError_t e = cudaMalloc(&ptr, want);
	if(e == cudaSuccess) cap = want;
	return e;
}
void DevBuf::release() { if(ptr) cudaFree(ptr); ptr = nullptr; cap = 0; }

cudaError_t PinnedBuf::reserve(size_t bytes) {
	if(bytes <= cap) return cudaSuccess;
	release();
	cudaError_t e = cudaHostAlloc(&ptr, bytes + bytes / 4, cudaHostAllocDefault);
	if(e == cudaSuccess) cap = bytes + bytes / 4;
	else ptr = nullptr;
	return e;
}
void PinnedBuf::release() { if(ptr) cudaFreeHost(ptr); ptr = nullptr; cap = 0; }

// ---------------------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------------------
extern "C" uint32_t pov_abi_version(void) { return POV_ABI_VERSION; }
extern "C" void pov_inverse_db_table(float out[256]) { make_inverse_db_table(out); }

extern "C" int pov_ctx_create(int device, pov_ctx** out, const char** error_out) {
	static thread_local char errbuf[256];
	auto fail = [&](const char* msg, cudaError_t e) {
		snprintf(errbuf, sizeof errbuf, "pov_ctx_create: %s: %s", msg, cudaGetErrorString(e));
		if(error_out) *error_out = errbuf;
		return (int) POV_ERR_CUDA;
	};
	if(!out) return POV_ERR_ARG;
	*out = nullptr;
	int count = 0;
	cudaError_t e = cudaGetDeviceCount(&count);
	if(e != cudaSuccess || count == 0) return fail("no CUDA device (this library has no CPU fallback)", e);
	if(device < 0 || device >= count) return fail("device ordinal out of range", cudaErrorInvalidDevice);
	cudaDeviceProp prop;
	if((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail("cudaGetDeviceProperties", e);
	if(prop.major != 10) {
		snprintf(errbuf, sizeof errbuf, "pov_ctx_create: device %d is sm_%d%d; this build holds sm_100a code only", device, prop.major, prop.minor);
		if(error_out) *error_out = errbuf;
		return POV_ERR_CUDA;
	}
	if((e = cudaSetDevice(device)) != cudaSuccess) return fail("cudaSetDevice", e);
	std::unique_ptr<pov_ctx> ctx(new pov_ctx());
	ctx->device = device;
	ctx->sm_count = prop.multiProcessorCount;
	if((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", e);
	if((e = cudaStreamCreateWithFlags(&ctx->out_stream, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", e);
	if((e = cudaEventCreateWithFlags(&ctx->ev_compute, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
	if((e = cudaEventCreateWithFlags(&ctx->ev_out, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
	float table[256];
	make_inverse_db_table(table);
	if((e = dev_upload((float**) &ctx->d_inv_db, table, 256, ctx->stream)) != cudaSuccess) return fail("upload inverse dB table", e);
	if((e = cudaStreamSynchronize(ctx->stream)) != cudaSuccess) return fail("sync", e);
	if((e = cudaMalloc((void**) &ctx->d_counter, 256)) != cudaSuccess) return fail("cudaMalloc work counter", e);
	if(const char* k = getenv("POV_KERNEL")) ctx->kernel_choice = !strcmp(k, "fused") ? 1 : !strcmp(k, "warp") ? 2 : 0;
	if(const char* de = getenv("POV_DEVICE_ENTROPY")) ctx->device_entropy = atoi(de) != 0;
	if(const char* sp = getenv("POV_ALLOW_SPANNING")) ctx->allow_spanning = atoi(sp) != 0;
	const char* rl = getenv("POV_RUN_LEN");
	ctx->run_len = rl ? (uint32_t) std::min(64, std::max(2, atoi(rl))) : 0;   // the fused kernel keeps <= 65 descriptors per run
	ctx->err[0] = 0;
	*out = ctx.release();
	return POV_OK;
}

static void free_setup(SetupRec& s) {
	cudaFree((void*) s.d_huff); cudaFree((void*) s.d_hbooks); cudaFree((void*) s.d_fsyntax);
	cudaFree((void*) s.d_floors); cudaFree((void*) s.d_mappings); cudaFree((void*) s.d_residues);
	cudaFree((void*) s.d_codebooks); cudaFree((void*) s.d_vq); cudaFree((void*) s.d_fast);
}

extern "C" void pov_ctx_destroy(pov_ctx* ctx) {
	if(!ctx) return;
	cudaSetDevice(ctx->device);
	cudaStreamSynchronize(ctx->stream);
	if(ctx->corpus && ctx->corpus_free) { ctx->corpus_free(ctx->corpus); ctx->corpus = nullptr; }
	for(auto& s : ctx->setups) free_setup(s);
	for(auto& kv : ctx->blk_tables) { cudaFree((void*) kv.second.d_rot); cudaFree((void*) kv.second.d_fft); cudaFree((void*) kv.second.d_fftp); cudaFree((void*) kv.second.d_fft8); cudaFree((void*) kv.second.d_slope); }
	cudaFree((void*) ctx->d_setups);
	cudaFree((void*) ctx->d_inv_db);
	cudaFree((void*) ctx->d_counter);
	ctx->mdct_in.release(); ctx->mdct_out.release();
	if(ctx->out_stream) { cudaStreamSynchronize(ctx->out_stream); cudaStreamDestroy(ctx->out_stream); }
	if(ctx->ev_compute) cudaEventDestroy(ctx->ev_compute);
	if(ctx->ev_out) cudaEventDestroy(ctx->ev_out);
	cudaStreamDestroy(ctx->stream);
	delete ctx;
}

extern "C" const char* pov_last_error(const pov_ctx* ctx) { return ctx ? ctx->err : "null context"; }
extern "C" void* pov_ctx_stream(pov_ctx* ctx) { return ctx ? (void*) ctx->stream : nullptr; }
extern "C" uint64_t pov_ctx_launch_count(const pov_ctx* ctx) { return ctx ? ctx->launches : 0; }
extern "C" void pov_ctx_set_device_entropy(pov_ctx* ctx, int on) { if(ctx) ctx->device_entropy = on != 0; }
extern "C" void pov_ctx_set_page_spanning(pov_ctx* ctx, int on) { if(ctx) ctx->allow_spanning = on != 0; }
extern "C" void pov_ctx_set_cut_damage(pov_ctx* ctx, int on) { if(ctx) ctx->cut_damage = on != 0; }
extern "C" void pov_ctx_io_bytes(const pov_ctx* ctx, uint64_t* h2d, uint64_t* d2h) {
	if(h2d) *h2d = ctx ? ctx->h2d_bytes : 0;
	if(d2h) *d2h = ctx ? ctx->d2h_bytes : 0;
}

// per-blocksize tables shared by all setups of a context
static int get_block_tables(pov_ctx* ctx, uint32_t n, BlockTables** out) {
	auto it = ctx->blk_tables.find(n);
	if(it != ctx->blk_tables.end()) { *out = &it->second; return POV_OK; }
	BlockTables t;
	std::vector<float> rot, fft, fftp, fft8, slope;
	make_rotation(n, rot);
	make_fft_twiddles(n, fft);
	make_fft_pass_tables(n, fftp);
	make_fft_r8_tables(n, fft8);
	make_rotation_consts(n, t.c1, t.c6);
	t.fft8_count = (uint32_t) (fft8.size() / 2);
	make_window_slope(n / 2, slope);
	t.h_slope = slope;
	CUDA_TRY(ctx, dev_upload((float**) &t.d_rot, rot.data(), rot.size(), ctx->stream));
	CUDA_TRY(ctx, dev_upload((float**) &t.d_fft, fft.data(), fft.size(), ctx->stream));
	CUDA_TRY(ctx, dev_upload((float**) &t.d_fftp, fftp.data(), fftp.size(), ctx->stream));
	CUDA_TRY(ctx, dev_upload((float**) &t.d_fft8, fft8.data(), fft8.size(), ctx->stream));
	CUDA_TRY(ctx, dev_upload((float**) &t.d_slope, slope.data(), slope.size(), ctx->stream));
	std::vector<float> tm;
	if(n == 2048) {
		make_tm_lane_tables(n, rot, slope, tm);
		CUDA_TRY(ctx, dev_upload((float**) &t.d_tm, tm.data(), tm.size(), ctx->stream));
	}
	CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	auto ins = ctx->blk_tables.emplace(n, std::move(t));
	*out = &ins.first->second;
	return POV_OK;
}

// canonical byte image of a setup (for de-duplication: a corpus of files typically shares a handful of setups)
static void serialize_setup(const pov_setup* s, std::string& out) {
	auto put = [&](const void* p, size_t n) { out.append((const char*) p, n); };
	put(&s->channels, 4); put(&s->sample_rate, 4); put(s->blocksize, 8);
	put(&s->n_codebooks, 4); put(&s->n_floors, 4); put(&s->n_residues, 4); put(&s->n_mappings, 4); put(&s->n_modes, 4);
	for(uint32_t i = 0; i < s->n_codebooks; ++i) {
		const pov_codebook& c = s->codebooks[i];
		put(&c.dim, 4); put(&c.n_entries, 4); put(&c.lookup_type, 4);
		if(c.lookup_type != 0 && c.vq) put(c.vq, sizeof(float) * (size_t) c.dim * c.n_entries);
		const uint8_t has_len = c.lengths != nullptr;
		put(&has_len, 1);
		if(c.lengths) put(c.lengths, c.n_entries);
	}
	{
		const uint8_t has_syntax = s->floor_syntax != nullptr;
		put(&has_syntax, 1);
		if(s->floor_syntax) put(s->floor_syntax, sizeof(pov_floor1_syntax) * (size_t) s->n_floors);
		for(uint32_t i = 0; i < s->n_residues; ++i) put(&s->residues[i].classbook, 4);
	}
	for(uint32_t i = 0; i < s->n_floors; ++i) {
		const pov_floor1& f = s->floors[i];
		put(&f.n_posts, 2); put(&f.multiplier, 1); put(f.xs, 2 * (size_t) std::min<uint32_t>(f.n_posts, POV_MAX_POSTS));
	}
	for(uint32_t i = 0; i < s->n_residues; ++i) {
		const pov_residue& r = s->residues[i];
		put(&r.type, 4); put(&r.begin, 4); put(&r.end, 4); put(&r.partition_size, 4); put(&r.n_class, 4);
		put(r.books, 8 * (size_t) std::min<uint32_t>(r.n_class, POV_MAX_CLASSES));
	}
	for(uint32_t i = 0; i < s->n_mappings; ++i) {
		const pov_mapping& m = s->mappings[i];
		put(&m.n_submaps, 4); put(&m.n_couplings, 4); put(m.mux, POV_MAX_CHANNELS);
		put(m.submap_floor, POV_MAX_SUBMAPS); put(m.submap_residue, POV_MAX_SUBMAPS);
		put(m.coupling_mag, std::min<uint32_t>(m.n_couplings, POV_MAX_COUPLINGS));
		put(m.coupling_ang, std::min<uint32_t>(m.n_couplings, POV_MAX_COUPLINGS));
	}
	for(uint32_t i = 0; i < s->n_modes; ++i) { put(&s->modes[i].blockflag, 1); put(&s->modes[i].mapping, 1); }
}

// Compact tables of the warp-autonomous kernel. Returns false when the setup is outside what kernel_warp.cu handles
// (those batches run on the CTA-per-run fused kernel instead).
static bool build_fast_tables(const pov_setup* s, const std::vector<DevFloor>& floors, const std::vector<DevMapping>& maps,
                              const uint32_t posts_cls[2], FastTables& ft, uint32_t& short_cap, uint32_t& long_cap, bool& wide) {
	memset(&ft, 0, sizeof ft);
	if(!warp_kernel_supports(s->blocksize[0], s->blocksize[1])) return false;
	if(s->channels > POV_MAX_CHANNELS || s->n_floors > POV_FAST_MAX_FLOORS || s->n_mappings > POV_FAST_MAX_MAPPINGS) return false;
	if(posts_cls[0] > POV_FAST_MAX_POSTS || posts_cls[1] > POV_FAST_MAX_POSTS) return false;
	short_cap = (posts_cls[0] + 3u) & ~3u;
	if(short_cap < 4) short_cap = 4;
	wide = posts_cls[0] > 32 || posts_cls[1] > 32;
	long_cap = wide ? 64u : 32u;             // (the wide kernel keeps 64 records per long curve whichever class has the big floor)
	ft.channels = s->channels;
	ft.short_posts_cap = short_cap;
	ft.long_posts_cap = long_cap;
	ft.wide = wide ? 1u : 0u;
	for(uint32_t i = 0; i < s->n_floors; ++i) {
		const DevFloor& f = floors[i];
		FastFloor& o = ft.floors[i];
		if(f.n_posts > POV_FAST_MAX_POSTS) {            // only reachable floors matter, but an unreachable big floor is not worth a special case
			bool used = false;
			for(uint32_t m = 0; m < s->n_mappings && !used; ++m)
				for(uint32_t c = 0; c < s->channels; ++c) if(maps[m].floor_of_ch[c] == i) used = true;
			if(used) return false;
			continue;
		}
		o.n_posts = f.n_posts; o.n_levels = f.n_levels; o.range = f.range; o.multiplier = f.multiplier;
		for(uint32_t k = 0; k < f.n_posts; ++k) {
			if(f.xs[k] > POV_FAST_MAX_X) return false;
			const uint32_t sidx = f.sorted_idx[k];
			o.post[k][0] = (uint32_t) f.lo[k] | ((uint32_t) f.hi[k] << 8) | ((uint32_t) f.level[k] << 16) | (sidx << 24);
			o.post[k][1] = (uint32_t) f.dxn[k] | ((uint32_t) f.adx[k] << 16);
			o.post[k][2] = (k >= 2) ? (uint32_t) ((0x100000000ull + f.adx[k] - 1) / f.adx[k]) : 0u;
			o.post[k][3] = f.xs[sidx];
			o.xs_sorted[k] = f.xs[sidx] | (sidx << 16);        // X of the k-th smallest post | its post number
		}
	}
	for(uint32_t m = 0; m < s->n_mappings; ++m) {
		const DevMapping& mp = maps[m];
		if(mp.n_couplings > POV_FAST_MAX_STEPS) return false;
		ft.ncoup[m] = (uint8_t) mp.n_couplings;
		for(uint32_t k = 0; k < mp.n_couplings; ++k) { ft.cmag[m][k] = mp.coupling_mag[k]; ft.cang[m][k] = mp.coupling_ang[k]; }
		for(uint32_t c = 0; c < s->channels; ++c) {
			ft.floor_of_ch[m][c] = mp.floor_of_ch[c];
			// Steps are applied k = n-1 .. 0 (hpp:1214). Walking them backwards in time (k = 0 .. n-1) from the final value of
			// channel c collects the steps that can reach it and the channels whose residue vectors it needs.
			uint32_t need = 1u << c;
			std::vector<uint32_t> steps;
			for(uint32_t k = 0; k < mp.n_couplings; ++k) {
				const uint32_t mg = mp.coupling_mag[k], an = mp.coupling_ang[k];
				if((need >> mg) & 1u || (need >> an) & 1u) { need |= (1u << mg) | (1u << an); steps.push_back(k); }
			}
			FastCouple& fc = ft.couple[m][c];
			uint8_t local[POV_MAX_CHANNELS];
			memset(local, 0xff, sizeof local);
			fc.nl = 0;
			fc.ch[fc.nl] = (uint8_t) c; local[c] = fc.nl++;
			for(uint32_t x = 0; x < s->channels; ++x)
				if(x != c && ((need >> x) & 1u)) {
					if(fc.nl >= POV_FAST_MAX_DEPS) return false;
					fc.ch[fc.nl] = (uint8_t) x; local[x] = fc.nl++;
				}
			fc.nsteps = (uint8_t) steps.size();
			for(size_t i = 0; i < steps.size(); ++i) {         // application order = descending k
				const uint32_t k = steps[steps.size() - 1 - i];
				fc.sm[i] = local[mp.coupling_mag[k]]; fc.sa[i] = local[mp.coupling_ang[k]];
			}
		}
	}
	for(uint32_t i = 0; i < s->n_modes; ++i) { ft.mode_flag[i] = s->modes[i].blockflag ? 1 : 0; ft.mode_map[i] = s->modes[i].mapping; }
	return warp_kernel_smem_bytes(s->blocksize[0], s->blocksize[1], short_cap, long_cap, nullptr, nullptr, nullptr) <= 227 * 1024;
}

extern "C" int pov_setup_register(pov_ctx* ctx, const pov_setup* s, uint32_t* id_out) try {
	if(!ctx || !s || !id_out) return POV_ERR_ARG;
	cudaSetDevice(ctx->device);
	if(s->abi_version != POV_ABI_VERSION) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: abi_version %u != %u", s->abi_version, POV_ABI_VERSION);
	if(s->channels < 1) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: channels == 0 (hpp:774)");
	if(s->channels > POV_MAX_CHANNELS) return pov_fail(ctx, POV_ERR_UNSUPPORTED, "pov_setup: %u channels > %u supported by this build", s->channels, POV_MAX_CHANNELS);
	if(!is_pow2_in(s->blocksize[0], 64, 8192) || !is_pow2_in(s->blocksize[1], 64, 8192) || s->blocksize[0] > s->blocksize[1])
		return pov_fail(ctx, POV_ERR_ARG, "pov_setup: blocksizes %u/%u invalid (hpp:1295-1298)", s->blocksize[0], s->blocksize[1]);
	if(s->n_modes < 1 || s->n_modes > POV_MAX_MODES || !s->modes) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: n_modes out of range (hpp:950)");
	if(s->n_mappings < 1 || !s->mappings || s->n_floors < 1 || !s->floors) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: needs >= 1 mapping and floor");
	if(s->n_codebooks > POV_MAX_CODEBOOKS) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: > 256 codebooks (hpp:905)");
	if(s->n_floors > 64 || s->n_residues > 64 || s->n_mappings > 64) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: > 64 floors/residues/mappings (hpp:923-941)");

	std::string image;
	serialize_setup(s, image);
	for(size_t i = 0; i < ctx->setups.size(); ++i)
		if(ctx->setups[i].image == image) { *id_out = (uint32_t) i; return POV_OK; }

	SetupRec rec;
	rec.channels = s->channels; rec.sample_rate = s->sample_rate;
	rec.blocksize[0] = s->blocksize[0]; rec.blocksize[1] = s->blocksize[1];
	DevSetup& d = rec.dev;
	memset(&d, 0, sizeof d);
	d.channels = s->channels;
	d.blocksize[0] = s->blocksize[0]; d.blocksize[1] = s->blocksize[1];
	d.log2bs[0] = ilog2u(s->blocksize[0]); d.log2bs[1] = ilog2u(s->blocksize[1]);
	d.n_floors = s->n_floors; d.n_mappings = s->n_mappings; d.n_modes = s->n_modes;
	d.n_residues = s->n_residues; d.n_codebooks = s->n_codebooks;

	// codebooks
	std::vector<DevCodebook> cbs(s->n_codebooks);
	std::vector<float> vq_all;
	std::vector<size_t> vq_off(s->n_codebooks, 0);
	uint32_t max_entries = 0;
	for(uint32_t i = 0; i < s->n_codebooks; ++i) {
		const pov_codebook& c = s->codebooks[i];
		if(c.dim < 1 || c.n_entries < 1) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: codebook %u has dim/entries == 0 (hpp:257,259)", i);
		if(c.lookup_type > 2) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: codebook %u lookup_type %u (hpp:299)", i, c.lookup_type);
		if(c.lookup_type != 0 && !c.vq) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: codebook %u has no VQ table", i);
		cbs[i].dim = c.dim; cbs[i].n_entries = c.n_entries; cbs[i].lookup_type = c.lookup_type; cbs[i].pad = 0; cbs[i].vq = nullptr;
		max_entries = std::max(max_entries, c.n_entries);
		if(c.lookup_type != 0) {
			vq_off[i] = vq_all.size();
			vq_all.insert(vq_all.end(), c.vq, c.vq + (size_t) c.dim * c.n_entries);
		}
	}
	d.entry_bits = (max_entries > 65536) ? 32 : 16;
	rec.entry_bits = d.entry_bits;
	// floors
	std::vector<DevFloor> floors(s->n_floors);
	uint32_t max_posts = 2;
	for(uint32_t i = 0; i < s->n_floors; ++i) {
		std::string msg;
		if(!make_floor_tables(s->floors[i], floors[i], msg)) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: floor %u: %s", i, msg.c_str());
		max_posts = std::max<uint32_t>(max_posts, floors[i].n_posts);
	}
	rec.max_posts = max_posts;
	// residues
	std::vector<DevResidue> residues(s->n_residues);
	for(uint32_t i = 0; i < s->n_residues; ++i) {
		const pov_residue& r = s->residues[i];
		if(r.type > 2) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: residue %u type %u (hpp:634)", i, r.type);
		if(r.begin > r.end) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: residue %u begin > end (hpp:638)", i);
		if(r.partition_size < 1 || r.n_class < 1 || r.n_class > POV_MAX_CLASSES) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: residue %u partition/class out of range", i);
		DevResidue& o = residues[i];
		o.type = r.type; o.begin = r.begin; o.end = r.end; o.partition_size = r.partition_size; o.n_class = r.n_class;
		memset(o.books, POV_NO_BOOK, sizeof o.books);
		for(uint32_t k = 0; k < r.n_class * 8; ++k) {
			const uint8_t bk = r.books[k];
			o.books[k] = bk;
			if(bk == POV_NO_BOOK) continue;
			if(bk >= s->n_codebooks) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: residue %u references codebook %u of %u", i, bk, s->n_codebooks);
			const uint32_t dim = s->codebooks[bk].dim;
			if(r.partition_size % dim) return pov_fail(ctx, POV_ERR_UNSUPPORTED, "pov_setup: residue %u: codebook %u dim %u does not divide partition size %u", i, bk, dim, r.partition_size);
		}
	}
	// mappings
	std::vector<DevMapping> maps(s->n_mappings);
	for(uint32_t i = 0; i < s->n_mappings; ++i) {
		const pov_mapping& m = s->mappings[i];
		DevMapping& o = maps[i];
		memset(&o, 0, sizeof o);
		if(m.n_submaps < 1 || m.n_submaps > POV_MAX_SUBMAPS) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: mapping %u: n_submaps %u (hpp:781)", i, m.n_submaps);
		if(m.n_couplings > POV_MAX_COUPLINGS) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: mapping %u: n_couplings %u (hpp:783)", i, m.n_couplings);
		o.n_submaps = m.n_submaps; o.n_couplings = m.n_couplings;
		for(uint32_t k = 0; k < m.n_submaps; ++k) {
			if(m.submap_floor[k] >= s->n_floors) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: mapping %u submap %u floor out of range (hpp:807)", i, k);
			if(s->n_residues && m.submap_residue[k] >= s->n_residues) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: mapping %u submap %u residue out of range (hpp:809)", i, k);
			o.submap_residue[k] = m.submap_residue[k];
		}
		for(uint32_t c = 0; c < s->channels; ++c) {
			if(m.mux[c] >= m.n_submaps) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: mapping %u mux[%u] out of range (hpp:799)", i, c);
			o.mux[c] = m.mux[c];
			o.floor_of_ch[c] = m.submap_floor[m.mux[c]];
		}
		for(uint32_t k = 0; k < m.n_couplings; ++k) {
			const uint8_t mg = m.coupling_mag[k], an = m.coupling_ang[k];
			if(mg == an || mg >= s->channels || an >= s->channels) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: mapping %u coupling %u invalid (hpp:788-790)", i, k);
			o.coupling_mag[k] = mg; o.coupling_ang[k] = an;
		}
	}
	for(uint32_t i = 0; i < s->n_modes; ++i) {
		if(s->modes[i].mapping >= s->n_mappings) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: mode %u mapping out of range (hpp:832)", i);
		d.mode_blockflag[i] = s->modes[i].blockflag ? 1 : 0;
		d.mode_mapping[i] = s->modes[i].mapping;
	}
	for(uint32_t i = 0; i < s->n_modes; ++i) {
		const pov_mapping& m = s->mappings[s->modes[i].mapping];
		const int cls = s->modes[i].blockflag ? 1 : 0;
		for(uint32_t k = 0; k < m.n_submaps; ++k)
			rec.posts_cls[cls] = std::max<uint32_t>(rec.posts_cls[cls], floors[m.submap_floor[k]].n_posts);
	}
	// k_residue_apply's need, from the submaps each mode decodes: the working vector of one submap (nch * n/2 floats, for
	// every residue type) and its 8 * partitions * vectors read cursors
	if(s->n_residues) {
		uint64_t acc_max = 0, cur_max = 0, both_max = 0;
		for(uint32_t mo = 0; mo < s->n_modes; ++mo) {
			const DevMapping& mp = maps[s->modes[mo].mapping];
			const uint32_t half = s->blocksize[s->modes[mo].blockflag ? 1 : 0] / 2;
			for(uint32_t sm = 0; sm < mp.n_submaps; ++sm) {
				uint32_t nch = 0;
				for(uint32_t c = 0; c < s->channels; ++c) nch += (mp.mux[c] == sm);
				const DevResidue& r = residues[mp.submap_residue[sm]];
				const uint32_t vch = r.type == 2 ? 1 : nch, vlen = r.type == 2 ? nch * half : half;
				const uint64_t parts = (std::min(r.end, vlen) - std::min(r.begin, vlen)) / r.partition_size;
				const uint64_t acc = (uint64_t) nch * half, cur = 8 * parts * vch;
				acc_max = std::max(acc_max, acc); cur_max = std::max(cur_max, cur); both_max = std::max(both_max, acc + cur);
			}
		}
		rec.res_smem = (uint32_t) (both_max * 4 + 64);
		rec.res_acc_smem = (uint32_t) (acc_max * 4 + 64);
		rec.res_cursors = (uint32_t) cur_max;
	}
	rec.n_modes = s->n_modes;
	memcpy(rec.mode_blockflag, d.mode_blockflag, sizeof rec.mode_blockflag);
	memcpy(rec.mode_mapping, d.mode_mapping, sizeof rec.mode_mapping);
	rec.floors_host = floors;
	rec.maps_host = maps;
	rec.residues_host = residues;
	rec.cb_dim.resize(s->n_codebooks);
	for(uint32_t i = 0; i < s->n_codebooks; ++i) rec.cb_dim[i] = s->codebooks[i].dim;

	// device copies
	BlockTables *t0 = nullptr, *t1 = nullptr;
	int rc;
	if((rc = get_block_tables(ctx, s->blocksize[0], &t0)) != POV_OK) return rc;
	if((rc = get_block_tables(ctx, s->blocksize[1], &t1)) != POV_OK) return rc;
	d.slope[0] = t0->d_slope; d.slope[1] = t1->d_slope;
	d.rot[0] = t0->d_rot; d.rot[1] = t1->d_rot;
	d.fft[0] = t0->d_fft; d.fft[1] = t1->d_fft;
	d.fftp[0] = t0->d_fftp; d.fftp[1] = t1->d_fftp;
	d.fft8[0] = t0->d_fft8; d.fft8[1] = t1->d_fft8;
	d.fft8_count[0] = t0->fft8_count; d.fft8_count[1] = t1->fft8_count;
	d.rotc1[0] = make_float2(t0->c1[0], t0->c1[1]); d.rotc1[1] = make_float2(t1->c1[0], t1->c1[1]);
	d.rotc6[0] = make_float2(t0->c6[0], t0->c6[1]); d.rotc6[1] = make_float2(t1->c6[0], t1->c6[1]);
	rec.table_float2 = t0->fft8_count + t1->fft8_count + s->blocksize[0] / 8 + s->blocksize[1] / 8;
	CUDA_TRY(ctx, dev_upload((float**) &rec.d_vq, vq_all.data(), vq_all.size(), ctx->stream));
	for(uint32_t i = 0; i < s->n_codebooks; ++i)
		if(cbs[i].lookup_type != 0) cbs[i].vq = rec.d_vq + vq_off[i];
	CUDA_TRY(ctx, dev_upload((DevCodebook**) &rec.d_codebooks, cbs.data(), cbs.size(), ctx->stream));
	CUDA_TRY(ctx, dev_upload((DevFloor**) &rec.d_floors, floors.data(), floors.size(), ctx->stream));
	CUDA_TRY(ctx, dev_upload((DevResidue**) &rec.d_residues, residues.data(), residues.size(), ctx->stream));
	CUDA_TRY(ctx, dev_upload((DevMapping**) &rec.d_mappings, maps.data(), maps.size(), ctx->stream));
	d.floors = rec.d_floors; d.mappings = rec.d_mappings; d.residues = rec.d_residues; d.codebooks = rec.d_codebooks;
	{
		FastTables ft;
		rec.fast_ok = build_fast_tables(s, floors, maps, rec.posts_cls, ft, rec.fast_short_cap, rec.fast_long_cap, rec.fast_wide);
		rec.fast_max_nl = 1;
		for(uint32_t m = 0; m < s->n_mappings && m < POV_FAST_MAX_MAPPINGS; ++m)
			for(uint32_t c = 0; c < s->channels; ++c) rec.fast_max_nl = std::max<uint32_t>(rec.fast_max_nl, ft.couple[m][c].nl);
		if(rec.fast_ok) CUDA_TRY(ctx, dev_upload((FastTables**) &rec.d_fast, &ft, 1, ctx->stream));
		CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));      // ft lives on this stack frame
	}
	// ---- device entropy decode (POV_INPUT_PACKETS): Huffman tables, floor syntax, per-mode worst-case arena sizes ----
	{
		bool ok = s->floor_syntax != nullptr && s->n_residues > 0 && s->n_residues <= 64 && s->n_codebooks <= 255;
		for(uint32_t i = 0; i < s->n_codebooks && ok; ++i) ok = s->codebooks[i].lengths != nullptr;
		std::vector<uint32_t> arena;
		std::vector<DevHuffBook> hb(s->n_codebooks);
		for(uint32_t i = 0; i < s->n_codebooks && ok; ++i) {
			HuffTables t;
			std::string why;
			if(!build_huff_tables(s->codebooks[i].lengths, s->codebooks[i].n_entries, POV_HUFF_LUT_BITS, t, why))
				return pov_fail(ctx, POV_ERR_ARG, "pov_setup: codebook %u: %s", i, why.c_str());
			memset(&hb[i], 0, sizeof hb[i]);
			hb[i].lut_off = (uint32_t) arena.size();
			arena.insert(arena.end(), t.lut.begin(), t.lut.end());
			hb[i].sorted_off = (uint32_t) arena.size();
			hb[i].n_sorted = (uint32_t) t.sorted_code.size();
			arena.insert(arena.end(), t.sorted_code.begin(), t.sorted_code.end());
			for(size_t k = 0; k < t.sorted_entry.size(); ++k) arena.push_back((t.sorted_entry[k] << 6) | t.sorted_len[k]);
			hb[i].n_entries = s->codebooks[i].n_entries; hb[i].dim = s->codebooks[i].dim; hb[i].lookup_type = s->codebooks[i].lookup_type;
			if(s->codebooks[i].n_entries >= (1u << 26)) ok = false;           // entry numbers share a word with the length
		}
		std::vector<DevFloorSyntax> fsx(s->n_floors);
		for(uint32_t i = 0; i < s->n_floors && ok; ++i) {
			const pov_floor1_syntax& in = s->floor_syntax[i];
			DevFloorSyntax& o = fsx[i];
			memset(&o, 0, sizeof o);
			if(in.n_partitions > 31 || in.n_classes > 16) { ok = false; break; }
			o.n_partitions = in.n_partitions; o.n_classes = in.n_classes;
			uint32_t rb = 0, rg = floors[i].range - 1;
			while(rg) { ++rb; rg >>= 1; }
			o.ybits = (uint8_t) rb;                                           // ilog(range - 1), hpp:494-497
			uint32_t count = 2;
			for(uint32_t k = 0; k < in.n_partitions; ++k) {
				if(in.partition_class[k] >= in.n_classes) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: floor %u: partition class out of range (hpp:429)", i);
				o.partition_class[k] = in.partition_class[k];
				count += in.class_dim[in.partition_class[k]];
			}
			if(count != s->floors[i].n_posts) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: floor %u: syntax describes %u posts, the floor has %u (hpp:519)", i, count, s->floors[i].n_posts);
			for(uint32_t k = 0; k < in.n_classes; ++k) {
				if(in.class_dim[k] < 1 || in.class_dim[k] > 8 || in.class_subclass_bits[k] > 3) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: floor %u: class %u out of range (hpp:433-434)", i, k);
				o.class_dim[k] = in.class_dim[k]; o.class_subclass_bits[k] = in.class_subclass_bits[k]; o.class_masterbook[k] = in.class_masterbook[k];
				if(in.class_subclass_bits[k] && in.class_masterbook[k] >= s->n_codebooks) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: floor %u: masterbook out of range", i);
				for(uint32_t b = 0; b < 8; ++b) {
					const int bk = (b < (1u << in.class_subclass_bits[k])) ? in.class_books[k][b] : -1;
					if(bk >= (int) s->n_codebooks) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: floor %u: subclass book out of range", i);
					o.class_books[k][b] = (int16_t) bk;
				}
			}
		}
		for(uint32_t i = 0; i < s->n_residues && ok; ++i) {
			if(s->residues[i].classbook >= s->n_codebooks) return pov_fail(ctx, POV_ERR_ARG, "pov_setup: residue %u: classbook out of range (hpp:700)", i);
			d.classbook[i] = s->residues[i].classbook;
		}
		// a submap without channels is fatal for every packet of its mapping in the reference (hpp:680): refuse the mode of decode
		for(uint32_t m = 0; m < s->n_mappings && ok; ++m)
			for(uint32_t sm = 0; sm < maps[m].n_submaps; ++sm) {
				bool any = false;
				for(uint32_t c = 0; c < s->channels; ++c) any |= (maps[m].mux[c] == sm);
				if(!any) ok = false;
			}
		if(ok) {
			// worst-case arena sizes of one packet per mode: Y slots of every channel; entries payload = per submap the header,
			// the classification bytes and, per pass, the largest vector count any class can code in a partition
			for(uint32_t mo = 0; mo < s->n_modes; ++mo) {
				const DevMapping& mp = maps[s->modes[mo].mapping];
				const uint32_t half = s->blocksize[s->modes[mo].blockflag ? 1 : 0] / 2;
				uint32_t ycap = 0;
				uint64_t ecap = 0;
				for(uint32_t c = 0; c < s->channels; ++c) ycap += floors[mp.floor_of_ch[c]].n_posts;
				for(uint32_t sm = 0; sm < mp.n_submaps; ++sm) {
					uint32_t nch = 0;
					for(uint32_t c = 0; c < s->channels; ++c) nch += (mp.mux[c] == sm);
					const DevResidue& r = residues[mp.submap_residue[sm]];
					const uint32_t vch = r.type == 2 ? 1 : nch, vlen = r.type == 2 ? nch * half : half;
					const uint32_t lb = std::min(r.begin, vlen), le = std::min(r.end, vlen), parts = (le - lb) / r.partition_size;
					uint64_t per_part = 0;
					for(uint32_t pass = 0; pass < 8; ++pass) {
						uint32_t mx = 0;
						for(uint32_t cl = 0; cl < r.n_class; ++cl) {
							const uint32_t bk = r.books[cl * 8 + pass];
							if(bk != POV_NO_BOOK && bk < s->n_codebooks) mx = std::max(mx, r.partition_size / s->codebooks[bk].dim);
						}
						per_part += mx;
					}
					ecap += 4 + (((uint64_t) vch * parts + 3) & ~3ull) + ((per_part * parts * vch * (d.entry_bits / 8) + 3) & ~3ull);
				}
				if(ecap > 0xFFFFFFF0ull) { ok = false; break; }
				rec.mode_ys_cap[mo] = ycap;
				rec.mode_ent_cap[mo] = (uint32_t) ecap;
			}
		}
		if(ok) {
			uint32_t mb = 0, v = s->n_modes - 1;
			while(v) { ++mb; v >>= 1; }
			d.mode_bits = mb;
			CUDA_TRY(ctx, dev_upload((uint32_t**) &rec.d_huff, arena.data(), arena.size(), ctx->stream));
			CUDA_TRY(ctx, dev_upload((DevHuffBook**) &rec.d_hbooks, hb.data(), hb.size(), ctx->stream));
			CUDA_TRY(ctx, dev_upload((DevFloorSyntax**) &rec.d_fsyntax, fsx.data(), fsx.size(), ctx->stream));
			CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
			d.huff = rec.d_huff; d.hbooks = rec.d_hbooks; d.fsyntax = rec.d_fsyntax;
		}
		rec.entropy_ok = ok;
	}
	rec.image.swap(image);
	ctx->setups.push_back(std::move(rec));

	// the device array of DevSetup is rebuilt (kernels index it by setup id)
	std::vector<DevSetup> all(ctx->setups.size());
	for(size_t i = 0; i < all.size(); ++i) all[i] = ctx->setups[i].dev;
	CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	if(ctx->d_setups) cudaFree((void*) ctx->d_setups);
	CUDA_TRY(ctx, dev_upload((DevSetup**) &ctx->d_setups, all.data(), all.size(), ctx->stream));
	CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	*id_out = (uint32_t) (ctx->setups.size() - 1);
	return POV_OK;
} POV_NOTHROW_END(ctx)

extern "C" int pov_setup_entry_bits(const pov_ctx* ctx, uint32_t id) {
	if(!ctx || id >= ctx->setups.size()) return -1;
	return (int) ctx->setups[id].entry_bits;
}

extern "C" int pov_window(uint32_t bs0, uint32_t bs1, int blockflag, int prev, int next, float* out, uint32_t n) try {
	if(!out || !is_pow2_in(bs0, 64, 8192) || !is_pow2_in(bs1, 64, 8192) || bs0 > bs1) return POV_ERR_ARG;
	std::vector<float> w;
	make_window(bs0, bs1, blockflag, prev, next, w);
	if(w.size() != n) return POV_ERR_ARG;
	memcpy(out, w.data(), n * sizeof(float));
	return POV_OK;
} catch(...) { return POV_ERR_ARG; }

extern "C" int pov_setup_get_window(const pov_ctx* ctx, uint32_t id, int blockflag, int prev, int next, float* out, uint32_t n) {
	if(!ctx || id >= ctx->setups.size() || !out) return POV_ERR_ARG;
	const SetupRec& s = ctx->setups[id];
	std::vector<float> w;
	make_window(s.blocksize[0], s.blocksize[1], blockflag, prev, next, w);
	if(w.size() != n) return POV_ERR_ARG;
	memcpy(out, w.data(), n * sizeof(float));
	return POV_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// batches
// ---------------------------------------------------------------------------------------------------------------
static void release_batch(pov_batch_handle* h) {
	h->d_streams.release(); h->d_packets.release(); h->d_ys.release(); h->d_payload.release(); h->d_spec_off.release();
	h->d_stage_off.release(); h->d_runs.release(); h->d_pcm.release(); h->d_status.release(); h->d_spectra.release();
	h->d_entries.release(); h->d_pk_off.release(); h->d_res_cursor.release();
	h->d_feat_rows.release(); h->d_feat_floors.release(); h->d_feat_out.release();
	h->st_final_ys.release(); h->st_flag.release(); h->st_floor.release(); h->st_floor_out.release();
	h->st_env.release(); h->st_mdct.release();
	h->h_derived.release();
	if(h->derived_copied) { cudaEventDestroy(h->derived_copied); h->derived_copied = nullptr; }
}

extern "C" void pov_batch_free(pov_ctx* ctx, pov_batch_handle* h) {
	if(!h) return;
	if(ctx) { cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream); }
	release_batch(h);
	delete h;
}

int pov_check_pcm_dev(pov_ctx* ctx, const void* p, size_t align, const char* fn) {
	if(!p) return pov_fail(ctx, POV_ERR_ARG, "%s: null pcm_dev", fn);
	if((uintptr_t) p % align) return pov_fail(ctx, POV_ERR_ARG, "%s: pcm_dev is not aligned to a %zu-byte sample", fn, align);
	cudaPointerAttributes a;
	if(cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void) cudaGetLastError(); return pov_fail(ctx, POV_ERR_ARG, "%s: pcm_dev is not a CUDA pointer", fn); }
	if((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != ctx->device)
		return pov_fail(ctx, POV_ERR_ARG, "%s: pcm_dev is not device memory of the context's device %d", fn, ctx->device);
	return POV_OK;
}

static int batch_upload(pov_ctx* ctx, const pov_batch* b, void* pcm_dev, pov_batch_handle** out);

extern "C" int pov_batch_upload(pov_ctx* ctx, const pov_batch* b, pov_batch_handle** out) try {
	return batch_upload(ctx, b, nullptr, out);
} POV_NOTHROW_END(ctx)

extern "C" int pov_batch_upload_into(pov_ctx* ctx, const pov_batch* b, void* pcm_dev, pov_batch_handle** out) try {
	if(!ctx || !b || !out) return POV_ERR_ARG;
	cudaSetDevice(ctx->device);
	const int rc = pov_check_pcm_dev(ctx, pcm_dev, pcm_elem_bytes(b->pcm_layout), "pov_batch_upload_into");
	return rc ? rc : batch_upload(ctx, b, pcm_dev, out);
} POV_NOTHROW_END(ctx)

// pcm_dev == nullptr: the handle's own PCM arena
static int batch_upload(pov_ctx* ctx, const pov_batch* b, void* pcm_dev, pov_batch_handle** out) {
	if(!ctx || !b || !out) return POV_ERR_ARG;
	cudaSetDevice(ctx->device);
	if(b->input_kind > POV_INPUT_PACKETS || (b->pcm_layout & ~POV_PCM_S16) > POV_PCM_INTERLEAVED) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: bad input_kind/pcm_layout");
	if(b->pcm_floats > SIZE_MAX / pcm_elem_bytes(b->pcm_layout)) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: PCM arena of %llu samples does not fit the address space", (unsigned long long) b->pcm_floats);
	if((b->n_streams && !b->streams) || (b->n_packets && !b->packets)) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: null arrays");
	if(b->input_kind == POV_INPUT_DENSE && ((uintptr_t) b->payload & 3)) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: dense payload must be 4-byte aligned");

	std::unique_ptr<pov_batch_handle> fresh;
	pov_batch_handle* h = *out;
	if(!h) { fresh.reset(new pov_batch_handle()); h = fresh.get(); }
	h->n_streams = b->n_streams; h->n_packets = b->n_packets;
	h->input_kind = b->input_kind; h->pcm_layout = b->pcm_layout; h->pcm_floats = b->pcm_floats;
	h->staged_ready = false;

	// ---- validation + derived arrays (one pass over the packets) ----
	const uint32_t P = b->n_packets;
	h->spec_off.resize(P); h->stage_off.resize(P); h->pk_n.resize(P); h->pk_setup.resize(P);
	h->pk_used.resize(P); h->pk_mode.resize(P);
	h->streams_host.assign(b->streams, b->streams + b->n_streams);
	const bool raw_packets = b->input_kind == POV_INPUT_PACKETS;
	h->pk_ys_off.resize(raw_packets ? P : 0); h->pk_ent_off.resize(raw_packets ? P : 0); h->pk_raw_off.resize(raw_packets ? P : 0);
	h->ys_cap = h->ent_cap = 0;
	h->runs.clear();
	uint32_t maxC = 1, maxbs = 64, minbs = 8192, maxposts = 2, res_smem = 0, res_acc_smem = 0, res_cursors = 0, posts_cls[2] = {2, 2};
	bool only_std = true;
	uint32_t table_float2 = 0;
	uint64_t dense_floats = 0, stage_floats = 0, expect_first = 0;
	const uint64_t payload_floats = b->payload_bytes / 4;
	// the persistent warp kernel handles batches whose streams all share one supported setup
	bool warp_ok = b->n_streams > 0 && ctx->kernel_choice != 1;
	for(uint32_t si = 0; si < b->n_streams && warp_ok; ++si) {
		const uint32_t id = b->streams[si].setup_id;
		if(id >= ctx->setups.size() || !ctx->setups[id].fast_ok) warp_ok = false;     // several setups: one launch per setup
	}
	h->warp_ok = warp_ok;
	h->warp_setup = warp_ok ? b->streams[0].setup_id : 0;
	bool any_wide = false;               // a stream whose floors have 33..64 posts: its runs hold at most 15 packets + halo
	for(uint32_t si = 0; si < b->n_streams && warp_ok; ++si) any_wide |= ctx->setups[b->streams[si].setup_id].fast_wide;
	// enough work for several items per warp: worth ordering the items so that the short ones come last
	const bool balance_tail = warp_ok && (uint64_t) P * ctx->setups[h->warp_setup].channels >= (uint64_t) ctx->sm_count * warp_kernel_warps() * warp_kernel_max_run(any_wide) * 4;
	uint32_t run_len = ctx->run_len;
	if(warp_ok) {
		// work items = runs x channels, taken dynamically by sm_count*16 warps: aim for >= 8 items per warp, keep the
		// halo overhead (one re-transformed packet per run) small; a run holds <= 32 packet descriptors, halo included
		const uint64_t C = ctx->setups[h->warp_setup].channels;
		const uint64_t want_items = (uint64_t) ctx->sm_count * warp_kernel_warps() * 8;
		const uint64_t max_run = warp_kernel_max_run(any_wide);
		const uint64_t auto_len = std::min<uint64_t>(max_run, std::max<uint64_t>(8, (uint64_t) P * C / want_items));
		run_len = run_len ? std::min<uint32_t>(run_len, (uint32_t) max_run) : (uint32_t) auto_len;
	} else if(run_len == 0) {
		// aim for >= ~8 CTAs per SM when the batch is big enough, keep the halo overhead <= 1/run_len
		const uint64_t want_runs = (uint64_t) ctx->sm_count * 8;
		run_len = (uint32_t) std::min<uint64_t>(32, std::max<uint64_t>(8, P / std::max<uint64_t>(1, want_runs)));
	}
	for(uint32_t si = 0; si < b->n_streams; ++si) {
		const pov_stream& st = b->streams[si];
		if(st.setup_id >= ctx->setups.size()) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: stream %u: unknown setup %u", si, st.setup_id);
		if(st.first_packet != expect_first || (uint64_t) st.first_packet + st.n_packets > P)
			return pov_fail(ctx, POV_ERR_ARG, "pov_batch: stream %u: packets must tile the packet array in stream order", si);
		expect_first += st.n_packets;
		const SetupRec& su = ctx->setups[st.setup_id];
		const uint32_t C = su.channels;
		if(raw_packets && !su.entropy_ok)
			return pov_fail(ctx, POV_ERR_UNSUPPORTED, "pov_batch: stream %u: setup %u cannot be entropy-decoded on the device (no codebook lengths / floor "
			                "syntax, floor0, or a submap without channels)", si, st.setup_id);
		// (subtraction form: none of these 64-bit sums may wrap)
		if(st.pcm_base > b->pcm_floats || st.pcm_frames > (b->pcm_floats - st.pcm_base) / C)
			return pov_fail(ctx, POV_ERR_ARG, "pov_batch: stream %u: PCM region exceeds pcm_floats", si);
		maxC = std::max(maxC, C); maxbs = std::max(maxbs, su.blocksize[1]); minbs = std::min(minbs, su.blocksize[0]);
		maxposts = std::max(maxposts, su.max_posts); res_smem = std::max(res_smem, su.res_smem);
		res_acc_smem = std::max(res_acc_smem, su.res_acc_smem); res_cursors = std::max(res_cursors, su.res_cursors);
		if(su.blocksize[0] != 256 || su.blocksize[1] != 2048) only_std = false;
		table_float2 = std::max(table_float2, su.table_float2);
		posts_cls[0] = std::max(posts_cls[0], su.posts_cls[0]); posts_cls[1] = std::max(posts_cls[1], su.posts_cls[1]);
		uint32_t n_prev = 0;
		for(uint32_t k = 0; k < st.n_packets; ++k) {
			const uint32_t p = st.first_packet + k;
			const pov_packet& pk = b->packets[p];
			if(pk.stream != si) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: stream field %u != %u", p, pk.stream, si);
			if(pk.mode >= su.n_modes) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: mode %u out of range (hpp:1146)", p, pk.mode);
			const uint32_t flag = su.mode_blockflag[pk.mode];
			const uint32_t n = su.blocksize[flag];
			if(pk.floor_used >> C) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: floor_used has bits beyond %u channels", p, C);
			const uint32_t max_emit = k ? n_prev / 4 + n / 4 : 0;
			if(pk.emit_frames > max_emit) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: emit_frames %u > %u (hpp:1026)", p, pk.emit_frames, max_emit);
			if(pk.pcm_off > st.pcm_frames || pk.emit_frames > st.pcm_frames - pk.pcm_off) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: PCM chunk outside the stream's %llu frames", p, (unsigned long long) st.pcm_frames);
			// Y lists
			const DevMapping& mp = su.maps_host[su.mode_mapping[pk.mode]];
			uint64_t ny = 0;
			for(uint32_t c = 0; c < C; ++c)
				if((pk.floor_used >> c) & 1) ny += su.floors_host[mp.floor_of_ch[c]].n_posts;
			if(!raw_packets && (pk.ys_off > b->n_ys || ny > b->n_ys - pk.ys_off)) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: Y lists outside the Y arena", p);
			if(raw_packets) {
				const uint64_t padded = ((uint64_t) pk.packet_bytes + 3) & ~3ull;
				if((pk.spec_off & 3) || pk.spec_off > b->payload_bytes || padded > b->payload_bytes - pk.spec_off)
					return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: raw packet outside the payload arena", p);
				h->pk_ys_off[p] = h->ys_cap; h->ys_cap += su.mode_ys_cap[pk.mode];
				h->pk_ent_off[p] = h->ent_cap; h->ent_cap += su.mode_ent_cap[pk.mode];
				h->pk_raw_off[p] = pk.spec_off;
				h->spec_off[p] = dense_floats;
				dense_floats += (uint64_t) C * (n / 2);
			} else if(b->input_kind == POV_INPUT_DENSE) {
				if(pk.spec_off & 3) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: spec_off must be a multiple of 4 floats (16-byte TMA source)", p);
				if(pk.spec_off > payload_floats || (uint64_t) C * (n / 2) > payload_floats - pk.spec_off) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: spectra outside the payload arena", p);
				h->spec_off[p] = pk.spec_off;
			} else {
				if((pk.spec_off & 3) || b->payload_bytes < 4 || pk.spec_off > b->payload_bytes - 4) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: residue payload offset invalid", p);
				if(su.residues_host.empty()) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: setup has no residues", p);
				h->spec_off[p] = dense_floats;
				dense_floats += (uint64_t) C * (n / 2);
			}
			h->stage_off[p] = stage_floats;
			stage_floats += (uint64_t) C * n;
			h->pk_n[p] = n; h->pk_setup[p] = st.setup_id;
			h->pk_used[p] = pk.floor_used; h->pk_mode[p] = pk.mode;
			n_prev = n;
		}
		// runs of <= run_len packets, each later run re-transforming one halo packet. For the persistent warp kernel the
		// last ~7 % / ~3.5 % of every stream are cut into half / quarter length runs (tiers 1, 2) that are handed out last:
		// the final wave of work items is then a quarter as long, which trims the idle tail of the launch.
		{
			const uint32_t t1 = (warp_ok && balance_tail && run_len >= 16) ? st.n_packets - st.n_packets * 7 / 100 : st.n_packets;
			const uint32_t t2 = (warp_ok && balance_tail && run_len >= 16) ? st.n_packets - st.n_packets * 35 / 1000 : st.n_packets;
			for(uint32_t k = 0; k < st.n_packets;) {
				const uint32_t tier = k >= t2 ? 2u : k >= t1 ? 1u : 0u;
				uint32_t len = tier == 2 ? run_len / 4 : tier == 1 ? run_len / 2 : run_len;
				if(tier == 0 && k + len > t1 && t1 > k) len = t1 - k;          // do not straddle a tier boundary
				if(tier == 1 && k + len > t2 && t2 > k) len = t2 - k;
				DevRun r;
				r.halo = k ? 1u : 0u;
				r.first_packet = st.first_packet + k - r.halo;
				r.n_packets = std::min(len, st.n_packets - k) + r.halo;
				r.pad = tier | (st.setup_id << 8);       // sort key below: work items grouped by setup, short tiers last
				h->runs.push_back(r);
				k += r.n_packets - r.halo;
			}
		}
	}
	if(expect_first != P) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: %u packets not covered by the stream table", (uint32_t) (P - expect_first));
	h->warp_groups.clear();
	if(warp_ok) {
		std::stable_sort(h->runs.begin(), h->runs.end(), [](const DevRun& a, const DevRun& b) { return a.pad < b.pad; });
		for(uint32_t i = 0; i < h->runs.size();) {
			const uint32_t sid = h->runs[i].pad >> 8;
			uint32_t j = i;
			while(j < h->runs.size() && (h->runs[j].pad >> 8) == sid) ++j;
			h->warp_groups.push_back({sid, i, j - i});
			i = j;
		}
	}
	if(h->warp_ok) {
		// the warp kernel keeps per-packet offsets relative to the run's first packet in 32 bits
		for(const DevRun& r : h->runs) {
			const uint64_t s0 = h->spec_off[r.first_packet], p0 = b->packets[r.first_packet].pcm_off;
			for(uint32_t k = 0; k < r.n_packets && h->warp_ok; ++k) {
				const int64_t ds = (int64_t) (h->spec_off[r.first_packet + k] - s0);
				const uint64_t pk = b->packets[r.first_packet + k].pcm_off;
				if(ds < INT32_MIN / 2 || ds > INT32_MAX / 2 || pk < p0 || pk - p0 > 0x7fffffffull) h->warp_ok = false;
			}
			if(!h->warp_ok) break;
		}
	}
	if(b->input_kind == POV_INPUT_ENTRIES) {
		// walk the payload headers on the host so that a malformed offset cannot send the kernel out of bounds
		for(uint32_t p = 0; p < P; ++p) {
			const SetupRec& su = ctx->setups[h->pk_setup[p]];
			const pov_packet& pk = b->packets[p];
			const DevMapping& mp = su.maps_host[su.mode_mapping[pk.mode]];
			uint64_t off = pk.spec_off;
			const uint32_t half = h->pk_n[p] / 2;
			for(uint32_t s = 0; s < mp.n_submaps; ++s) {
				uint32_t nch = 0;
				for(uint32_t c = 0; c < su.channels; ++c) nch += (mp.mux[c] == s);
				const DevResidue& rs = su.residues_host[mp.submap_residue[s]];
				const uint32_t vch = rs.type == 2 ? 1 : nch, vlen = rs.type == 2 ? nch * half : half;
				const uint32_t lb = std::min(rs.begin, vlen), le = std::min(rs.end, vlen);
				const uint32_t parts = (le - lb) / rs.partition_size;
				if(b->payload_bytes < 4 || off > b->payload_bytes - 4) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: residue payload truncated", p);
				uint32_t ne;
				memcpy(&ne, (const uint8_t*) b->payload + off, 4);
				// sizes are < 2^37 each, off <= payload_bytes: the sum cannot wrap
				const uint64_t cls_bytes = ((uint64_t) vch * parts + 3) & ~3ull, ent_bytes = ((uint64_t) ne * (su.entry_bits / 8) + 3) & ~3ull;
				if(cls_bytes + ent_bytes > b->payload_bytes - off - 4) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: residue payload truncated", p);
				// classification numbers index the (class, pass) book table: hpp:715-722 produces values < n_class by construction
				const uint8_t* cls = (const uint8_t*) b->payload + off + 4;
				for(uint64_t i = 0; i < (uint64_t) vch * parts; ++i)
					if(cls[i] >= rs.n_class) return pov_fail(ctx, POV_ERR_ARG, "pov_batch: packet %u: residue classification %u >= %u classes", p, cls[i], rs.n_class);
				off += 4 + cls_bytes + ent_bytes;
			}
		}
	}
	h->max_channels = maxC; h->max_blocksize = maxbs; h->min_blocksize = std::min(minbs, maxbs);
	h->floor_cap = (maxposts + 3u) & ~3u;
	h->floor_cap_cls[0] = (posts_cls[0] + 3u) & ~3u; h->floor_cap_cls[1] = (posts_cls[1] + 3u) & ~3u;
	h->res_smem = res_smem; h->res_acc_smem = res_acc_smem; h->res_cursors = res_cursors;
	h->only_256_2048 = only_std && b->n_streams > 0;
	h->table_float2 = table_float2;
	h->stage_floats = stage_floats;
	h->dense_floats = dense_floats;
	h->fused_ok = fused_smem_bytes(maxC, maxbs, h->min_blocksize, h->floor_cap_cls, h->table_float2) <= 227 * 1024;

	// ---- device copies ----
	cudaStream_t st = ctx->stream;
	auto up = [&](DevBuf& buf, const void* src, size_t bytes) -> cudaError_t {
		cudaError_t e = buf.reserve(std::max<size_t>(bytes, 16));
		if(e != cudaSuccess || bytes == 0) return e;
		ctx->h2d_bytes += bytes;
		return cudaMemcpyAsync(buf.ptr, src, bytes, cudaMemcpyHostToDevice, st);
	};
	CUDA_TRY(ctx, up(h->d_streams, b->streams, sizeof(pov_stream) * b->n_streams));
	CUDA_TRY(ctx, up(h->d_packets, b->packets, sizeof(pov_packet) * P));
	if(raw_packets) {
		CUDA_TRY(ctx, h->d_ys.reserve(std::max<size_t>(sizeof(uint16_t) * h->ys_cap, 16)));
		CUDA_TRY(ctx, h->d_entries.reserve(std::max<size_t>(h->ent_cap, 16)));
	} else CUDA_TRY(ctx, up(h->d_ys, b->ys, sizeof(uint16_t) * b->n_ys));
	CUDA_TRY(ctx, up(h->d_payload, b->payload, b->payload_bytes));
	{
		const size_t b_spec = sizeof(uint64_t) * P, o_runs = (b_spec + 15) & ~(size_t) 15, b_runs = sizeof(DevRun) * h->runs.size();
		const size_t o_pk = (o_runs + b_runs + 15) & ~(size_t) 15, b_pk = raw_packets ? 3 * sizeof(uint64_t) * P : 0;
		const size_t need = std::max<size_t>(o_pk + b_pk, 16);
		if(h->derived_copied) CUDA_TRY(ctx, cudaEventSynchronize(h->derived_copied));     // the previous upload through this handle has read them
		else CUDA_TRY(ctx, cudaEventCreateWithFlags(&h->derived_copied, cudaEventDisableTiming));
		CUDA_TRY(ctx, h->h_derived.reserve(need));
		uint8_t* hd = (uint8_t*) h->h_derived.ptr;
		if(b_spec) memcpy(hd, h->spec_off.data(), b_spec);
		if(b_runs) memcpy(hd + o_runs, h->runs.data(), b_runs);
		if(b_pk) {
			memcpy(hd + o_pk, h->pk_ys_off.data(), b_pk / 3);
			memcpy(hd + o_pk + b_pk / 3, h->pk_ent_off.data(), b_pk / 3);
			memcpy(hd + o_pk + 2 * (b_pk / 3), h->pk_raw_off.data(), b_pk / 3);
			CUDA_TRY(ctx, up(h->d_pk_off, hd + o_pk, b_pk));
		}
		CUDA_TRY(ctx, up(h->d_spec_off, hd, b_spec));
		CUDA_TRY(ctx, up(h->d_runs, hd + o_runs, b_runs));
		CUDA_TRY(ctx, cudaEventRecord(h->derived_copied, st));
	}
	if(pcm_dev) h->d_pcm.release();          // (cudaFree waits for the device: the previous run has written its arena)
	else CUDA_TRY(ctx, h->d_pcm.reserve(std::max<size_t>(pcm_elem_bytes(b->pcm_layout) * b->pcm_floats, 16)));
	h->pcm_ext = pcm_dev;
	CUDA_TRY(ctx, h->d_status.reserve(std::max<size_t>(sizeof(uint32_t) * P, 16)));
	CUDA_TRY(ctx, cudaMemsetAsync(h->d_status.ptr, 0, sizeof(uint32_t) * P, st));
	if(b->input_kind != POV_INPUT_DENSE) CUDA_TRY(ctx, h->d_spectra.reserve(std::max<size_t>(sizeof(float) * dense_floats, 16)));
	if(fresh) *out = fresh.release();
	return POV_OK;
}

static DevBatchView make_view(pov_ctx* ctx, pov_batch_handle* h) {
	DevBatchView v;
	v.setups = ctx->d_setups;
	v.streams = (const pov_stream*) h->d_streams.ptr;
	v.packets = (const pov_packet*) h->d_packets.ptr;
	v.ys = (const uint16_t*) h->d_ys.ptr;
	v.spec_off = (const uint64_t*) h->d_spec_off.ptr;
	if(h->input_kind == POV_INPUT_DENSE) { v.spectra = (const float*) h->d_payload.ptr; v.payload = nullptr; }
	else if(h->input_kind == POV_INPUT_ENTRIES) { v.spectra = (const float*) h->d_spectra.ptr; v.payload = (const uint8_t*) h->d_payload.ptr; }
	else { v.spectra = (const float*) h->d_spectra.ptr; v.payload = (const uint8_t*) h->d_entries.ptr; }   // (what k_packet_decode writes)
	v.inv_db = ctx->d_inv_db;
	v.pcm = h->pcm();
	v.status = (uint32_t*) h->d_status.ptr;
	v.n_streams = h->n_streams; v.n_packets = h->n_packets;
	v.pcm_layout = h->pcm_layout & ~POV_PCM_S16; v.pcm_s16 = (h->pcm_layout & POV_PCM_S16) ? 1u : 0u;
	return v;
}

static int run_residue_if_needed(pov_ctx* ctx, pov_batch_handle* h, const DevBatchView& v) {
	if(h->input_kind == POV_INPUT_DENSE) return POV_OK;
	if(h->input_kind == POV_INPUT_PACKETS) {
		// entropy decode on the device: raw packet bytes -> floor_used + Y lists + entries payload (then as POV_INPUT_ENTRIES)
		DevBatchView raw = v;
		raw.payload = (const uint8_t*) h->d_payload.ptr;
		const uint64_t* off = (const uint64_t*) h->d_pk_off.ptr;
		CUDA_TRY(ctx, launch_packet_decode(raw, (pov_packet*) h->d_packets.ptr, (uint16_t*) h->d_ys.ptr, (uint8_t*) h->d_entries.ptr, off, off + h->n_packets,
		                                   off + 2 * (size_t) h->n_packets, h->n_packets, ctx->stream, &ctx->launches));
	}
	if(h->res_smem <= residue_apply_max_dynamic_smem()) {
		CUDA_TRY(ctx, launch_residue_apply(v, (float*) h->d_spectra.ptr, h->res_smem, nullptr, 0, h->n_packets, ctx->stream, &ctx->launches));
		return POV_OK;
	}
	// The cursors do not fit next to the working vector (small partitions of long multichannel blocks): they go to a global
	// scratch of res_cursors words per block, at most 256 MB of it, and the blocks loop over the packets.
	const uint64_t per = std::max<uint32_t>(h->res_cursors, 1);
	const uint32_t grid = (uint32_t) std::max<uint64_t>(1, std::min<uint64_t>(h->n_packets, (256ull << 20) / (4 * per)));
	CUDA_TRY(ctx, h->d_res_cursor.reserve(4 * per * grid));
	CUDA_TRY(ctx, launch_residue_apply(v, (float*) h->d_spectra.ptr, h->res_acc_smem, (uint32_t*) h->d_res_cursor.ptr, (uint32_t) per, grid,
	                                   ctx->stream, &ctx->launches));
	return POV_OK;
}

static int prepare_stage_buffers(pov_ctx* ctx, pov_batch_handle* h, DevStageBuffers& sb) {
	const size_t cps = (size_t) h->n_packets * h->max_channels;
	CUDA_TRY(ctx, h->d_stage_off.reserve(std::max<size_t>(sizeof(uint64_t) * h->n_packets, 16)));
	CUDA_TRY(ctx, cudaMemcpyAsync(h->d_stage_off.ptr, h->stage_off.data(), sizeof(uint64_t) * h->n_packets, cudaMemcpyHostToDevice, ctx->stream));
	CUDA_TRY(ctx, h->st_final_ys.reserve(std::max<size_t>(cps * POV_MAX_POSTS * 4, 16)));
	CUDA_TRY(ctx, h->st_flag.reserve(std::max<size_t>(cps * POV_MAX_POSTS, 16)));
	CUDA_TRY(ctx, h->st_floor.reserve(std::max<size_t>(h->stage_floats * 2, 16)));
	CUDA_TRY(ctx, h->st_floor_out.reserve(std::max<size_t>(h->stage_floats * 4, 16)));
	CUDA_TRY(ctx, h->st_env.reserve(std::max<size_t>(h->stage_floats * 2, 16)));
	CUDA_TRY(ctx, h->st_mdct.reserve(std::max<size_t>(h->stage_floats * 4, 16)));
	CUDA_TRY(ctx, cudaMemsetAsync(h->st_final_ys.ptr, 0, cps * POV_MAX_POSTS * 4, ctx->stream));
	CUDA_TRY(ctx, cudaMemsetAsync(h->st_flag.ptr, 0, cps * POV_MAX_POSTS, ctx->stream));
	sb.stage_off = (const uint64_t*) h->d_stage_off.ptr;
	sb.final_ys = (uint32_t*) h->st_final_ys.ptr;
	sb.step2_flag = (uint8_t*) h->st_flag.ptr;
	sb.floor = (uint16_t*) h->st_floor.ptr;
	sb.floor_outputs = (float*) h->st_floor_out.ptr;
	sb.after_envelope = (float*) h->st_env.ptr;
	sb.pcm_after_mdct = (float*) h->st_mdct.ptr;
	return POV_OK;
}

extern "C" int pov_batch_run_staged(pov_ctx* ctx, pov_batch_handle* h) try {
	if(!ctx || !h) return POV_ERR_ARG;
	cudaSetDevice(ctx->device);
	DevBatchView v = make_view(ctx, h);
	int rc = run_residue_if_needed(ctx, h, v);
	if(rc) return rc;
	DevStageBuffers sb;
	if((rc = prepare_stage_buffers(ctx, h, sb)) != POV_OK) return rc;
	CUDA_TRY(ctx, launch_staged(v, sb, h->max_channels, ctx->stream, &ctx->launches));
	h->staged_ready = true;
	return POV_OK;
} POV_NOTHROW_END(ctx)

static int run_batch(pov_ctx* ctx, pov_batch_handle* h, unsigned char* dbg_floor);
extern "C" int pov_batch_run(pov_ctx* ctx, pov_batch_handle* h) try {
	return run_batch(ctx, h, nullptr);
} POV_NOTHROW_END(ctx)

// The production kernel's own floor1 step-1 result, for parity tests: runs the batch on k_warp_synth with its floor hook on
// and returns [n_packets][channels][72] bytes — 64 final Ys in ascending-x order (clamped to 255) | 64-bit step-2 mask —
// for every channel-packet whose floor was decoded (others: unspecified).
extern "C" int pov_batch_fetch_fast_floor(pov_ctx* ctx, pov_batch_handle* h, uint8_t* out, uint64_t out_bytes) try {
	if(!ctx || !h || !out) return POV_ERR_ARG;
	if(!h->warp_ok) return pov_fail(ctx, POV_ERR_UNSUPPORTED, "pov_batch_fetch_fast_floor: this batch does not run on the warp kernel");
	const uint64_t need = (uint64_t) h->n_packets * h->max_channels * 72;
	if(out_bytes != need) return pov_fail(ctx, POV_ERR_ARG, "pov_batch_fetch_fast_floor: %llu bytes expected", (unsigned long long) need);
	cudaSetDevice(ctx->device);
	CUDA_TRY(ctx, h->d_feat_out.reserve(std::max<size_t>(need, 16)));
	CUDA_TRY(ctx, cudaMemsetAsync(h->d_feat_out.ptr, 0, need, ctx->stream));
	const int rc = run_batch(ctx, h, (unsigned char*) h->d_feat_out.ptr);
	if(rc) return rc;
	CUDA_TRY(ctx, cudaMemcpyAsync(out, h->d_feat_out.ptr, need, cudaMemcpyDeviceToHost, ctx->stream));
	CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return POV_OK;
} POV_NOTHROW_END(ctx)

static int run_batch(pov_ctx* ctx, pov_batch_handle* h, unsigned char* dbg_floor) {
	if(!ctx || !h) return POV_ERR_ARG;
	if(ctx->kernel_choice == 2 && !h->warp_ok) return pov_fail(ctx, POV_ERR_UNSUPPORTED, "POV_KERNEL=warp: this batch is outside what the warp kernel supports");
	if(!h->warp_ok && !h->fused_ok) return pov_batch_run_staged(ctx, h);   // working set beyond one SM's shared memory: staged kernels
	cudaSetDevice(ctx->device);
	DevBatchView v = make_view(ctx, h);
	int rc = run_residue_if_needed(ctx, h, v);
	if(rc) return rc;
	if(h->warp_ok) {
		for(const WarpGroup& g : h->warp_groups) {      // one persistent launch per setup (its tables live in shared memory)
			const SetupRec& su = ctx->setups[g.setup];
			CUDA_TRY(ctx, launch_warp(v, (const DevRun*) h->d_runs.ptr + g.first_run, g.n_runs, su.channels, su.d_fast, su.blocksize[0], su.blocksize[1],
			                          su.fast_short_cap, su.fast_long_cap, su.fast_max_nl, su.dev.slope, su.dev.rot, su.dev.fft8, su.dev.fftp,
			                          ctx->blk_tables.count(2048) ? ctx->blk_tables[2048].d_tm : nullptr, dbg_floor, ctx->d_counter, ctx->sm_count, ctx->stream,
			                          &ctx->launches));
		}
		return POV_OK;
	}
	CUDA_TRY(ctx, launch_fused(v, (const DevRun*) h->d_runs.ptr, (uint32_t) h->runs.size(), h->max_channels, h->max_blocksize,
	                           h->min_blocksize, h->floor_cap_cls, h->table_float2, h->only_256_2048, ctx->stream, &ctx->launches));
	return POV_OK;
}

extern "C" const char* pov_batch_kernel_name(const pov_ctx* ctx, const pov_batch_handle* h) {
	if(!ctx || !h) return "none";
	if(h->warp_ok) return "k_warp_synth";
	return h->fused_ok ? "k_fused_synth" : "staged";
}

extern "C" int pov_batch_sync(pov_ctx* ctx, pov_batch_handle* h) {
	if(!ctx || !h) return POV_ERR_ARG;
	cudaSetDevice(ctx->device);
	CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return POV_OK;
}

cudaError_t pov_copy_out_async(pov_ctx* ctx, void* dst, const void* src, size_t bytes, bool fork, bool join) {
	cudaError_t e = cudaSuccess;
	if(fork) {
		if((e = cudaEventRecord(ctx->ev_compute, ctx->stream)) != cudaSuccess) return e;
		if((e = cudaStreamWaitEvent(ctx->out_stream, ctx->ev_compute, 0)) != cudaSuccess) return e;
	}
	if(bytes && (e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->out_stream)) != cudaSuccess) return e;
	ctx->d2h_bytes += bytes;
	if(join) {
		if((e = cudaEventRecord(ctx->ev_out, ctx->out_stream)) != cudaSuccess) return e;
		if((e = cudaStreamWaitEvent(ctx->stream, ctx->ev_out, 0)) != cudaSuccess) return e;
	}
	return e;
}

static int fetch_pcm(pov_ctx* ctx, pov_batch_handle* h, void* out, uint64_t n_values, int sync, bool s16, const char* fn) {
	if(!ctx || !h || (!out && n_values)) return POV_ERR_ARG;
	if(((h->pcm_layout & POV_PCM_S16) != 0) != s16)
		return pov_fail(ctx, POV_ERR_ARG, "%s: the batch's PCM arena holds %s samples", fn, s16 ? "float32" : "int16 (POV_PCM_S16)");
	if(n_values > h->pcm_floats) return pov_fail(ctx, POV_ERR_ARG, "%s: %llu samples requested, arena holds %llu", fn, (unsigned long long) n_values, (unsigned long long) h->pcm_floats);
	cudaSetDevice(ctx->device);
	if(n_values) CUDA_TRY(ctx, pov_copy_out_async(ctx, out, h->pcm(), n_values * pcm_elem_bytes(h->pcm_layout)));
	if(sync) CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return POV_OK;
}

extern "C" int pov_batch_fetch_pcm(pov_ctx* ctx, pov_batch_handle* h, float* out, uint64_t n_floats, int sync) try {
	return fetch_pcm(ctx, h, out, n_floats, sync, false, "pov_batch_fetch_pcm");
} POV_NOTHROW_END(ctx)

extern "C" int pov_batch_fetch_pcm_s16(pov_ctx* ctx, pov_batch_handle* h, int16_t* out, uint64_t n_values, int sync) try {
	return fetch_pcm(ctx, h, out, n_values, sync, true, "pov_batch_fetch_pcm_s16");
} POV_NOTHROW_END(ctx)

extern "C" void* pov_batch_pcm_dev(pov_batch_handle* h) { return h ? h->pcm() : nullptr; }

extern "C" int pov_batch_status(pov_ctx* ctx, pov_batch_handle* h, uint32_t* out, uint32_t n) try {
	if(!ctx || !h) return POV_ERR_ARG;
	cudaSetDevice(ctx->device);
	std::vector<uint32_t> tmp(h->n_packets);
	CUDA_TRY(ctx, cudaMemcpyAsync(tmp.data(), h->d_status.ptr, sizeof(uint32_t) * h->n_packets, cudaMemcpyDeviceToHost, ctx->stream));
	ctx->d2h_bytes += sizeof(uint32_t) * h->n_packets;
	CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	if(out) memcpy(out, tmp.data(), sizeof(uint32_t) * std::min<uint32_t>(n, h->n_packets));
	for(uint32_t p = 0; p < h->n_packets; ++p)
		if(tmp[p]) return pov_fail(ctx, POV_ERR_STREAM, "audio packet %u: check failed: %s", p, pov_status_text(tmp[p]));
	return POV_OK;
} POV_NOTHROW_END(ctx)

const char* pov_status_text(uint32_t status) {
	return (status & POV_PKT_FLOOR_PREDICTED) ? "predicted <= range (hpp:536)"
	     : (status & POV_PKT_FLOOR_RANGE)     ? "floor[i] < 256 (hpp:587)"
	                                          : "temp.size() > 0 (hpp:739,748: VQ entry out of range)";
}

extern "C" int pov_batch_fetch_stage(pov_ctx* ctx, pov_batch_handle* h, uint32_t packet, uint32_t channel, int stage,
                                     void* out, uint64_t out_bytes) try {
	if(!ctx || !h || !out) return POV_ERR_ARG;
	if(packet >= h->n_packets) return pov_fail(ctx, POV_ERR_ARG, "pov_batch_fetch_stage: packet out of range");
	const SetupRec& su = ctx->setups[h->pk_setup[packet]];
	if(channel >= su.channels) return pov_fail(ctx, POV_ERR_ARG, "pov_batch_fetch_stage: channel out of range");
	if(stage != POV_STAGE_AFTER_RESIDUE && !h->staged_ready) return pov_fail(ctx, POV_ERR_ARG, "pov_batch_fetch_stage: run pov_batch_run_staged first");
	cudaSetDevice(ctx->device);
	const uint32_t n = h->pk_n[packet];
	const uint64_t so = h->stage_off[packet];
	const uint64_t slot = ((uint64_t) packet * h->max_channels + channel) * POV_MAX_POSTS;
	const void* src = nullptr;
	uint64_t bytes = 0;
	std::vector<uint16_t> tmp16;
	switch(stage) {
		case POV_STAGE_FINAL_YS: src = (const uint32_t*) h->st_final_ys.ptr + slot; bytes = out_bytes; if(bytes > POV_MAX_POSTS * 4) bytes = 0; break;
		case POV_STAGE_STEP2_FLAG: src = (const uint8_t*) h->st_flag.ptr + slot; bytes = out_bytes; if(bytes > POV_MAX_POSTS) bytes = 0; break;
		case POV_STAGE_FLOOR: {
			if(out_bytes != (uint64_t) n * 4) return pov_fail(ctx, POV_ERR_ARG, "pov_batch_fetch_stage: size mismatch");
			tmp16.resize(n);
			CUDA_TRY(ctx, cudaMemcpyAsync(tmp16.data(), (const uint16_t*) h->st_floor.ptr + so + (uint64_t) channel * n, n * 2, cudaMemcpyDeviceToHost, ctx->stream));
			CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
			for(uint32_t i = 0; i < n; ++i) ((uint32_t*) out)[i] = tmp16[i];
			return POV_OK;
		}
		case POV_STAGE_FLOOR_OUTPUTS: src = (const float*) h->st_floor_out.ptr + so + (uint64_t) channel * n; bytes = (uint64_t) n * 4; break;
		case POV_STAGE_AFTER_RESIDUE: {
			const float* base = (h->input_kind == POV_INPUT_DENSE) ? (const float*) h->d_payload.ptr : (const float*) h->d_spectra.ptr;
			src = base + h->spec_off[packet] + (uint64_t) channel * (n / 2); bytes = (uint64_t) n * 2; break;
		}
		case POV_STAGE_AFTER_ENVELOPE: src = (const float*) h->st_env.ptr + so / 2 + (uint64_t) channel * (n / 2); bytes = (uint64_t) n * 2; break;
		case POV_STAGE_PCM_AFTER_MDCT: src = (const float*) h->st_mdct.ptr + so + (uint64_t) channel * n; bytes = (uint64_t) n * 4; break;
		default: return pov_fail(ctx, POV_ERR_ARG, "pov_batch_fetch_stage: unknown stage %d", stage);
	}
	if(bytes == 0 || bytes != out_bytes) return pov_fail(ctx, POV_ERR_ARG, "pov_batch_fetch_stage: size mismatch (%llu vs %llu)", (unsigned long long) out_bytes, (unsigned long long) bytes);
	CUDA_TRY(ctx, cudaMemcpyAsync(out, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
	CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return POV_OK;
} POV_NOTHROW_END(ctx)

// bulk access for the dump writer: whole stage arrays in one copy
int pov_batch_fetch_stage_all(pov_ctx* ctx, pov_batch_handle* h, StageHost& out) {
	if(!h->staged_ready) return pov_fail(ctx, POV_ERR_ARG, "staged path has not run");
	cudaSetDevice(ctx->device);
	const size_t cps = (size_t) h->n_packets * h->max_channels;
	out.final_ys.resize(cps * POV_MAX_POSTS); out.step2.resize(cps * POV_MAX_POSTS);
	out.floor.resize(h->stage_floats); out.floor_out.resize(h->stage_floats);
	out.env.resize(h->stage_floats / 2); out.mdct.resize(h->stage_floats);
	const uint64_t res_floats = (h->input_kind == POV_INPUT_DENSE) ? h->d_payload.cap / 4 : h->dense_floats;
	(void) res_floats;
	cudaStream_t st = ctx->stream;
	CUDA_TRY(ctx, cudaMemcpyAsync(out.final_ys.data(), h->st_final_ys.ptr, out.final_ys.size() * 4, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx, cudaMemcpyAsync(out.step2.data(), h->st_flag.ptr, out.step2.size(), cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx, cudaMemcpyAsync(out.floor.data(), h->st_floor.ptr, out.floor.size() * 2, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx, cudaMemcpyAsync(out.floor_out.data(), h->st_floor_out.ptr, out.floor_out.size() * 4, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx, cudaMemcpyAsync(out.env.data(), h->st_env.ptr, out.env.size() * 4, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx, cudaMemcpyAsync(out.mdct.data(), h->st_mdct.ptr, out.mdct.size() * 4, cudaMemcpyDeviceToHost, st));
	if(h->input_kind == POV_INPUT_ENTRIES) {
		out.residue.resize(h->dense_floats);
		CUDA_TRY(ctx, cudaMemcpyAsync(out.residue.data(), h->d_spectra.ptr, out.residue.size() * 4, cudaMemcpyDeviceToHost, st));
	}
	CUDA_TRY(ctx, cudaStreamSynchronize(st));
	return POV_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// drop-in for mdct_backward (src/mdct.h:105)
// ---------------------------------------------------------------------------------------------------------------
// ---------------------------------------------------------------------------------------------------------------
// feature matrices for RETURNN-style front ends (SURVEY.md §8f-3)
// ---------------------------------------------------------------------------------------------------------------
extern "C" int pov_batch_features(pov_ctx* ctx, pov_batch_handle* h, uint32_t stream, int kind, uint32_t output_dim,
                                  float* out, uint64_t rows_cap, uint64_t* rows_out) try {
	if(!ctx || !h || !rows_out) return POV_ERR_ARG;
	if(kind < POV_FEAT_FLOOR_FINAL_YS || kind > POV_FEAT_RESIDUE_YS_WITH_FLOOR) return pov_fail(ctx, POV_ERR_ARG, "pov_batch_features: unknown kind %d", kind);
	const bool all_streams = stream == POV_ALL_STREAMS;
	if(!all_streams && stream >= h->n_streams) return pov_fail(ctx, POV_ERR_ARG, "pov_batch_features: stream out of range");
	if(h->n_streams == 0) { *rows_out = 0; return POV_OK; }
	if(all_streams) {
		for(uint32_t i = 1; i < h->n_streams; ++i)
			if(h->streams_host[i].setup_id != h->streams_host[0].setup_id)
				return pov_fail(ctx, POV_ERR_ARG, "pov_batch_features: POV_ALL_STREAMS needs one setup for the whole batch");
		stream = 0;
	}
	if(output_dim < 1 || output_dim > 4096) return pov_fail(ctx, POV_ERR_ARG, "pov_batch_features: output_dim out of range");
	cudaSetDevice(ctx->device);
	int rc = POV_OK;
	if(!h->staged_ready && (rc = pov_batch_run_staged(ctx, h)) != POV_OK) return rc;
	const SetupRec& su = ctx->setups[h->streams_host[stream].setup_id];
	const uint32_t C = su.channels, nf = (uint32_t) su.floors_host.size();
	// which floors were decoded: the host's descriptors, or what k_packet_decode found in the packets
	std::vector<uint16_t> used(h->pk_used);
	if(h->input_kind == POV_INPUT_PACKETS) {
		std::vector<pov_packet> tmp(h->n_packets);
		CUDA_TRY(ctx, cudaMemcpyAsync(tmp.data(), h->d_packets.ptr, sizeof(pov_packet) * h->n_packets, cudaMemcpyDeviceToHost, ctx->stream));
		CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
		ctx->d2h_bytes += sizeof(pov_packet) * h->n_packets;
		for(uint32_t p = 0; p < h->n_packets; ++p) used[p] = tmp[p].floor_used;
	}
	uint32_t biggest = 0;                 // demo_live_extract.py:313 / :442: the first floor with the most posts
	for(uint32_t i = 1; i < nf; ++i) if(su.floors_host[i].n_posts > su.floors_host[biggest].n_posts) biggest = i;
	if((kind == POV_FEAT_RESIDUE_YS || kind == POV_FEAT_RESIDUE_YS_WITH_FLOOR) && output_dim < su.floors_host[biggest].n_posts)
		return pov_fail(ctx, POV_ERR_ARG, "pov_batch_features: output_dim %u < %u posts of the biggest floor (the reference asserts, demo_live_extract.py:486)",
		                output_dim, su.floors_host[biggest].n_posts);
	std::vector<FeatRow> rows;
	for(uint32_t si = stream; si < (all_streams ? h->n_streams : stream + 1); ++si) {
	const pov_stream& st = h->streams_host[si];
	uint64_t base = ~0ull;                 // (the reader's floor_base starts as None for every file)
	uint32_t base_n = 0;
	for(uint32_t k = 0; k < st.n_packets; ++k) {
		const uint32_t p = st.first_packet + k, n = h->pk_n[p];
		const DevMapping& mp = su.maps_host[su.mode_mapping[h->pk_mode[p]]];
		if(kind <= POV_FEAT_FLOOR_FINAL_YS_RENDERED) {
			for(uint32_t c = 0; c < C; ++c) {
				if(!((used[p] >> c) & 1)) continue;
				FeatRow r;
				memset(&r, 0, sizeof r);
				r.src = kind == POV_FEAT_FLOOR_FINAL_YS ? (uint64_t) p * h->max_channels + c : h->stage_off[p] + (uint64_t) c * n;
				r.floor = mp.floor_of_ch[c]; r.n = n; r.base = ~0ull;
				rows.push_back(r);
			}
		} else {
			for(uint32_t c = 0; c < C; ++c)           // "floor1 floor" entries of this packet come before its "after_residue" entries
				if(((used[p] >> c) & 1) && mp.floor_of_ch[c] == biggest) { base = h->stage_off[p] + (uint64_t) c * n; base_n = n; }
			const uint32_t recent = mp.floor_of_ch[C - 1];     // the last "floor_number" entry before the residues (demo_live_extract.py:455)
			if(recent != biggest) continue;
			for(uint32_t c = 0; c < C; ++c) {
				FeatRow r;
				memset(&r, 0, sizeof r);
				r.src = h->spec_off[p] + (uint64_t) c * (n / 2);
				r.floor = recent; r.n = n;
				r.base = kind == POV_FEAT_RESIDUE_YS_WITH_FLOOR ? base : ~0ull; r.base_n = base_n;
				rows.push_back(r);
			}
		}
	}
	}
	*rows_out = rows.size();
	if(!out) return POV_OK;                                  // size query
	if(rows.size() > rows_cap) return pov_fail(ctx, POV_ERR_ARG, "pov_batch_features: %llu rows, room for %llu", (unsigned long long) rows.size(), (unsigned long long) rows_cap);
	if(rows.empty()) return POV_OK;
	std::vector<FeatFloor> ff(nf);
	for(uint32_t i = 0; i < nf; ++i) {
		memset(&ff[i], 0, sizeof(FeatFloor));
		ff[i].tag = (float) (((double) i + 1.0) / (double) nf - 0.5);
		ff[i].multiplier = su.floors_host[i].multiplier; ff[i].n_posts = su.floors_host[i].n_posts;
		for(uint32_t k = 0; k < su.floors_host[i].n_posts; ++k) ff[i].xs[k] = su.floors_host[i].xs[k];
	}
	CUDA_TRY(ctx, h->d_feat_rows.reserve(rows.size() * sizeof(FeatRow)));
	CUDA_TRY(ctx, h->d_feat_floors.reserve(ff.size() * sizeof(FeatFloor)));
	CUDA_TRY(ctx, h->d_feat_out.reserve(rows.size() * (size_t) output_dim * sizeof(float)));
	CUDA_TRY(ctx, cudaMemcpyAsync(h->d_feat_rows.ptr, rows.data(), rows.size() * sizeof(FeatRow), cudaMemcpyHostToDevice, ctx->stream));
	CUDA_TRY(ctx, cudaMemcpyAsync(h->d_feat_floors.ptr, ff.data(), ff.size() * sizeof(FeatFloor), cudaMemcpyHostToDevice, ctx->stream));
	ctx->h2d_bytes += rows.size() * sizeof(FeatRow) + ff.size() * sizeof(FeatFloor);
	const float* residue = (h->input_kind == POV_INPUT_DENSE) ? (const float*) h->d_payload.ptr : (const float*) h->d_spectra.ptr;
	CUDA_TRY(ctx, launch_features(kind, (const FeatRow*) h->d_feat_rows.ptr, rows.size(), (const FeatFloor*) h->d_feat_floors.ptr, output_dim,
	                              (const uint32_t*) h->st_final_ys.ptr, (const uint16_t*) h->st_floor.ptr, residue, (float*) h->d_feat_out.ptr,
	                              ctx->stream, &ctx->launches));
	CUDA_TRY(ctx, cudaMemcpyAsync(out, h->d_feat_out.ptr, rows.size() * (size_t) output_dim * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
	ctx->d2h_bytes += rows.size() * (size_t) output_dim * sizeof(float);
	CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));       // rows / ff live on this stack frame
	return POV_OK;
} POV_NOTHROW_END(ctx)

extern "C" int pov_mdct_backward_batch(pov_ctx* ctx, uint32_t n, uint64_t count, const float* in, float* out) try {
	if(!ctx || (count && (!in || !out))) return POV_ERR_ARG;
	if(!is_pow2_in(n, 64, 8192)) return pov_fail(ctx, POV_ERR_ARG, "pov_mdct_backward_batch: n = %u is not a power of two in 64..8192 (hpp:1295)", n);
	if(count > 0x7fffffffull) return pov_fail(ctx, POV_ERR_ARG, "pov_mdct_backward_batch: count too large for one call");
	cudaSetDevice(ctx->device);
	BlockTables* t = nullptr;
	int rc = get_block_tables(ctx, n, &t);
	if(rc) return rc;
	if(count == 0) return POV_OK;
	CUDA_TRY(ctx, ctx->mdct_in.reserve(count * (n / 2) * sizeof(float)));
	CUDA_TRY(ctx, ctx->mdct_out.reserve(count * n * sizeof(float)));
	CUDA_TRY(ctx, cudaMemcpyAsync(ctx->mdct_in.ptr, in, count * (n / 2) * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
	CUDA_TRY(ctx, launch_mdct_backward(nullptr, n, count, (const float*) ctx->mdct_in.ptr, (float*) ctx->mdct_out.ptr, t->d_rot, t->d_fft, ctx->stream, &ctx->launches));
	CUDA_TRY(ctx, cudaMemcpyAsync(out, ctx->mdct_out.ptr, count * n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
	CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return POV_OK;
} POV_NOTHROW_END(ctx)
