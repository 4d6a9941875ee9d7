// Host-side state behind the opaque handles of include/pov_synth.h.
#ifndef POV_API_INTERNAL_H
#define POV_API_INTERNAL_H

#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <string>
#include <vector>

#include "pov_internal.h"

struct DevBuf {
	void* ptr = nullptr;
	size_t cap = 0;
	cudaError_t reserve(size_t bytes);
	void release();
};

// Growable pinned host buffer: the source or destination of asynchronous copies (a pageable one makes the "async" copy wait
// for the stream). reserve() grows it to bytes + bytes / 4 and does not keep the contents.
struct PinnedBuf {
	void* ptr = nullptr;
	size_t cap = 0;
	cudaError_t reserve(size_t bytes);
	void release();
};

struct BlockTables {              // per blocksize n: DCT-IV rotation, FFT twiddles, rising slope of n/2 samples
	const float2* d_rot = nullptr;
	const float2* d_fft = nullptr;
	const float2* d_fftp = nullptr;
	const float2* d_fft8 = nullptr;
	uint32_t fft8_count = 0;
	float c1[2] = {1, 0}, c6[2] = {1, 0};
	const float*  d_slope = nullptr;
	std::vector<float> h_slope;
	const float*  d_tm = nullptr;     // n == 2048: lane rows of the tensor-memory FFT (make_tm_lane_tables)
};

struct SetupRec {
	uint32_t channels = 0, sample_rate = 0, blocksize[2] = {0, 0};
	uint32_t n_modes = 0, entry_bits = 16, max_posts = 2;
	// k_residue_apply, per packet of the worst mode: dynamic shared memory with the read cursors in it (res_smem), without
	// them (res_acc_smem: the working vector only), and the cursor count (res_cursors, global scratch when they do not fit)
	uint32_t res_smem = 0, res_acc_smem = 0, res_cursors = 0;
	uint32_t posts_cls[2] = {2, 2};   // largest floor (posts) reachable from short / long modes
	uint32_t table_float2 = 0;        // float2 slots of the fused kernel's shared-memory tables for this setup
	uint8_t mode_blockflag[POV_MAX_MODES] = {0};
	uint8_t mode_mapping[POV_MAX_MODES] = {0};
	std::vector<DevFloor> floors_host;
	std::vector<DevMapping> maps_host;
	std::vector<DevResidue> residues_host;
	std::vector<uint32_t> cb_dim;
	DevSetup dev;
	const DevFloor* d_floors = nullptr;
	const DevMapping* d_mappings = nullptr;
	const DevResidue* d_residues = nullptr;
	const DevCodebook* d_codebooks = nullptr;
	const float* d_vq = nullptr;
	// warp-autonomous kernel (kernel_warp.cu): eligible setups carry their compact tables
	bool fast_ok = false;
	uint32_t fast_short_cap = 4, fast_long_cap = 32;
	bool fast_wide = false;           // a reachable floor has 33..64 posts: shorter runs (72-byte Y records)
	uint32_t fast_max_nl = 1;         // largest channel set a coupling program of this setup needs
	const FastTables* d_fast = nullptr;
	// device entropy decode (POV_INPUT_PACKETS): tables + per-mode arena capacities of one packet
	bool entropy_ok = false;
	const uint32_t* d_huff = nullptr;
	const DevHuffBook* d_hbooks = nullptr;
	const DevFloorSyntax* d_fsyntax = nullptr;
	uint32_t mode_ys_cap[POV_MAX_MODES] = {0};       // uint16 slots: every channel's Y list
	uint32_t mode_ent_cap[POV_MAX_MODES] = {0};      // bytes of the entries payload in the worst case (multiple of 4)
	std::string image;            // canonical bytes, for de-duplication
};

struct pov_ctx {
	int device = 0;
	int sm_count = 148;
	cudaStream_t stream = nullptr;
	// Asynchronous copies back to the host run on a stream of their own, joined with `stream` by events: an operation that
	// follows a device-to-host copy in stream order is submitted to the copy engine's queue, i.e. behind every copy-out that
	// any other stream submitted before it (measured: the next chunk's copy-in + kernels waited for three foreign copy-outs).
	cudaStream_t out_stream = nullptr;
	cudaEvent_t ev_compute = nullptr, ev_out = nullptr;
	uint64_t launches = 0;
	uint64_t h2d_bytes = 0, d2h_bytes = 0;   // what this context copied between host and device (pov_ctx_io_bytes)
	uint32_t run_len = 0;         // 0 = automatic
	int kernel_choice = 0;        // POV_KERNEL: 0 automatic, 1 force the CTA-per-run fused kernel, 2 require the warp kernel
	bool allow_spanning = false;  // accept packets that span pages (the reference refuses them, hpp:89)
	bool device_entropy = true;   // whole-file / corpus decode: audio packets are entropy-decoded on the device (POV_DEVICE_ENTROPY=0: on the host)
	bool cut_damage = false;      // corpus decode: cut damaged streams and go on (pov_ctx_set_cut_damage)
	std::vector<pov_file_report> corpus_files;   // pov_corpus_report: the last corpus call's per-file report
	std::vector<uint64_t> corpus_valid;          // and its valid frames per stream-table record
	bool corpus_report_ok = false;               // that call succeeded (every corpus entry point resets it first)
	uint32_t* d_counter = nullptr; // work counter of the persistent kernel
	const float* d_inv_db = nullptr;
	const DevSetup* d_setups = nullptr;
	std::vector<SetupRec> setups;
	std::map<uint32_t, BlockTables> blk_tables;
	std::map<std::string, uint32_t> setup_by_key;   // raw header bytes of a parsed stream -> setup id (front end)
	DevBuf mdct_in, mdct_out;
	void* corpus = nullptr;                 // what pov_decode_corpus keeps between calls (front_end.cpp: sibling context, slots, pinned pool)
	void (*corpus_free)(void*) = nullptr;
	char err[512] = {0};
};

// Bytes of one PCM arena element for a pov_batch::pcm_layout value: int16 with POV_PCM_S16, float otherwise.
inline size_t pcm_elem_bytes(uint32_t pcm_layout) { return (pcm_layout & POV_PCM_S16) ? sizeof(int16_t) : sizeof(float); }

struct WarpGroup { uint32_t setup, first_run, n_runs; };   // runs of one setup: one launch of the persistent warp kernel

struct pov_batch_handle {
	uint32_t n_streams = 0, n_packets = 0, input_kind = 0, pcm_layout = 0;   // pcm_layout as uploaded (POV_PCM_S16 included)
	uint64_t pcm_floats = 0, stage_floats = 0, dense_floats = 0;
	uint32_t max_channels = 1, max_blocksize = 64, min_blocksize = 64, floor_cap = 4, res_smem = 0, res_acc_smem = 0, res_cursors = 0;
	uint32_t floor_cap_cls[2] = {4, 4};
	uint32_t table_float2 = 0;
	bool fused_ok = true, staged_ready = false, only_256_2048 = false;
	bool warp_ok = false;         // every stream uses one setup that kernel_warp.cu supports
	uint32_t warp_setup = 0;
	std::vector<WarpGroup> warp_groups;
	std::vector<uint64_t> spec_off, stage_off;
	std::vector<uint64_t> pk_ys_off, pk_ent_off, pk_raw_off;     // POV_INPUT_PACKETS: capacity-based places of a packet's Y lists / entries payload
	uint64_t ys_cap = 0, ent_cap = 0;
	std::vector<uint32_t> pk_n, pk_setup;
	std::vector<uint16_t> pk_used;                   // floor_used as the host saw it (POV_INPUT_PACKETS: decoded on the device instead)
	std::vector<uint8_t> pk_mode;
	std::vector<pov_stream> streams_host;
	DevBuf d_feat_rows, d_feat_floors, d_feat_out;   // pov_batch_features
	std::vector<DevRun> runs;
	DevBuf d_streams, d_packets, d_ys, d_payload, d_spec_off, d_stage_off, d_runs, d_pcm, d_status, d_spectra;
	void* pcm_ext = nullptr;                         // pov_batch_upload_into: the caller's PCM memory (then d_pcm is empty)
	void* pcm() const { return pcm_ext ? pcm_ext : d_pcm.ptr; }
	DevBuf d_entries, d_pk_off;                      // POV_INPUT_PACKETS: entries payload written by k_packet_decode; ys_off | ent_off
	DevBuf d_res_cursor;                             // k_residue_apply's read cursors when they do not fit its shared memory
	DevBuf st_final_ys, st_flag, st_floor, st_floor_out, st_env, st_mdct;
	// pinned copy of the derived arrays (spec_off | runs): sources of asynchronous copies, so they must outlive the copy (derived_copied)
	PinnedBuf h_derived;
	cudaEvent_t derived_copied = nullptr;
};

struct StageHost {                // whole stage arrays on the host (debug dump writer)
	std::vector<uint32_t> final_ys;
	std::vector<uint8_t> step2;
	std::vector<uint16_t> floor;
	std::vector<float> floor_out, env, mdct, residue;
};

// Device -> host copy on the context's copy-out stream. fork: ordered after everything queued on ctx->stream so far; join:
// work queued on ctx->stream afterwards waits for the copy (and cudaStreamSynchronize(ctx->stream) covers it).
cudaError_t pov_copy_out_async(pov_ctx* ctx, void* dst, const void* src, size_t bytes, bool fork = true, bool join = true);
int pov_fail(pov_ctx* ctx, int code, const char* fmt, ...);
// Entry points are function-try-blocks that end in POV_NOTHROW_END: no exception crosses the C boundary.
int pov_fail_exception(pov_ctx* ctx);
#define POV_NOTHROW_END(ctx) catch(...) { return pov_fail_exception(ctx); }
int pov_batch_fetch_stage_all(pov_ctx* ctx, pov_batch_handle* h, StageHost& out);
// Device memory of the context's GPU, aligned to `align` bytes: where pov_batch_upload_into / pov_decode_corpus_device may write.
int pov_check_pcm_dev(pov_ctx* ctx, const void* p, size_t align, const char* fn);
// The reference's check that a non-zero packet status word (POV_PKT_*) reports, as error text.
const char* pov_status_text(uint32_t status);

#endif
