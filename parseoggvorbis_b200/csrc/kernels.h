// Launchers of the CUDA kernels (kernels_staged.cu, kernel_fused.cu). All pointers are device pointers.
#ifndef POV_KERNELS_H
#define POV_KERNELS_H

#include <cuda_runtime.h>
#include "pov_internal.h"

namespace pov {

struct DevBatchView {
	const DevSetup*   setups;        // [n_setups]
	const pov_stream* streams;       // [n_streams]
	const pov_packet* packets;       // [n_packets]
	const uint16_t*   ys;
	const float*      spectra;       // dense after_residue vectors (input arena, or output of the residue kernel)
	const uint64_t*   spec_off;      // per packet: float offset of its [C][n/2] block inside `spectra`
	const uint8_t*    payload;       // residue payload arena (POV_INPUT_ENTRIES) or nullptr
	const float*      inv_db;        // floor1_inverse_dB_table[256] (src/inverse_db_table.h:13-78), device copy
	void*             pcm;           // PCM arena: float, or int16_t when pcm_s16
	uint32_t*         status;        // [n_packets]
	uint32_t n_streams, n_packets, pcm_layout;   // pcm_layout: POV_PCM_PLANAR | POV_PCM_INTERLEAVED (without POV_PCM_S16)
	uint32_t pcm_s16;                // the kernels store PCM as int16 (pcm_out.cuh: pcm_s16)
};

// Staged (debug) path: every intermediate is materialised.
struct DevStageBuffers {
	const uint64_t* stage_off;   // per packet: float offset of its [C][n] block in the n-sized stage arrays
	uint32_t* final_ys;          // [n_packets*C][POV_MAX_POSTS]
	uint8_t*  step2_flag;        // [n_packets*C][POV_MAX_POSTS]
	uint16_t* floor;             // n-sized
	float*    floor_outputs;     // n-sized
	float*    after_envelope;    // n/2-sized (offset stage_off/2)
	float*    pcm_after_mdct;    // n-sized
};

// cursor_scratch == nullptr: one block per packet, read cursors in shared memory after the working vector. Otherwise `grid`
// blocks loop over the packets and block i keeps its cursors at cursor_scratch + i * cursor_stride.
cudaError_t launch_residue_apply(const DevBatchView& b, float* spectra_out, size_t smem_bytes, uint32_t* cursor_scratch,
                                 uint32_t cursor_stride, uint32_t grid, cudaStream_t st, uint64_t* launches);
size_t residue_apply_max_dynamic_smem();   // the current device's opt-in limit less k_residue_apply's static tables
cudaError_t launch_staged(const DevBatchView& b, const DevStageBuffers& sb, uint32_t max_channels, cudaStream_t st,
                          uint64_t* launches);
cudaError_t launch_fused(const DevBatchView& b, const DevRun* runs, uint32_t n_runs, uint32_t max_channels,
                         uint32_t max_blocksize, uint32_t min_blocksize, const uint32_t floor_cap[2], uint32_t table_float2,
                         bool only_256_2048,
                         cudaStream_t st, uint64_t* launches);
size_t fused_smem_bytes(uint32_t max_channels, uint32_t max_blocksize, uint32_t min_blocksize, const uint32_t floor_cap[2],
                        uint32_t table_float2);
// Warp-autonomous persistent kernel (kernel_warp.cu): single-setup batches with blocksizes 256/2048.
bool warp_kernel_supports(uint32_t bs0, uint32_t bs1);     // block size pairs the warp kernel is instantiated for
size_t warp_kernel_smem_bytes(uint32_t bs0, uint32_t bs1, uint32_t short_posts_cap, uint32_t long_posts_cap, uint32_t* group_short_out, uint32_t* curve_bytes_out,
                              uint32_t* short_stride_out);
uint32_t warp_kernel_max_run(bool wide);   // packets per run without the halo (wide: a floor of 33..64 posts is reachable)
uint32_t warp_kernel_warps(void);     // resident warps per SM
cudaError_t launch_warp(const DevBatchView& b, const DevRun* runs, uint32_t n_runs, uint32_t channels, const FastTables* d_tabs,
                        uint32_t bs0, uint32_t bs1, uint32_t short_posts_cap, uint32_t long_posts_cap, uint32_t max_nl, const float* const slope[2], const float2* const rot[2],
                        const float2* const tw8[2], const float2* const fp[2], const float* tmtab, unsigned char* dbg_floor, uint32_t* d_counter, int sm_count,
                        cudaStream_t st, uint64_t* launches);
// One row of a feature matrix (pov_batch_features; reference: demo_live_extract.py:262-505): where its values come from.
struct FeatRow {
	uint64_t src;        // kinds 0: index of the channel-packet's final_ys slot; 1: float offset of its rendered floor (u16);
	                     // 2, 3: float offset of its after_residue vector
	uint64_t base;       // kind 3: float offset of the rendered floor that scales the row, ~0 = none
	uint32_t floor;      // floor number (row of the per-floor tables)
	uint32_t n;          // block size of the source (and, kind 3, of the base floor in base_n)
	uint32_t base_n;
	uint32_t pad;
};
struct FeatFloor { float tag; uint32_t multiplier, n_posts, pad; uint16_t xs[POV_MAX_POSTS]; };   // tag = (floor + 1) / floors - 0.5
cudaError_t launch_features(int kind, const FeatRow* rows, uint64_t n_rows, const FeatFloor* floors, uint32_t output_dim,
                            const uint32_t* final_ys, const uint16_t* floor, const float* residue, float* out, cudaStream_t st, uint64_t* launches);
cudaError_t launch_packet_decode(const DevBatchView& b, pov_packet* packets, uint16_t* ys_out, uint8_t* ent_out, const uint64_t* ys_off,
                                 const uint64_t* ent_off, const uint64_t* raw_off, uint32_t n_packets, cudaStream_t st, uint64_t* launches);
// Cut mode of the corpus decode (kernel_cut.cu): one logical stream of a chunk, where the synthesis wrote it. Blocks
// [tile_first, tile_first + channels * tiles) of the launch work on it, tiles = max(1, ceil(frames / kCutTile)).
constexpr uint64_t kCutTile = 32768;               // frames per block
struct CutDesc {
	uint64_t base, stride, frames;                 // sample index of channel 0, samples between channels, frames
	uint64_t tile_first;
	uint32_t first_packet, n_packets;              // the stream's packets (and status words) in the chunk's batch
	uint32_t walk_bad;                             // stream-relative packet whose host walk failed, or 0xFFFFFFFF
	uint32_t channels;
	uint64_t tiles;
};
struct CutResult {
	uint64_t valid_frames;                         // pcm_off of the first damaged packet, or frames
	uint32_t packet;                               // that packet (stream-relative), 0xFFFFFFFF: none
	uint32_t status;                               // its status word (0: only its host walk failed)
};
// descs ascending by tile_first, n_tiles = last tile_first + its blocks; pcm: float, or int16_t when s16.
cudaError_t launch_cut_damaged(void* pcm, bool s16, const CutDesc* descs, uint32_t n_descs, uint64_t n_tiles, const uint32_t* status,
                               const pov_packet* packets, CutResult* results, cudaStream_t st, uint64_t* launches);
cudaError_t launch_mdct_backward(const DevSetup* dummy, uint32_t n, uint64_t count, const float* in, float* out,
                                 const float2* rot, const float2* fft, cudaStream_t st, uint64_t* launches);

}  // namespace pov

// float64 sum of a float arena into *(double*) d_sum, or (s16) exact int64 sum of an int16 arena into *(uint64_t*) d_sum
cudaError_t pov_checksum_launch(const void* pcm, bool s16, uint64_t n, void* d_sum, cudaStream_t st, uint64_t* launches);
#endif
