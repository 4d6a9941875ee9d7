// Polyphase resampler of the device corpus decode (kernel_resample.cu; contract in include/pov_synth.h, pov_resample).
#ifndef POV_RESAMPLE_H
#define POV_RESAMPLE_H

#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

namespace pov {

// One logical stream of a chunk: where its decoded channels are in the slot's float32 arena, where its output goes, and its
// filter. Blocks [tile_first, tile_first + out_channels * ceil(out_frames / tile)) of the launch work on it.
struct ResampleDesc {
	uint64_t in_base, in_stride, in_frames;      // arena sample index of channel 0, samples between channels, frames
	uint64_t out_base, out_stride, out_frames;   // the caller's region (sample indices)
	uint64_t tile_first;
	const float* taps;                           // [K][L]: taps[k * L + phase] = h[phase + k * L], 0 past N (null for a copy)
	uint32_t in_channels, out_channels, mono;
	uint32_t L, M, hl, K;                        // L = M = 1: copy
	uint32_t tile;                               // output frames per block
	float inv_c;                                 // 1.0f / in_channels (mono)
	uint32_t pad;
};

// Filter of in_rate -> out_rate reduced by the gcd. Returns false past POV_RESAMPLE_MAX_PHASES (L, M still set). With
// `h`, the N = 2 hl + 1 float32 taps (empty for a copy).
bool resample_design(uint32_t in_rate, uint32_t out_rate, uint32_t* L, uint32_t* M, uint32_t* hl, std::vector<float>* h);
uint64_t resample_frames(uint64_t frames, uint32_t L, uint32_t M);     // ceil(frames L / M)
uint32_t resample_tile(uint32_t L, uint32_t M);                         // output frames per block for this ratio

// One launch for a chunk: descs on the device, n_tiles = last tile_first + its tiles. out: float, or int16_t when s16.
cudaError_t launch_resample(const float* arena, const ResampleDesc* descs, uint32_t n_descs, uint64_t n_tiles, void* out, bool s16,
                            cudaStream_t st, uint64_t* launches);

}  // namespace pov
#endif
