// Output sample type of the PCM stores (kernel_warp.cu, kernel_fused.cu, kernels_staged.cu): float32 as computed, or signed
// 16-bit (POV_PCM_S16) converted at the store, so that no float32 PCM reaches HBM on that path.
#ifndef POV_PCM_OUT_CUH
#define POV_PCM_OUT_CUH

#include <stdint.h>

// The one conversion rule of POV_PCM_S16: s = clamp(round_half_even(x * 32768), -32768, 32767), NaN -> 0.
// The multiplication by 2^15 is exact (±inf saturates), so s depends on x alone. On finite input this is what libvorbisfile's
// ov_read gives on x86-64 (multiply by 32768, SSE conversion to nearest-even, clip); for NaN ov_read gives -32768, this gives 0
// (the PTX saturating conversion's result).
__device__ __forceinline__ int16_t pcm_s16(float x) {
	short s;
	asm("cvt.rni.sat.s16.f32 %0, %1;" : "=h"(s) : "f"(__fmul_rn(x, 32768.0f)));
	return (int16_t) s;
}

template <class T> __device__ __forceinline__ T pcm_value(float x);
template <> __device__ __forceinline__ float pcm_value<float>(float x) { return x; }
template <> __device__ __forceinline__ int16_t pcm_value<int16_t>(float x) { return pcm_s16(x); }

// Four consecutive samples at dst (aligned to four samples: 16 bytes for float, 8 for int16): plain / streaming store.
__device__ __forceinline__ short4 pcm_pack4(float4 v) { return make_short4(pcm_s16(v.x), pcm_s16(v.y), pcm_s16(v.z), pcm_s16(v.w)); }
__device__ __forceinline__ void pcm_store4(float* dst, float4 v) { *reinterpret_cast<float4*>(dst) = v; }
__device__ __forceinline__ void pcm_store4(int16_t* dst, float4 v) { *reinterpret_cast<short4*>(dst) = pcm_pack4(v); }
__device__ __forceinline__ void pcm_store4_cs(float* dst, float4 v) { __stcs(reinterpret_cast<float4*>(dst), v); }
__device__ __forceinline__ void pcm_store4_cs(int16_t* dst, float4 v) { __stcs(reinterpret_cast<short4*>(dst), pcm_pack4(v)); }

#endif
