// Polyphase FIR resampler and mono downmix of the device corpus decode (pov_decode_corpus_device_resampled): reads a chunk's
// decoded float32 arena and writes the caller's regions. The filter is scipy.signal.resample_poly's default design, computed
// here on the host; the contract is in include/pov_synth.h (pov_resample).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <numeric>
#include <vector>

#include "pcm_out.cuh"
#include "../../include/pov_synth.h"
#include "resample.h"

namespace pov {

constexpr int kResThreads = 256;
constexpr int kResQ = 4;                   // outputs per thread and block: tiles of at most 1024 output frames
constexpr int kResWindow = 8192;           // floats of staged input per block (32 KB)

// ---------------------------------------------------------------------------------------------------------------
// host: filter design
// ---------------------------------------------------------------------------------------------------------------
static double bessel_i0(double x) {        // power series; every term is positive, so it converges to full precision
	const double q = 0.25 * x * x;
	double sum = 1.0, term = 1.0;
	for(int k = 1; k < 500; ++k) {
		term *= q / ((double) k * k);
		sum += term;
		if(term < sum * 1e-18) break;
	}
	return sum;
}

bool resample_design(uint32_t in_rate, uint32_t out_rate, uint32_t* L, uint32_t* M, uint32_t* hl, std::vector<float>* h) {
	const uint32_t g = std::gcd(in_rate, out_rate);
	*L = out_rate / g; *M = in_rate / g; *hl = 0;
	if(h) h->clear();
	if(*L == 1 && *M == 1) return true;
	const uint32_t R = *L > *M ? *L : *M;
	if(R > POV_RESAMPLE_MAX_PHASES) return false;
	*hl = 10 * R;
	if(!h) return true;
	const uint32_t N = 2 * *hl + 1;
	const double fc = 1.0 / R, i0b = bessel_i0(5.0), pi = 3.14159265358979323846;
	std::vector<double> v(N);
	double sum = 0;
	for(uint32_t n = 0; n < N; ++n) {
		const double m = (double) n - (double) *hl, x = fc * m, r = m / (double) *hl;
		const double sinc = x == 0.0 ? 1.0 : sin(pi * x) / (pi * x);
		v[n] = fc * sinc * bessel_i0(5.0 * sqrt(fmax(0.0, 1.0 - r * r))) / i0b;
		sum += v[n];
	}
	h->resize(N);
	for(uint32_t n = 0; n < N; ++n) (*h)[n] = (float) (v[n] / sum * (double) *L);
	return true;
}

uint64_t resample_frames(uint64_t frames, uint32_t L, uint32_t M) { return (frames * L + M - 1) / M; }

// The block's input window spans at most ceil((tile - 1) M / L) + 1 samples; keeping that within half the staged window leaves
// the other half for taps, so a long filter is applied in a few passes over k (each pass restages the window).
uint32_t resample_tile(uint32_t L, uint32_t M) {
	const uint32_t full = kResThreads * kResQ;
	if(L == 1 && M == 1) return full;
	const uint64_t t = (uint64_t) (kResWindow / 2 - 2) * L / M + 1;
	return t < full ? (uint32_t) t : full;
}

// ---------------------------------------------------------------------------------------------------------------
// device
// ---------------------------------------------------------------------------------------------------------------
// One block per (stream, output channel, tile of output frames). Thread t owns outputs j0 + t + q * 256 (q < 4), so the
// stores are coalesced; consecutive outputs have different phases, so every FMA takes one shared-memory load (the staged
// input) and one read-only load (the tap, [K][L] layout: a warp's taps of one k lie in one row of L floats).
template <class OutT>
__global__ void __launch_bounds__(kResThreads) k_resample(const float* __restrict__ arena, const ResampleDesc* __restrict__ descs,
                                                          uint32_t n_descs, OutT* __restrict__ out) {
	__shared__ float win[kResWindow];
	const uint64_t blk = blockIdx.x;
	uint32_t lo = 0, hi = n_descs;                       // the last descriptor with tile_first <= blk
	while(hi - lo > 1) {
		const uint32_t mid = (lo + hi) >> 1;
		if(descs[mid].tile_first <= blk) lo = mid; else hi = mid;
	}
	const ResampleDesc& d = descs[lo];
	const uint64_t tiles = (d.out_frames + d.tile - 1) / d.tile, local = blk - d.tile_first;
	const uint32_t oc = (uint32_t) (local / tiles);
	const uint64_t j0 = (local % tiles) * d.tile;
	const uint32_t n = (uint32_t) min((uint64_t) d.tile, d.out_frames - j0);
	const uint32_t C = d.in_channels, mono = d.mono;
	const uint64_t in_frames = d.in_frames, in_stride = d.in_stride;
	const float inv_c = d.inv_c;
	const float* x = arena + d.in_base + (mono ? 0 : oc * in_stride);
	OutT* y = out + d.out_base + oc * d.out_stride + j0;
	auto input = [&](int64_t i) -> float {             // decoded (and downmixed) input sample i, zero outside the stream
		if(i < 0 || (uint64_t) i >= in_frames) return 0.f;
		float s = x[i];
		if(mono) {
			for(uint32_t c = 1; c < C; ++c) s = __fadd_rn(s, x[c * in_stride + i]);
			s = __fmul_rn(s, inv_c);
		}
		return s;
	};
	const uint32_t L = d.L, M = d.M, K = d.K;
	if(L == 1 && M == 1) {
		for(uint32_t t = threadIdx.x; t < n; t += kResThreads) y[t] = pcm_value<OutT>(input((int64_t) (j0 + t)));
		return;
	}
	const uint64_t b0 = (j0 * M + d.hl) / L;
	const uint32_t span = (uint32_t) (((j0 + n - 1) * M + d.hl) / L - b0) + 1;      // <= kResWindow / 2 (resample_tile)
	const uint32_t ks = kResWindow - span;
	uint32_t rel[kResQ], ph[kResQ];
	float acc[kResQ];
#pragma unroll
	for(int q = 0; q < kResQ; ++q) {
		const uint32_t t = threadIdx.x + q * kResThreads;
		const uint64_t p = (j0 + t) * M + d.hl;
		rel[q] = t < n ? (uint32_t) (p / L - b0) : 0;    // (outputs past the tile compute on sample 0 and are not stored)
		ph[q] = t < n ? (uint32_t) (p % L) : 0;
		acc[q] = 0.f;
	}
	const float* __restrict__ taps = d.taps;
	for(uint32_t k0 = 0; k0 < K; k0 += ks) {
		const uint32_t k1 = min(K, k0 + ks);
		const int64_t first = (int64_t) b0 - (int64_t) (k1 - 1);       // win[i] = input(first + i)
		const uint32_t len = span + (k1 - k0) - 1;
		if(k0) __syncthreads();
		for(uint32_t i = threadIdx.x; i < len; i += kResThreads) win[i] = input(first + i);
		__syncthreads();
		for(uint32_t k = k0; k < k1; ++k) {              // output q, tap k: input b0 + rel[q] - k = first + rel[q] + k1 - 1 - k
			const float* tk = taps + (uint64_t) k * L;
			const uint32_t o = k1 - 1 - k;
#pragma unroll
			for(int q = 0; q < kResQ; ++q) acc[q] = fmaf(win[rel[q] + o], __ldg(tk + ph[q]), acc[q]);
		}
	}
#pragma unroll
	for(int q = 0; q < kResQ; ++q) {
		const uint32_t t = threadIdx.x + q * kResThreads;
		if(t < n) y[t] = pcm_value<OutT>(acc[q]);
	}
}

cudaError_t launch_resample(const float* arena, const ResampleDesc* descs, uint32_t n_descs, uint64_t n_tiles, void* out, bool s16,
                            cudaStream_t st, uint64_t* launches) {
	if(n_tiles == 0) return cudaSuccess;
	if(n_tiles > 0x7FFFFFFFull) return cudaErrorInvalidConfiguration;
	if(s16) k_resample<int16_t><<<(unsigned) n_tiles, kResThreads, 0, st>>>(arena, descs, n_descs, (int16_t*) out);
	else k_resample<float><<<(unsigned) n_tiles, kResThreads, 0, st>>>(arena, descs, n_descs, (float*) out);
	if(launches) ++*launches;
	return cudaGetLastError();
}

}  // namespace pov

extern "C" int pov_resample_filter(uint32_t in_rate, uint32_t out_rate, uint32_t* up, uint32_t* down, uint32_t* half_len,
                                   float* taps, uint32_t taps_cap) try {
	if(!up || !down || !half_len || in_rate == 0) return POV_ERR_ARG;
	uint32_t L = 1, M = 1, hl = 0;
	if(out_rate == 0) { *up = 1; *down = 1; *half_len = 0; return POV_OK; }
	if(!pov::resample_design(in_rate, out_rate, &L, &M, &hl, nullptr)) { *up = L; *down = M; *half_len = 10 * (L > M ? L : M); return POV_ERR_UNSUPPORTED; }
	*up = L; *down = M; *half_len = hl;
	if(!taps || hl == 0) return POV_OK;
	if(taps_cap < 2 * hl + 1) return POV_ERR_ARG;
	std::vector<float> h;
	pov::resample_design(in_rate, out_rate, &L, &M, &hl, &h);
	for(size_t i = 0; i < h.size(); ++i) taps[i] = h[i];
	return POV_OK;
} catch(...) { return POV_ERR_ARG; }
