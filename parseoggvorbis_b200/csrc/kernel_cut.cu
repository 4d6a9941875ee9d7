// Cut mode of the corpus decode (pov_ctx_set_cut_damage; contract in include/pov_synth.h, "Cut mode"): after a chunk's
// synthesis, find each stream's first damaged packet and zero the stream from that packet's first frame on.
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.h"

namespace pov {

constexpr int kCutThreads = 256;
constexpr uint32_t kCutNone = 0xFFFFFFFFu;

// Block -> (stream, channel, tile). Every block finds its stream's first damaged packet p: the first non-zero status word, or
// the packet whose host walk failed. The block of channel 0, tile 0 writes the stream's result; a block whose tile lies before
// the cut exits after the scan, the others zero their part of [pcm_off[p], frames). The grid depends on the streams only, so a
// clean chunk costs one launch in which every block reads about one status word per packet of its stream (L2-resident).
template <class T>
__global__ void __launch_bounds__(kCutThreads) k_cut_damaged(T* __restrict__ pcm, const CutDesc* __restrict__ descs, uint32_t n_descs,
                                                            const uint32_t* __restrict__ status, const pov_packet* __restrict__ packets,
                                                            CutResult* __restrict__ results) {
	__shared__ uint32_t s_first;
	const uint64_t b = blockIdx.x;
	uint32_t lo = 0, hi = n_descs;                       // the last descriptor with tile_first <= b
	while(hi - lo > 1) {
		const uint32_t mid = (lo + hi) / 2;
		if(descs[mid].tile_first <= b) lo = mid; else hi = mid;
	}
	const CutDesc& d = descs[lo];
	const uint64_t rel = b - d.tile_first;
	const uint64_t c = rel / d.tiles, t = rel - c * d.tiles;
	if(threadIdx.x == 0) s_first = kCutNone;
	__syncthreads();
	// warp w scans the 32-packet groups w, w + 8, ... in order: its first hit is its lowest damaged packet
	const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	for(uint32_t g = warp * 32; g < d.n_packets; g += kCutThreads) {
		const uint32_t i = g + lane;
		const bool bad = i < d.n_packets && (status[d.first_packet + i] != 0 || i == d.walk_bad);
		const uint32_t m = __ballot_sync(0xFFFFFFFFu, bad);
		if(m) {
			if(lane == 0) atomicMin(&s_first, g + __ffs(m) - 1);
			break;
		}
	}
	__syncthreads();
	const uint32_t p = s_first;
	const uint64_t cut = p == kCutNone ? d.frames : packets[d.first_packet + p].pcm_off;
	if(rel == 0 && threadIdx.x == 0) {
		CutResult r;
		r.valid_frames = cut; r.packet = p; r.status = p == kCutNone ? 0u : status[d.first_packet + p];
		results[lo] = r;
	}
	const uint64_t f0 = max(cut, t * kCutTile), f1 = min(d.frames, (t + 1) * kCutTile);
	if(f0 >= f1) return;
	T* y = pcm + d.base + c * d.stride + f0;
	const uint64_t n = f1 - f0;
	// scalar up to the first 16-byte boundary, 16-byte stores, scalar tail
	constexpr uint32_t kVec = 16 / sizeof(T);
	const uint64_t head = min(n, (uint64_t) (((16 - ((uintptr_t) y & 15)) & 15) / sizeof(T)));
	const uint64_t nvec = (n - head) / kVec;
	for(uint64_t i = threadIdx.x; i < head; i += kCutThreads) y[i] = T(0);
	uint4* v = reinterpret_cast<uint4*>(y + head);
	for(uint64_t i = threadIdx.x; i < nvec; i += kCutThreads) v[i] = make_uint4(0, 0, 0, 0);
	for(uint64_t i = head + nvec * kVec + threadIdx.x; i < n; i += kCutThreads) y[i] = T(0);
}

cudaError_t launch_cut_damaged(void* pcm, bool s16, const CutDesc* descs, uint32_t n_descs, uint64_t n_tiles, const uint32_t* status,
                               const pov_packet* packets, CutResult* results, cudaStream_t st, uint64_t* launches) {
	if(n_tiles == 0) return cudaSuccess;
	if(n_tiles > 0x7FFFFFFFull) return cudaErrorInvalidConfiguration;
	if(s16) k_cut_damaged<int16_t><<<(unsigned) n_tiles, kCutThreads, 0, st>>>((int16_t*) pcm, descs, n_descs, status, packets, results);
	else k_cut_damaged<float><<<(unsigned) n_tiles, kCutThreads, 0, st>>>((float*) pcm, descs, n_descs, status, packets, results);
	if(launches) ++*launches;
	return cudaGetLastError();
}

}  // namespace pov
