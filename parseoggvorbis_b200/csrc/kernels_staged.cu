// Staged device path: one kernel per reference stage, every intermediate written to HBM so that the debug dump
// (pov_batch_fetch_stage / "ParseOggVorbis-header-v1") can be produced from device results. The production
// path is kernel_fused.cu; both share floor_core.cuh / fft_core.cuh.
//
// Stage -> reference lines (paths relative to the reference root):
//   k_floor1        src/ParseOggVorbis.hpp:521-591
//   k_residue_apply src/ParseOggVorbis.hpp:685-694, 696-757 (adds only; Huffman walk done by the host front-end)
//   k_couple_dot    src/ParseOggVorbis.hpp:1174-1180, 1213-1255
//   k_imdct         src/mdct.h:105 mdct_backward (contract; algorithm in fft_core.cuh)
//   k_ola           src/ParseOggVorbis.hpp:1008-1059 (gather form)
#include "kernels.h"
#include "fft_core.cuh"
#include "floor_core.cuh"
#include "pcm_out.cuh"

namespace pov {

__device__ __forceinline__ const DevSetup& setup_of(const DevBatchView& b, const pov_packet& pk) {
	return b.setups[b.streams[pk.stream].setup_id];
}

// ---------------------------------------------------------------------------------------------------------------
// floor1: one warp per (packet, channel)
// ---------------------------------------------------------------------------------------------------------------
constexpr int kFloorWarps = 4;

__global__ void __launch_bounds__(kFloorWarps * 32) k_floor1(DevBatchView b, DevStageBuffers sb, uint32_t max_channels) {
	__shared__ __align__(16) unsigned char scratch[kFloorWarps][floor_scratch_stride(POV_MAX_POSTS)];
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const uint64_t cp = (uint64_t) blockIdx.x * kFloorWarps + warp;
	const uint32_t p = (uint32_t) (cp / max_channels), c = (uint32_t) (cp % max_channels);
	if(p >= b.n_packets) return;
	const pov_packet pk = b.packets[p];
	const DevSetup& su = setup_of(b, pk);
	if(c >= su.channels) return;
	const uint32_t flag = su.mode_blockflag[pk.mode];
	const uint32_t n = su.blocksize[flag];
	const DevMapping& mp = su.mappings[su.mode_mapping[pk.mode]];
	uint16_t* fl_out = sb.floor + sb.stage_off[p] + (uint64_t) c * n;
	float* fo_out = sb.floor_outputs + sb.stage_off[p] + (uint64_t) c * n;
	if(!((pk.floor_used >> c) & 1)) {
		for(uint32_t x = lane; x < n; x += 32) { fl_out[x] = 0; fo_out[x] = 0.f; }  // hpp:1159 zero-initialised
		return;
	}
	const DevFloor* F = &su.floors[mp.floor_of_ch[c]];
	// this channel's Y list: after the lists of the lower-numbered used channels
	uint64_t yo = pk.ys_off;
	for(uint32_t cc = 0; cc < c; ++cc)
		if((pk.floor_used >> cc) & 1) yo += su.floors[mp.floor_of_ch[cc]].n_posts;
	FloorScratch S;
	S.bind(scratch[warp], POV_MAX_POSTS);
	uint32_t st = floor1_unwrap_warp(F, b.ys + yo, S, lane);
	const uint64_t slot = ((uint64_t) p * max_channels + c) * POV_MAX_POSTS;
	for(int i = lane; i < F->n_posts; i += 32) {
		sb.final_ys[slot + i] = S.fy[i];
		sb.step2_flag[slot + i] = S.flag[i];
	}
	bool over = false;
	floor1_render_warp(S, 0, n, lane, [&](uint32_t x, uint32_t y) {
		fl_out[x] = (uint16_t) min(y, 0xFFFFu);
		if(y >= 256) over = true;
		fo_out[x] = __ldg(&b.inv_db[y & 255]);
	});
	if(__any_sync(0xffffffffu, over)) st |= POV_PKT_FLOOR_RANGE;
	if(st && lane == 0) atomicOr(&b.status[p], st);
}

// ---------------------------------------------------------------------------------------------------------------
// residue VQ application: one block per packet. Entries are in the reference's decode order (pass, partition,
// channel, vector); an exclusive scan of the per-(pass,partition,channel) vector counts gives every partition
// its read cursor, so partitions are independent while each bin still receives its <= 8 addends in pass order.
// The cursors live in shared memory after the submap's working vector, or, when g_cursor is set (too many partitions
// for shared memory), in g_cursor + blockIdx.x * cursor_stride; the blocks then loop over the packets.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kResThreads = 256;

__global__ void __launch_bounds__(kResThreads) k_residue_apply(DevBatchView b, float* __restrict__ spectra_out,
                                                               uint32_t* __restrict__ g_cursor, uint32_t cursor_stride) {
	extern __shared__ __align__(16) unsigned char res_smem[];
	__shared__ uint32_t s_scan[kResThreads / 32];
	__shared__ uint32_t s_carry;
	// setup tables the inner loops index for every bin and pass: kept in shared memory so that the dependent chain of a
	// (bin, pass) is shared-memory lookups plus two global loads (entry number, VQ value)
	__shared__ const float* s_vq[POV_MAX_CODEBOOKS];
	__shared__ uint32_t s_nent[POV_MAX_CODEBOOKS];          // 0: no lookup table (lookup_type 0) -> every entry is invalid
	__shared__ uint16_t s_dim[POV_MAX_CODEBOOKS];
	__shared__ uint8_t s_books[POV_MAX_CLASSES * 8];
	for(uint32_t p = blockIdx.x; p < b.n_packets; p += gridDim.x) {
		__syncthreads();                                         // the previous packet is done with the shared tables
		const pov_packet pk = b.packets[p];
		const DevSetup& su = setup_of(b, pk);
		const uint32_t C = su.channels;
		const uint32_t n = su.blocksize[su.mode_blockflag[pk.mode]], half = n / 2;
		const DevMapping& mp = su.mappings[su.mode_mapping[pk.mode]];
		float* out = spectra_out + b.spec_off[p];
		float* acc = reinterpret_cast<float*>(res_smem);                 // [nch*half] working vector of one submap
		const uint32_t n_books = min(su.n_codebooks, (uint32_t) POV_MAX_CODEBOOKS);
		for(uint32_t i = threadIdx.x; i < n_books; i += blockDim.x) {
			const DevCodebook cb = su.codebooks[i];
			s_vq[i] = cb.vq;
			s_nent[i] = cb.lookup_type ? cb.n_entries : 0u;
			s_dim[i] = (uint16_t) min(cb.dim, 0xFFFFu);
		}

		// nonzero propagate (hpp:1174-1180) decides which channels the residue touches
		uint32_t used = pk.floor_used;
		for(uint32_t k = 0; k < mp.n_couplings; ++k) {
			const uint32_t m = mp.coupling_mag[k], a = mp.coupling_ang[k];
			if(((used >> m) | (used >> a)) & 1) used |= (1u << m) | (1u << a);
		}
		const uint8_t* pl = b.payload + pk.spec_off;
		uint32_t bad = 0;
		for(uint32_t s = 0; s < mp.n_submaps; ++s) {
			uint32_t chs[POV_MAX_CHANNELS], nch = 0;
			for(uint32_t c = 0; c < C; ++c) if(mp.mux[c] == s) chs[nch++] = c;
			const DevResidue& rs = su.residues[mp.submap_residue[s]];
			// type 2 decodes ONE interleaved vector of length nch*half that is always "used" (hpp:685-694)
			const uint32_t rtype = rs.type;
			const uint32_t vch = (rtype == 2) ? 1u : nch;
			const uint32_t vlen = (rtype == 2) ? nch * half : half;
			const uint32_t lb = min(rs.begin, vlen), le = min(rs.end, vlen);
			const uint32_t psize = rs.partition_size;
			const uint32_t parts = (le - lb) / psize;
			uint32_t* cursor = g_cursor ? g_cursor + (size_t) blockIdx.x * cursor_stride          // [8*parts*vch] exclusive offsets
			                            : reinterpret_cast<uint32_t*>(acc + (size_t) nch * half);
			const uint32_t n_entries = *reinterpret_cast<const uint32_t*>(pl);
			const uint8_t* cls = pl + 4;
			const uint32_t cls_bytes = (vch * parts + 3u) & ~3u;
			const uint8_t* ent = cls + cls_bytes;
			const bool ent16 = su.entry_bits == 16;
			const uint32_t ent_bytes = (n_entries * (su.entry_bits / 8) + 3u) & ~3u;
			pl = ent + ent_bytes;

			__syncthreads();                                     // previous submap done with s_books / acc; book tables visible
			for(uint32_t i = threadIdx.x; i < rs.n_class * 8u; i += blockDim.x) s_books[i] = rs.books[i];
			for(uint32_t i = threadIdx.x; i < vch * vlen; i += blockDim.x) acc[i] = 0.f;
			if(threadIdx.x == 0) s_carry = 0;
			__syncthreads();
			// vector counts in decode order (pass, partition, channel) + block-wide exclusive scan: warp shuffles, one
			// shared-memory hop between the warps
			const uint32_t items = 8 * parts * vch;
			const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
			for(uint32_t base = 0; base < items; base += blockDim.x) {
				const uint32_t it = base + threadIdx.x;
				uint32_t cnt = 0;
				if(it < items) {
					const uint32_t j = it % vch, part = (it / vch) % parts, pass = it / (vch * parts);
					const bool ch_used = (rtype == 2) ? true : ((used >> chs[j]) & 1);
					if(ch_used) {
						const uint32_t book = s_books[cls[j * parts + part] * 8 + pass];
						if(book != POV_NO_BOOK && book < n_books) cnt = psize / s_dim[book];
					}
				}
				uint32_t incl = cnt;
	#pragma unroll
				for(int o = 1; o < 32; o <<= 1) {
					const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
					if((int) lane >= o) incl += v;
				}
				if(lane == 31) s_scan[warp] = incl;
				__syncthreads();
				uint32_t before = s_carry;
				for(uint32_t w = 0; w < warp; ++w) before += s_scan[w];
				if(it < items) cursor[it] = before + incl - cnt;
				__syncthreads();
				if(threadIdx.x == blockDim.x - 1) s_carry = before + incl;
				__syncthreads();
			}
			// apply: one thread per BIN. A bin receives at most one addend per pass (hpp:734-752), so it can gather its own
			// addends in pass order: the same additions, in the same order, as the reference's vector-by-vector accumulation
			// (which starts from the zero-initialised vector), with every thread of the block busy instead of one per partition.
			for(uint32_t idx = threadIdx.x; idx < parts * vch * psize; idx += blockDim.x) {
				const uint32_t o = idx % psize, w = idx / psize;
				const uint32_t j = w % vch, part = w / vch;
				const bool ch_used = (rtype == 2) ? true : ((used >> chs[j]) & 1);
				if(!ch_used) continue;
				const uint32_t cl = cls[j * parts + part];
				float sum = 0.f;
	#pragma unroll
				for(uint32_t pass = 0; pass < 8; ++pass) {
					const uint32_t book = s_books[cl * 8 + pass];
					if(book == POV_NO_BOOK) continue;
					if(book >= n_books) { bad |= POV_PKT_VQ_ENTRY; continue; }
					const uint32_t dim = s_dim[book];
					const uint32_t nvec = psize / dim;
					// type 0: v[k + l*nvec] (hpp:734-743); types 1/2: v[k*dim + l] (hpp:744-752)
					uint32_t k, l;
					if(rtype == 0) { if(nvec == 0) continue; l = o / nvec; k = o - l * nvec; if(l >= dim) continue; }
					else { k = o / dim; l = o - k * dim; if(k >= nvec) continue; }
					const uint32_t cur = cursor[(pass * parts + part) * vch + j] + k;
					if(cur >= n_entries) { bad |= POV_PKT_VQ_ENTRY; continue; }
					const uint32_t e = ent16 ? reinterpret_cast<const uint16_t*>(ent)[cur] : reinterpret_cast<const uint32_t*>(ent)[cur];
					if(e >= s_nent[book]) { bad |= POV_PKT_VQ_ENTRY; continue; }
					sum += __ldg(&s_vq[book][(size_t) e * dim + l]);
				}
				acc[(size_t) j * vlen + lb + part * psize + o] = sum;
			}
			__syncthreads();
			// scatter to the channel-major dense layout (de-interleave for type 2, hpp:690-692)
			if(rtype == 2) {
				for(uint32_t i = threadIdx.x; i < nch * half; i += blockDim.x) {
					const uint32_t j = i % nch, bin = i / nch;
					out[(size_t) chs[j] * half + bin] = acc[i];
				}
			} else {
				for(uint32_t i = threadIdx.x; i < nch * half; i += blockDim.x) {
					const uint32_t j = i / half, bin = i % half;
					out[(size_t) chs[j] * half + bin] = acc[i];
				}
			}
		}
		if(bad) atomicOr(&b.status[p], bad);
	}
}

// ---------------------------------------------------------------------------------------------------------------
// nonzero propagate + inverse coupling + floor multiply: one block per packet, one thread per bin
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void uncouple(float& m, float& a) {   // hpp:1220-1239
	const float mv = m, av = a;
	if(mv > 0.f) {
		if(av > 0.f) a = mv - av;
		else { a = mv; m = mv + av; }
	} else {
		if(av > 0.f) a = mv + av;
		else { a = mv; m = mv - av; }
	}
}

__global__ void __launch_bounds__(256) k_couple_dot(DevBatchView b, DevStageBuffers sb) {
	const uint32_t p = blockIdx.x;
	const pov_packet pk = b.packets[p];
	const DevSetup& su = setup_of(b, pk);
	const uint32_t C = su.channels;
	const uint32_t n = su.blocksize[su.mode_blockflag[pk.mode]], half = n / 2;
	const DevMapping& mp = su.mappings[su.mode_mapping[pk.mode]];
	uint32_t used = pk.floor_used;
	for(uint32_t k = 0; k < mp.n_couplings; ++k) {
		const uint32_t m = mp.coupling_mag[k], a = mp.coupling_ang[k];
		if(((used >> m) | (used >> a)) & 1) used |= (1u << m) | (1u << a);
	}
	const float* in = b.spectra + b.spec_off[p];
	const float* fo = sb.floor_outputs + sb.stage_off[p];
	float* out = sb.after_envelope + sb.stage_off[p] / 2;
	for(uint32_t i = threadIdx.x; i < half; i += blockDim.x) {
		float v[POV_MAX_CHANNELS];
#pragma unroll
		for(uint32_t c = 0; c < POV_MAX_CHANNELS; ++c) v[c] = (c < C) ? in[(size_t) c * half + i] : 0.f;
		for(uint32_t k = mp.n_couplings; k > 0; --k) {
			const uint32_t m = mp.coupling_mag[k - 1], a = mp.coupling_ang[k - 1];
			float mv = 0.f, av = 0.f;
#pragma unroll
			for(uint32_t c = 0; c < POV_MAX_CHANNELS; ++c) { if(c == m) mv = v[c]; if(c == a) av = v[c]; }
			uncouple(mv, av);
#pragma unroll
			for(uint32_t c = 0; c < POV_MAX_CHANNELS; ++c) { if(c == m) v[c] = mv; if(c == a) v[c] = av; }
		}
#pragma unroll
		for(uint32_t c = 0; c < POV_MAX_CHANNELS; ++c) {
			if(c >= C) continue;
			float r = v[c];
			if((used >> c) & 1) r = __fmul_rn(r, fo[(size_t) c * n + i]);   // hpp:1247-1252
			out[(size_t) c * half + i] = r;
		}
	}
}

// ---------------------------------------------------------------------------------------------------------------
// inverse MDCT of one channel-packet per block (staged / drop-in mdct_backward path)
// ---------------------------------------------------------------------------------------------------------------
template <int Q>
__device__ void imdct_block(const float* __restrict__ X, float* __restrict__ y, const float2* __restrict__ rot,
                            const float2* __restrict__ W, float2* T, float* D) {
	constexpr int M = 2 * Q;
	for(int j = threadIdx.x; j < Q; j += blockDim.x)
		T[tpad(j)] = cmul(make_float2(X[2 * j], X[M - 1 - 2 * j]), __ldg(&rot[j]));
	__syncthreads();
	fft_passes_except_last<Q>(T, 1, W);
	for(int t = threadIdx.x; t < Q / 8; t += blockDim.x) pass_last_to_D<Q>(T, t, rot, D);
	__syncthreads();
	for(int m = threadIdx.x; m < 2 * M; m += blockDim.x) y[m] = frame_from_D(D, M, m);
	__syncthreads();
}

__device__ __forceinline__ void imdct_dispatch(uint32_t n, const float* X, float* y, const float2* rot, const float2* W,
                                               float2* T, float* D) {
	switch(n) {
		case 64:   imdct_block<16>(X, y, rot, W, T, D); break;
		case 128:  imdct_block<32>(X, y, rot, W, T, D); break;
		case 256:  imdct_block<64>(X, y, rot, W, T, D); break;
		case 512:  imdct_block<128>(X, y, rot, W, T, D); break;
		case 1024: imdct_block<256>(X, y, rot, W, T, D); break;
		case 2048: imdct_block<512>(X, y, rot, W, T, D); break;
		case 4096: imdct_block<1024>(X, y, rot, W, T, D); break;
		case 8192: imdct_block<2048>(X, y, rot, W, T, D); break;
		default: break;
	}
}

constexpr int kImdctThreads = 128;
constexpr int kImdctSmemFloat2 = 2048 + 256;   // Q=2048 padded
constexpr int kImdctSmemD = 4096;

__global__ void __launch_bounds__(kImdctThreads) k_imdct_staged(DevBatchView b, DevStageBuffers sb, uint32_t max_channels) {
	extern __shared__ __align__(16) unsigned char imdct_smem[];
	float2* T = reinterpret_cast<float2*>(imdct_smem);
	float* D = reinterpret_cast<float*>(T + kImdctSmemFloat2);
	const uint32_t p = blockIdx.x / max_channels, c = blockIdx.x % max_channels;
	const pov_packet pk = b.packets[p];
	const DevSetup& su = setup_of(b, pk);
	if(c >= su.channels) return;
	const uint32_t flag = su.mode_blockflag[pk.mode];
	const uint32_t n = su.blocksize[flag];
	const float* X = sb.after_envelope + sb.stage_off[p] / 2 + (size_t) c * (n / 2);
	float* y = sb.pcm_after_mdct + sb.stage_off[p] + (size_t) c * n;
	imdct_dispatch(n, X, y, su.rot[flag], su.fft[flag], T, D);
}

__global__ void __launch_bounds__(kImdctThreads) k_mdct_backward(uint32_t n, const float* __restrict__ in,
                                                                 float* __restrict__ out, const float2* rot, const float2* W) {
	extern __shared__ __align__(16) unsigned char imdct_smem[];
	float2* T = reinterpret_cast<float2*>(imdct_smem);
	float* D = reinterpret_cast<float*>(T + kImdctSmemFloat2);
	imdct_dispatch(n, in + (size_t) blockIdx.x * (n / 2), out + (size_t) blockIdx.x * n, rot, W, T, D);
}

// ---------------------------------------------------------------------------------------------------------------
// window + overlap-add + emit, gather form: one block per (packet, channel)
//   PCM[centre(prev) + j] = (0 + prev[n_prev/2 + j] * w_prev[..]) + cur[j + n/4 - n_prev/4] * w_cur[..]
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void slope_lengths(const DevSetup& su, const pov_packet& pk, int& left, int& right) {
	const uint32_t flag = su.mode_blockflag[pk.mode];
	// hpp:844-847: short blocks always use blocksize0 slopes; long blocks follow their own prev/next flags
	left = (int) ((flag && (pk.window_flags & 1)) ? su.blocksize[1] : su.blocksize[0]) / 2;
	right = (int) ((flag && (pk.window_flags & 2)) ? su.blocksize[1] : su.blocksize[0]) / 2;
}

template <class TPcm>
__global__ void __launch_bounds__(256) k_ola_staged(DevBatchView b, DevStageBuffers sb, uint32_t max_channels) {
	const uint32_t p = blockIdx.x / max_channels, c = blockIdx.x % max_channels;
	const pov_packet pk = b.packets[p];
	const pov_stream st = b.streams[pk.stream];
	const DevSetup& su = b.setups[st.setup_id];
	if(c >= su.channels || p == st.first_packet || pk.emit_frames == 0) return;   // hpp:1021
	const pov_packet pv = b.packets[p - 1];
	const int n = su.blocksize[su.mode_blockflag[pk.mode]], np = su.blocksize[su.mode_blockflag[pv.mode]];
	int lc, rc, lp, rp;
	slope_lengths(su, pk, lc, rc);
	slope_lengths(su, pv, lp, rp);
	const float* sl_c_l = su.slope[lc == (int) su.blocksize[1] / 2 ? 1 : 0];
	const float* sl_c_r = su.slope[rc == (int) su.blocksize[1] / 2 ? 1 : 0];
	const float* sl_p_l = su.slope[lp == (int) su.blocksize[1] / 2 ? 1 : 0];
	const float* sl_p_r = su.slope[rp == (int) su.blocksize[1] / 2 ? 1 : 0];
	const float* ycur = sb.pcm_after_mdct + sb.stage_off[p] + (size_t) c * n;
	const float* yprev = sb.pcm_after_mdct + sb.stage_off[p - 1] + (size_t) c * np;
	const int shift = n / 4 - np / 4;
	for(uint32_t j = threadIdx.x; j < pk.emit_frames; j += blockDim.x) {
		float acc = 0.f;
		const int ip = np / 2 + (int) j;
		if(ip < np) acc = __fadd_rn(acc, __fmul_rn(yprev[ip], window_at(np, ip, lp, rp, sl_p_l, sl_p_r)));
		const int ic = (int) j + shift;
		if(ic >= 0 && ic < n) acc = __fadd_rn(acc, __fmul_rn(ycur[ic], window_at(n, ic, lc, rc, sl_c_l, sl_c_r)));
		const uint64_t f = pk.pcm_off + j;
		const uint64_t o = (b.pcm_layout == POV_PCM_PLANAR) ? st.pcm_base + (uint64_t) c * st.pcm_frames + f
		                                                    : st.pcm_base + f * su.channels + c;
		reinterpret_cast<TPcm*>(b.pcm)[o] = pcm_value<TPcm>(acc);
	}
}

// ---------------------------------------------------------------------------------------------------------------
// sum of a PCM arena in float64 (corpus decode reports it as a checksum of everything that was delivered)
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_checksum(const float* __restrict__ pcm, uint64_t n, double* __restrict__ sum) {
	double acc = 0;
	for(uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) acc += (double) pcm[i];
	for(int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
	__shared__ double part[8];
	if((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
	__syncthreads();
	if(threadIdx.x == 0) {
		double t = 0;
		for(int i = 0; i < 8; ++i) t += part[i];
		atomicAdd(sum, t);
	}
}

// exact integer sum of an int16 PCM arena (POV_PCM_S16): two's-complement accumulation in 64 bits, independent of the order
__global__ void __launch_bounds__(256) k_checksum_s16(const int16_t* __restrict__ pcm, uint64_t n, unsigned long long* __restrict__ sum) {
	long long acc = 0;
	for(uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) acc += pcm[i];
	for(int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
	__shared__ long long part[8];
	if((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
	__syncthreads();
	if(threadIdx.x == 0) {
		long long t = 0;
		for(int i = 0; i < 8; ++i) t += part[i];
		atomicAdd(sum, (unsigned long long) t);
	}
}

// ---------------------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------------------
size_t residue_apply_max_dynamic_smem() {
	int dev = 0, optin = 0;
	cudaFuncAttributes fa;
	if(cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess ||
	   cudaFuncGetAttributes(&fa, k_residue_apply) != cudaSuccess)
		return 48 * 1024 - 8 * 1024;
	return (size_t) optin > fa.sharedSizeBytes ? (size_t) optin - fa.sharedSizeBytes : 0;
}

cudaError_t launch_residue_apply(const DevBatchView& b, float* spectra_out, size_t smem, uint32_t* cursor_scratch,
                                 uint32_t cursor_stride, uint32_t grid, cudaStream_t st, uint64_t* launches) {
	if(b.n_packets == 0) return cudaSuccess;
	// smem = max over the batch's submaps of (nch * n/2 floats [+ 8 * partitions * vectors cursors]), computed at upload
	if(smem > 48 * 1024) {
		cudaError_t e = cudaFuncSetAttribute(k_residue_apply, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
		if(e != cudaSuccess) return e;
	}
	k_residue_apply<<<grid, kResThreads, smem, st>>>(b, spectra_out, cursor_scratch, cursor_stride);
	if(launches) ++*launches;
	return cudaGetLastError();
}

cudaError_t launch_staged(const DevBatchView& b, const DevStageBuffers& sb, uint32_t max_channels, cudaStream_t st,
                          uint64_t* launches) {
	if(b.n_packets == 0) return cudaSuccess;
	const uint64_t cps = (uint64_t) b.n_packets * max_channels;
	k_floor1<<<(unsigned) ((cps + kFloorWarps - 1) / kFloorWarps), kFloorWarps * 32, 0, st>>>(b, sb, max_channels);
	k_couple_dot<<<b.n_packets, 256, 0, st>>>(b, sb);
	const size_t smem = kImdctSmemFloat2 * sizeof(float2) + kImdctSmemD * sizeof(float);
	k_imdct_staged<<<(unsigned) cps, kImdctThreads, smem, st>>>(b, sb, max_channels);
	if(b.pcm_s16) k_ola_staged<int16_t><<<(unsigned) cps, 256, 0, st>>>(b, sb, max_channels);
	else k_ola_staged<float><<<(unsigned) cps, 256, 0, st>>>(b, sb, max_channels);
	if(launches) *launches += 4;
	return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------
// Feature matrices (SURVEY.md §8f-3): what the reference's Python readers compute from a debug dump
// (demo_live_extract.py: read_floor_ys :262-408, read_residue_ys :410-505, default arguments), gathered on the device
// from the staged kernels' intermediates. One warp per row, lanes over the columns; the expressions keep the readers'
// float32 operation order so that kinds 0-2 come out bit for bit.
//   0 floor_final_ys           [tag | (final_y * multiplier - 127.5) / 127.5 ...]          one row per decoded floor curve
//   1 floor_final_ys_rendered  [tag | (floor[x_i] - 127.5) / 127.5 ...]                     x_i = the floor's X list, bitstream order
//   2 residue_ys               [after_residue[min(x_i, n/2 - 1)] ...]                       packets of the floor with most posts
//   3 residue_ys_with_floor    the same times exp(floor[min(x_i, n - 1)] / 255 - 1)
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_features(int kind, const FeatRow* __restrict__ rows, uint64_t n_rows, const FeatFloor* __restrict__ floors, uint32_t dim,
                           const uint32_t* __restrict__ final_ys, const uint16_t* __restrict__ floor, const float* __restrict__ residue,
                           float* __restrict__ out) {
	const uint64_t r = (uint64_t) blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
	if(r >= n_rows) return;
	const int lane = threadIdx.x & 31;
	const FeatRow row = rows[r];
	const FeatFloor& F = floors[row.floor];
	float* o = out + r * dim;
	for(uint32_t c = lane; c < dim; c += 32) {
		float v = 0.f;
		if(kind <= 1) {
			if(c == 0) v = F.tag;
			else if(c - 1 < F.n_posts) {
				const uint32_t i = c - 1;
				const float y = kind == 0 ? __fmul_rn((float) final_ys[row.src * POV_MAX_POSTS + i], (float) F.multiplier)
				                          : (float) floor[row.src + F.xs[i]];
				v = __fdiv_rn(__fsub_rn(y, 127.5f), 127.5f);
			}
		} else if(c < F.n_posts) {
			const uint32_t x = min((uint32_t) F.xs[c], row.n / 2 - 1);
			v = residue[row.src + x];
			if(kind == 3 && row.base != ~0ull) {
				const uint32_t xb = min((uint32_t) F.xs[c], row.base_n - 1);
				const float fb = __fdiv_rn((float) floor[row.base + xb], 255.0f);
				v = __fmul_rn(v, expf(__fsub_rn(fb, 1.0f)));
			}
		}
		o[c] = v;
	}
}

cudaError_t launch_features(int kind, const FeatRow* rows, uint64_t n_rows, const FeatFloor* floors, uint32_t output_dim,
                            const uint32_t* final_ys, const uint16_t* floor, const float* residue, float* out, cudaStream_t st, uint64_t* launches) {
	if(n_rows == 0) return cudaSuccess;
	k_features<<<(unsigned) ((n_rows + 7) / 8), 256, 0, st>>>(kind, rows, n_rows, floors, output_dim, final_ys, floor, residue, out);
	if(launches) ++*launches;
	return cudaGetLastError();
}

cudaError_t launch_mdct_backward(const DevSetup*, uint32_t n, uint64_t count, const float* in, float* out,
                                 const float2* rot, const float2* fft, cudaStream_t st, uint64_t* launches) {
	if(count == 0) return cudaSuccess;
	const size_t smem = kImdctSmemFloat2 * sizeof(float2) + kImdctSmemD * sizeof(float);
	k_mdct_backward<<<(unsigned) count, kImdctThreads, smem, st>>>(n, in, out, rot, fft);
	if(launches) ++*launches;
	return cudaGetLastError();
}

}  // namespace pov

cudaError_t pov_checksum_launch(const void* pcm, bool s16, uint64_t n, void* d_sum, cudaStream_t st, uint64_t* launches) {
	if(n == 0) return cudaSuccess;
	const unsigned blocks = (unsigned) ((n + 256ull * 16 - 1) / (256ull * 16) > 1184 ? 1184 : (n + 256ull * 16 - 1) / (256ull * 16));
	if(s16) pov::k_checksum_s16<<<blocks ? blocks : 1, 256, 0, st>>>((const int16_t*) pcm, n, (unsigned long long*) d_sum);
	else pov::k_checksum<<<blocks ? blocks : 1, 256, 0, st>>>((const float*) pcm, n, (double*) d_sum);
	if(launches) ++*launches;
	return cudaGetLastError();
}
