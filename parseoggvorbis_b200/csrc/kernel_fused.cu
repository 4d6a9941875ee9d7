// Production path: ONE kernel from coded floor posts + residue spectra to PCM.
//
//   floor1 unwrap/render -> nonzero propagate -> inverse coupling -> floor multiply -> inverse MDCT
//   -> window -> overlap-add -> planar/interleaved PCM
// (reference: VorbisStream::parse_audio stages 4.3.2-4.3.7 + VorbisStreamDecodeState, src/ParseOggVorbis.hpp:
//  521-591, 1174-1180, 1213-1268, 1008-1059; the IMDCT contract is src/mdct.h:105.)
//
// Why fused: unfused, every channel-packet of blocksize n moves 2n B of spectrum in, 4n B of frame out, 4n B
// of frame back in and 2n B of PCM out. Here HBM sees the spectrum once (TMA bulk copy into shared memory,
// double buffered) and the PCM once (coalesced 128-bit stores): 4n B per channel-packet = 8 B per PCM sample,
// the algorithmic minimum of SURVEY.md §8(d). Everything in between lives in shared memory and registers.
//
// Work decomposition: one CTA per *run* = up to K consecutive packets of one stream, all channels. The overlap
// of consecutive frames is carried in shared memory (the D array of the previous frame); the first packet of a
// run is a halo that is transformed again instead of exchanged, so runs are independent (no inter-CTA traffic).
// Inside a run the CTA advances in *steps*: one long packet, or a group of consecutive short packets that
// together fill the same buffers (batching by blocksize class).
#include "kernels.h"
#include "fft_core.cuh"
#include "floor_core.cuh"
#include "pcm_out.cuh"
#include <stdlib.h>

namespace pov {

// ---- mbarrier / TMA bulk copy (sm_90+ PTX; SASS: UBLKCP + SYNCS) ----------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
	asm volatile(
		"{\n\t.reg .pred p;\n\t"
		"WAIT_LOOP:\n\t"
		"mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
		"@p bra.uni WAIT_DONE;\n\t"
		"bra.uni WAIT_LOOP;\n\t"
		"WAIT_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
	             ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void uncouple_f(float& m, float& a) {   // hpp:1220-1239, branch-free
	// t = +a when m > 0, -a otherwise; the four cases collapse to:  a > 0 ? (m, m - t) : (m + t, m)
	const float mv = m, av = a;
	const float t = (mv > 0.f) ? av : -av;
	const bool p = av > 0.f;
	const float diff = mv - t, sum = mv + t;
	a = p ? diff : mv;
	m = p ? mv : sum;
}

struct StepInfo {
	uint32_t first;      // global index of the step's first packet
	uint32_t count;      // packets in the step
	uint32_t flag;       // blocksize class (0 short / 1 long)
};

struct FusedParams {
	DevBatchView b;
	const DevRun* runs;
	uint32_t floor_cap[2];   // posts capacity (multiple of 4) of a curve block, per blocksize class
	uint32_t scratch_cap;    // posts capacity of the per-warp unwrap scratch (only allocated when > 32)
	uint32_t group_short;    // max short packets per step
	uint32_t slot_floats;    // floats of one spectra buffer = C_max * blocksize1/2
	uint32_t curve_bytes;    // size of the curve-block region
	uint32_t table_float2;   // float2 slots of the shared-memory twiddle/rotation tables
};

// Compact per-packet descriptor kept in shared memory for the whole run (loaded once in the prologue), so that the
// per-step control flow never waits on global memory.
struct PktCtx { uint32_t used, emit, wflags, mode; uint64_t ys_off, pcm_off; };
constexpr int kMaxRunPackets = 65;     // run_len <= 64 plus one halo packet (api.cu clamps POV_RUN_LEN)
struct StepCtx { uint32_t first, count, flag, mode; };    // first = index inside the run

// Elementwise stage for C channels (compile time): floor curve evaluation + coupling + floor multiply + DCT-IV
// pre-rotation. Item = (packet g of the step, quad q): complex points j = 2q, 2q+1 and their mirrors Q-1-j, which
// together consume the bins 4q..4q+3 and M-4-4q..M-1-4q of every channel (two aligned 128-bit loads per spectrum).
template <int C>
__device__ __forceinline__ void stage_spectral(const float* __restrict__ raw, unsigned char* __restrict__ curves, uint32_t curve_stride,
                                               uint32_t floor_cap, const float* __restrict__ invdb, float2* __restrict__ T,
                                               int npk, int log2quads, const float2* __restrict__ rot, float2 c1, float2 c6,
                                               const DevMapping* __restrict__ mp) {
	const int quads = 1 << log2quads, Q = 4 * quads, M = 2 * Q;
	const int tstride = Q + Q / 8;
	const int ncoup = (C > 1) ? (int) mp->n_couplings : 0;
	for(int it = threadIdx.x; it < (npk << log2quads); it += blockDim.x) {
		const int g = it >> log2quads, q = it & (quads - 1);
		const float* R0 = raw + (size_t) (g * C) * M;
		float4 lo[C], hi[C];                 // bins 4q..4q+3 and M-4-4q..M-1-4q
#pragma unroll
		for(int c = 0; c < C; ++c) {
			lo[c] = *reinterpret_cast<const float4*>(R0 + c * M + 4 * q);
			hi[c] = *reinterpret_cast<const float4*>(R0 + c * M + M - 4 - 4 * q);
		}
		if(C == 2) {
			// two channels can only be coupled with each other: no channel search needed
			for(int k = ncoup - 1; k >= 0; --k) {
				if(mp->coupling_mag[k] == 0) {
					uncouple_f(lo[0].x, lo[C - 1].x); uncouple_f(lo[0].y, lo[C - 1].y); uncouple_f(lo[0].z, lo[C - 1].z); uncouple_f(lo[0].w, lo[C - 1].w);
					uncouple_f(hi[0].x, hi[C - 1].x); uncouple_f(hi[0].y, hi[C - 1].y); uncouple_f(hi[0].z, hi[C - 1].z); uncouple_f(hi[0].w, hi[C - 1].w);
				} else {
					uncouple_f(lo[C - 1].x, lo[0].x); uncouple_f(lo[C - 1].y, lo[0].y); uncouple_f(lo[C - 1].z, lo[0].z); uncouple_f(lo[C - 1].w, lo[0].w);
					uncouple_f(hi[C - 1].x, hi[0].x); uncouple_f(hi[C - 1].y, hi[0].y); uncouple_f(hi[C - 1].z, hi[0].z); uncouple_f(hi[C - 1].w, hi[0].w);
				}
			}
		} else if(C > 2) {
			for(int k = ncoup - 1; k >= 0; --k) {
				const int m = mp->coupling_mag[k], a = mp->coupling_ang[k];
				float4 ml = make_float4(0.f, 0.f, 0.f, 0.f), mh = ml, al = ml, ah = ml;
#pragma unroll
				for(int c = 0; c < C; ++c) {
					if(c == m) { ml = lo[c]; mh = hi[c]; }
					if(c == a) { al = lo[c]; ah = hi[c]; }
				}
				uncouple_f(ml.x, al.x); uncouple_f(ml.y, al.y); uncouple_f(ml.z, al.z); uncouple_f(ml.w, al.w);
				uncouple_f(mh.x, ah.x); uncouple_f(mh.y, ah.y); uncouple_f(mh.z, ah.z); uncouple_f(mh.w, ah.w);
#pragma unroll
				for(int c = 0; c < C; ++c) {
					if(c == m) { lo[c] = ml; hi[c] = mh; }
					if(c == a) { lo[c] = al; hi[c] = ah; }
				}
			}
		}
		// rotations w[2q], w[2q+1] and w[Q-2-2q], w[Q-1-2q] from ONE shared-memory entry:
		//   w[j+1] = w[j] * exp(-i pi/M),   w[Q-1-j] = -i * conj(w[j]) * exp(+i pi 6/(8M))
		const float2 r0 = rot[2 * q];
		const float2 r1 = cmul(r0, c1);
		const float2 rq1 = cmul(make_float2(-r0.y, -r0.x), c6);      // w[Q-1-2q]
		const float2 rq2 = cmul(make_float2(-r1.y, -r1.x), c6);      // w[Q-2-2q]
		const float4 wl = make_float4(r0.x, r0.y, r1.x, r1.y);
		const float4 wh = make_float4(rq2.x, rq2.y, rq1.x, rq1.y);
		float2* T0 = T + (size_t) (g * C) * tstride;
		const int j1 = 2 * q, j2 = Q - 2 - 2 * q;
		const int p1 = j1 + (j1 >> 3), p2 = j2 + (j2 >> 3);       // (even, odd) index pairs never straddle a pad slot
#pragma unroll
		for(int c = 0; c < C; ++c) {
			CurveV3 Cv;
			Cv.bind(curves + (size_t) (g * C + c) * curve_stride, floor_cap);
			float4 fl, fh;
			const uint32_t mode = Cv.hdr[0];
			if(mode == 0) {
				fl = curve_quad(Cv, (uint32_t) (4 * q), invdb);
				fh = curve_quad(Cv, (uint32_t) (M - 4 - 4 * q), invdb);
			} else {
				const float fill = (mode == 1) ? 1.f : 0.f;
				fl = make_float4(fill, fill, fill, fill); fh = fl;
			}
			// hpp:1252 residue *= floor (one rounding each)
			const float l0 = __fmul_rn(lo[c].x, fl.x), l1 = __fmul_rn(lo[c].y, fl.y), l2 = __fmul_rn(lo[c].z, fl.z), l3 = __fmul_rn(lo[c].w, fl.w);
			const float h0 = __fmul_rn(hi[c].x, fh.x), h1 = __fmul_rn(hi[c].y, fh.y), h2 = __fmul_rn(hi[c].z, fh.z), h3 = __fmul_rn(hi[c].w, fh.w);
			// t[j] = (X[2j] + i X[M-1-2j]) * w[j]
			float2* Tc = T0 + c * tstride;
			Tc[p1]     = cmul(make_float2(l0, h3), make_float2(wl.x, wl.y));       // j = 2q
			Tc[p1 + 1] = cmul(make_float2(l2, h1), make_float2(wl.z, wl.w));       // j = 2q+1
			Tc[p2]     = cmul(make_float2(h0, l3), make_float2(wh.x, wh.y));       // j = Q-2-2q: X[M-4-4q], X[4q+3]
			Tc[p2 + 1] = cmul(make_float2(h2, l1), make_float2(wh.z, wh.w));       // j = Q-1-2q: X[M-2-4q], X[4q+1]
		}
	}
}

// Last pass + post-rotation with the D array split in halves: lo = D[0..M/2) (second half of the frame, needed by the
// NEXT packet), hi = D[M/2..M) (first half of the frame, consumed by this packet's overlap-add).
template <int Q>
__device__ __forceinline__ void pass_last_split(const float2* __restrict__ T, int t, const float2* __restrict__ rot,
                                                float* __restrict__ lo, float* __restrict__ hi) {
	constexpr int M = 2 * Q;
	float2 a[8];
	const float2* p = T + 9 * t;
#pragma unroll
	for(int m = 0; m < 8; ++m) a[m] = p[m];
	dft8(a);
	const int k0 = freq_of_pos<Q>(8 * t);           // k0 < Q/8; k = k0 + m*Q/8
	// w[k0 + m*Q/8] = w[k0] * exp(-i pi m/16)  (Q/M = 1/2), w[k0] from shared memory
	const float2 r0 = rot[k0];
	constexpr float kVr[8] = {1.f, 0.98078528040323044913f, 0.92387953251128675613f, 0.83146961230254523708f,
	                          0.70710678118654752440f, 0.55557023301960222474f, 0.38268343236508977173f, 0.19509032201612826785f};
	constexpr float kVi[8] = {0.f, -0.19509032201612826785f, -0.38268343236508977173f, -0.55557023301960222474f,
	                          -0.70710678118654752440f, -0.83146961230254523708f, -0.92387953251128675613f, -0.98078528040323044913f};
#pragma unroll
	for(int m = 0; m < 8; ++m) {
		const float2 wm = (m == 0) ? r0 : cmul(r0, make_float2(kVr[m], kVi[m]));
		const float2 c = cmul(a[m], wm);
		// D[2k] = Re, D[M-1-2k] = -Im;  2k < M/2  <=>  m < 4
		if(m < 4) { lo[2 * k0 + m * (Q / 4)] = c.x; hi[(M / 2 - 1 - 2 * k0) - m * (Q / 4)] = -c.y; }
		else      { hi[2 * k0 + m * (Q / 4) - M / 2] = c.x; lo[(M - 1 - 2 * k0) - m * (Q / 4)] = -c.y; }
	}
}

// bar.sync on a named barrier: only the `count` threads of one FFT meet (ids 1..15; 0 is __syncthreads)
__device__ __forceinline__ void named_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }

template <int Q, int L>
__device__ __forceinline__ void passes_radix8_group(float2* Tf, int t, const float2* tw8, int bar_id) {
	if constexpr(L >= 64) {
		pass_radix8_s<Q, L>(Tf, t, tw8);
		named_sync(bar_id, FftGeom<Q>::kItems);
		passes_radix8_group<Q, L / 8>(Tf, t, tw8, bar_id);
	}
}

template <int Q, int L>
__device__ __forceinline__ void passes_radix8_block(float2* T, int nf, const float2* tw8) {
	if constexpr(L >= 64) {
		for(int w = threadIdx.x; w < nf * FftGeom<Q>::kItems; w += blockDim.x) {
			const int f = w / FftGeom<Q>::kItems, t = w - f * FftGeom<Q>::kItems;
			pass_radix8_s<Q, L>(T + f * FftGeom<Q>::kStride, t, tw8);
		}
		__syncthreads();
		passes_radix8_block<Q, L / 8>(T, nf, tw8);
	}
}

// rot / tw8: shared-memory tables of this blocksize class; TWP: global per-pass table, used by the first small-radix
// pass only (block sizes whose log2(Q) is not a multiple of 3).
template <int Q>
__device__ __forceinline__ void stage_fft(float2* T, float* Dlo, float* Dhi, int nf, const float2* rot, const float2* tw8, const float2* TWP) {
	constexpr int kItems = FftGeom<Q>::kItems;
	if(kItems >= 32 && nf * kItems == (int) blockDim.x && nf <= 15) {
		// one work item per thread and every FFT owns whole warps: the passes of one FFT only synchronise its own
		// kItems threads (named barrier), the other FFTs of the CTA run ahead independently
		const int f = threadIdx.x / kItems, t = threadIdx.x - f * kItems;
		float2* Tf = T + (size_t) f * FftGeom<Q>::kStride;
		if constexpr(FftGeom<Q>::kFirstRadix != 8) {
			pass_first_small_p<Q>(Tf, t, TWP);
			named_sync(1 + f, kItems);
		}
		passes_radix8_group<Q, PassTables<Q>::kL1>(Tf, t, tw8, 1 + f);
		pass_last_split<Q>(Tf, t, rot, Dlo + (size_t) f * Q, Dhi + (size_t) f * Q);
		return;
	}
	if constexpr(FftGeom<Q>::kFirstRadix != 8) {
		for(int w = threadIdx.x; w < nf * kItems; w += blockDim.x) {
			const int f = w / kItems, t = w - f * kItems;
			pass_first_small_p<Q>(T + f * FftGeom<Q>::kStride, t, TWP);
		}
		__syncthreads();
	}
	passes_radix8_block<Q, PassTables<Q>::kL1>(T, nf, tw8);
	for(int w = threadIdx.x; w < nf * kItems; w += blockDim.x) {
		const int f = w / kItems, t = w - f * kItems;
		pass_last_split<Q>(T + (size_t) f * FftGeom<Q>::kStride, t, rot, Dlo + (size_t) f * Q, Dhi + (size_t) f * Q);
	}
}

// floors with more than 32 posts: shared-memory unwrap (floor_core.cuh floor1_unwrap_warp) + record build in chunks
static __device__ __noinline__ uint32_t floor1_curve_generic(const DevFloor* F, const uint16_t* ys, const CurveV3& Cv, uint32_t cells, uint32_t n,
                                                      int lane, unsigned char* scratch, uint32_t scratch_cap) {
	FloorScratch W;
	W.bind(scratch, scratch_cap);
	uint32_t stt = floor1_unwrap_warp(F, ys, W, lane);
	stt |= floor1_range_check_warp(W, n, lane);
	const uint32_t ns = *W.nseg;
	if(lane == 0) Cv.hdr[0] = 0;
	for(uint32_t base = 0; base < ns; base += 32) {
		const uint32_t sg = base + lane;
		const bool have = sg < ns;
		const uint32_t x0 = have ? W.segx[sg] : 0u, y0 = have ? W.segy[sg] : 0u;
		const uint32_t x1 = (sg + 1 < ns) ? W.segx[sg + 1] : 0u, y1 = (sg + 1 < ns) ? W.segy[sg + 1] : 0u;
		curve_build_warp(Cv, ns, x0, y0, x1, y1, have, base, cells, lane, base == 0);
	}
	curve_scan_cells_warp(Cv, cells, lane);
	return stt;
}

// floor1 unwrap + curve records of one (packet, channel) curve of a step, by one warp. Out of line on purpose: it is
// reached from three places and the kernel is instruction-cache bound.
struct FloorTaskArgs {
	const uint16_t* ys; uint32_t* status; const DevFloor* floors; const DevMapping* mappings; const uint8_t* mode_map;
	const PktCtx* pk; unsigned char* curves; unsigned char* fscr;
	uint32_t floor_cap[2], scratch_cap, bs[2]; int C;
};
static __device__ __noinline__ void floor_task_fn(const FloorTaskArgs& A, uint32_t first, uint32_t flag, uint32_t mode, int f, int warp, int lane) {
	const int C = A.C;
	const int n = (int) A.bs[flag ? 1 : 0];
	const uint32_t cells = (uint32_t) n / 8;
	const uint32_t fcap = A.floor_cap[flag ? 1 : 0];
	const uint32_t curve_stride = CurveV3::bytes(fcap, cells);
	const DevMapping* mp = &A.mappings[A.mode_map[mode]];
	const int g = f / C, c = f - g * C;
	CurveV3 Cv;
	Cv.bind(A.curves + (size_t) f * curve_stride, fcap);
	const PktCtx& pc = A.pk[first + g];
	const uint32_t used = pc.used;
	if(!((used >> c) & 1)) {
		// no curve decoded: the reference multiplies by its zero-initialised floor buffer if the channel became
		// "used" through coupling (hpp:1159,1247) and leaves the residue untouched otherwise
		uint32_t prop = used;
		for(uint32_t k = 0; k < mp->n_couplings; ++k) {   // hpp:1174-1180
			const uint32_t m = mp->coupling_mag[k], a = mp->coupling_ang[k];
			if(((prop >> m) | (prop >> a)) & 1) prop |= (1u << m) | (1u << a);
		}
		if(lane == 0) Cv.hdr[0] = ((prop >> c) & 1) ? 2u : 1u;
		return;
	}
	const DevFloor* F = &A.floors[mp->floor_of_ch[c]];
	uint64_t yo = pc.ys_off;
	for(int cc = 0; cc < c; ++cc)
		if((used >> cc) & 1) yo += A.floors[mp->floor_of_ch[cc]].n_posts;
	uint32_t stt;
	if(F->n_posts <= 32) stt = floor1_curve_warp32(F, A.ys + yo, Cv, cells, (uint32_t) n, lane);
	else stt = floor1_curve_generic(F, A.ys + yo, Cv, cells, (uint32_t) n, lane, A.fscr + (size_t) warp * floor_scratch_stride(A.scratch_cap), A.scratch_cap);
	if(stt && lane == 0) atomicOr(&A.status[first + g], stt);
}

// Geometry of one emitting packet for the overlap-add stage (all block-uniform).
struct OlaGeom {
	int Hp, H;          // quarter sizes: Hp = n_prev/4, H = n/4 (= length of the lo / hi halves of D)
	int shift;          // index in the current frame of the chunk's first sample: n/4 - n_prev/4
	int lb, lc;         // current frame: left slope begins at lb, has length lc
	int rbp, pr;        // previous frame, relative to its second half: falling slope begins at rbp, has length pr
	const float* slL;   // rising slope table of length lc
	const float* slR;   // rising slope table of length pr (read mirrored)
};

// Overlap-add of one uniform region [j0, j1) (multiples of 4) of the chunk:
//   out = (0 + prev[n_prev/2 + j] * w_prev) + cur[j + shift] * w_cur        (hpp:1008-1017 in gather form)
// plo = lo half of the previous frame's D, chi = hi half of the current frame's D. Inside a region the case of both
// terms is fixed (every boundary is a multiple of 16), so all branches below are block-uniform.
template <class TPcm>
__device__ __forceinline__ void ola_region(const OlaGeom& G, const float* __restrict__ plo, const float* __restrict__ chi,
                                           TPcm* __restrict__ dst, int j0, int j1, int tid, int nthreads) {
	const bool has_p = j0 < G.rbp + G.pr, p_rev = j0 < G.Hp, p_slope = j0 >= G.rbp;
	const int ic0 = j0 + G.shift;
	const bool has_c = ic0 >= G.lb, c_rev = ic0 >= G.H, c_slope = ic0 < G.lb + G.lc;
#pragma unroll 2
	for(int j = j0 + 4 * tid; j < j1; j += 4 * nthreads) {
		float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
		if(has_p) {
			// second half of the previous frame: -D[Hp-1-i] for i < Hp, -D[i-Hp] beyond
			float4 y;
			if(p_rev) { const float4 t = *reinterpret_cast<const float4*>(plo + G.Hp - 4 - j); y = make_float4(t.w, t.z, t.y, t.x); }
			else y = *reinterpret_cast<const float4*>(plo + j - G.Hp);
			float4 w = make_float4(1.f, 1.f, 1.f, 1.f);
			if(p_slope) { const float4 t = __ldg(reinterpret_cast<const float4*>(G.slR + G.pr - 4 - (j - G.rbp))); w = make_float4(t.w, t.z, t.y, t.x); }
			acc.x = __fadd_rn(acc.x, __fmul_rn(-y.x, w.x)); acc.y = __fadd_rn(acc.y, __fmul_rn(-y.y, w.y));
			acc.z = __fadd_rn(acc.z, __fmul_rn(-y.z, w.z)); acc.w = __fadd_rn(acc.w, __fmul_rn(-y.w, w.w));
		}
		if(has_c) {
			// first half of the current frame: D[H+i] for i < H, -D[3H-1-i] beyond
			const int ic = j + G.shift;
			float4 y;
			if(c_rev) { const float4 t = *reinterpret_cast<const float4*>(chi + 2 * G.H - 4 - ic); y = make_float4(-t.w, -t.z, -t.y, -t.x); }
			else y = *reinterpret_cast<const float4*>(chi + ic);
			float4 w = make_float4(1.f, 1.f, 1.f, 1.f);
			if(c_slope) w = __ldg(reinterpret_cast<const float4*>(G.slL + ic - G.lb));
			acc.x = __fadd_rn(acc.x, __fmul_rn(y.x, w.x)); acc.y = __fadd_rn(acc.y, __fmul_rn(y.y, w.y));
			acc.z = __fadd_rn(acc.z, __fmul_rn(y.z, w.z)); acc.w = __fadd_rn(acc.w, __fmul_rn(y.w, w.w));
		}
		pcm_store4(dst + j, acc);
	}
}

// scalar version for ragged tails / unaligned destinations / interleaved output
__device__ __forceinline__ float ola_one(const OlaGeom& G, const float* __restrict__ plo, const float* __restrict__ chi, int j) {
	float acc = 0.f;
	if(j < G.rbp + G.pr) {
		const float y = (j < G.Hp) ? -plo[G.Hp - 1 - j] : -plo[j - G.Hp];
		const float w = (j >= G.rbp) ? __ldg(G.slR + G.pr - 1 - (j - G.rbp)) : 1.f;
		acc = __fadd_rn(acc, __fmul_rn(y, w));
	}
	const int ic = j + G.shift;
	if(ic >= G.lb) {
		const float y = (ic < G.H) ? chi[ic] : -chi[2 * G.H - 1 - ic];
		const float w = (ic < G.lb + G.lc) ? __ldg(G.slL + ic - G.lb) : 1.f;
		acc = __fadd_rn(acc, __fmul_rn(y, w));
	}
	return acc;
}

// kSpec = true: the batch only holds 256/2048 setups, so only those two FFT sizes are instantiated (smaller code).
// TPcm: float, or int16_t for POV_PCM_S16 (converted at the store, pcm_out.cuh).
template <int kThreads, int kMinBlocks, bool kSpec, class TPcm>
__global__ void __launch_bounds__(kThreads, kMinBlocks) k_fused_synth(FusedParams P) {
	extern __shared__ __align__(128) unsigned char smem[];
	__shared__ __align__(8) uint64_t s_bar;
	__shared__ float s_invdb[256];
	__shared__ uint8_t s_mode_flag[POV_MAX_MODES], s_mode_map[POV_MAX_MODES];
	__shared__ PktCtx s_pk[kMaxRunPackets];

	const DevBatchView& b = P.b;
	const DevRun run = P.runs[blockIdx.x];
	const pov_packet pk0 = b.packets[run.first_packet];
	const pov_stream st = b.streams[pk0.stream];
	const DevSetup* __restrict__ su = &b.setups[st.setup_id];
	const int C = (int) su->channels;
	constexpr int nwarps = kThreads >> 5;
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const uint32_t bs0 = su->blocksize[0], bs1 = su->blocksize[1];
	const DevFloor* __restrict__ floors = su->floors;
	const DevMapping* __restrict__ mappings = su->mappings;

	// ---- shared memory carve-up (floats): raw[slot] | T[1.125*slot] | Dlo[2][slot/2] | Dhi[slot/2] | curves | scratch
	const uint32_t slot = P.slot_floats;
	float* raw = reinterpret_cast<float*>(smem);
	float2* T = reinterpret_cast<float2*>(raw + slot);
	float* Dlo = reinterpret_cast<float*>(T) + (size_t) slot + slot / 8;
	float* Dhi = Dlo + slot;
	// One curve-block region is enough: it is read in stage 2 of a step and rewritten (for the next step) in stage 4.
	unsigned char* curves = reinterpret_cast<unsigned char*>(Dhi + slot / 2);
	// twiddle + rotation tables of both blocksize classes (copied from global once per CTA): tw8[0] | tw8[1] | rot[0] | rot[1]
	float2* tab = reinterpret_cast<float2*>(curves + P.curve_bytes);
	const uint32_t tw8n0 = su->fft8_count[0], tw8n1 = su->fft8_count[1];
	float2* s_tw8[2] = {tab, tab + tw8n0};
	float2* s_rot[2] = {tab + tw8n0 + tw8n1, tab + tw8n0 + tw8n1 + bs0 / 8};
	unsigned char* fscr = reinterpret_cast<unsigned char*>(tab + P.table_float2);    // per-warp unwrap scratch, only when scratch_cap > 32

	const int run_n = (int) run.n_packets;           // <= kMaxRunPackets
	for(int i = threadIdx.x; i < 256; i += kThreads) s_invdb[i] = __ldg(&b.inv_db[i]);
	for(int i = threadIdx.x; i < (int) POV_MAX_MODES; i += kThreads) { s_mode_flag[i] = su->mode_blockflag[i]; s_mode_map[i] = su->mode_mapping[i]; }
	for(uint32_t i = threadIdx.x; i < tw8n0; i += kThreads) s_tw8[0][i] = __ldg(&su->fft8[0][i]);
	for(uint32_t i = threadIdx.x; i < tw8n1; i += kThreads) s_tw8[1][i] = __ldg(&su->fft8[1][i]);
	for(uint32_t i = threadIdx.x; i < bs0 / 8; i += kThreads) s_rot[0][i] = __ldg(&su->rot[0][i]);
	for(uint32_t i = threadIdx.x; i < bs1 / 8; i += kThreads) s_rot[1][i] = __ldg(&su->rot[1][i]);
	const float2 rc1[2] = {su->rotc1[0], su->rotc1[1]}, rc6[2] = {su->rotc6[0], su->rotc6[1]};
	for(int i = threadIdx.x; i < run_n; i += kThreads) {
		const pov_packet pk = b.packets[run.first_packet + i];
		PktCtx c;
		c.used = pk.floor_used; c.emit = pk.emit_frames; c.wflags = pk.window_flags; c.mode = pk.mode;
		c.ys_off = pk.ys_off; c.pcm_off = pk.pcm_off;
		s_pk[i] = c;
	}
	if(threadIdx.x == 0) {
		mbar_init(&s_bar, 1);
		mbar_fence_init();
	}
	__syncthreads();

	const int gshort = (bs0 == bs1) ? 1 : (int) P.group_short;

	// Step starting at run-relative packet `first`: one long packet, or up to gshort consecutive short packets of one
	// mode (same mapping, same floors). Evaluated redundantly by every thread from shared memory (block-uniform).
	auto make_step = [&](int first) {
		StepCtx s;
		s.first = (uint32_t) first; s.count = 0; s.flag = 0; s.mode = 0;
		if(first >= run_n) return s;
		s.mode = s_pk[first].mode;
		s.flag = s_mode_flag[s.mode];
		s.count = 1;
		if(!s.flag && bs0 != bs1)
			while((int) s.count < gshort && first + (int) s.count < run_n && s_pk[first + s.count].mode == s.mode) ++s.count;
		return s;
	};
	auto issue_loads = [&](const StepCtx& sx) {     // one elected thread: TMA bulk copies of the step's spectra
		const uint32_t half = (sx.flag ? bs1 : bs0) / 2;
		const uint32_t bytes = (uint32_t) C * half * 4u;
		mbar_expect_tx(&s_bar, bytes * sx.count);
#pragma unroll 1
		for(uint32_t g = 0; g < sx.count; ++g)
			tma_bulk_g2s(raw + (size_t) g * C * half, b.spectra + b.spec_off[run.first_packet + sx.first + g], bytes, &s_bar);
	};
	FloorTaskArgs fa;
	fa.ys = b.ys; fa.status = b.status + run.first_packet; fa.floors = floors; fa.mappings = mappings; fa.mode_map = s_mode_map;
	fa.pk = s_pk; fa.curves = curves; fa.fscr = fscr;
	fa.floor_cap[0] = P.floor_cap[0]; fa.floor_cap[1] = P.floor_cap[1]; fa.scratch_cap = P.scratch_cap;
	fa.bs[0] = bs0; fa.bs[1] = bs1; fa.C = C;
	auto floor_task = [&](const StepCtx& sx, int f) { floor_task_fn(fa, sx.first, sx.flag, sx.mode, f, warp, lane); };

	StepCtx cur = make_step(0);
	if(threadIdx.x == 0 && cur.count) issue_loads(cur);
	// prologue: curves of the first step (later steps get theirs during the previous step's overlap-add stage)
	for(int f = warp; f < (int) cur.count * C; f += nwarps) floor_task(cur, f);
	uint32_t phase = 0;
	// overlap carried from the previous packet: the lo half of its D array and its geometry
	int prev_valid = 0, prev_n = 0, prev_right = 0;
	const float* prev_lo = nullptr;    // channel 0; channels are prev_n/4 apart
	int step_idx = 0;

	while(cur.count) {
		const int buf = step_idx & 1;
		const int npk = (int) cur.count;
		const int first = (int) cur.first;
		const uint32_t flag = cur.flag;
		const StepCtx nxt = make_step(first + npk);

		const int n = (int) (flag ? bs1 : bs0), Q = n / 4;
		const int log2Q = 31 - __clz(Q);
		const int nf = npk * C;
		const DevMapping* mp = &mappings[s_mode_map[cur.mode]];
		float* Dlo_cur = Dlo + (size_t) buf * (slot / 2);
		const uint32_t cells = (uint32_t) n / 8;
		const uint32_t fcap = flag ? P.floor_cap[1] : P.floor_cap[0];
		const uint32_t curve_stride = CurveV3::bytes(fcap, cells);

		// ---- wait for this step's spectra (TMA): one warp polls, the barrier releases everyone; it also publishes the
		//      curve blocks of this step, which were built during the previous step's stage 4 (or the prologue) ----
		if(warp == 0) mbar_wait(&s_bar, phase);
		phase ^= 1;
		__syncthreads();

		// ---- stage 2: floor evaluation + coupling + floor multiply + pre-rotation -> T ----
		{
			const float2* rot = flag ? s_rot[1] : s_rot[0];
			const float2 c1 = flag ? rc1[1] : rc1[0], c6 = flag ? rc6[1] : rc6[0];
			const int lq = log2Q - 2;
			if constexpr(kThreads == 128) {      // the 128-thread variant is only launched for <= 2 channels
				if(C == 1) stage_spectral<1>(raw, curves, curve_stride, fcap, s_invdb, T, npk, lq, rot, c1, c6, mp);
				else stage_spectral<2>(raw, curves, curve_stride, fcap, s_invdb, T, npk, lq, rot, c1, c6, mp);
			} else switch(C) {
				case 1: stage_spectral<1>(raw, curves, curve_stride, fcap, s_invdb, T, npk, lq, rot, c1, c6, mp); break;
				case 2: stage_spectral<2>(raw, curves, curve_stride, fcap, s_invdb, T, npk, lq, rot, c1, c6, mp); break;
				case 3: stage_spectral<3>(raw, curves, curve_stride, fcap, s_invdb, T, npk, lq, rot, c1, c6, mp); break;
				case 4: stage_spectral<4>(raw, curves, curve_stride, fcap, s_invdb, T, npk, lq, rot, c1, c6, mp); break;
				case 5: stage_spectral<5>(raw, curves, curve_stride, fcap, s_invdb, T, npk, lq, rot, c1, c6, mp); break;
				case 6: stage_spectral<6>(raw, curves, curve_stride, fcap, s_invdb, T, npk, lq, rot, c1, c6, mp); break;
				case 7: stage_spectral<7>(raw, curves, curve_stride, fcap, s_invdb, T, npk, lq, rot, c1, c6, mp); break;
				default: stage_spectral<8>(raw, curves, curve_stride, fcap, s_invdb, T, npk, lq, rot, c1, c6, mp); break;
			}
		}
		__syncthreads();
		// the spectra buffer is free again: prefetch the next step's spectra behind stages 3-4
		if(threadIdx.x == 0 && nxt.count) issue_loads(nxt);

		// ---- stage 3: FFT passes + post-rotation -> D (lo / hi halves) ----
		{
			const float2* rot = flag ? s_rot[1] : s_rot[0];
			const float2* tw8 = flag ? s_tw8[1] : s_tw8[0];
			const float2* TWP = su->fftp[flag];
			if constexpr(kSpec) {
				if(flag) stage_fft<512>(T, Dlo_cur, Dhi, nf, rot, tw8, TWP);
				else stage_fft<64>(T, Dlo_cur, Dhi, nf, rot, tw8, TWP);
			} else switch(Q) {
				case 16:   stage_fft<16>(T, Dlo_cur, Dhi, nf, rot, tw8, TWP); break;
				case 32:   stage_fft<32>(T, Dlo_cur, Dhi, nf, rot, tw8, TWP); break;
				case 64:   stage_fft<64>(T, Dlo_cur, Dhi, nf, rot, tw8, TWP); break;
				case 128:  stage_fft<128>(T, Dlo_cur, Dhi, nf, rot, tw8, TWP); break;
				case 256:  stage_fft<256>(T, Dlo_cur, Dhi, nf, rot, tw8, TWP); break;
				case 512:  stage_fft<512>(T, Dlo_cur, Dhi, nf, rot, tw8, TWP); break;
				case 1024: stage_fft<1024>(T, Dlo_cur, Dhi, nf, rot, tw8, TWP); break;
				default:   stage_fft<2048>(T, Dlo_cur, Dhi, nf, rot, tw8, TWP); break;
			}
		}
		__syncthreads();

		// ---- stage 4: the NEXT step's floor curves (a few warps) overlapped with this step's window + overlap-add +
		//      emit (hpp:1008-1059 in gather form, the other warps) ----
		const int nft = (int) nxt.count * C;                     // curves of the next step
		int ola_tid = (int) threadIdx.x, ola_n = kThreads;
		if(nft > 0) {
			if(nft < nwarps) {
				// the top nft warps take one curve each, the others share the overlap-add
				if(warp >= nwarps - nft) { floor_task(nxt, nwarps - 1 - warp); ola_n = 0; }
				else ola_n = 32 * (nwarps - nft);
			} else {
				for(int f = warp; f < nft; f += nwarps) floor_task(nxt, f);
			}
		}
		for(int g = 0; g < npk; ++g) {
			const PktCtx& pc = s_pk[first + g];
			const uint32_t wflags = pc.wflags, emit = pc.emit;
			// hpp:844-847: short blocks always use blocksize0 slopes; long blocks follow their own prev/next flags
			const int lc = (int) ((flag && (wflags & 1)) ? bs1 : bs0) / 2;
			const int rc = (int) ((flag && (wflags & 2)) ? bs1 : bs0) / 2;
			const float* cur_lo = Dlo_cur + (size_t) g * C * Q;
			const float* cur_hi = Dhi + (size_t) g * C * Q;
			const bool emits = prev_valid && emit > 0 && (run.first_packet + (uint32_t) (first + g)) != st.first_packet;
			if(emits && ola_n > 0) {
				OlaGeom G;
				G.Hp = prev_n / 4; G.H = Q;
				G.shift = Q - prev_n / 4;
				G.lc = lc; G.lb = Q - lc / 2;
				G.pr = prev_right; G.rbp = prev_n / 4 - prev_right / 2;
				G.slL = su->slope[lc == (int) bs1 / 2 ? 1 : 0];
				G.slR = su->slope[prev_right == (int) bs1 / 2 ? 1 : 0];
				const bool planar = (b.pcm_layout == POV_PCM_PLANAR);
				const uint64_t chan_base = st.pcm_base + pc.pcm_off;
				if(planar && (emit & 3u) == 0 && ((chan_base | st.pcm_frames) & 3ull) == 0) {
					// 128-bit path. The chunk is cut at the (block-uniform) points where either term changes its case.
					int bnd[6] = {G.Hp, G.rbp, G.rbp + G.pr, G.lb - G.shift, G.lb + G.lc - G.shift, G.H - G.shift};
					int j0 = 0;
					while(j0 < (int) emit) {
						int j1 = (int) emit;
#pragma unroll
						for(int k = 0; k < 6; ++k) if(bnd[k] > j0 && bnd[k] < j1) j1 = bnd[k];
						for(int c = 0; c < C; ++c)
							ola_region(G, prev_lo + (size_t) c * G.Hp, cur_hi + (size_t) c * Q,
							           reinterpret_cast<TPcm*>(b.pcm) + chan_base + (uint64_t) c * st.pcm_frames, j0, j1, ola_tid, ola_n);
						j0 = j1;
					}
				} else {
					const uint32_t total = emit * (uint32_t) C;
					for(uint32_t e = (uint32_t) ola_tid; e < total; e += (uint32_t) ola_n) {
						uint32_t c, j;
						if(planar) { c = e / emit; j = e - c * emit; } else { j = e / (uint32_t) C; c = e - j * (uint32_t) C; }
						const float v = ola_one(G, prev_lo + (size_t) c * G.Hp, cur_hi + (size_t) c * Q, (int) j);
						const uint64_t fidx = pc.pcm_off + j;
						const uint64_t o = planar ? st.pcm_base + (uint64_t) c * st.pcm_frames + fidx : st.pcm_base + fidx * (uint64_t) C + c;
						reinterpret_cast<TPcm*>(b.pcm)[o] = pcm_value<TPcm>(v);
					}
				}
			}
			prev_valid = 1; prev_n = n; prev_right = rc; prev_lo = cur_lo;
		}
		// No barrier needed here: the next step starts with one; its stage 2 is the first reader of the curve blocks built
		// above and the first writer of T; Dhi and Dlo[buf^1] are not written again before two more barriers.
		cur = nxt;
		++step_idx;
	}
}

static uint32_t fused_threads(uint32_t max_channels, uint32_t max_blocksize) {
	// one 8-point work item per thread per pass for the long block: C * n/32 threads -> 128, 256 or 512
	const uint32_t want = max_channels * (max_blocksize / 32);
	if(want <= 128 && max_channels <= 2) return 128;
	if(want <= 256) return 256;
	return 512;
}

static void fused_layout(uint32_t max_channels, uint32_t max_blocksize, uint32_t min_blocksize, const uint32_t floor_cap[2],
                         uint32_t table_float2, FusedParams& P, uint32_t& threads, size_t& smem) {
	P.table_float2 = (table_float2 + 1u) & ~1u;
	threads = fused_threads(max_channels, max_blocksize);
	uint32_t group = max_blocksize / min_blocksize;
	if(group > 8) group = 8;
	if(group < 1) group = 1;
	P.group_short = group;
	P.floor_cap[0] = floor_cap[0]; P.floor_cap[1] = floor_cap[1];
	P.scratch_cap = floor_cap[0] > floor_cap[1] ? floor_cap[0] : floor_cap[1];
	P.slot_floats = max_channels * (max_blocksize / 2);
	const size_t long_bytes = (size_t) max_channels * CurveV3::bytes(floor_cap[1], max_blocksize / 8);
	const size_t short_bytes = (size_t) group * max_channels * CurveV3::bytes(floor_cap[0], min_blocksize / 8);
	// a setup with blocksize0 == blocksize1 runs every packet as a "short" step of one packet with the long geometry
	const size_t same_bytes = (size_t) max_channels * CurveV3::bytes(P.scratch_cap, max_blocksize / 8);
	size_t cb = long_bytes > short_bytes ? long_bytes : short_bytes;
	if(same_bytes > cb) cb = same_bytes;
	P.curve_bytes = (uint32_t) ((cb + 15) & ~(size_t) 15);
	const size_t slot = P.slot_floats;
	const size_t floats = slot + (slot + slot / 8) + slot + slot / 2;       // raw | T | Dlo[2] | Dhi
	smem = floats * sizeof(float) + P.curve_bytes + (size_t) P.table_float2 * sizeof(float2) + 128;
	if(P.scratch_cap > 32) smem += (size_t) (threads / 32) * floor_scratch_stride(P.scratch_cap);
}

size_t fused_smem_bytes(uint32_t max_channels, uint32_t max_blocksize, uint32_t min_blocksize, const uint32_t floor_cap[2],
                        uint32_t table_float2) {
	FusedParams P;
	uint32_t threads;
	size_t smem;
	fused_layout(max_channels, max_blocksize, min_blocksize, floor_cap, table_float2, P, threads, smem);
	return smem;
}

template <int kThreads, int kMinBlocks, bool kSpec, class TPcm>
static cudaError_t launch_variant(const FusedParams& P, uint32_t n_runs, size_t smem, cudaStream_t st) {
	cudaError_t e = cudaFuncSetAttribute(k_fused_synth<kThreads, kMinBlocks, kSpec, TPcm>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
	if(e != cudaSuccess) return e;
	// The twiddle / rotation / window tables (~15 KB for 256/2048) are read through L1 by every CTA: leave L1 enough
	// room for them instead of maximising resident CTAs (tuning knob: POV_SMEM_CARVEOUT = percent of the 228 KB).
	static const int carve = [] { const char* e = getenv("POV_SMEM_CARVEOUT"); return e ? atoi(e) : 100; }();
	cudaFuncSetAttribute(k_fused_synth<kThreads, kMinBlocks, kSpec, TPcm>, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
	k_fused_synth<kThreads, kMinBlocks, kSpec, TPcm><<<n_runs, kThreads, smem, st>>>(P);
	return cudaGetLastError();
}

template <class TPcm>
static cudaError_t launch_fused_as(const FusedParams& P, uint32_t threads, bool only_256_2048, uint32_t n_runs, size_t smem, cudaStream_t st) {
	if(threads == 128) return only_256_2048 ? launch_variant<128, 5, true, TPcm>(P, n_runs, smem, st) : launch_variant<128, 5, false, TPcm>(P, n_runs, smem, st);
	if(threads == 256) return only_256_2048 ? launch_variant<256, 2, true, TPcm>(P, n_runs, smem, st) : launch_variant<256, 2, false, TPcm>(P, n_runs, smem, st);
	return launch_variant<512, 1, false, TPcm>(P, n_runs, smem, st);
}

cudaError_t launch_fused(const DevBatchView& b, const DevRun* runs, uint32_t n_runs, uint32_t max_channels,
                         uint32_t max_blocksize, uint32_t min_blocksize, const uint32_t floor_cap[2], uint32_t table_float2,
                         bool only_256_2048, cudaStream_t st, uint64_t* launches) {
	if(n_runs == 0) return cudaSuccess;
	FusedParams P;
	uint32_t threads;
	size_t smem;
	fused_layout(max_channels, max_blocksize, min_blocksize, floor_cap, table_float2, P, threads, smem);
	P.b = b;
	P.runs = runs;
	if(smem > 227 * 1024) return cudaErrorInvalidConfiguration;
	const cudaError_t e = b.pcm_s16 ? launch_fused_as<int16_t>(P, threads, only_256_2048, n_runs, smem, st)
	                                : launch_fused_as<float>(P, threads, only_256_2048, n_runs, smem, st);
	if(launches) ++*launches;
	return e;
}

}  // namespace pov
