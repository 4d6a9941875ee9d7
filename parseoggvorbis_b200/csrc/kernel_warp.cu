// Production path for every pair of block sizes from {256, 512, 1024, 2048}: a persistent, warp-autonomous synthesis kernel.
//
//   floor1 unwrap/render -> nonzero propagate -> inverse coupling -> floor multiply -> inverse MDCT
//   -> window -> overlap-add -> PCM
// (reference: VorbisStream::parse_audio stages 4.3.2-4.3.7 + VorbisStreamDecodeState, src/ParseOggVorbis.hpp:
//  521-591, 1174-1180, 1213-1268, 1008-1059; the IMDCT contract is src/mdct.h:105.)
//
// Design (see DESIGN.md "kernel_warp"):
//   * One CTA per SM, 20 warps (96 registers each), resident for the whole launch. Every table a packet needs (inverse-dB table, window
//     slopes, FFT twiddles, DCT-IV rotations, floor neighbour tables, coupling programs) is brought
//     into shared memory ONCE per CTA with TMA bulk copies and shared by all warps.
//   * The unit of work is (run of <= 31 consecutive packets of one stream, one channel), taken from a global atomic
//     counter. ONE WARP owns it from the coded floor posts to the PCM stores: there is no CTA-wide barrier after the
//     prologue, only __syncwarp. A warp that needs other channels for the inverse coupling simply loads them too
//     (they are L1/L2 hits: the sibling warp reads the same lines), so warps never exchange data.
//   * The Q = n/4 point complex FFT of a long block lives in registers: 16 points per lane, three radix-8 passes,
//     two transposes through a warp-private shared buffer whose layouts make every access conflict free.
//     Spectra are read straight from HBM with 128-bit loads arranged so that the bins a pair of pre-rotated points and
//     their mirror images need arrive in the same lane (points 2q, 2q+1, Q-2-2q, Q-1-2q are handled together); the
//     post-rotation pairs butterflies k and Q-1-k to emit the D array with 64-bit stores. Smaller FFTs (Q = 64..256) use
//     Q/16 lanes each and are transformed several packets at a time.
//   * Overlap-add exploits the TDAC symmetry: one lane produces samples j..j+3 and n/2-4-j..n/2-1-j from the same four
//     128-bit shared loads, halving the shared-memory traffic of the window stage.
// HBM traffic is the algorithmic minimum: every spectrum is read once, every PCM sample written once (+ one halo
// packet per run).
#include "kernels.h"
#include "fft_core.cuh"
#include "pcm_out.cuh"
#include <stdlib.h>
#include <algorithm>
#include <type_traits>

namespace pov {
// POV_EXP_*: knock-out switches for timing experiments (tools/build_variant.sh, DESIGN.md §3): each removes one routine from the
// kernel so that its marginal cost can be read off the launch time. Such a build computes garbage and says so at compile time;
// the Makefile never sets them.
#if defined(POV_EXP_SAME_SPECTRUM) || defined(POV_EXP_NO_FLOOR_EVAL) || defined(POV_EXP_NO_UNWRAP) || defined(POV_EXP_NO_RECORDS) || \
    defined(POV_EXP_NO_SPECTRAL) || defined(POV_EXP_NO_FFT) || defined(POV_EXP_NO_OLA) || defined(POV_EXP_NO_PREFETCH)
#pragma message("k_warp_synth: timing-experiment build (POV_EXP_*): output is wrong by construction, never ship this object")
#endif
#ifdef POV_EXP_SAME_SPECTRUM      // timing experiment only (wrong output): every step reads the run's first spectrum, i.e. L1 / L2 hits
#define POV_EXP_SPEC_REL(x) 0
#else
#define POV_EXP_SPEC_REL(x) (x)
#endif

namespace wk {

#ifndef POV_WARP_WARPS
#define POV_WARP_WARPS 20
#endif
constexpr int kWarps = POV_WARP_WARPS;
constexpr int kThreads = kWarps * 32;
constexpr int kRegionF2 = 576;          // float2 slots of one FFT work region (long: 8*72, short: 8 FFTs * 72)
constexpr int kSlotF2 = kRegionF2 / 2;  // the work area of a warp is three half regions A | B | C: even steps transform in
                                        // A+B and leave their overlap half (D lo) in A, odd steps use B+C and leave it in C;
                                        // the other half (D hi, consumed by the same step's overlap-add) always lands in B
#ifndef POV_WARP_TMEM
#define POV_WARP_TMEM 1        // tensor memory: 0 = unused (round-1 layout), 1 = per-lane factor tables (default), 2 = tables + the FFT exchanges (fft512_tm; measured slower, DESIGN.md)
#endif
#ifndef POV_TM_SPLIT_LD
#define POV_TM_SPLIT_LD 1
#endif
#ifndef POV_TM_SPLIT_ST
#define POV_TM_SPLIT_ST 0
#endif
#ifndef POV_SPECTRAL_UNROLL
#define POV_SPECTRAL_UNROLL 1  // quads of the spectral stage unrolled per loop iteration (2 measured: see profiles/r02_ab_kernel_variants.log)
#endif
constexpr int kSpectralUnroll = POV_SPECTRAL_UNROLL;
#ifndef POV_OLA_UNROLL
#define POV_OLA_UNROLL 4
#endif
constexpr int kOlaUnroll = POV_OLA_UNROLL;   // iterations of ola_long_long unrolled (the hot code of 20 warps in different phases competes for the instruction cache)
#ifndef POV_WARP_PKT_CAP
#define POV_WARP_PKT_CAP 32
#endif
#ifndef POV_WARP_CURVE_MAX
#define POV_WARP_CURVE_MAX 2048
#endif
constexpr int kPktCap = POV_WARP_PKT_CAP;   // packets per run, halo included (<= 32: one lane per packet in unwrap_run)
constexpr uint32_t kCurveMax = POV_WARP_CURVE_MAX;   // bytes of curve blocks a warp may hold (bounds the short-packet group)
constexpr uint32_t FULL = 0xffffffffu;

struct __align__(16) WPkt { uint32_t meta, emit, pcm_rel; int32_t spec_rel; };   // 16 bytes; offsets relative to the run's first packet

struct Params {
	DevBatchView b;
	const DevRun* runs;
	uint32_t n_runs, n_items, C;
	uint32_t* counter;
	const FastTables* tabs;
	const float* slope[2];
	const float2* rot[2];
	const float2* tw8[2];
	const float2* fp[2];         // twiddles of the first radix-2 / radix-4 pass (block sizes 512 and 1024)
	const float* tmtab;          // [32][kTxTable] lane rows of the tensor-memory FFT (block size 2048; make_tm_lane_tables)
	unsigned char* dbg_floor;    // null, or [n_packets][C][72]: this kernel's own floor1 step-1 result per channel-packet (parity tests)
	uint32_t group_short;        // short packets per step (<= 8)
	uint32_t curve_bytes;        // per-warp curve area
	uint32_t short_curve_stride; // bytes of one short-block curve block
};

// ---- shared memory map (bytes), per pair of FFT sizes Q0 = blocksize0/4, Q1 = blocksize1/4 in {64, 128, 256, 512} ------
__host__ __device__ constexpr int tw8_count(int Q) { return Q == 512 ? 288 : 32; }      // float2 of make_fft_r8_tables: Q = 512 has the L = 512 and L = 64 passes
__host__ __device__ constexpr int fp_count(int Q) { return (Q == 128 || Q == 256) ? Q : 0; }   // first radix-2 / radix-4 pass (make_fft_pass_tables)
template <int Q0, int Q1> struct Map {
	static constexpr int kOffTabs   = 0;
	static constexpr int kOffInvDb  = kOffTabs + (int) sizeof(FastTables);
	static constexpr int kOffSlope0 = kOffInvDb + 1024 + 16;               // invdb[256] = 0.0f (curve of a channel multiplied by zero)
	static constexpr int kOffSlope1 = kOffSlope0 + 2 * Q0 * 4;
	static constexpr int kOffTw1    = kOffSlope1 + 2 * Q1 * 4;
	static constexpr int kOffTw0    = kOffTw1 + tw8_count(Q1) * 8;
	static constexpr int kOffRot1   = kOffTw0 + tw8_count(Q0) * 8;
	static constexpr int kOffRot0   = kOffRot1 + Q1 * 8;
	static constexpr int kOffFp1    = kOffRot0 + Q0 * 8;
	static constexpr int kOffFp0    = kOffFp1 + fp_count(Q1) * 8;
	static constexpr int kOffRecip  = kOffFp0 + fp_count(Q0) * 8;           // ceil(2^32 / d), d <= POV_FAST_MAX_X
	static constexpr int kOffBar    = kOffRecip + (POV_FAST_MAX_X + 4) * 4;      // mbarrier (8 bytes) | tensor-memory base address (4 bytes)
	static constexpr int kOffWarps  = kOffBar + 16;
	static_assert(kOffWarps % 16 == 0, "warp areas must stay 16-byte aligned");
};
constexpr int kOffInvDb = (int) sizeof(FastTables);    // the same for every geometry
constexpr int kFsStride = 36;           // per packet: final Y of every post in ascending-x order (uint8 x 32) + step2 mask (uint32)
constexpr int kWorkBytes = 3 * kSlotF2 * 8;
constexpr int kWarpFixedBytes = kWorkBytes + kPktCap * (int) sizeof(WPkt) + kPktCap * kFsStride;

extern __shared__ __align__(128) unsigned char g_smem[];     // the kernel's dynamic shared memory (map above)

// ---- mbarrier / TMA bulk copy (SASS: UBLKCP + SYNCS) ----------------------------------------------------------------
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
// Shared-memory arguments of the out-of-line routines travel as 32-bit shared-window addresses: inside the callee the
// pointer is rebuilt with a shared->generic conversion that the compiler folds, so every access is a plain LDS/STS
// (a generic pointer argument would cost a window-base subtraction per access).
template <class T> __device__ __forceinline__ T* sptr(uint32_t a) { return reinterpret_cast<T*>(__cvta_shared_to_generic((size_t) a)); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {   // TMA bulk prefetch (size multiple of 16)
	asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// ---- tensor memory (TMEM) as a second table store --------------------------------------------------------------------
// The rotation, twiddle and window factors a lane needs are the same for every packet (they depend on the lane's
// fixed place in the FFT only), so each lane keeps its own copy in ITS row of tensor memory (tcgen05.ld/st .32x32b:
// thread t <-> TMEM lane t of the warp's 32-lane quarter, registers <-> consecutive columns). tcgen05.ld does not go
// through the LSU / shared-memory data pipe that bounds this kernel: measured on B200 (tools/probes/tmem_probe.cu), 20
// warps read 268 B/clk/SM from TMEM alone and 122 B/clk/SM from TMEM *while* shared memory delivers its full
// 122-128 B/clk/SM. Column map of a quarter (floats), whole-warp FFT (Q = 512) only:
constexpr uint32_t kTmSpec = 0;     // 4 x [w[j] pair of quad q = lane + 32 m | pair of quad Q/2-1-q]      spectral stage
constexpr uint32_t kTmTw1  = 32;    // [W^j, W^2j, W^3j, W^4j] of butterflies lane and 63 - lane             pass over j2
constexpr uint32_t kTmTw2  = 48;    // [W^j, W^2j, W^3j, W^4j] of j0 = lane % 8                              pass over j1
constexpr uint32_t kTmRot  = 56;    // w[lane + 64 k], k < 8 | w[63 - lane + 64 k]                           post-rotation
constexpr uint32_t kTmWin  = 88;    // 4 x [slope[4 lane + 128 i ..+3] | slope[2Q - 4 - (4 lane + 128 i) ..+3]]  overlap-add
constexpr uint32_t kTmCols = 128;   // allocation (power of two >= 32)
template <uint32_t kCols>
__device__ __forceinline__ void tm_alloc(uint32_t* slot_smem) {      // one warp; the base address lands in shared memory
	asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_smem)), "n"(kCols) : "memory");
	asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tm_dealloc(uint32_t base) {
	asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tm_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tm_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tm_st8(uint32_t taddr, const float (&v)[8]) {
	asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
	             ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// Issue / complete split: the load is started early and its registers are only touched after tm_wait8, which carries the
// eight values as in-out operands so that no use can be scheduled above the wait.
__device__ __forceinline__ void tm_ld8(uint32_t taddr, float (&v)[8]) {
	asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
	             : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "r"(taddr));
}
__device__ __forceinline__ void tm_wait8(float (&v)[8]) {
	asm volatile("tcgen05.wait::ld.sync.aligned;"
	             : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]));
}

__device__ __forceinline__ void uncouple_f(float& m, float& a) {   // hpp:1220-1239, branch-free
	const float mv = m, av = a;
	const float t = (mv > 0.f) ? av : -av;
	const bool p = av > 0.f;
	const float diff = mv - t, sum = mv + t;
	a = p ? diff : mv;
	m = p ? mv : sum;
}
__device__ __forceinline__ void uncouple2(float2& m, float2& a) { uncouple_f(m.x, a.x); uncouple_f(m.y, a.y); }
// The same step when only one of the two results is needed (the last step of a channel's coupling program):
//   new magnitude = a > 0 ? m : m + t,  new angle = a > 0 ? m - t : m,  t = m > 0 ? a : -a
__device__ __forceinline__ float uncouple_mag(float m, float a) {
	const float v = fminf(a, 0.f);
	return m + ((m > 0.f) ? v : -v);
}
__device__ __forceinline__ float uncouple_ang(float m, float a) {
	const float v = fmaxf(a, 0.f);
	return m - ((m > 0.f) ? v : -v);
}

// ---- floor curve block (warp private, shared memory) ------------------------------------------------------------
// 8-byte segment record (a, b) of the segment [x0, x1) that starts at (x0, y0): the curve is y(x) = (a + x * b) >> 20 with
//   S = ceil(2^20 * |dy| / dx),  b = +S (ascending) or -S (descending, two's complement),
//   a = (y0 << 20) + (descending ? 2^20 - 1 : 0) - x0 * b        (all modulo 2^32; the true value stays below 2^31)
// i.e. y0 + floor(k S / 2^20) going up and y0 - floor(k S / 2^20) = ceil-form (y0 2^20 - k S + 2^20 - 1) >> 20 going down,
// k = x - x0, which are the reference's y0 +/- floor(k |dy| / dx) (Utils.hpp:122-137):
// Exact: with k < dx <= 2^10 the excess k * (S - 2^20 |dy|/dx) / 2^20 < dx / 2^20 <= 1/dx can never carry the
// fractional part of k*|dy|/dx (<= 1 - 1/dx) over the next integer. |dy| <= 1023 keeps S below 2^30. Curves that
// violate these bounds also violate hpp:587 and are reported through the packet status word (samples unspecified, as in
// the reference, which aborts the stream there). The flat tail after the last post is (y0 << 20, 0).
// Block layout: uint2 rec[cap] | uint2 tab[n/64] (rank table, see build_records).
// floor1 step 1 (amplitude unwrap, hpp:521-559) for ALL packets of a run at once: lane p owns packet p and walks its
// posts serially (the neighbour DAG makes the posts of one curve sequential, but the <= 32 curves of a run are
// independent). The final Y values leave as bytes in POST order, with the step2 flags as a bit mask over posts, 36 bytes per
// packet; the hpp:536 / hpp:587 checks are evaluated here with full-width values and reported per packet.
// scratch: [posts][32 lanes] uint16, aliasing the (idle) FFT work regions.
// kWide: floors of 33..64 posts (libvorbis' high-quality setups): 64-bit flag masks, 72-byte Y records (64 bytes + mask), so
// a run then holds at most 16 packets (the record area of a warp is the same 1152 bytes).
template <bool kWide>
__device__ __forceinline__ void unwrap_run(const FastTables* __restrict__ tb, const WPkt* __restrict__ wp, const pov_packet* __restrict__ pk0, int run_n, int ch,
                                        const uint16_t* __restrict__ ys, uint16_t* __restrict__ scratch, unsigned char* __restrict__ fs,
                                        uint32_t* __restrict__ status, uint32_t n0, uint32_t n1, int lane) {
	const bool have = lane < run_n;
	const uint32_t meta = have ? wp[lane].meta : 0u;
	const uint32_t mode = meta & 0xffu, used = meta >> 16;
	const uint32_t mapping = tb->mode_map[mode];
	const bool act = have && ((used >> ch) & 1u);
	const FastFloor* F = &tb->floors[tb->floor_of_ch[mapping][ch]];
	const int posts = act ? (int) F->n_posts : 0;
	const int maxposts = __reduce_max_sync(FULL, posts);
	if(maxposts == 0) return;
	// Y list of this channel inside the packet: after the lists of the used channels before it (hpp:498-518 order)
	uint64_t yo = have ? pk0[lane].ys_off : 0ull;
	for(int cc = 0; cc < ch; ++cc)
		if((used >> cc) & 1u) yo += tb->floors[tb->floor_of_ch[mapping][cc]].n_posts;
	const uint16_t* yp = ys + yo;
	const uint32_t range = F->range;
	using MaskT = typename std::conditional<kWide, uint64_t, uint32_t>::type;
	constexpr int kStride = kWide ? 72 : 36, kMaskAt = kWide ? 64 : 32;
	MaskT flags = 3u;
	MaskT over = 0u;                        // posts whose final Y, scaled by the multiplier, is >= 256 (hpp:587 once they are flagged)
	uint32_t bad = 0u;
	const uint32_t mult = F->multiplier;
	unsigned char* out = fs + lane * kStride;
	uint16_t* col = scratch + lane;
	// All coded values of this lane's packet first, eight independent loads at a time: one memory round trip per eight posts
	// instead of one per post inside the serial walk below. col[i] holds the coded value of post i until step i replaces it
	// by the final one (steps only read final values of posts before them).
	for(int i0 = 0; i0 < maxposts; i0 += 8) {
		uint16_t v[8];
#pragma unroll
		for(int k = 0; k < 8; ++k) v[k] = (i0 + k < posts) ? __ldg(yp + i0 + k) : (uint16_t) 0;
#pragma unroll
		for(int k = 0; k < 8; ++k) if(i0 + k < posts) col[(i0 + k) * 32] = v[k];
	}
	if(act) {
		const uint32_t a = col[0], b2 = col[32];
		out[0] = (unsigned char) min(a, 255u); out[1] = (unsigned char) min(b2, 255u);
		if(min(a * mult, 0xFFFFu) >= 256u) over |= 1u;
		if(min(b2 * mult, 0xFFFFu) >= 256u) over |= 2u;
	}
	for(int i = 2; i < maxposts; ++i) {
		if(i < posts) {
			const uint4 t = *reinterpret_cast<const uint4*>(F->post[i]);
			const uint32_t lo = t.x & 0xffu, hi = (t.x >> 8) & 0xffu;
			const uint32_t y0 = col[lo * 32], y1 = col[hi * 32];
			const uint32_t val = col[i * 32];
			const bool up = y1 >= y0;
			const uint32_t ady = up ? (y1 - y0) : (y0 - y1);
			// floor(ady * dxn / adx) by multiplication with m = ceil(2^32/adx): e = ady * dxn < 2^32 and m - 2^32/adx < 1 put the
			// estimate at most one above the quotient, never below (adx >= 2: a post lies strictly between its neighbours)
			const uint32_t e = ady * (t.y & 0xffffu), adx = t.y >> 16;
			uint32_t off = __umulhi(e, t.z);
			if(off * adx > e) --off;
			const uint32_t predicted = up ? y0 + off : y0 - off;
			if(predicted > range) bad |= POV_PKT_FLOOR_PREDICTED;
			const uint32_t high_room = range - predicted, low_room = predicted;
			const uint32_t room = min(high_room, low_room) * 2;
			uint32_t fin = predicted;
			if(val != 0) {
				flags |= ((MaskT) 1 << lo) | ((MaskT) 1 << hi) | ((MaskT) 1 << i);
				if(val >= room) fin = (high_room > low_room) ? val - low_room + predicted : predicted - val + high_room - 1;
				else fin = (val & 1) ? predicted - (val + 1) / 2 : predicted + val / 2;
			}
			fin = min(fin, 0xFFFFu);
			col[i * 32] = (uint16_t) fin;
			out[i] = (unsigned char) min(fin, 255u);
			if(min(fin * mult, 0xFFFFu) >= 256u) over |= (MaskT) 1 << i;
		}
	}
	// hpp:587 CHECK(floor[i] < 256) over the n bins the reference renders: segments are monotone, so the maxima are at rendered
	// end points. Every X of an ordinary floor lies below n (X <= n/2): then the flagged posts are all there is to check.
	// A floor with posts at or beyond n (legal, never produced by an encoder) takes the walk in ascending-x order below: posts
	// beyond n are not rendered, and the segment cut by bin n-1 needs y(n-1).
	const uint32_t n = tb->mode_flag[mode] ? n1 : n0;
	const bool beyond = act && F->xs_sorted[posts - 1] >= n;             // (low 16 bits: X; see build_records)
	if(!beyond) { if(over & flags) bad |= POV_PKT_FLOOR_RANGE; }
	if(__any_sync(FULL, beyond)) {
		uint32_t xp = 0u, ypv = 0u;
		bool havep = false;
		for(int sidx = 0; sidx < maxposts; ++sidx) {
			if(beyond && sidx < posts) {
				const uint32_t e = F->xs_sorted[sidx], si = e >> 16, x = e & 0xffffu;
				const uint32_t y = col[si * 32];
				if((flags >> si) & 1u) {
					const uint32_t yv = min(y * mult, 0xFFFFu);
					if(x < n && yv >= 256u) bad |= POV_PKT_FLOOR_RANGE;
					if(havep && xp < n && x > n - 1) {
						const bool down = yv < ypv;
						const uint32_t ady = down ? ypv - yv : yv - ypv, dx = x - xp;
						const uint32_t q = (uint32_t) (((uint64_t) (n - 1 - xp) * ady) / dx);
						if((down ? ypv - q : ypv + q) >= 256u) bad |= POV_PKT_FLOOR_RANGE;
					}
					xp = x; ypv = yv; havep = true;
				}
			}
		}
	}
	if(act) {
		*reinterpret_cast<MaskT*>(out + kMaskAt) = flags;
		if(bad) atomicOr(status + lane, bad);
	}
	__syncwarp();
}

// floor1 step 2 set-up (hpp:563-585) of one curve by one warp: segment records + rank table from the final Ys.
// Rank table: for every 32-bin word w of the curve, tab[w] = (bitmap of the flagged posts inside the word,
// number of flagged posts before the word - 1); the record that contains bin x is
//   tab[x >> 5].y + popc(tab[x >> 5].x & (0xFFFFFFFF >> (31 - (x & 31)))).
template <bool kWide>
__device__ __forceinline__ void build_records(const FastFloor* __restrict__ F, const unsigned char* __restrict__ fsp, unsigned char* __restrict__ curve,
                                           uint32_t rec_cap, uint32_t nwords, const uint32_t* __restrict__ recip, int lane) {
	using MaskT = typename std::conditional<kWide, uint64_t, uint32_t>::type;
	constexpr int kMaskAt = kWide ? 64 : 32, kRounds = kWide ? 2 : 1;
	const int posts = (int) F->n_posts;
	const MaskT flags = *reinterpret_cast<const MaskT*>(fsp + kMaskAt);     // step2 flags by post number
	uint2* rec = reinterpret_cast<uint2*>(curve);
	uint2* tab = rec + rec_cap;
	uint32_t* bits = reinterpret_cast<uint32_t*>(tab);          // word w at bits[2w] while the bitmap is collected
	if((uint32_t) lane < nwords) bits[2 * lane] = 0u;
	__syncwarp();
	// ascending-x order is made here, one lane per post (unwrap_run leaves post order): xs_sorted[p] = X | post number << 16 of
	// the p-th smallest X; the flag mask in that order is a ballot
	uint32_t xs_[kRounds], yb_[kRounds];
	bool f_[kRounds];
	MaskT mask = 0;
#pragma unroll
	for(int h = 0; h < kRounds; ++h) {
		const int p = lane + 32 * h;
		const bool have = p < posts;
		const uint32_t e = have ? F->xs_sorted[p] : 0u;
		xs_[h] = e & 0xffffu;
		yb_[h] = have ? fsp[e >> 16] : 0u;
		f_[h] = have && ((flags >> (e >> 16)) & 1u);
		mask |= (MaskT) __ballot_sync(FULL, f_[h]) << (32 * h);
	}
#pragma unroll
	for(int h = 0; h < kRounds; ++h) {                          // post p = lane + 32 h (ascending-x order)
		const int p = lane + 32 * h;
		const uint32_t yb = yb_[h];
		const uint32_t x0 = xs_[h];
		const bool f = f_[h];
		const uint32_t rank = kWide ? (uint32_t) __popcll((uint64_t) mask & (((uint64_t) 1 << p) - 1u)) : (uint32_t) __popc((uint32_t) mask & ((1u << p) - 1u));
		const uint32_t y0 = min(yb * F->multiplier, 1023u);
		// the next flagged post (the segment's right end): (x1, y1) straight from the tables, no shuffle
		const MaskT above = (p == (kWide ? 63 : 31)) ? (MaskT) 0 : (MaskT) (mask & ~(((MaskT) 2 << p) - 1u));
		const bool last = above == 0;
		const int np = last ? p : (kWide ? __ffsll((long long) above) : __ffs((int) above)) - 1;
		uint32_t x1, y1;
		if constexpr(kWide) {
			const uint32_t en = f ? F->xs_sorted[np] : 0u;
			x1 = en & 0xffffu; y1 = f ? min((uint32_t) fsp[en >> 16] * F->multiplier, 1023u) : 0u;
		} else {                                                  // one round: the next post is another lane's (x0, y0)
			const uint32_t pn = __shfl_sync(FULL, x0 | (y0 << 16), np);
			x1 = pn & 0xffffu; y1 = pn >> 16;
		}
		if(f) {
			uint2 r;
			if(last) r = make_uint2(y0 << 20, 0u);
			else {
				const bool down = y1 < y0;
				const uint32_t ady = down ? y0 - y1 : y1 - y0, adx = x1 - x0;
				// slope = ceil(2^20 |dy| / dx) = floor(N / dx), N = (|dy| << 20) + dx - 1 < 2^31: the table quotient is exact or one too big
				const uint32_t N = (ady << 20) + adx - 1u;
				uint32_t q = __umulhi(N, recip[adx]);
				if(q * adx > N) --q;
				if(adx == 1u) q = N;
				const uint32_t b = down ? 0u - q : q;
				r = make_uint2((y0 << 20) + (down ? 0xFFFFFu : 0u) - x0 * b, b);
			}
			rec[rank] = r;
			if((x0 >> 5) < nwords) atomicOr(&bits[2 * (x0 >> 5)], 1u << (x0 & 31u));
		}
	}
	__syncwarp();
	{
		const uint32_t w = ((uint32_t) lane < nwords) ? bits[2 * lane] : 0u;
		uint32_t incl = __popc(w);
#pragma unroll
		for(int o = 1; o < 32; o <<= 1) {
			const uint32_t v = __shfl_up_sync(FULL, incl, o);
			if(lane >= o) incl += v;
		}
		if((uint32_t) lane < nwords) bits[2 * lane + 1] = incl - __popc(w) - 1u;
	}
	__syncwarp();
}

// Curve block of a channel without a decoded floor: one flat segment at table index y (255 -> 1.0f: the reference
// skips the multiplication, hpp:1247; 256 -> 0.0f: multiplied by its zero-initialised floor buffer, hpp:1159).
__device__ __forceinline__ void flat_curve(unsigned char* __restrict__ curve, uint32_t rec_cap, uint32_t nwords, uint32_t y, int lane) {
	uint2* rec = reinterpret_cast<uint2*>(curve);
	uint2* tab = rec + rec_cap;
	if(lane == 0) rec[0] = make_uint2(y << 20, 0u);
	if((uint32_t) lane < nwords) tab[lane] = make_uint2(lane == 0 ? 1u : 0u, lane == 0 ? 0xFFFFFFFFu : 0u);
	__syncwarp();
}

// Four consecutive bins x..x+3 (x a multiple of 4) of a curve as inverse-dB table values (hpp:586-589): one rank-table
// and one record read for the quad; the bitmap tells which of the bins x+1..x+3 start a new segment.
__device__ __forceinline__ float4 curve_quad(const uint2* __restrict__ rec, const uint2* __restrict__ tab, uint32_t x,
                                             const float* __restrict__ invdb) {
	const uint2 t = tab[x >> 5];
	const uint32_t sh = x & 31u;                                         // <= 28
	uint32_t s = t.y + __popc(t.x & (0xFFFFFFFFu >> (31u - sh)));
	const uint32_t cross = t.x >> (sh + 1u);                             // bit b-1: bin x+b starts a segment (b = 1..3)
	uint2 r = rec[s];
	float out[4];
#pragma unroll
	for(int b = 0; b < 4; ++b) {
		if(b > 0 && ((cross >> (b - 1)) & 1u)) r = rec[++s];
		out[b] = invdb[(r.x + (x + (uint32_t) b) * r.y) >> 20];
	}
	return make_float4(out[0], out[1], out[2], out[3]);
}

// ---- FFT geometry ----------------------------------------------------------------------------------------------------
// The spectral stage leaves the pre-rotated points in natural order (point j at slot j of the FFT's buffer). Then
// Q = 512 = 8*8*8: j = 64 j2 + 8 j1 + j0, k = k0 + 8 k1 + 64 k2
//   pass 1 (over j2): lane l owns butterflies (j1,j0) = l and 63-l         in: j + 64 j2        out A1[k0*72 + 8 j1 + j0]
//   pass 2 (over j1): lane l owns butterflies (k0 = l/8 (+4), j0 = l%8)     in: A1               out A2[j0*66 + k0 + 8 k1]
//   pass 3 (over j0): lane l owns butterflies (k0 + 8 k1) = l and 63-l      in: A2               out D as float2[Q]
// Q = 64 = 8*8 (4 lanes per FFT, 8 FFTs per warp, FFT f at f*72): j = 8 j1 + j0, k = k0 + 8 k1
//   pass 1 (over j1): lane u owns butterflies j0 = u and 7-u                in: j0 + 8 j1        out A1[k0*9 + j0]
//   pass 2 (over j0): lane u owns butterflies k0 = u and 7-u                in: A1               out D as float2[Q] at f*64
// Every access of a pass is either contiguous over the lanes or hits 16 distinct 8-byte bank pairs per half warp.
// Every pass has one call site per block class and is inlined (no call ABI, strides become immediates); the hot loop of
// the 20 independently running warps is ~1700 instructions, just inside the 32 KB L1.5 instruction cache.
__device__ __forceinline__ void twiddle8w(float2* a, float2 w1, float2 w2, float2 w3, float2 w4);
__device__ __forceinline__ void twiddle8(float2* a, const float2* __restrict__ tw, int half) {   // tw: (W^j, W^2j); tw + half: (W^3j, W^4j)
	const float4 w12 = *reinterpret_cast<const float4*>(tw), w34 = *reinterpret_cast<const float4*>(tw + half);
	twiddle8w(a, make_float2(w12.x, w12.y), make_float2(w12.z, w12.w), make_float2(w34.x, w34.y), make_float2(w34.z, w34.w));
}
__device__ __forceinline__ void twiddle8w(float2* a, float2 w1, float2 w2, float2 w3, float2 w4) {
	a[1] = cmul(a[1], w1);
	a[2] = cmul(a[2], w2);
	a[3] = cmul(a[3], w3);
	a[4] = cmul(a[4], w4);
	a[5] = cmul(a[5], cmul(w4, w1));
	a[6] = cmul(a[6], cmul(w4, w2));
	a[7] = cmul(a[7], cmul(w4, w3));
}

// Radix-8 DIF pass of two butterflies per lane: inputs in*[m*sin], outputs out*[k*sout] (twiddled by tw*).
// All addresses are shared-window byte addresses, strides are in float2 units. Twiddles of butterfly j: (W^j, W^2j) at
// tw, (W^3j, W^4j) at tw + twhalf (the table keeps the two halves apart so that lanes read consecutive 16-byte words).
template <int kTm = 0>
__device__ __forceinline__ void r8_pass(uint32_t inA_, uint32_t inB_, int sin, uint32_t twA_, uint32_t twB_, int twhalf, uint32_t outA_, uint32_t outB_, int sout, uint32_t tm = 0) {
	const float2* inA = sptr<const float2>(inA_); const float2* inB = sptr<const float2>(inB_);
	float2* outA = sptr<float2>(outA_); float2* outB = sptr<float2>(outB_);
	float2 a[8], b[8];
	float wa[8], wb[8];               // kTm: twiddles from this lane's tensor-memory row (1: a and b differ, 2: shared by both)
	// the tensor-memory loads go out before the shared-memory ones: their latency (~100+ cycles) then runs under the first
	// butterfly (measured 2.203 against 2.208 ms; the same in the spectral stage costs a spill and 10 %)
	if constexpr(kTm != 0) tm_ld8(tm, wa);
	if constexpr(kTm == 1) tm_ld8(tm + 8, wb);
#pragma unroll
	for(int m = 0; m < 8; ++m) { a[m] = inA[m * sin]; b[m] = inB[m * sin]; }
	__syncwarp();
	dft8(a);
	if constexpr(kTm != 0) {
		tm_wait8(wa);
		twiddle8w(a, make_float2(wa[0], wa[1]), make_float2(wa[2], wa[3]), make_float2(wa[4], wa[5]), make_float2(wa[6], wa[7]));
	} else twiddle8(a, sptr<const float2>(twA_), twhalf);
	dft8(b);
	if constexpr(kTm == 1) {
		tm_wait8(wb);
		twiddle8w(b, make_float2(wb[0], wb[1]), make_float2(wb[2], wb[3]), make_float2(wb[4], wb[5]), make_float2(wb[6], wb[7]));
	} else if constexpr(kTm == 2) {
		twiddle8w(b, make_float2(wa[0], wa[1]), make_float2(wa[2], wa[3]), make_float2(wa[4], wa[5]), make_float2(wa[6], wa[7]));
	} else twiddle8(b, sptr<const float2>(twB_), twhalf);
#pragma unroll
	for(int k = 0; k < 8; ++k) { outA[k * sout] = a[k]; outB[k * sout] = b[k]; }
	__syncwarp();
}

// Last pass + post-rotation of butterflies kkA and kkB = J-1-kkA (rotA = rot + kkA, rotB = rot + kkB):
//   c[k] = X[k] * w[k];  D2[k] = (D[2k], D[2k+1]) = (Re c[k], -Im c[Q-1-k]);  Q-1-(kkA + J k2) = kkB + J (7-k2)
template <bool kTm = false>
__device__ __forceinline__ void last_pass(uint32_t inA_, uint32_t inB_, int sin, uint32_t rotA_, uint32_t rotB_, int J,
                                       uint32_t loA_, uint32_t loB_, uint32_t hiA_, uint32_t hiB_, uint32_t tm = 0) {
	const float2* inA = sptr<const float2>(inA_); const float2* inB = sptr<const float2>(inB_);
	const float2* rotA = sptr<const float2>(rotA_); const float2* rotB = sptr<const float2>(rotB_);
	float2* loA = sptr<float2>(loA_); float2* loB = sptr<float2>(loB_);      // D2[kk + J k2], k2 < 4  (D lo half: next packet's overlap)
	float2* hiA = sptr<float2>(hiA_); float2* hiB = sptr<float2>(hiB_);      // D2[kk + J k2], k2 >= 4 (D hi half), indexed by k2 - 4
	float2 a[8], b[8];
	float r0[8], r1[8];
	if constexpr(kTm) { tm_ld8(tm, r0); tm_ld8(tm + 8, r1); }      // (before the shared-memory loads: see r8_pass)
#pragma unroll
	for(int m = 0; m < 8; ++m) { a[m] = inA[m * sin]; b[m] = inB[m * sin]; }
	__syncwarp();
	if constexpr(kTm) {
		// rotation factors from this lane's tensor-memory row: [w[kkA + J k], k < 8 | w[kkB + J k], k < 8], 8 floats at a time
		dft8(a);
		tm_wait8(r0);
		tm_wait8(r1);
#pragma unroll
		for(int k = 0; k < 4; ++k) { a[k] = cmul(a[k], make_float2(r0[2 * k], r0[2 * k + 1])); a[k + 4] = cmul(a[k + 4], make_float2(r1[2 * k], r1[2 * k + 1])); }
		dft8(b);
		tm_ld8(tm + 16, r0);
		tm_ld8(tm + 24, r1);
		tm_wait8(r0);
		tm_wait8(r1);
#pragma unroll
		for(int k = 0; k < 4; ++k) { b[k] = cmul(b[k], make_float2(r0[2 * k], r0[2 * k + 1])); b[k + 4] = cmul(b[k + 4], make_float2(r1[2 * k], r1[2 * k + 1])); }
	} else {
		dft8(a);
		dft8(b);
#pragma unroll
		for(int k = 0; k < 8; ++k) {
			a[k] = cmul(a[k], rotA[J * k]);
			b[k] = cmul(b[k], rotB[J * k]);
		}
	}
#pragma unroll
	for(int k = 0; k < 4; ++k) {
		loA[J * k] = make_float2(a[k].x, -b[7 - k].y);
		loB[J * k] = make_float2(b[k].x, -a[7 - k].y);
		hiA[J * k] = make_float2(a[k + 4].x, -b[3 - k].y);
		hiB[J * k] = make_float2(b[k + 4].x, -a[3 - k].y);
	}
	__syncwarp();
}

// First pass of a Q = R*64 point FFT with R = 2 or 4 (block sizes 512 and 1024): radix-R DIF over the stride-64 index,
// x[j + 64 r] -> sub-FFT r' at T + 72 r' + j, twiddled by W_Q^(j r') (table: R factors per j, make_fft_pass_tables).
// Lane u of the Q/16 lanes of the FFT handles j = u + (Q/16) i, i < 1024/Q... i.e. 16/R butterflies of R points.
template <int R>
__device__ __forceinline__ void first_pass_small(uint32_t Tf_, uint32_t fp_, int u) {
	constexpr int LPF = 4 * R, NB = 16 / R;
	float2* T = sptr<float2>(Tf_);
	const float2* fp = sptr<const float2>(fp_);
	float2 x[NB][R];
#pragma unroll
	for(int i = 0; i < NB; ++i)
#pragma unroll
		for(int r = 0; r < R; ++r) x[i][r] = T[u + LPF * i + 64 * r];
	__syncwarp();
#pragma unroll
	for(int i = 0; i < NB; ++i) {
		const int j = u + LPF * i;
		if(R == 2) {
			dft2(x[i][0], x[i][1]);
			x[i][1] = cmul(x[i][1], fp[2 * j + 1]);
		} else {
			dft4(x[i][0], x[i][1], x[i][2], x[i][3]);
			const float4 w01 = *reinterpret_cast<const float4*>(fp + 4 * j), w23 = *reinterpret_cast<const float4*>(fp + 4 * j + 2);
			x[i][1] = cmul(x[i][1], make_float2(w01.z, w01.w));
			x[i][2] = cmul(x[i][2], make_float2(w23.x, w23.y));
			x[i][3] = cmul(x[i][3], make_float2(w23.z, w23.w));
		}
#pragma unroll
		for(int r = 0; r < R; ++r) T[72 * r + j] = x[i][r];
	}
	__syncwarp();
}

// ---- lane <-> register exchanges of the 512-point FFT through tensor memory ------------------------------------------
// tcgen05.st .32x32b writes register i of thread t to (TMEM lane t, column i); tcgen05.ld .16x256b hands thread t the
// elements (lane 16 I + t/4 + 8 h, column 8 k + 2 (t%4) + b) as register 4 k + 2 h + b (I = which 16-lane half: two
// instructions) — maps measured on B200 by tools/probes/tmem_probe.cu. One store + two loads therefore move two lane bits
// into the register index and two register bits into the lane index: a 4 x 4 transpose between lane groups and registers
// that never touches shared memory or the LSU pipe. Which register goes to which column is free (it is only a naming of
// registers), so the bits that leave can be any function of the register index; the FFT below sends them XORed with a bit
// that stays behind, which is what puts the outputs k and Q-1-k into the same lane at the end (see fft512_tm).
__device__ __forceinline__ void tm_st32(uint32_t taddr, const float (&c)[32]) {
	asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
	             :: "r"(taddr), "f"(c[0]), "f"(c[1]), "f"(c[2]), "f"(c[3]), "f"(c[4]), "f"(c[5]), "f"(c[6]), "f"(c[7]), "f"(c[8]), "f"(c[9]), "f"(c[10]), "f"(c[11]), "f"(c[12]), "f"(c[13]), "f"(c[14]), "f"(c[15]), "f"(c[16]), "f"(c[17]), "f"(c[18]), "f"(c[19]), "f"(c[20]), "f"(c[21]), "f"(c[22]), "f"(c[23]), "f"(c[24]), "f"(c[25]), "f"(c[26]), "f"(c[27]), "f"(c[28]), "f"(c[29]), "f"(c[30]), "f"(c[31]) : "memory");
}
__device__ __forceinline__ void tm_ld16(uint32_t taddr, float (&r)[16]) {
	asm volatile("tcgen05.ld.sync.aligned.16x256b.x4.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
	             : "=f"(r[0]), "=f"(r[1]), "=f"(r[2]), "=f"(r[3]), "=f"(r[4]), "=f"(r[5]), "=f"(r[6]), "=f"(r[7]), "=f"(r[8]), "=f"(r[9]), "=f"(r[10]), "=f"(r[11]), "=f"(r[12]), "=f"(r[13]), "=f"(r[14]), "=f"(r[15]) : "r"(taddr));
}
__device__ __forceinline__ void tm_st16(uint32_t taddr, const float* c) {
	asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
	             :: "r"(taddr), "f"(c[0]), "f"(c[1]), "f"(c[2]), "f"(c[3]), "f"(c[4]), "f"(c[5]), "f"(c[6]), "f"(c[7]), "f"(c[8]), "f"(c[9]), "f"(c[10]), "f"(c[11]), "f"(c[12]), "f"(c[13]), "f"(c[14]), "f"(c[15]) : "memory");
}
__device__ __forceinline__ void tm_ld16h(uint32_t taddr, float (&r)[8]) {        // 16 lanes x 16 columns
	asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
	             : "=f"(r[0]), "=f"(r[1]), "=f"(r[2]), "=f"(r[3]), "=f"(r[4]), "=f"(r[5]), "=f"(r[6]), "=f"(r[7]) : "r"(taddr));
}
__device__ __forceinline__ void tm_wait32(float (&a)[16], float (&b)[16]) {
	asm volatile("tcgen05.wait::ld.sync.aligned;"
	             : "+f"(a[0]), "+f"(a[1]), "+f"(a[2]), "+f"(a[3]), "+f"(a[4]), "+f"(a[5]), "+f"(a[6]), "+f"(a[7]), "+f"(a[8]), "+f"(a[9]), "+f"(a[10]), "+f"(a[11]), "+f"(a[12]), "+f"(a[13]), "+f"(a[14]), "+f"(a[15]), "+f"(b[0]), "+f"(b[1]), "+f"(b[2]), "+f"(b[3]), "+f"(b[4]), "+f"(b[5]), "+f"(b[6]), "+f"(b[7]), "+f"(b[8]), "+f"(b[9]), "+f"(b[10]), "+f"(b[11]), "+f"(b[12]), "+f"(b[13]), "+f"(b[14]), "+f"(b[15]));
}
// column (in complex units, 0..15) that complex register `reg` is stored to before exchange kX:
//   kX = 1: registers 2 k0 + j0            -> (r, j0 | k0_0 ^ r, k0_1 ^ r), r = k0_2
//   kX = 2, 3: registers 8 d1 + 4 r + 2 j0 + d0 (d = output digit of the radix-4 pass just done) -> (r, j0 | d1 ^ r, d0 ^ r)
template <int kX> __host__ __device__ constexpr int tm_colmap(int reg) {
	if(kX == 1) {
		const int k0 = reg >> 1, j0 = reg & 1, r = k0 >> 2;
		return (r << 3) | (j0 << 2) | (((k0 & 1) ^ r) << 1) | (((k0 >> 1) & 1) ^ r);
	}
	const int d1 = reg >> 3, r = (reg >> 2) & 1, j0 = (reg >> 1) & 1, d0 = reg & 1;
	return (r << 3) | (j0 << 2) | ((d1 ^ r) << 1) | (d0 ^ r);
}
template <int kX>
__device__ __forceinline__ void tm_exchange(uint32_t xa, float2 (&v)[16]) {
	float c[32];
#pragma unroll
	for(int reg = 0; reg < 16; ++reg) { c[2 * tm_colmap<kX>(reg)] = v[reg].x; c[2 * tm_colmap<kX>(reg) + 1] = v[reg].y; }
#if POV_TM_SPLIT_ST
	tm_st16(xa, c);
	tm_st16(xa + 16u, c + 16);
#else
	tm_st32(xa, c);
#endif
#ifndef POV_TM_NOFENCE
	tm_wait_st();
#endif
	__syncwarp();
#if POV_TM_SPLIT_LD
	// four loads of 16 lanes x 16 columns: complex register 8 I + 4 cg + 2 k + h <- column group cg (two 256-bit atoms each)
	float q0[8], q1[8], q2[8], q3[8];
	tm_ld16h(xa, q0);
	tm_ld16h(xa + 16u, q1);
	tm_ld16h(xa + (16u << 16), q2);
	tm_ld16h(xa + (16u << 16) + 16u, q3);
	tm_wait8(q0); tm_wait8(q1); tm_wait8(q2); tm_wait8(q3);
#pragma unroll
	for(int i = 0; i < 4; ++i) {
		v[i] = make_float2(q0[2 * i], q0[2 * i + 1]); v[4 + i] = make_float2(q1[2 * i], q1[2 * i + 1]);
		v[8 + i] = make_float2(q2[2 * i], q2[2 * i + 1]); v[12 + i] = make_float2(q3[2 * i], q3[2 * i + 1]);
	}
#else
	float r0[16], r1[16];
	tm_ld16(xa, r0);
	tm_ld16(xa + (16u << 16), r1);
	tm_wait32(r0, r1);
#pragma unroll
	for(int i = 0; i < 8; ++i) { v[i] = make_float2(r0[2 * i], r0[2 * i + 1]); v[8 + i] = make_float2(r1[2 * i], r1[2 * i + 1]); }
#endif
}

// Column map of a lane's table row for the exchange variant (host_tables.cpp: make_tm_lane_tables):
constexpr uint32_t kTxSpec = 0, kTxTw1 = 32, kTxTw2 = 48, kTxTw3 = 64, kTxRot = 80, kTxWin = 112, kTxTable = 144;
constexpr uint32_t kTxCols = 512;          // tables + one 32-column exchange area per warp of a lane quarter (5 x 32)

// 512-point FFT + post-rotation with all three exchanges in tensor memory. In: the pre-rotated points in natural order at T
// (shared memory). Out: D2[k] = (D[2k], D[2k+1]) = (Re c[k], -Im c[Q-1-k]), c = X w, lo half (k < 256) at `lo`, hi half at
// `hi`, each half in STORAGE order: the quad (D2[2i], D2[2i+1]) of true index tq = i lives at quad
//   sq = [tq6][tq3][tq1][tq0][tq2][tq5][tq4]       (bits of tq, most significant first)
// which makes the 128-bit stores below and the 128-bit loads of the overlap-add conflict free (model: tools/model).
//   pass 1: radix 8 over j8 j7 j6, registers 2 m + j0 <- points 64 m + 2 lane + j0 (eight 128-bit loads)
//   pass 2: radix 4 over j5 j4;  pass 3: radix 4 over j3 j2;  pass 4: radix 4 over j1 j0
__device__ __forceinline__ void fft512_tm(uint32_t Ts, int lane, uint32_t tm, uint32_t xa, uint32_t lo, uint32_t hi) {
	const float4* T4 = sptr<const float4>(Ts);
	float2 v[16];
#pragma unroll
	for(int m = 0; m < 8; ++m) {
		const float4 q = T4[32 * m + lane];
		v[2 * m] = make_float2(q.x, q.y); v[2 * m + 1] = make_float2(q.z, q.w);
	}
	__syncwarp();
	{
		float2 a[8], b[8];
		float wa[8], wb[8];
#pragma unroll
		for(int m = 0; m < 8; ++m) { a[m] = v[2 * m]; b[m] = v[2 * m + 1]; }
		dft8(a);
		tm_ld8(tm + kTxTw1, wa);
		tm_wait8(wa);
		twiddle8w(a, make_float2(wa[0], wa[1]), make_float2(wa[2], wa[3]), make_float2(wa[4], wa[5]), make_float2(wa[6], wa[7]));
		dft8(b);
		tm_ld8(tm + kTxTw1 + 8, wb);
		tm_wait8(wb);
		twiddle8w(b, make_float2(wb[0], wb[1]), make_float2(wb[2], wb[3]), make_float2(wb[4], wb[5]), make_float2(wb[6], wb[7]));
#pragma unroll
		for(int k = 0; k < 8; ++k) { v[2 * k] = a[k]; v[2 * k + 1] = b[k]; }
	}
	tm_exchange<1>(xa, v);
	// registers 8 I + 4 r + 2 j0 + h, (I, h) = (j5, j4): radix 4 over d = 2 I + h in place, then W_64^(e d), e = (j3 j2 j1 j0)
#pragma unroll
	for(int pass = 0; pass < 2; ++pass) {
#pragma unroll
		for(int k = 0; k < 4; ++k) dft4(v[2 * k], v[2 * k + 1], v[8 + 2 * k], v[9 + 2 * k]);
#pragma unroll
		for(int j0 = 0; j0 < 2; ++j0) {          // twiddles (W^e, W^2e, W^3e, -) of the butterflies with this j0 (k = 2 r + j0)
			float w[8];
			tm_ld8(tm + (pass == 0 ? kTxTw2 : kTxTw3) + 8u * j0, w);
			tm_wait8(w);
#pragma unroll
			for(int k = j0; k < 4; k += 2) {
				v[2 * k + 1] = cmul(v[2 * k + 1], make_float2(w[0], w[1]));
				v[8 + 2 * k] = cmul(v[8 + 2 * k], make_float2(w[2], w[3]));
				v[9 + 2 * k] = cmul(v[9 + 2 * k], make_float2(w[4], w[5]));
			}
		}
		if(pass == 0) tm_exchange<2>(xa, v); else tm_exchange<3>(xa, v);
	}
	// registers 8 j1 + 4 r + 2 j0 + h: radix 4 over (j1 j0) in place -> R = 8 k3_1 + 4 r + 2 k3_0 + h, h = k0_0 ^ r
#pragma unroll
	for(int r = 0; r < 2; ++r)
#pragma unroll
		for(int h = 0; h < 2; ++h) dft4(v[4 * r + h], v[4 * r + 2 + h], v[8 + 4 * r + h], v[8 + 4 * r + 2 + h]);
	// post-rotation c[k] = X[k] w[k] (factors in register order from the lane's row)
#pragma unroll
	for(int g = 0; g < 4; ++g) {
		float w[8];
		tm_ld8(tm + kTxRot + 8u * g, w);
		tm_wait8(w);
#pragma unroll
		for(int i = 0; i < 4; ++i) v[4 * g + i] = cmul(v[4 * g + i], make_float2(w[2 * i], w[2 * i + 1]));
	}
	// D2[k] = (Re c[k], -Im c[Q-1-k]); Q-1-k sits in register R ^ 14 of the same lane; registers R, R+1 (h = 0, 1) hold k, k+1
	// (r = 0) or k+1, k (r = 1): one 128-bit store per pair. Lane part of the storage quad: [t3][r][t4][t2][t1][t0] ^ r...r
	const uint32_t ls = (uint32_t) (((lane & 8) << 2) | ((lane & 16) >> 1) | (lane & 7));
	const uint32_t a0 = ls * 16u, a1 = ((ls ^ 0x2Fu) | 0x10u) * 16u;
#pragma unroll
	for(int k31 = 0; k31 < 2; ++k31)
#pragma unroll
		for(int r = 0; r < 2; ++r)
#pragma unroll
			for(int k30 = 0; k30 < 2; ++k30) {
				const int R0 = 8 * k31 + 4 * r + 2 * k30;
				const int e0 = r ? R0 + 1 : R0, e1 = r ? R0 : R0 + 1;
				const float4 out = make_float4(v[e0].x, -v[e0 ^ 14].y, v[e1].x, -v[e1 ^ 14].y);
				*sptr<float4>((k31 ? hi : lo) + (uint32_t) (k30 << 6) * 16u + (r ? a1 : a0)) = out;
			}
	__syncwarp();
}

// All FFT passes of one step for block class Q (compile time): natural-order points at Tf -> D halves at lo / hi.
//   Q = 64:            r8 over j1                    -> A1[k0*9 + j0]              -> last pass (J = 8)
//   Q = 128, 256:      radix-R first pass (R = Q/64) -> R sub-FFTs at T + 72 r'
//                      r8 over j1 inside each        -> A2[j0*(J+2) + r' + R k1]   -> last pass (J = 8R)
//   Q = 512:           r8 over j2 (R = 8)            -> A1[k0*72 + j], then as above
// f = FFT index inside the warp (0 for Q = 512), u = lane inside the FFT, tw / fp / rot = shared-window table addresses.
template <int Q, bool kTm = false>
__device__ __forceinline__ void fft_passes(uint32_t Tfs, int u, uint32_t tws, uint32_t fps, uint32_t rots, uint32_t lo, uint32_t hi, uint32_t tm = 0) {
	static_assert(!kTm || Q == 512, "tensor-memory tables are laid out for the whole-warp FFT");
	constexpr int R = Q / 64, J = Q / 8;
	const uint32_t uu = (uint32_t) u, u2 = (uint32_t) J - 1u - uu;
	if constexpr(R == 1) {
		r8_pass(Tfs + uu * 8, Tfs + u2 * 8, 8, tws + uu * 16, tws + u2 * 16, 16, Tfs + uu * 8, Tfs + u2 * 8, 9);
		last_pass(Tfs + uu * 72, Tfs + u2 * 72, 1, rots + uu * 8, rots + u2 * 8, J, lo + uu * 8, lo + u2 * 8, hi + uu * 8, hi + u2 * 8);
	} else {
		constexpr int S2 = J + 2;
		if constexpr(R == 8) r8_pass<kTm ? 1 : 0>(Tfs + uu * 8, Tfs + u2 * 8, 64, tws + uu * 16, tws + u2 * 16, 128, Tfs + uu * 8, Tfs + u2 * 8, 72, tm + kTmTw1);
		else first_pass_small<R>(Tfs, fps, u);
		// pass over j1 inside the sub-FFTs: lane owns (r' = u/8, j0 = u%8) and (r' + R/2, j0); its twiddles are the L = 64 pass
		constexpr uint32_t kTw64 = (R == 8) ? 256u : 0u;
		const uint32_t j0 = uu & 7u, rp = uu >> 3;
		r8_pass<kTm ? 2 : 0>(Tfs + (rp * 72 + j0) * 8, Tfs + ((rp + R / 2) * 72 + j0) * 8, 8, tws + (kTw64 + j0 * 2) * 8, tws + (kTw64 + j0 * 2) * 8, 16,
		                     Tfs + (j0 * S2 + rp) * 8, Tfs + (j0 * S2 + rp + R / 2) * 8, R, tm + kTmTw2);
		last_pass<kTm>(Tfs + uu * 8, Tfs + u2 * 8, S2, rots + uu * 8, rots + u2 * 8, J, lo + uu * 8, lo + u2 * 8, hi + uu * 8, hi + u2 * 8, tm + kTmRot);
	}
}

// Spectral stage of the FFT this lane belongs to: nonzero propagate + inverse coupling + floor multiply + DCT-IV
// pre-rotation. Lane u handles points u + J*m and their mirrors Q-1-(u + J*m), m = 0..7: the bins (2j, 2j+1) and
// (M-2-2j, M-1-2j) arrive with two 64-bit loads per channel and feed both points.
// src*: spectra ([n/2] floats) of the local channels of this lane's packet (src0 = this warp's channel);
// fmode: 0 evaluate the curve, 1 multiply by 1 (hpp:1247 skipped), 2 multiply by 0.
template <int NL, bool GEN>
__device__ __forceinline__ void spectral_stage(const float* __restrict__ base, int o0, int o1, int o2, int o3, uint32_t curve_, uint32_t rec_cap,
                                               uint32_t rot_, int Q, uint32_t Tf_, int u, uint32_t cp_, uint32_t tm) {
	// Lane u handles the quads q = u + (Q/16) m, m = 0..3: bins 4q..4q+3 and M-4-4q..M-1-4q arrive with two 128-bit loads
	// per channel and yield the points 2q, 2q+1 and their mirrors Q-2-2q, Q-1-2q (two 128-bit stores, natural order).
	const int LPF = Q >> 4, M = 2 * Q;
	const uint2* rec = sptr<const uint2>(curve_);
	const uint2* tab = rec + rec_cap;
	const float* invdb = reinterpret_cast<const float*>(g_smem + kOffInvDb);
	const float4* rot4 = sptr<const float4>(rot_);        // rot4[j/2] = (w[j], w[j+1]), j even
	float4* T4 = sptr<float4>(Tf_);
	const FastCouple* cp = sptr<const FastCouple>(cp_);
	// coupling program in registers (the loop below stores to shared memory, so nothing would be hoisted otherwise)
	const int nsteps = (NL > 1) ? (int) cp->nsteps : 0;
	const bool last_mag = (NL > 1 && nsteps > 0) ? (cp->sm[nsteps - 1] == 0) : false;
	const int off[4] = {o0, o1, o2, o3};
	// (no hand-written register prefetch: with 20 warps per SM the loads of a whole iteration issued together hide
	// their latency behind the other warps, and the 16 registers it would cost are what keeps the kernel spill free)
	// this lane's first quad and its mirror, as pointers: a load is then one 32-bit offset and one wide multiply-add
	const float* const lane_lo = base + 4 * u;
	const float* const lane_hi = base + (M - 4 - 4 * u);
#pragma unroll kSpectralUnroll
	for(int m = 0; m < 4; ++m) {
		const int q = u + LPF * m, d = 4 * LPF * m;
		float4 lo[NL], hi[NL];
#pragma unroll
		for(int i = 0; i < NL; ++i) {
			lo[i] = __ldg(reinterpret_cast<const float4*>(lane_lo + (off[i] + d)));
			hi[i] = __ldg(reinterpret_cast<const float4*>(lane_hi + (off[i] - d)));
		}
		// the floor evaluation needs none of the loaded values: it runs while the loads are in flight
#ifdef POV_EXP_NO_FLOOR_EVAL      // timing experiment only (wrong output)
		const float4 fl = make_float4(1.f, 1.f, 1.f, 1.f), fh = fl;
#else
		const float4 fl = curve_quad(rec, tab, (uint32_t) (4 * q), invdb);
		const float4 fh = curve_quad(rec, tab, (uint32_t) (M - 4 - 4 * q), invdb);
#endif
		if(NL > 1 && !GEN) {
			// single coupling step between two channels: only this warp's channel (local index 0) is needed
			if(last_mag) {
				lo[0].x = uncouple_mag(lo[0].x, lo[NL - 1].x); lo[0].y = uncouple_mag(lo[0].y, lo[NL - 1].y);
				lo[0].z = uncouple_mag(lo[0].z, lo[NL - 1].z); lo[0].w = uncouple_mag(lo[0].w, lo[NL - 1].w);
				hi[0].x = uncouple_mag(hi[0].x, hi[NL - 1].x); hi[0].y = uncouple_mag(hi[0].y, hi[NL - 1].y);
				hi[0].z = uncouple_mag(hi[0].z, hi[NL - 1].z); hi[0].w = uncouple_mag(hi[0].w, hi[NL - 1].w);
			} else {
				lo[0].x = uncouple_ang(lo[NL - 1].x, lo[0].x); lo[0].y = uncouple_ang(lo[NL - 1].y, lo[0].y);
				lo[0].z = uncouple_ang(lo[NL - 1].z, lo[0].z); lo[0].w = uncouple_ang(lo[NL - 1].w, lo[0].w);
				hi[0].x = uncouple_ang(hi[NL - 1].x, hi[0].x); hi[0].y = uncouple_ang(hi[NL - 1].y, hi[0].y);
				hi[0].z = uncouple_ang(hi[NL - 1].z, hi[0].z); hi[0].w = uncouple_ang(hi[NL - 1].w, hi[0].w);
			}
		} else if(NL > 1) {
			for(int st = 0; st < nsteps; ++st) {
				const int mi = cp->sm[st], ai = cp->sa[st];
				float4 ml = lo[0], mh = hi[0], al = lo[0], ah = hi[0];
#pragma unroll
				for(int i = 0; i < NL; ++i) {
					if(i == mi) { ml = lo[i]; mh = hi[i]; }
					if(i == ai) { al = lo[i]; ah = hi[i]; }
				}
				uncouple_f(ml.x, al.x); uncouple_f(ml.y, al.y); uncouple_f(ml.z, al.z); uncouple_f(ml.w, al.w);
				uncouple_f(mh.x, ah.x); uncouple_f(mh.y, ah.y); uncouple_f(mh.z, ah.z); uncouple_f(mh.w, ah.w);
#pragma unroll
				for(int i = 0; i < NL; ++i) {
					if(i == mi) { lo[i] = ml; hi[i] = mh; }
					if(i == ai) { lo[i] = al; hi[i] = ah; }
				}
			}
		}
		// hpp:1252 residue *= floor (one rounding each)
		const float l0 = __fmul_rn(lo[0].x, fl.x), l1 = __fmul_rn(lo[0].y, fl.y), l2 = __fmul_rn(lo[0].z, fl.z), l3 = __fmul_rn(lo[0].w, fl.w);
		const float h0 = __fmul_rn(hi[0].x, fh.x), h1 = __fmul_rn(hi[0].y, fh.y), h2 = __fmul_rn(hi[0].z, fh.z), h3 = __fmul_rn(hi[0].w, fh.w);
		// t[j] = (X[2j] + i X[M-1-2j]) * w[j] for j = 2q, 2q+1 and Q-2-2q, Q-1-2q
		float4 wl, wh;
		if(tm) {                      // tm != 0: whole-warp FFT, rotation factors from this lane's tensor-memory row (warp uniform)
			float wr[8];
			tm_ld8(tm + kTmSpec + 8u * (uint32_t) m, wr);
			tm_wait8(wr);
			wl = make_float4(wr[0], wr[1], wr[2], wr[3]); wh = make_float4(wr[4], wr[5], wr[6], wr[7]);
		} else { wl = rot4[q]; wh = rot4[(Q >> 1) - 1 - q]; }
		const float2 t0 = cmul(make_float2(l0, h3), make_float2(wl.x, wl.y));
		const float2 t1 = cmul(make_float2(l2, h1), make_float2(wl.z, wl.w));
		const float2 t2 = cmul(make_float2(h0, l3), make_float2(wh.x, wh.y));
		const float2 t3 = cmul(make_float2(h2, l1), make_float2(wh.z, wh.w));
		T4[q] = make_float4(t0.x, t0.y, t1.x, t1.y);
		T4[(Q >> 1) - 1 - q] = make_float4(t2.x, t2.y, t3.x, t3.y);
	}
}

// picks the instantiation: <1> no coupling, <2,false> the stereo case (one step), generic otherwise. kMaxNL (1, 2 or 4) is
// the largest channel set any coupling program of the setup needs: variants beyond it are not even compiled in.
template <int kMaxNL>
__device__ __forceinline__ void spectral_dispatch(const FastCouple* cp, const float* base, int half, uint32_t curve_, uint32_t rec_cap,
                                                  uint32_t rot_, int Q, uint32_t Tf_, int u, uint32_t tm) {
	const int o0 = (int) cp->ch[0] * half, o1 = (int) cp->ch[1] * half, o2 = (int) cp->ch[2] * half, o3 = (int) cp->ch[3] * half;
	const uint32_t cps = smem_u32(cp);
	const int nl = cp->nl;
	if(kMaxNL == 1 || nl == 1) spectral_stage<1, false>(base, o0, o0, o0, o0, curve_, rec_cap, rot_, Q, Tf_, u, cps, tm);
	else if(kMaxNL >= 2 && nl == 2 && cp->nsteps == 1) spectral_stage<2, false>(base, o0, o1, o0, o0, curve_, rec_cap, rot_, Q, Tf_, u, cps, tm);
	else if(kMaxNL >= 2 && nl == 2) spectral_stage<2, true>(base, o0, o1, o0, o0, curve_, rec_cap, rot_, Q, Tf_, u, cps, tm);
	else if(kMaxNL >= 3 && nl == 3) spectral_stage<3, true>(base, o0, o1, o2, o0, curve_, rec_cap, rot_, Q, Tf_, u, cps, tm);
	else if(kMaxNL >= 3) spectral_stage<4, true>(base, o0, o1, o2, o3, curve_, rec_cap, rot_, Q, Tf_, u, cps, tm);
}

// ---- overlap-add ---------------------------------------------------------------------------------------------------
struct OlaGeom {
	int Hp, H;          // quarter sizes: Hp = n_prev/4, H = n/4 (= length of the lo / hi halves of D)
	int shift;          // index in the current frame of the chunk's first sample: n/4 - n_prev/4
	int lb, lc;         // current frame: left slope begins at lb, has length lc
	int rbp, pr;        // previous frame, relative to its second half: falling slope begins at rbp, has length pr
	const float* slL;   // rising slope table of length lc
	const float* slR;   // rising slope table of length pr (read mirrored)
	bool pperm, cperm;  // the previous / current frame's D halves are in the storage order of fft512_tm
};
// float index inside a D half of fft512_tm's storage order (quad bits [6][3][1][0][2][5][4] of the true quad index)
__device__ __forceinline__ int dperm(int idx) {
	return (idx & 0x113) | ((idx & 0x20) << 2) | ((idx & 0x0C) << 3) | ((idx & 0xC0) >> 4);
}

// One sample of the chunk:  out = prev[n_prev/2 + j] * w_prev + cur[j + shift] * w_cur   (hpp:1008-1017 in gather form)
// plo = lo half of the previous frame's D, chi = hi half of the current frame's D.
__device__ __forceinline__ float ola_one(const OlaGeom& G, const float* __restrict__ plo, const float* __restrict__ chi, int j) {
	float acc = 0.f;
	if(j < G.rbp + G.pr) {
		const int ip = (j < G.Hp) ? G.Hp - 1 - j : j - G.Hp;
		const float y = -plo[G.pperm ? dperm(ip) : ip];
		const float w = (j >= G.rbp) ? G.slR[G.pr - 1 - (j - G.rbp)] : 1.f;
		acc = __fadd_rn(acc, __fmul_rn(y, w));
	}
	const int ic = j + G.shift;
	if(ic >= G.lb) {
		const int ii = (ic < G.H) ? ic : 2 * G.H - 1 - ic;
		const float yy = chi[G.cperm ? dperm(ii) : ii];
		const float y = (ic < G.H) ? yy : -yy;
		const float w = (ic < G.lb + G.lc) ? G.slL[ic - G.lb] : 1.f;
		acc = __fadd_rn(acc, __fmul_rn(y, w));
	}
	return acc;
}

// Long block after a long block, both slopes long: every sample has both terms and both windows. Lane produces
// out[j..j+3] and out[1020-j..1023-j] (j < 512) from the same four vectors (TDAC symmetry of both frames and windows).
// kTm = 1: window slopes from tensor memory. kTm = 2: also the D halves in the storage order of fft512_tm — lane L reads
// storage quad 32 i + L (and its mirror 127 - that), which holds the true quad tq = [sq6][sq1][sq0][sq5][sq2][sq4][sq3].
template <int Q, bool kStrided, int kTm, class TPcm>
__device__ __forceinline__ void ola_long_long(const float* __restrict__ plo, const float* __restrict__ chi, const float* __restrict__ sl,
                                              TPcm* __restrict__ dst, int stride, int lane, uint32_t tm, float* __restrict__ stage = nullptr) {
	// n = 4Q: the chunk has 2Q samples, half of them (Q) below the centre; 8 samples per lane and iteration
#pragma unroll kOlaUnroll
	for(int i = 0; i < Q / 128; ++i) {
		const int js = 4 * lane + 128 * i;                                   // position in the stored halves
		const int j = (kTm == 2) ? 4 * ((((lane & 3) << 4) | (lane & 4) | (lane >> 3)) + ((i & 2) << 5) + ((i & 1) << 3)) : js;   // true position
		float ww[8];
		const float4 p = *reinterpret_cast<const float4*>(plo + (Q - 4) - js);
		const float4 c = *reinterpret_cast<const float4*>(chi + js);
		float4 wa, wb;
		if constexpr(kTm != 0) {      // window slopes from this lane's tensor-memory row
			tm_ld8(tm + (kTm == 2 ? kTxWin : kTmWin) + 8u * (uint32_t) i, ww);
			tm_wait8(ww);
			wa = make_float4(ww[0], ww[1], ww[2], ww[3]); wb = make_float4(ww[4], ww[5], ww[6], ww[7]);
		} else {
			wa = *reinterpret_cast<const float4*>(sl + j);
			wb = *reinterpret_cast<const float4*>(sl + (2 * Q - 4) - j);
		}
		float4 o1, o2;
		o1.x = __fadd_rn(__fmul_rn(-p.w, wb.w), __fmul_rn(c.x, wa.x));
		o1.y = __fadd_rn(__fmul_rn(-p.z, wb.z), __fmul_rn(c.y, wa.y));
		o1.z = __fadd_rn(__fmul_rn(-p.y, wb.y), __fmul_rn(c.z, wa.z));
		o1.w = __fadd_rn(__fmul_rn(-p.x, wb.x), __fmul_rn(c.w, wa.w));
		o2.x = __fadd_rn(__fmul_rn(-p.x, wa.w), __fmul_rn(-c.w, wb.x));
		o2.y = __fadd_rn(__fmul_rn(-p.y, wa.z), __fmul_rn(-c.z, wb.y));
		o2.z = __fadd_rn(__fmul_rn(-p.z, wa.y), __fmul_rn(-c.y, wb.z));
		o2.w = __fadd_rn(__fmul_rn(-p.w, wa.x), __fmul_rn(-c.x, wb.w));
		if constexpr(!kStrided) {
			pcm_store4_cs(dst + j, o1);
			pcm_store4_cs(dst + (2 * Q - 4) - j, o2);
		} else {
			// interleaved PCM: sample j of this channel lives at dst[j * channels]. The lane's four samples would be four stores
			// 16 * channels bytes apart from the next lane's; through a 512-byte stage (the step's curve block, dead by now) every
			// store instruction covers 32 consecutive frames instead, i.e. a quarter of the sectors.
			if constexpr(kTm == 2) {          // (fft512_tm's storage order: lanes are not frame-consecutive; plain strided stores)
				TPcm* a = dst + (size_t) j * stride;
				TPcm* b = dst + (size_t) ((2 * Q - 4) - j) * stride;
				a[0] = pcm_value<TPcm>(o1.x); a[stride] = pcm_value<TPcm>(o1.y); a[2 * stride] = pcm_value<TPcm>(o1.z); a[3 * stride] = pcm_value<TPcm>(o1.w);
				b[0] = pcm_value<TPcm>(o2.x); b[stride] = pcm_value<TPcm>(o2.y); b[2 * stride] = pcm_value<TPcm>(o2.z); b[3 * stride] = pcm_value<TPcm>(o2.w);
				continue;
			}
			*reinterpret_cast<float4*>(stage + 4 * lane) = o1;
			__syncwarp();
			TPcm* a = dst + (size_t) (128 * i + lane) * stride;
#pragma unroll
			for(int k = 0; k < 4; ++k) a[(size_t) (32 * k) * stride] = pcm_value<TPcm>(stage[32 * k + lane]);
			__syncwarp();
			*reinterpret_cast<float4*>(stage + 124 - 4 * lane) = o2;
			__syncwarp();
			TPcm* b = dst + (size_t) ((2 * Q - 128) - 128 * i + lane) * stride;
#pragma unroll
			for(int k = 0; k < 4; ++k) b[(size_t) (32 * k) * stride] = pcm_value<TPcm>(stage[32 * k + lane]);
			__syncwarp();
		}
	}
}

// Curve mode of channel c of a packet: 0 = decoded curve, 1 = untouched (multiply by 1), 2 = multiply by the
// reference's zero-initialised floor buffer (channel became "used" through the propagate rule, hpp:1174-1180, 1159, 1247).
__device__ __forceinline__ int curve_mode(const FastTables* tb, uint32_t mapping, uint32_t used, int c) {
	if((used >> c) & 1u) return 0;
	uint32_t prop = used;
	const int nc = tb->ncoup[mapping];
	for(int k = 0; k < nc; ++k) {
		const uint32_t m = tb->cmag[mapping][k], a = tb->cang[mapping][k];
		if(((prop >> m) | (prop >> a)) & 1u) prop |= (1u << m) | (1u << a);
	}
	return ((prop >> c) & 1u) ? 2 : 1;
}

// kWide: a floor of 33..64 posts is reachable (compile time, so that the common case keeps its constants: 32 records per long
// curve, 36-byte Y records, 32-bit step-2 masks); instantiated with the generic coupling class only.
// TPcm: float, or int16_t for POV_PCM_S16 (converted at the store, pcm_out.cuh). A template parameter like kPlanar: a run-time
// flag of comparable weight (the 64-post floors) measured 6.5 % slower (DESIGN.md §3).
template <int Q0, int Q1, bool kPlanar, class TPcm, int kMaxNL, bool kWide>
__global__ void __launch_bounds__(kThreads, 1) k_warp_synth(const Params P) {
	using M = Map<Q0, Q1>;
	constexpr int N0 = 4 * Q0, N1 = 4 * Q1;              // block sizes
	constexpr int LPF0 = Q0 / 16, LPF1 = Q1 / 16;        // lanes per FFT
	unsigned char* const smem = g_smem;
	const FastTables* tb = reinterpret_cast<const FastTables*>(smem + M::kOffTabs);
	const float* s_slope0 = reinterpret_cast<const float*>(smem + M::kOffSlope0);
	const float* s_slope1 = reinterpret_cast<const float*>(smem + M::kOffSlope1);
	const float2* s_tw1 = reinterpret_cast<const float2*>(smem + M::kOffTw1);
	const float2* s_tw0 = reinterpret_cast<const float2*>(smem + M::kOffTw0);
	const float2* s_rot1 = reinterpret_cast<const float2*>(smem + M::kOffRot1);
	const float2* s_rot0 = reinterpret_cast<const float2*>(smem + M::kOffRot0);
	uint32_t* s_recip = reinterpret_cast<uint32_t*>(smem + M::kOffRecip);
	uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + M::kOffBar);

	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const DevBatchView& b = P.b;

	// ---- prologue: tables -> shared memory (TMA bulk copies) ----
	if(threadIdx.x == 0) {
		mbar_init(s_bar, 1);
		mbar_fence_init();
		constexpr uint32_t total = (uint32_t) sizeof(FastTables) + 1024u + 2u * Q0 * 4u + 2u * Q1 * 4u + tw8_count(Q1) * 8u + tw8_count(Q0) * 8u +
		                           Q1 * 8u + Q0 * 8u + fp_count(Q1) * 8u + fp_count(Q0) * 8u;
		mbar_expect_tx(s_bar, total);
		tma_bulk_g2s(smem + M::kOffTabs, P.tabs, (uint32_t) sizeof(FastTables), s_bar);
		tma_bulk_g2s(smem + M::kOffInvDb, b.inv_db, 1024u, s_bar);
		tma_bulk_g2s(smem + M::kOffSlope0, P.slope[0], 2u * Q0 * 4u, s_bar);
		tma_bulk_g2s(smem + M::kOffSlope1, P.slope[1], 2u * Q1 * 4u, s_bar);
		tma_bulk_g2s(smem + M::kOffTw1, P.tw8[1], tw8_count(Q1) * 8u, s_bar);
		tma_bulk_g2s(smem + M::kOffTw0, P.tw8[0], tw8_count(Q0) * 8u, s_bar);
		tma_bulk_g2s(smem + M::kOffRot1, P.rot[1], Q1 * 8u, s_bar);
		tma_bulk_g2s(smem + M::kOffRot0, P.rot[0], Q0 * 8u, s_bar);
		if(fp_count(Q1)) tma_bulk_g2s(smem + M::kOffFp1, P.fp[1], fp_count(Q1) * 8u, s_bar);
		if(fp_count(Q0)) tma_bulk_g2s(smem + M::kOffFp0, P.fp[0], fp_count(Q0) * 8u, s_bar);
	}
	if(threadIdx.x < 4) reinterpret_cast<float*>(smem + M::kOffInvDb + 1024)[threadIdx.x] = 0.f;
	for(uint32_t d = threadIdx.x; d <= POV_FAST_MAX_X; d += kThreads)
		s_recip[d] = (d < 2) ? 0xFFFFFFFFu : (uint32_t) ((0x100000000ull + d - 1) / d);
	// Tensor memory (one CTA per SM, so the allocation never waits): per-lane factor tables of the whole-warp (512-point) FFT and,
	// in mode 2, one exchange area per warp. POV_WARP_TMEM: 0 = unused, 1 = tables, 2 = tables + FFT exchanges (fft512_tm).
	constexpr int kTm = (Q1 == 512) ? POV_WARP_TMEM : 0;
	constexpr uint32_t kCols = (kTm == 2) ? kTxCols : kTmCols;
	uint32_t* s_tmbase = reinterpret_cast<uint32_t*>(smem + M::kOffBar + 8);
	if constexpr(kTm != 0) { if(warp == kWarps - 1) tm_alloc<kCols>(s_tmbase); tm_fence_before(); }
	__syncthreads();
	mbar_wait(s_bar, 0);
	uint32_t tmw = 0, tmx = 0;           // this warp's window into tensor memory (lanes 32 (warp % 4) .. +31) and its exchange area
	if constexpr(kTm != 0) {
		tm_fence_after();
		tmw = *s_tmbase + ((uint32_t) ((warp & 3) * 32) << 16);
		tmx = tmw + kTxTable + 32u * (uint32_t) (warp >> 2);
		if(warp < 4) {                   // one warp per lane quarter writes the rows (thread t <-> TMEM lane t)
			if constexpr(kTm == 2) {
				const float4* row = reinterpret_cast<const float4*>(P.tmtab + (size_t) lane * kTxTable);
				for(uint32_t c = 0; c < kTxTable; c += 8) {
					const float4 x = __ldg(row + c / 4), y = __ldg(row + c / 4 + 1);
					const float v[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
					tm_st8(tmw + c, v);
				}
			} else {
				const float4* rot4 = reinterpret_cast<const float4*>(s_rot1);
				const float4* tw4 = reinterpret_cast<const float4*>(s_tw1);
				const float4* sl4 = reinterpret_cast<const float4*>(s_slope1);
				auto put2 = [&](uint32_t col, float4 x, float4 y) {
					const float v[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
					tm_st8(tmw + col, v);
				};
				const int l2 = 63 - lane, j0 = lane & 7;
				for(int m = 0; m < 4; ++m) put2(kTmSpec + 8u * m, rot4[lane + 32 * m], rot4[(Q1 >> 1) - 1 - (lane + 32 * m)]);
				put2(kTmTw1, tw4[lane], tw4[lane + 64]);
				put2(kTmTw1 + 8, tw4[l2], tw4[l2 + 64]);
				put2(kTmTw2, tw4[128 + j0], tw4[136 + j0]);
				for(int h = 0; h < 2; ++h) {
					const int kk = h ? l2 : lane;
					for(int g = 0; g < 2; ++g) {
						const float2 r0 = s_rot1[kk + 64 * (4 * g)], r1 = s_rot1[kk + 64 * (4 * g + 1)], r2 = s_rot1[kk + 64 * (4 * g + 2)], r3 = s_rot1[kk + 64 * (4 * g + 3)];
						put2(kTmRot + 16u * h + 8u * g, make_float4(r0.x, r0.y, r1.x, r1.y), make_float4(r2.x, r2.y, r3.x, r3.y));
					}
				}
				for(int i = 0; i < 4; ++i) put2(kTmWin + 8u * i, sl4[lane + 32 * i], sl4[(Q1 >> 1) - 1 - (lane + 32 * i)]);
			}
			tm_wait_st();
		}
		tm_fence_before();
		__syncthreads();
		tm_fence_after();
	}

	// ---- warp-private areas ----
	const uint32_t warp_bytes = (uint32_t) kWarpFixedBytes + P.curve_bytes;
	unsigned char* wbase = smem + M::kOffWarps + (size_t) warp * warp_bytes;
	float2* slotA = reinterpret_cast<float2*>(wbase);        // work area: three half regions A | B | C (see kSlotF2)
	WPkt* wp = reinterpret_cast<WPkt*>(wbase + kWorkBytes);
	unsigned char* fs = wbase + kWorkBytes + kPktCap * (int) sizeof(WPkt);
	unsigned char* curves = wbase + kWarpFixedBytes;

	const int C = (int) P.C;
	constexpr bool planar = kPlanar;       // PCM layout is a template parameter: the interleaved address arithmetic stays out of the planar kernel

	for(;;) {
		// (claiming the next item one run ahead, to take the atomic's round trip off the path, was measured slower: 2.274 against
		// 2.232 ms — the items held back at the tail cost more than the latency that four other warps per scheduler already hide)
		uint32_t item = 0;
		if(lane == 0) item = atomicAdd(P.counter, 1u);
		item = __shfl_sync(FULL, item, 0);
		if(item >= P.n_items) break;
		const uint32_t run_idx = item / (uint32_t) C;
		const int ch = (int) (item - run_idx * (uint32_t) C);
		const DevRun run = P.runs[run_idx];
		const int run_n = (int) run.n_packets;        // <= kPktCap
		__syncwarp();
		const pov_packet* pk0 = b.packets + run.first_packet;
		const uint64_t spec0 = b.spec_off[run.first_packet], pcm0 = pk0->pcm_off;
		if(lane < run_n) {
			const pov_packet pk = pk0[lane];
			WPkt w;
			w.meta = (uint32_t) pk.mode | ((uint32_t) pk.window_flags << 8) | ((uint32_t) pk.floor_used << 16);
			w.emit = pk.emit_frames;
			w.pcm_rel = (uint32_t) (pk.pcm_off - pcm0);                                       // host guarantees 32-bit deltas
			w.spec_rel = (int32_t) (int64_t) (b.spec_off[run.first_packet + lane] - spec0);
			wp[lane] = w;
		}
		const float* spec_base = b.spectra + spec0;
		// where this run's first chunk starts in the PCM arena, for this channel (one pointer instead of the stream record):
		//   planar:      pcm_base + ch * pcm_frames + frame,  + 1 per frame;   interleaved: pcm_base + frame * C + ch,  + C per frame
		TPcm* out0;
		bool first_of_stream;                   // the run starts at its stream's first packet, which only primes the overlap (hpp:1021)
		{
			const pov_stream st = b.streams[pk0->stream];
			out0 = reinterpret_cast<TPcm*>(b.pcm) + (planar ? st.pcm_base + (uint64_t) ch * st.pcm_frames + pcm0 : st.pcm_base + pcm0 * (uint64_t) C + (uint64_t) ch);
			first_of_stream = run.first_packet == st.first_packet;
		}
		__syncwarp();
#ifndef POV_EXP_NO_UNWRAP         // (defined: timing experiment only, wrong output)
		unwrap_run<kWide>(tb, wp, pk0, run_n, ch, b.ys, reinterpret_cast<uint16_t*>(slotA), fs, b.status + run.first_packet, (uint32_t) N0, (uint32_t) N1, lane);
#endif
		if(P.dbg_floor) {
			// parity hook: the production kernel's integer floor stage as it is — final Ys (ascending x, clamped to 255) and the
			// step-2 mask of every packet of the run — copied out for comparison with the reference's "floor1 final_ys" /
			// "floor1 step2_flag" (pov_batch_fetch_fast_floor). 72 bytes per channel-packet: 64 Ys | 64-bit mask.
			constexpr int kS = kWide ? 72 : kFsStride, kM = kWide ? 64 : 32;
			if(lane < run_n) {
				unsigned char* d = P.dbg_floor + ((size_t) (run.first_packet + lane) * C + ch) * 72;
				const unsigned char* src = fs + lane * kS;
				const uint32_t meta = wp[lane].meta;
				const FastFloor* Fd = &tb->floors[tb->floor_of_ch[tb->mode_map[meta & 0xffu]][ch]];
				const int np = ((meta >> 16) >> ch) & 1u ? (int) Fd->n_posts : 0;
				unsigned long long fl = 0, sm = 0;
				for(int i = 0; i < (kWide ? 8 : 4); ++i) fl |= (unsigned long long) src[kM + i] << (8 * i);
				for(int i = 0; i < 64; ++i) {                 // the records hold post order; the dump is in ascending-x order
					const uint32_t si = i < np ? Fd->xs_sorted[i] >> 16 : 0u;
					d[i] = i < np ? src[si] : (unsigned char) 0;
					if(i < np && ((fl >> si) & 1ull)) sm |= 1ull << i;
				}
				for(int i = 0; i < 8; ++i) d[64 + i] = (unsigned char) (sm >> (8 * i));
			}
			__syncwarp();
		}

		// State carried from step to step, packed into one register (the FFT in between needs every register it can get):
		//   bit 0 step parity (which half regions the step uses) | bit 1 a previous frame exists | bit 2 it was a long block |
		//   bit 3 its right slope is long | bit 4 its D lo half is in fft512_tm's storage order | bit 5 the run starts at its
		//   stream's first packet | bits 8.. index of the step's first packet in the run.
		// The previous frame's D lo half always sits in the survivor slot of the previous step (slot A or C by its parity).
		uint32_t stt = first_of_stream ? 32u : 0u;
		while((int) (stt >> 8) < run_n) {
			const int first = (int) (stt >> 8);
			const int par = (int) (stt & 1u);
			const uint32_t meta0 = wp[first].meta;
			const uint32_t mode = meta0 & 0xffu;
			const int flag = tb->mode_flag[mode];
			const uint32_t mapping = tb->mode_map[mode];
			const FastCouple* cp = &tb->couple[mapping][ch];
			const FastFloor* F = &tb->floors[tb->floor_of_ch[mapping][ch]];
			float2* T = slotA + par * kSlotF2;                       // A+B or B+C
			float2* surv = slotA + par * (2 * kSlotF2);              // A or C: where this step's last D lo half stays
			float2* slotB = slotA + kSlotF2;
			// A long FFT of Q1 < 512 points needs fewer than 32 lanes: such long packets are transformed 512/Q1 at a time, exactly
			// like the groups of short packets (D of FFT f packed at T + Q f, last lo half moved to the survivor slot).
			constexpr bool kLongGrouped = LPF1 < 32;
			constexpr int kGroupLong = 32 / LPF1;
			const bool grouped = !flag || kLongGrouped;
			int count = 1;
			{
				const int cap = flag ? (kLongGrouped ? kGroupLong : 1) : (int) P.group_short;
				while(count < cap && first + count < run_n && (wp[first + count].meta & 0xffu) == mode) ++count;
			}

			// pull the next step's spectra towards L2 while this step computes: one 128-byte line per lane and channel
			if(first + count < run_n) {
				const WPkt& nw = wp[first + count];
				const uint32_t nmode = nw.meta & 0xffu;
				const uint32_t nhalf = tb->mode_flag[nmode] ? 2u * Q1 : 2u * Q0;
				const FastCouple* ncp = &tb->couple[tb->mode_map[nmode]][ch];
#ifndef POV_EXP_NO_PREFETCH
				if(lane < (int) ncp->nl) prefetch_l2_bulk(spec_base + nw.spec_rel + (int) (ncp->ch[lane] * nhalf), nhalf * 4u);
#endif
			}
			// ================= one 2048-sample packet or a group of smaller packets: Q/16 lanes per FFT, same code for all classes,
			//                   geometry in registers (256/2048: the whole warp is one 512-point FFT, or eight 64-point FFTs) ====
			const int Qs = flag ? Q1 : Q0;
			const int lpf = flag ? LPF1 : LPF0;
			// lpf is a power of two; lanes whose FFT index f is beyond the group (f >= count) still walk the passes on their own
			// (unused) part of the work area, so that every lane reaches the warp barriers
			const int u = lane & (lpf - 1);
			const int f = lane / lpf;                    // 0 for a whole-warp FFT
			constexpr uint32_t kLongCap = kWide ? 64u : 32u;              // records of a long curve (= FastTables::long_posts_cap)
			constexpr uint32_t kLongCurveBytes = kLongCap * 8u + (uint32_t) (Q1 / 16) * 8u;
			const uint32_t cstride = flag ? (kLongGrouped ? kLongCurveBytes : 0u) : P.short_curve_stride, rcap = flag ? kLongCap : tb->short_posts_cap,
			               nwords = (uint32_t) Qs / 16u;
			for(int g = 0; g < count; ++g) {
				const int md = curve_mode(tb, mapping, wp[first + g].meta >> 16, ch);
				unsigned char* cv = curves + (size_t) g * cstride;
#ifdef POV_EXP_NO_RECORDS         // timing experiment only (wrong output)
				if(md == 0) flat_curve(cv, rcap, nwords, 200u, lane);
#else
				if(md == 0) build_records<kWide>(F, fs + (first + g) * (kWide ? 72 : kFsStride), cv, rcap, nwords, s_recip, lane);
#endif
				else flat_curve(cv, rcap, nwords, md == 1 ? 255u : 256u, lane);
			}
			// FFT buffer of FFT f: Q/64 sub-FFT rows of 72 slots (one row for Q = 64)
			const uint32_t Ts = smem_u32(T), Tfs = Ts + (uint32_t) f * (uint32_t) ((Qs >> 6) * 72 * 8);
			const uint32_t rots = smem_u32(flag ? s_rot1 : s_rot0), tws = smem_u32(flag ? s_tw1 : s_tw0);
			// (a whole-warp FFT has f = 0 in every lane: the call below is warp uniform there, which the tensor-memory loads need)
#ifdef POV_EXP_NO_SPECTRAL        // timing experiment only (wrong output)
			if(f < count && P.n_items == 0xffffffffu)
#else
			if(f < count)
#endif
				spectral_dispatch<kMaxNL>(cp, spec_base + POV_EXP_SPEC_REL(wp[first + f].spec_rel), 2 * Qs, smem_u32(curves + (size_t) f * cstride), rcap, rots, Qs, Tfs, u,
				                          (kTm != 0 && flag) ? tmw : 0u);
			__syncwarp();
			// last pass output: long: lo half -> survivor slot, hi half -> slot B; short: D of FFT f packed at T + Q0 f (lo | hi)
#ifdef POV_EXP_NO_FFT             // timing experiment only (wrong output)
			if(P.n_items != 0xffffffffu) { __syncwarp(); }
			else
#endif
			if(flag && !kLongGrouped) {
				if constexpr(kTm == 2) fft512_tm(Ts, lane, tmw, tmx, smem_u32(surv), smem_u32(slotB));
				else fft_passes<Q1, kTm == 1>(Tfs, u, tws, smem_u32(smem + M::kOffFp1), rots, smem_u32(surv), smem_u32(slotB), tmw);
			}
			else if(flag) {
				const uint32_t lo = Ts + (uint32_t) f * (uint32_t) (Q1 * 8);
				fft_passes<Q1>(Tfs, u, tws, smem_u32(smem + M::kOffFp1), rots, lo, lo + (uint32_t) (Q1 / 2 * 8));
			} else {
				const uint32_t lo = Ts + (uint32_t) f * (uint32_t) (Q0 * 8);
				fft_passes<Q0>(Tfs, u, tws, smem_u32(smem + M::kOffFp0), rots, lo, lo + (uint32_t) (Q0 / 2 * 8));
			}

			// ================= window + overlap-add + emit (hpp:1008-1059 in gather form) =================
			const int n = flag ? N1 : N0, Q = n / 4;
			const float* Dstep = reinterpret_cast<const float*>(T);
			int prev_valid = (int) ((stt >> 1) & 1u), prev_n = (stt & 4u) ? N1 : N0, prev_right = (stt & 8u) ? N1 / 2 : N0 / 2;
			bool prev_perm = (stt & 16u) != 0;
			const float* prev_lo = reinterpret_cast<const float*>(slotA + (par ^ 1) * (2 * kSlotF2));
			for(int g = 0; g < count; ++g) {
				const WPkt& w = wp[first + g];
				const uint32_t wflags = (w.meta >> 8) & 0xffu, emit = w.emit;
				// hpp:844-847: short blocks always use blocksize0 slopes; long blocks follow their own prev/next flags
				const int lc = (flag && (wflags & 1u)) ? N1 / 2 : N0 / 2;
				const int rc = (flag && (wflags & 2u)) ? N1 / 2 : N0 / 2;
				const float* cur_lo = !grouped ? reinterpret_cast<const float*>(surv) : Dstep + (size_t) g * 2 * Q;
				const float* cur_hi = !grouped ? reinterpret_cast<const float*>(slotB) : cur_lo + Q;
				const bool emits = prev_valid && emit > 0 && !((stt & 32u) && first + g == 0);
#ifdef POV_EXP_NO_OLA
				if(emits && P.n_items == 0xffffffffu) {
#else
				if(emits) {
#endif
					TPcm* const dst = out0 + (planar ? (size_t) w.pcm_rel : (size_t) w.pcm_rel * (size_t) C);
					if(flag && prev_n == N1 && lc == N1 / 2 && prev_right == N1 / 2 && emit == (uint32_t) (N1 / 2) && (!planar || ((size_t) dst & (4 * sizeof(TPcm) - 1)) == 0)) {
						if constexpr(planar) ola_long_long<Q1, false, kTm>(prev_lo, cur_hi, s_slope1, dst, 1, lane, tmw);
						else ola_long_long<Q1, true, kTm>(prev_lo, cur_hi, s_slope1, dst, C, lane, tmw, reinterpret_cast<float*>(curves));
					} else {
						OlaGeom G;
						G.Hp = prev_n / 4; G.H = Q;
						G.shift = Q - prev_n / 4;
						G.lc = lc; G.lb = Q - lc / 2;
						G.pr = prev_right; G.rbp = prev_n / 4 - prev_right / 2;
						G.slL = (lc == N1 / 2) ? s_slope1 : s_slope0;
						G.slR = (prev_right == N1 / 2) ? s_slope1 : s_slope0;
						G.pperm = (kTm == 2) && prev_perm; G.cperm = (kTm == 2) && flag && !kLongGrouped;     // (compile-time false unless kTm == 2)
						for(uint32_t j = (uint32_t) lane; j < emit; j += 32u) {
							const float v = ola_one(G, prev_lo, cur_hi, (int) j);
							dst[planar ? (size_t) j : (size_t) j * (size_t) C] = pcm_value<TPcm>(v);
						}
					}
				}
				prev_valid = 1; prev_n = n; prev_right = rc; prev_lo = cur_lo;
				prev_perm = (kTm == 2) && flag && !kLongGrouped;
			}
			if(grouped && prev_lo != reinterpret_cast<const float*>(surv)) {
				// grouped step: move the last packet's D lo half (Q/2 float2) into the survivor slot (ranges may overlap:
				// every lane reads all of its elements before anyone writes)
				constexpr int kPer0 = (Q0 / 2 + 31) / 32, kPer1 = kLongGrouped ? (Q1 / 2 + 31) / 32 : 1;
				constexpr int kPer = kPer0 > kPer1 ? kPer0 : kPer1;
				const int per = flag ? kPer1 : kPer0;       // elements beyond Q/2 are never read back, but stay inside the work area
				float2 v[kPer];
				__syncwarp();
#pragma unroll
				for(int i = 0; i < kPer; ++i) if(i < per) v[i] = reinterpret_cast<const float2*>(prev_lo)[lane + 32 * i];
				__syncwarp();
#pragma unroll
				for(int i = 0; i < kPer; ++i) if(i < per) surv[lane + 32 * i] = v[i];
				__syncwarp();
				prev_lo = reinterpret_cast<const float*>(surv);
			}
			stt = ((uint32_t) (first + count) << 8) | (stt & 32u) | (prev_perm ? 16u : 0u) | (prev_right == N1 / 2 ? 8u : 0u) | (prev_n == N1 ? 4u : 0u) | 2u |
			      (uint32_t) (par ^ 1);
		}
	}
	if constexpr(kTm != 0) {
		tm_fence_before();
		__syncthreads();
		if(warp == kWarps - 1) tm_dealloc<kCols>(*s_tmbase);
	}
}

}  // namespace wk

// ---- host side: geometry selection, shared-memory budget, launch -----------------------------------------------------
static bool supported_block(uint32_t n) { return n == 256 || n == 512 || n == 1024 || n == 2048; }

bool warp_kernel_supports(uint32_t bs0, uint32_t bs1) {
	// instantiated pairs (Vorbis encoders use 256/2048 at 44.1-48 kHz, 512/1024 or 256/1024 at 16-22 kHz, 256/512 at 8 kHz)
	if(!supported_block(bs0) || !supported_block(bs1) || bs0 >= bs1) return false;
	return true;
}

template <int Q0, int Q1> static size_t smem_for(uint32_t cb) {
	return (size_t) wk::Map<Q0, Q1>::kOffWarps + (size_t) wk::kWarps * ((size_t) wk::kWarpFixedBytes + cb);
}

size_t warp_kernel_smem_bytes(uint32_t bs0, uint32_t bs1, uint32_t short_posts_cap, uint32_t long_posts_cap, uint32_t* group_short_out,
                              uint32_t* curve_bytes_out, uint32_t* short_stride_out) {
	const uint32_t Q0 = bs0 / 4, Q1 = bs1 / 4;
	const uint32_t stride = short_posts_cap * 8u + (Q0 / 16u) * 8u;       // records + rank-table words of one short curve
	uint32_t group = 512u / Q0;                                           // short FFTs a warp transforms at once (Q0/16 lanes each)
	uint32_t cb = long_posts_cap * 8u + (Q1 / 16u) * 8u;                  // one long curve: records (32 or 64) + rank table
	if(Q1 < 512u) cb *= 512u / Q1;                                         // long packets of < 512 points are grouped too (kLongGrouped)
	while(group > 1 && group * stride > wk::kCurveMax) --group;
	const uint32_t cb_long = cb;
	auto total = [&](uint32_t g) -> size_t {
		uint32_t c = std::max(cb_long, g * stride);
		c = (c + 15u) & ~15u;
		switch(Q0 * 1024u + Q1) {
			case 64u * 1024u + 128u:  return smem_for<64, 128>(c);
			case 64u * 1024u + 256u:  return smem_for<64, 256>(c);
			case 64u * 1024u + 512u:  return smem_for<64, 512>(c);
			case 128u * 1024u + 256u: return smem_for<128, 256>(c);
			case 128u * 1024u + 512u: return smem_for<128, 512>(c);
			case 256u * 1024u + 512u: return smem_for<256, 512>(c);
			default: return (size_t) 1 << 30;
		}
	};
	// a setup with big short-block floors keeps the kernel by transforming fewer short packets per step rather than losing it
	while(group > 1 && total(group) > 227u * 1024u) --group;
	cb = (std::max(cb_long, group * stride) + 15u) & ~15u;
	if(group_short_out) *group_short_out = group;
	if(curve_bytes_out) *curve_bytes_out = cb;
	if(short_stride_out) *short_stride_out = stride;
	return total(group);
}

// packets of a run (halo excluded): the Y records of a run share 1152 bytes: 32 of 36 bytes, or 16 of 72 (floors of 33..64 posts)
uint32_t warp_kernel_max_run(bool wide) { return wide ? (uint32_t) (wk::kPktCap * wk::kFsStride / 72) - 1u : (uint32_t) wk::kPktCap - 1u; }
uint32_t warp_kernel_warps(void) { return (uint32_t) wk::kWarps; }

template <int Q0, int Q1, bool kPlanar, class TPcm, int kMaxNL, bool kWide = false>
static cudaError_t launch_one(const wk::Params& P, uint32_t grid, size_t smem, cudaStream_t st) {
	cudaError_t e = cudaFuncSetAttribute(wk::k_warp_synth<Q0, Q1, kPlanar, TPcm, kMaxNL, kWide>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
	if(e != cudaSuccess) return e;
	wk::k_warp_synth<Q0, Q1, kPlanar, TPcm, kMaxNL, kWide><<<grid, wk::kThreads, smem, st>>>(P);
	return cudaGetLastError();
}

template <int Q0, int Q1, class TPcm>
static cudaError_t launch_geom(const wk::Params& P, uint32_t max_nl, bool wide, uint32_t grid, size_t smem, cudaStream_t st) {
	if(wide) return P.b.pcm_layout == POV_PCM_PLANAR ? launch_one<Q0, Q1, true, TPcm, 4, true>(P, grid, smem, st) : launch_one<Q0, Q1, false, TPcm, 4, true>(P, grid, smem, st);
	const int cls = max_nl <= 1 ? 1 : max_nl == 2 ? 2 : 4;
	if(P.b.pcm_layout == POV_PCM_PLANAR) {
		if(cls == 1) return launch_one<Q0, Q1, true, TPcm, 1>(P, grid, smem, st);
		if(cls == 2) return launch_one<Q0, Q1, true, TPcm, 2>(P, grid, smem, st);
		return launch_one<Q0, Q1, true, TPcm, 4>(P, grid, smem, st);
	}
	if(cls == 1) return launch_one<Q0, Q1, false, TPcm, 1>(P, grid, smem, st);
	if(cls == 2) return launch_one<Q0, Q1, false, TPcm, 2>(P, grid, smem, st);
	return launch_one<Q0, Q1, false, TPcm, 4>(P, grid, smem, st);
}

template <int Q0, int Q1>
static cudaError_t launch_geom(const wk::Params& P, uint32_t max_nl, bool wide, uint32_t grid, size_t smem, cudaStream_t st) {
	return P.b.pcm_s16 ? launch_geom<Q0, Q1, int16_t>(P, max_nl, wide, grid, smem, st) : launch_geom<Q0, Q1, float>(P, max_nl, wide, grid, smem, st);
}

cudaError_t launch_warp(const DevBatchView& b, const DevRun* runs, uint32_t n_runs, uint32_t channels, const FastTables* d_tabs,
                        uint32_t bs0, uint32_t bs1, uint32_t short_posts_cap, uint32_t long_posts_cap, uint32_t max_nl, const float* const slope[2], const float2* const rot[2],
                        const float2* const tw8[2], const float2* const fp[2], const float* tmtab, unsigned char* dbg_floor, uint32_t* d_counter, int sm_count,
                        cudaStream_t st, uint64_t* launches) {
	if(n_runs == 0) return cudaSuccess;
	wk::Params P;
	P.b = b; P.runs = runs; P.n_runs = n_runs; P.C = channels; P.n_items = n_runs * channels;
	P.counter = d_counter; P.tabs = d_tabs; P.tmtab = tmtab; P.dbg_floor = dbg_floor;
	for(int k = 0; k < 2; ++k) { P.slope[k] = slope[k]; P.rot[k] = rot[k]; P.tw8[k] = tw8[k]; P.fp[k] = fp[k]; }
	const size_t smem = warp_kernel_smem_bytes(bs0, bs1, short_posts_cap, long_posts_cap, &P.group_short, &P.curve_bytes, &P.short_curve_stride);
	if(smem > 227 * 1024) return cudaErrorInvalidConfiguration;
	cudaError_t e = cudaMemsetAsync(d_counter, 0, sizeof(uint32_t), st);
	if(e != cudaSuccess) return e;
	uint32_t grid = (uint32_t) sm_count;
	const uint32_t need = (P.n_items + wk::kWarps - 1) / wk::kWarps;
	if(grid > need) grid = need;
	switch((bs0 / 4) * 1024u + bs1 / 4) {
		case 64u * 1024u + 128u:  e = launch_geom<64, 128>(P, max_nl, long_posts_cap > 32, grid, smem, st); break;
		case 64u * 1024u + 256u:  e = launch_geom<64, 256>(P, max_nl, long_posts_cap > 32, grid, smem, st); break;
		case 64u * 1024u + 512u:  e = launch_geom<64, 512>(P, max_nl, long_posts_cap > 32, grid, smem, st); break;
		case 128u * 1024u + 256u: e = launch_geom<128, 256>(P, max_nl, long_posts_cap > 32, grid, smem, st); break;
		case 128u * 1024u + 512u: e = launch_geom<128, 512>(P, max_nl, long_posts_cap > 32, grid, smem, st); break;
		case 256u * 1024u + 512u: e = launch_geom<256, 512>(P, max_nl, long_posts_cap > 32, grid, smem, st); break;
		default: return cudaErrorInvalidConfiguration;
	}
	if(launches) ++*launches;
	return e;
}

}  // namespace pov
