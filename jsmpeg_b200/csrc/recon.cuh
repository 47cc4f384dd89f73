// recon.cuh -- stage 2 device code: one 8x8 block = one thread (sm_100a).
//
// Included by recon.cu (kernel shell + launcher).  Like walk.cuh the same text compiles for the host
// when JSMPEG_WALK_EMU is defined (tests/emu/walk_emu.cpp): the TMA copy and the packed-saturate /
// dot-product instructions get plain C stand-ins, so that the CPU test-suite can run the whole hot
// path -- walk, expand, reconstruct -- against the oracle's planes.
#pragma once
#include "common.cuh"

namespace {


constexpr int THREADS = 128;
constexpr int ROW_PITCH = 144;                       // bytes per staged block: 128 + 16 (bank spread)
constexpr int WARP_STAGE = 32 * ROW_PITCH + 16;      // + the warp's mbarrier
constexpr int MAX_TASKS = 80;       // per launch; (80 * 48 B) + 16 < 4 KB of kernel parameters
constexpr int MAX_TASKS_RGBA = 60;  // the RGBA variant's parameters: (60 * (48 + 16) B) + 16 < 4 KB


struct CompactTask {
	const mb_record_t *hdr;
	const int16_t *coef;
	uint8_t *cur;        // Y at 0, Cr at coded_size, Cb at coded_size * 5 / 4; readable for coded_width + 64 bytes past the end
	const uint8_t *fwd;
	int32_t mb_width, mb_height;
	uint32_t row_magic;  // floor(2^32 / (6 mb_width)) + 1: slot / (6 mb_width) == umulhi(slot, row_magic) for every slot of a picture
	uint32_t flags;      // (none defined)
};

template <int N>
struct ReconParamsT {
	CompactTask t[N];
	int32_t n_tasks;
};
using ReconParams = ReconParamsT<MAX_TASKS>;

// B pictures (the opt-in extension; the reference skips them, mpeg1.js:181-184): a second reference.
// fwd = the older, bwd = the newer of the stream's two most recent I/P pictures.
struct CompactTaskB : CompactTask {
	const uint8_t *bwd;
};
constexpr int MAX_TASKS_B = 64;  // (64 * 56 B) + 16 < 4 KB of kernel parameters
struct ReconParamsB {
	CompactTaskB t[MAX_TASKS_B];
	int32_t n_tasks;
};

#ifndef JSMPEG_WALK_EMU
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ uint32_t umulhi_u32(uint32_t a, uint32_t b) { return __umulhi(a, b); }
#else
static inline void prefetch_l2(const void *) {}
static inline uint32_t umulhi_u32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
#endif

// PREMULTIPLIER_MATRIX (src/mpeg1.js:1026-1035) = outer product of these AAN scales, rounded as the
// reference's table is; kept as a constexpr so that every use folds into an immediate.
__device__ constexpr int PM[64] = {
    32, 44, 42, 38, 32, 25, 17, 9,  44, 62, 58, 52, 44, 35, 24, 12, 42, 58, 55, 49, 42, 33, 23, 12,
    38, 52, 49, 44, 38, 30, 20, 10, 32, 44, 42, 38, 32, 25, 17, 9,  25, 35, 33, 30, 25, 20, 14, 7,
    17, 24, 23, 20, 17, 14, 9,  5,  9,  12, 12, 10, 9,  7,  5,  2};

// One 8-point pass of the reference IDCT on v[o], v[o+s], ... v[o+7s].
// Column pass: no scaling; row pass: (v + 128) >> 8.
template <bool ROW, int O, int S>
__device__ __forceinline__ void idct8(int (&v)[64]) {
	const int b1 = v[O + 4 * S];
	const int b3 = v[O + 2 * S] + v[O + 6 * S];
	const int b4 = v[O + 5 * S] - v[O + 3 * S];
	const int t1 = v[O + 1 * S] + v[O + 7 * S];
	const int t2 = v[O + 3 * S] + v[O + 5 * S];
	const int b6 = v[O + 1 * S] - v[O + 7 * S];
	const int b7 = t1 + t2;
	const int m0 = v[O];
	const int x4 = ((b6 * 473 - b4 * 196 + 128) >> 8) - b7;
	const int x0 = x4 - (((t1 - t2) * 362 + 128) >> 8);
	const int x1 = m0 - b1;
	const int x2 = (((v[O + 2 * S] - v[O + 6 * S]) * 362 + 128) >> 8) - b3;
	const int x3 = m0 + b1;
	const int y3 = x1 + x2, y4 = x3 + b3, y5 = x1 - x2, y6 = x3 - b3;
	const int y7 = -x0 - ((b4 * 473 + b6 * 196 + 128) >> 8);
	if (ROW) {
		v[O] = (b7 + y4 + 128) >> 8;         v[O + 1 * S] = (x4 + y3 + 128) >> 8;
		v[O + 2 * S] = (y5 - x0 + 128) >> 8; v[O + 3 * S] = (y6 - y7 + 128) >> 8;
		v[O + 4 * S] = (y6 + y7 + 128) >> 8; v[O + 5 * S] = (x0 + y5 + 128) >> 8;
		v[O + 6 * S] = (y3 - x4 + 128) >> 8; v[O + 7 * S] = (y4 - b7 + 128) >> 8;
	} else {
		v[O] = b7 + y4;         v[O + 1 * S] = x4 + y3; v[O + 2 * S] = y5 - x0; v[O + 3 * S] = y6 - y7;
		v[O + 4 * S] = y6 + y7; v[O + 5 * S] = x0 + y5; v[O + 6 * S] = y3 - x4; v[O + 7 * S] = y4 - b7;
	}
}

template <int I>
__device__ __forceinline__ void idct_columns(int (&v)[64]) {
	if constexpr (I < 8) {
		idct8<false, I, 8>(v);
		idct_columns<I + 1>(v);
	}
}
template <int I>
__device__ __forceinline__ void idct_rows(int (&v)[64]) {
	if constexpr (I < 8) {
		idct8<true, I * 8, 1>(v);
		idct_rows<I + 1>(v);
	}
}

__device__ __forceinline__ uint32_t pack_sat_u8x4(int a, int b, int c, int d) {
	// PTX: d[7:0] = sat(b_op), d[15:8] = sat(a_op), d[31:16] = c_op[15:0]
#ifndef JSMPEG_WALK_EMU
	uint32_t hi, r;
	const uint32_t zero = 0;
	asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(hi) : "r"(d), "r"(c), "r"(zero));
	asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(b), "r"(a), "r"(hi));
	return r;
#else
	auto sat = [](int x) { return (uint32_t)(x < 0 ? 0 : (x > 255 ? 255 : x)); };
	return sat(a) | sat(b) << 8 | sat(c) << 16 | sat(d) << 24;
#endif
}

// packed predicted samples p (4 per word) + 4 residuals -> 4 saturated output samples
__device__ __forceinline__ uint32_t add_sat4(uint32_t p, int r0, int r1, int r2, int r3) {
	return pack_sat_u8x4((int)(p & 255u) + r0, (int)((p >> 8) & 255u) + r1, (int)((p >> 16) & 255u) + r2, (int)(p >> 24) + r3);
}

// 9 consecutive samples starting at flat index i of a plane whose base is 4-byte aligned:
// a = samples 0..3, b = 4..7, c (low byte) = sample 8.
__device__ __forceinline__ void row9(const uint8_t *__restrict__ plane, int i, uint32_t &a, uint32_t &b, uint32_t &c) {
	const uint32_t *w = reinterpret_cast<const uint32_t *>(plane) + (i >> 2);
	const uint32_t w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2);
	const uint32_t sh = (uint32_t)(i & 3) * 8u;
	a = __funnelshift_r(w0, w1, sh);
	b = __funnelshift_r(w1, w2, sh);
	c = w2 >> sh;
}

// dp4a with unsigned bytes in `a` and signed bytes in `b`: sum_i a.b[i] * b.b[i] + c (integer dot
// product unit, off the ALU pipe that bounds this kernel)
__device__ __forceinline__ int dp4a_us(uint32_t a, uint32_t b, int c) {
#ifndef JSMPEG_WALK_EMU
	int d;
	asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
	return d;
#else
	for (int i = 0; i < 4; i++) c += (int)((a >> (8 * i)) & 255u) * (int)(int8_t)((b >> (8 * i)) & 255u);
	return c;
#endif
}

// Prediction of the 8 rows of one block + residual.  The four half-pel cases of the reference
// (copy, (a+b+1)>>1 horizontally or vertically, (a+b+c+d+2)>>2; src/mpeg1.js:481-556) are ONE
// formula with per-thread tap weights:
//     (wA*A + wB*B + wC*C + wD*D + 2) >> 2,   (wA,wB,wC,wD) = (4,0,0,0) | (2,2,0,0) | (2,0,2,0) | (1,1,1,1)
// ((4A+2)>>2 = A, (2A+2B+2)>>2 = (A+B+1)>>1).  Per output sample: one PRMT gathers the four taps
// into a word, one dp4a applies the weights (accumulator preloaded with the rounding 2).
// The lanes of a warp hold blocks of different macroblocks, i.e. different parities: the weights
// are data, the instruction stream is the same for every lane.
// FULLPEL (warp-uniform: no lane has a half-pel component) is the plain copy: one dp4a per sample
// selects the byte and adds the residual.
// v = the residual, all zero for a block that is not coded.
// KEEP: the packed rows are also handed back (the fused RGBA epilogue converts them).
template <bool FULLPEL, bool KEEP>
__device__ __forceinline__ void predict_rows(const uint8_t *__restrict__ splane, int src, int stride, uint32_t weights,
                                             const int (&v)[64], uint8_t *__restrict__ dst, uint2 (&rows)[8]) {
	uint32_t a0, a1, a2;
	row9(splane, src, a0, a1, a2);
#pragma unroll
	for (int r = 0; r < 8; r++) {
		uint32_t c0 = 0, c1 = 0, c2 = 0;
		int s[8];
		if (FULLPEL) {
			if (r < 7) row9(splane, src + (r + 1) * stride, c0, c1, c2);
#pragma unroll
			for (int x = 0; x < 4; x++) {
				s[x] = dp4a_us(a0, 1u << (8 * x), v[r * 8 + x]);
				s[4 + x] = dp4a_us(a1, 1u << (8 * x), v[r * 8 + 4 + x]);
			}
		} else {
			row9(splane, src + (r + 1) * stride, c0, c1, c2);  // row 8 is inside the plane (checked by the caller)
			const uint32_t sa0 = __funnelshift_r(a0, a1, 8), sa1 = __funnelshift_r(a1, a2, 8);  // samples 1..4, 5..8
			const uint32_t sc0 = __funnelshift_r(c0, c1, 8), sc1 = __funnelshift_r(c1, c2, 8);
			// taps (A, B, C, D) = (row[x], row[x+1], next[x], next[x+1]) as one word per sample.  The residual
			// rides in the accumulator: (sum + 2 + 4 res) >> 2 == ((sum + 2) >> 2) + res exactly, and 4 res + 2
			// is a multiply-add on the FMA pipe instead of an add on the ALU pipe that bounds this kernel.
			int acc[8];
#pragma unroll
			for (int x = 0; x < 8; x++) acc[x] = v[r * 8 + x] * 4 + 2;
			s[0] = dp4a_us(__byte_perm(a0, c0, 0x5410), weights, acc[0]);
			s[1] = dp4a_us(__byte_perm(a0, c0, 0x6521), weights, acc[1]);
			s[2] = dp4a_us(__byte_perm(a0, c0, 0x7632), weights, acc[2]);
			s[3] = dp4a_us(__byte_perm(sa0, sc0, 0x7632), weights, acc[3]);
			s[4] = dp4a_us(__byte_perm(a1, c1, 0x5410), weights, acc[4]);
			s[5] = dp4a_us(__byte_perm(a1, c1, 0x6521), weights, acc[5]);
			s[6] = dp4a_us(__byte_perm(a1, c1, 0x7632), weights, acc[6]);
			s[7] = dp4a_us(__byte_perm(sa1, sc1, 0x7632), weights, acc[7]);
#pragma unroll
			for (int x = 0; x < 8; x++) s[x] >>= 2;
		}
		uint2 out;
		out.x = pack_sat_u8x4(s[0], s[1], s[2], s[3]);
		out.y = pack_sat_u8x4(s[4], s[5], s[6], s[7]);
		*reinterpret_cast<uint2 *>(dst + r * stride) = out;
		if (KEEP) rows[r] = out;
		a0 = c0; a1 = c1; a2 = c2;
	}
}

// ---- B pictures: prediction from two references (ISO 11172-2 2.4.4.3) ------------------------------------------
// per byte (a + b + 1) >> 1: the "//" of the standard on samples (halves rounded up)
__device__ __forceinline__ uint32_t avg_round_u8x4(uint32_t a, uint32_t b) {
#ifndef JSMPEG_WALK_EMU
	return __vavgu4(a, b);
#else
	uint32_t r = 0;
	for (int i = 0; i < 4; i++) r |= ((((a >> (8 * i)) & 255u) + ((b >> (8 * i)) & 255u) + 1u) >> 1) << (8 * i);
	return r;
#endif
}

// One row of 8 predicted samples (packed) from rows a (this row) and c (the next one) of one reference with the
// lane's tap weights -- the formula of predict_rows, without residual: (wA*A + wB*B + wC*C + wD*D + 2) >> 2.
__device__ __forceinline__ uint2 predict_row_packed(uint32_t a0, uint32_t a1, uint32_t a2, uint32_t c0, uint32_t c1, uint32_t c2,
                                                    uint32_t weights) {
	const uint32_t sa0 = __funnelshift_r(a0, a1, 8), sa1 = __funnelshift_r(a1, a2, 8);
	const uint32_t sc0 = __funnelshift_r(c0, c1, 8), sc1 = __funnelshift_r(c1, c2, 8);
	int s[8];
	s[0] = dp4a_us(__byte_perm(a0, c0, 0x5410), weights, 2);
	s[1] = dp4a_us(__byte_perm(a0, c0, 0x6521), weights, 2);
	s[2] = dp4a_us(__byte_perm(a0, c0, 0x7632), weights, 2);
	s[3] = dp4a_us(__byte_perm(sa0, sc0, 0x7632), weights, 2);
	s[4] = dp4a_us(__byte_perm(a1, c1, 0x5410), weights, 2);
	s[5] = dp4a_us(__byte_perm(a1, c1, 0x6521), weights, 2);
	s[6] = dp4a_us(__byte_perm(a1, c1, 0x7632), weights, 2);
	s[7] = dp4a_us(__byte_perm(sa1, sc1, 0x7632), weights, 2);
	uint2 out;  // (sums of at most four bytes + 2) >> 2 fit a byte: plain packing
	out.x = (uint32_t)(s[0] >> 2) | (uint32_t)(s[1] >> 2) << 8 | (uint32_t)(s[2] >> 2) << 16 | (uint32_t)(s[3] >> 2) << 24;
	out.y = (uint32_t)(s[4] >> 2) | (uint32_t)(s[5] >> 2) << 8 | (uint32_t)(s[6] >> 2) << 16 | (uint32_t)(s[7] >> 2) << 24;
	return out;
}

// The 8 rows of one block of a B picture: forward and / or backward prediction (each rounded on its own, like
// copyMacroblock, mpeg1.js:481-556), their rounded average when both are used, + residual, saturate, store.
// A direction that is not used is read at the block's own position (in bounds) and ignored.
template <bool KEEP>
__device__ __forceinline__ void predict_rows_b(const uint8_t *__restrict__ fplane, int fsrc, uint32_t fweights, bool use_f,
                                               const uint8_t *__restrict__ bplane, int bsrc, uint32_t bweights, bool use_b,
                                               int stride, const int (&v)[64], uint8_t *__restrict__ dst, uint2 (&rows)[8]) {
	uint32_t f0, f1, f2, b0, b1, b2;
	row9(fplane, fsrc, f0, f1, f2);
	row9(bplane, bsrc, b0, b1, b2);
#pragma unroll
	for (int r = 0; r < 8; r++) {
		uint32_t g0, g1, g2, c0, c1, c2;
		row9(fplane, fsrc + (r + 1) * stride, g0, g1, g2);  // row 8 is inside the allocation (checked by the caller / the pad)
		row9(bplane, bsrc + (r + 1) * stride, c0, c1, c2);
		const uint2 pf = predict_row_packed(f0, f1, f2, g0, g1, g2, fweights);
		const uint2 pb = predict_row_packed(b0, b1, b2, c0, c1, c2, bweights);
		uint2 p;
		p.x = use_f ? (use_b ? avg_round_u8x4(pf.x, pb.x) : pf.x) : pb.x;
		p.y = use_f ? (use_b ? avg_round_u8x4(pf.y, pb.y) : pf.y) : pb.y;
		uint2 out;
		out.x = add_sat4(p.x, v[r * 8 + 0], v[r * 8 + 1], v[r * 8 + 2], v[r * 8 + 3]);
		out.y = add_sat4(p.y, v[r * 8 + 4], v[r * 8 + 5], v[r * 8 + 6], v[r * 8 + 7]);
		*reinterpret_cast<uint2 *>(dst + r * stride) = out;
		if (KEEP) rows[r] = out;
		f0 = g0; f1 = g1; f2 = g2;
		b0 = c0; b1 = c1; b2 = c2;
	}
}

// one predicted sample by flat index with per-tap bounds check: any tap outside the plane zeroes it (SURVEY Q11)
__device__ __forceinline__ int tap_px(const uint8_t *__restrict__ plane, int i, int stride, bool oh, bool ov, int plane_size) {
	const int taps[4] = {i, i + 1, i + stride, i + stride + 1};
	const bool use[4] = {true, oh, ov, oh && ov};
	int sum = 0, n = 0;
	bool in = true;
	for (int k = 0; k < 4; k++) {
		if (!use[k]) continue;
		if (taps[k] < 0 || taps[k] >= plane_size) { in = false; continue; }
		sum += plane[taps[k]];
		n++;
	}
	return !in ? 0 : (n == 4 ? (sum + 2) >> 2 : (n == 2 ? (sum + 1) >> 1 : sum));
}

#ifndef JSMPEG_WALK_EMU
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
#else
static inline uint32_t smem_u32(const void *) { return 0; }
#endif

// One 8x8 block: slot first_slot + tid of picture `ty` of the launch (see above); `stage` = the CTA's
// staging area (one WARP_STAGE per warp), tid = the thread's index in the CTA.
// WARP-CONVERGENT: the 32 lanes of a warp call it together (collectives inside).
//
// Latency plan (round 2; the kernel was stalled on memory it asked for too late -- long-scoreboard 2.7
// warps per issue at 4.5 resident warps per scheduler, profiles/r2_reconstruct.md):
//   t0  the header load starts;  the header and the coefficient record of the CTA that will run here two
//       pictures of the launch later are pulled into L2
//   t0' header there: the records of the coded blocks are requested (TMA).  (Requesting every slot's record
//       before the header is known, for pictures with most blocks coded, was built and measured: 11.90 ms per
//       60 launches against 11.92 -- nothing, for 3.5 % more DRAM traffic; removed.)
//   t1  header there: the nine reference rows of a predicted block are pulled into L2 (no registers)
//   t2  records there: IDCT (some 700 instructions) -- the reference rows arrive meanwhile
//   t3  prediction reads hit L2, + residual, store
// block (mb_row, mb_col, b) of picture `ty`; the 32 lanes of the warp call it together, wstage = the warp's staging
// area.  KEEP: the block's eight packed output rows come back in `rows` (also for a macroblock that is not present:
// the samples it keeps).
// BIDIR (B pictures, PARAMS = ReconParamsB): the record's MBF_MOTION_* bits say which of t.fwd / t.bwd a predicted
// block uses; everything up to the prediction is the same code.
template <bool KEEP, bool BIDIR = false, class PARAMS>
__device__ __forceinline__ void reconstruct_at(const PARAMS &params, int ty, int mb_row, int mb_col, int b, bool in_picture,
                                               int lane, uint8_t *wstage, uint2 (&rows)[8]) {
	const auto &t = params.t[ty];
	const int W = t.mb_width;
	const int mb = mb_row * W + mb_col;

	const uint32_t mbar = smem_u32(wstage + 32 * ROW_PITCH);
	const uint32_t my_row = smem_u32(wstage + lane * ROW_PITCH);
	const int16_t *cblk = t.coef + ((size_t)mb * 6 + b) * 64;

	// ---- coefficient records of the warp's blocks: one TMA bulk copy per lane
	// `want` = this lane's record is copied; warp-uniform `copy_mask` = which lanes' are
	auto request_records = [&](bool want, unsigned copy_mask) {
#ifndef JSMPEG_WALK_EMU
		if (lane == 0) {
			asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar));
			// the initialised barrier must be visible to the async proxy (the TMA unit) before the copies name it:
			// the proxy fence of the CUDA guide's single-CTA pattern.  (fence.mbarrier_init.release.cluster, used
			// until round 2, is cluster-scoped: ptxas adds CCTL.IVALL to it, an invalidation of the SM's whole L1.)
			asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
			asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(128u * (uint32_t)__popc(copy_mask)) : "memory");
		}
		__syncwarp();
		if (want)
			asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], 128, [%2];"
			             ::"r"(my_row), "l"(cblk), "r"(mbar) : "memory");
#else
		(void)mbar; (void)copy_mask;
		if (want) memcpy(wstage + lane * ROW_PITCH, cblk, 128);  // the emulated "TMA": the lane's record into its staging row
#endif
	};
	uint2 rec = make_uint2(0, 0);
	uint32_t rec_bwd = 0;  // BIDIR: the backward vector (mb_record_t::mv_bwd)
	if constexpr (BIDIR) {
		if (in_picture) {
			const uint4 r4 = __ldg(reinterpret_cast<const uint4 *>(t.hdr + mb));
			rec = make_uint2(r4.x, r4.y);
			rec_bwd = r4.w;
		}
	} else {
		if (in_picture) rec = __ldg(reinterpret_cast<const uint2 *>(t.hdr + mb));
	}
	if (ty + 2 < params.n_tasks) {  // the CTA that runs on this SM next but one: its header and record, into L2
		const auto &t2 = params.t[ty + 2];
		if (in_picture && mb < t2.mb_width * t2.mb_height) {
			prefetch_l2(t2.hdr + mb);
			prefetch_l2(t2.coef + ((size_t)mb * 6 + b) * 64);
		}
	}
	const int flags = rec.y & 0xff;
	const bool present = flags & MBF_PRESENT;  // an untouched macroblock keeps the two-pictures-old content (SURVEY Q12)
	const bool intra = flags & MBF_INTRA;
	const int bit = 0x20 >> b;
	const bool coded = present && ((rec.y >> 8) & bit);
	const bool dc_only = coded && ((rec.y >> 16) & bit);
	const bool full = coded && !dc_only;
	const bool warp_full = __any_sync(0xffffffffu, full);  // warp-uniform: some lane needs the transform

	const unsigned coded_mask = __ballot_sync(0xffffffffu, coded);
	if (coded_mask) request_records(coded, coded_mask);  // only what is coded (the DC-only blocks' value too)
	const bool copying = coded_mask != 0;                 // warp-uniform

	const int stride_y = W * 16;
	const int ysize = stride_y * t.mb_height * 16;
	int stride, plane_off, plane_size, origin;
	if (b < 4) {
		stride = stride_y; plane_off = 0; plane_size = ysize;
		origin = (mb_row * 16 + (b >> 1) * 8) * stride + mb_col * 16 + (b & 1) * 8;
	} else {
		stride = stride_y >> 1; plane_size = ysize >> 2;
		plane_off = b == 4 ? ysize + plane_size : ysize;  // Cb is the third plane, Cr the second
		origin = mb_row * 8 * stride + mb_col * 8;
	}

	// motion vector of this block's plane, and whether ANY lane of the warp needs half-pel taps
	int mh = (int)(int16_t)(rec.x & 0xffffu), mv = (int)(int16_t)(rec.x >> 16);
	if (b >= 4) { mh /= 2; mv /= 2; }  // truncation toward zero (mpeg1.js:562-565, SURVEY Q9)
	const bool oh = mh & 1, ov = mv & 1;
	const bool warp_halfpel = __any_sync(0xffffffffu, present && !intra && (oh || ov));
	const int src = origin + (mv >> 1) * stride + (mh >> 1);  // flat index (mpeg1.js:479, 567)
	const uint8_t *splane = t.fwd + plane_off;
	// every tap the prediction USES lies inside the plane.  (What the row loads touch beyond them -- the
	// rest of the last word, row 8 of a lane without a vertical half -- is inside the allocation: planes
	// are contiguous and followed by coded_width + 64 readable bytes.)
	const bool inside = src >= 0 && src + 7 * stride + 7 + (ov ? stride : 0) + (oh ? 1 : 0) < plane_size;
	// BIDIR: which references the block uses (a record with neither bit predicts forward, like the oracle), and the
	// same geometry for the backward one
	const bool use_b = BIDIR && (flags & MBF_MOTION_BWD);
	const bool use_f = !use_b || (flags & MBF_MOTION_FWD);
	int src_b = origin;
	bool ohb = false, ovb = false, inside_b = true;
	if constexpr (BIDIR) {
		int bh = (int)(int16_t)(rec_bwd & 0xffffu), bv = (int)(int16_t)(rec_bwd >> 16);
		if (b >= 4) { bh /= 2; bv /= 2; }
		if (!use_b) bh = bv = 0;
		ohb = bh & 1; ovb = bv & 1;
		src_b = origin + (bv >> 1) * stride + (bh >> 1);
		inside_b = src_b >= 0 && src_b + 7 * stride + 7 + (ovb ? stride : 0) + (ohb ? 1 : 0) < plane_size;
		if (present && !intra && use_b && inside_b) {
#pragma unroll
			for (int r = 0; r < 9; r++) prefetch_l2(t.bwd + plane_off + src_b + r * stride + 4);
		}
	}
	if (present && !intra && inside && (!BIDIR || use_f)) {  // t1: the reference rows, into L2, while the records travel and the IDCT runs
		// (Sharing the rows out among the lanes -- lane l asks for row l & 7 of its own block, two instructions
		// instead of nine -- was measured: 12.03 ms per 60 launches against 11.87, the neighbours' vectors differ too often.)
#pragma unroll
		for (int r = 0; r < 9; r++) prefetch_l2(splane + src + r * stride + 4);
	}

	if (copying) {  // t2: wait for the warp's copies (phase 0 of a barrier used once)
#ifndef JSMPEG_WALK_EMU
		uint32_t done = 0;
		while (!done)
			asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
			             : "=r"(done) : "r"(mbar) : "memory");
#endif
	}
	uint8_t *dst = t.cur + plane_off + origin;
	auto reload_rows = [&]() {  // what is in the plane now (rare paths of the RGBA variant)
#pragma unroll
		for (int r = 0; r < 8; r++) rows[r] = *reinterpret_cast<const uint2 *>(dst + r * stride);
	};
	if (!present) {
		if (KEEP && in_picture) reload_rows();
		return;
	}

	// ---- residual: 64 values in registers
	// One path per WARP.  A block with nothing but coefficient 0 takes the reference's scalar shortcut
	// (mpeg1.js:838-853: every sample = (block[0] + 128) >> 8) -- and the full transform of such a block gives
	// exactly that: column 0 comes out as eight copies of block[0], every row then as (block[0] + 128) >> 8
	// (all other terms are (0 * k + 128) >> 8 = 0).  An uncoded block is the transform of zeros.  So in a warp
	// with at least one block that needs the transform, every lane runs it -- the DC-only lanes on their staged
	// record (zeros behind coefficient 0, the expand kernel writes whole records), the uncoded lanes on a row
	// they zero themselves -- instead of the warp running the transform AND the 64-register fill one after the other.
	int v[64];
	if (warp_full) {
		if (!coded) {  // present, nothing coded: a residual of zeros
#ifndef JSMPEG_WALK_EMU
#pragma unroll
			for (int i = 0; i < 8; i++) asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(my_row + i * 16), "r"(0u) : "memory");
#else
			memset(wstage + lane * ROW_PITCH, 0, 128);
#endif
		}
#pragma unroll
		for (int i = 0; i < 8; i++) {
			uint4 q;
#ifndef JSMPEG_WALK_EMU
			asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w) : "r"(my_row + i * 16) : "memory");
#else
			(void)my_row;
			memcpy(&q, wstage + lane * ROW_PITCH + i * 16, 16);
#endif
			// dp2a: (lo16 * b0 + hi16 * b1): one instruction per coefficient, no unpacking on the ALU pipe
			v[i * 8 + 0] = __dp2a_lo((int)q.x, PM[i * 8 + 0], 0); v[i * 8 + 1] = __dp2a_lo((int)q.x, PM[i * 8 + 1] << 8, 0);
			v[i * 8 + 2] = __dp2a_lo((int)q.y, PM[i * 8 + 2], 0); v[i * 8 + 3] = __dp2a_lo((int)q.y, PM[i * 8 + 3] << 8, 0);
			v[i * 8 + 4] = __dp2a_lo((int)q.z, PM[i * 8 + 4], 0); v[i * 8 + 5] = __dp2a_lo((int)q.z, PM[i * 8 + 5] << 8, 0);
			v[i * 8 + 6] = __dp2a_lo((int)q.w, PM[i * 8 + 6], 0); v[i * 8 + 7] = __dp2a_lo((int)q.w, PM[i * 8 + 7] << 8, 0);
		}
		idct_columns<0>(v);
		idct_rows<0>(v);
	} else {
		int dc = 0;
		if (coded) {  // mpeg1.js:838-841, 850-853: the staged record's first value
			int16_t c0;
#ifndef JSMPEG_WALK_EMU
			asm volatile("ld.shared.s16 %0, [%1];" : "=h"(c0) : "r"(my_row));
#else
			memcpy(&c0, wstage + lane * ROW_PITCH, 2);
#endif
			dc = ((int)c0 * PM[0] + 128) >> 8;
		}
#pragma unroll
		for (int i = 0; i < 64; i++) v[i] = dc;
	}

	if (intra) {
#pragma unroll
		for (int r = 0; r < 8; r++) {
			uint2 out;
			out.x = pack_sat_u8x4(v[r * 8 + 0], v[r * 8 + 1], v[r * 8 + 2], v[r * 8 + 3]);
			out.y = pack_sat_u8x4(v[r * 8 + 4], v[r * 8 + 5], v[r * 8 + 6], v[r * 8 + 7]);
			*reinterpret_cast<uint2 *>(dst + r * stride) = out;
			if (KEEP) rows[r] = out;
		}
		return;
	}

	if constexpr (BIDIR) {
		// ---- B picture: forward and / or backward prediction (+ their rounded average) + residual
		const uint8_t *bplane = t.bwd + plane_off;
		const int fsrc = use_f ? src : origin;  // (an unused direction is read at the block's own position and ignored)
		if ((!use_f || inside) && (!use_b || inside_b)) {
			const uint32_t fw = (use_f && oh) ? (ov ? 0x01010101u : 0x00000202u) : ((use_f && ov) ? 0x00020002u : 0x00000004u);
			const uint32_t bw = ohb ? (ovb ? 0x01010101u : 0x00000202u) : (ovb ? 0x00020002u : 0x00000004u);
			predict_rows_b<KEEP>(splane, fsrc, fw, use_f, bplane, src_b, bw, use_b, stride, v, dst, rows);
			return;
		}
		// a vector leaves its plane: per-tap bounds check, any outside tap zeroes that prediction's sample (SURVEY Q11)
#pragma unroll 1
		for (int r = 0; r < 8; r++) {
			uint32_t p[2] = {0, 0};
			for (int x = 0; x < 8; x++) {
				const int pf = use_f ? tap_px(splane, src + r * stride + x, stride, oh, ov, plane_size) : 0;
				const int pb = use_b ? tap_px(bplane, src_b + r * stride + x, stride, ohb, ovb, plane_size) : 0;
				const int px = (use_f && use_b) ? (pf + pb + 1) >> 1 : (use_b ? pb : pf);
				p[x >> 2] |= (uint32_t)px << (8 * (x & 3));
			}
			int rr[8];
#pragma unroll
			for (int x = 0; x < 8; x++) {
				int acc = 0;
#pragma unroll
				for (int q = 0; q < 8; q++) acc = (q == r) ? v[q * 8 + x] : acc;
				rr[x] = acc;
			}
			uint2 out;
			out.x = add_sat4(p[0], rr[0], rr[1], rr[2], rr[3]);
			out.y = add_sat4(p[1], rr[4], rr[5], rr[6], rr[7]);
			*reinterpret_cast<uint2 *>(dst + r * stride) = out;
		}
		if (KEEP) reload_rows();
		return;
	}

	// ---- prediction from the forward picture + residual
	if (inside) {
		// tap weights of this lane: bytes (wA, wB, wC, wD)
		const uint32_t weights = oh ? (ov ? 0x01010101u : 0x00000202u) : (ov ? 0x00020002u : 0x00000004u);
		if (warp_halfpel) predict_rows<false, KEEP>(splane, src, stride, weights, v, dst, rows);
		else predict_rows<true, KEEP>(splane, src, stride, weights, v, dst, rows);
		return;
	}
	// vector leaves the plane: per-tap bounds check, any outside tap zeroes the sample (SURVEY Q11)
#pragma unroll 1
	for (int r = 0; r < 8; r++) {
		uint32_t p[2] = {0, 0};
		for (int x = 0; x < 8; x++) {
			const int i = src + r * stride + x;
			const int taps[4] = {i, i + 1, i + stride, i + stride + 1};
			const bool use[4] = {true, (bool)oh, (bool)ov, oh && ov};
			int sum = 0, n = 0;
			bool inside = true;
			for (int k = 0; k < 4; k++) {
				if (!use[k]) continue;
				if (taps[k] < 0 || taps[k] >= plane_size) { inside = false; continue; }
				sum += splane[taps[k]];
				n++;
			}
			const int px = !inside ? 0 : (n == 4 ? (sum + 2) >> 2 : (n == 2 ? (sum + 1) >> 1 : sum));
			p[x >> 2] |= (uint32_t)px << (8 * (x & 3));
		}
		// v[] is indexed dynamically only on this rare path (spills to local memory are fine here)
		int rr[8];
#pragma unroll
		for (int x = 0; x < 8; x++) {
			int acc = 0;
#pragma unroll
			for (int q = 0; q < 8; q++) acc = (q == r) ? v[q * 8 + x] : acc;
			rr[x] = acc;
		}
		uint2 out;
		if (coded) {
			out.x = add_sat4(p[0], rr[0], rr[1], rr[2], rr[3]);
			out.y = add_sat4(p[1], rr[4], rr[5], rr[6], rr[7]);
		} else {
			out.x = p[0]; out.y = p[1];
		}
		*reinterpret_cast<uint2 *>(dst + r * stride) = out;
	}
	if (KEEP) reload_rows();
}

// The plain kernel's numbering: slot first_slot + tid of picture `ty`; `stage` = the CTA's staging area (one
// WARP_STAGE per warp).  The 32 lanes of a warp hold 32 horizontally adjacent blocks of one plane row:
// [luma top 2W | luma bottom 2W | Cb W | Cr W] per macroblock row.
template <bool BIDIR = false, class PARAMS>
__device__ __forceinline__ void reconstruct_block(const PARAMS &params, int ty, int first_slot, int tid, uint8_t *stage) {
	const auto &t = params.t[ty];
	const int W = t.mb_width;
	const int slots_per_row = 6 * W;
	const int slot = first_slot + tid;
	const bool in_picture = slot < slots_per_row * t.mb_height;
	const int mb_row = in_picture ? (int)umulhi_u32((uint32_t)slot, t.row_magic) : 0;
	const int s = in_picture ? slot - mb_row * slots_per_row : 0;
	int b, mb_col;
	if (s < 4 * W) {
		const int by = s >= 2 * W;
		const int bx = s - by * 2 * W;
		mb_col = bx >> 1;
		b = by * 2 + (bx & 1);
	} else {
		const int c = s - 4 * W;
		const int second = c >= W;
		mb_col = c - second * W;
		b = 4 + second;  // block 4 -> Cb plane, block 5 -> Cr plane (mpeg1.js:829-834, SURVEY Q8)
	}
	uint2 unused[8];
	reconstruct_at<false, BIDIR>(params, ty, mb_row, mb_col, b, in_picture, tid & 31, stage + (tid >> 5) * WARP_STAGE, unused);
}

#ifndef JSMPEG_WALK_EMU  // (a CTA-wide barrier: outside what the one-warp host emulation runs)
// ---- fused planar -> RGBA epilogue (SURVEY 8f rank 2, src/canvas2d.js:53-122) ------------------------------------
// A CTA of three warps owns 16 macroblocks of one macroblock row: warp 0 their 32 top luma blocks, warp 1 the 32
// bottom ones, warp 2 the 16 Cb and the 16 Cr blocks.  All reconstruct (and write their planes, the next picture
// needs them); the chroma warp also leaves its 16 x 8 x 8 samples twice in shared memory; after one barrier the
// luma threads convert their own 8 x 8 samples, still in registers, with the 4 x 4 chroma samples that cover them,
// and write 8 rows of 32 RGBA bytes.  The planes are never read back.
//     r = Cr + (Cr * 103 >> 8) - 179,  g = (Cb * 88 >> 8) - 44 + (Cr * 183 >> 8) - 91,  b = Cb + (Cb * 198 >> 8) - 227
//     R = clamp(Y + r), G = clamp(Y - g), B = clamp(Y + b), A = 255
// (canvas2d.js names its parameters (y, cb, cr) but is CALLED with (Y, Cr, Cb), mpeg1.js:217 -- its `ccb` is a Cr
// sample, SURVEY Q8.)  Only (width >> 1) x (height >> 1) quads are converted (canvas2d.js:77-78); the odd edge of
// the image keeps the opaque white the buffer is created with (canvas2d.js:24-29).
constexpr int RGBA_THREADS = 96, RGBA_MBS = 16;

struct RgbaTarget {
	uint8_t *rgba;          // display size, RGBA8888
	int32_t width, height;  // display size
};

__device__ __forceinline__ uint32_t rgba_px(int y, int r, int g, int b) {
	auto c = [](int v) { return (uint32_t)min(255, max(0, v)); };  // Uint8ClampedArray
	return c(y + r) | (c(y - g) << 8) | (c(y + b) << 16) | 0xff000000u;
}

template <bool BIDIR = false, class PARAMS>
__device__ __forceinline__ void reconstruct_rgba_block(const PARAMS &params, const RgbaTarget &out, int ty, int mb_row, int first_mb_col,
                                                       int tid, uint8_t *stage, uint8_t (*chroma)[8][RGBA_MBS * 8]) {
	const auto &t = params.t[ty];
	const int warp = tid >> 5, lane = tid & 31;
	int b, local;  // local = macroblock within the CTA's 16
	if (warp < 2) { b = warp * 2 + (lane & 1); local = lane >> 1; }
	else { b = 4 + (lane >> 4); local = lane & 15; }
	const int mb_col = first_mb_col + local;
	// the grid covers the launch's widest and tallest picture: a CTA outside this one's rows or columns only joins the barrier
	const bool in_picture = mb_col < t.mb_width && mb_row < t.mb_height;
	uint2 rows[8];
#pragma unroll
	for (int r = 0; r < 8; r++) rows[r] = make_uint2(0u, 0u);
	reconstruct_at<true, BIDIR>(params, ty, mb_row, in_picture ? mb_col : 0, b, in_picture, lane, stage + warp * WARP_STAGE, rows);
	if (warp == 2) {
		// plane 0 = Cb (block 4), plane 1 = Cr (block 5)
#pragma unroll
		for (int r = 0; r < 8; r++) *reinterpret_cast<uint2 *>(&chroma[b - 4][r][local * 8]) = rows[r];
	}
	__syncthreads();
	if (warp == 2 || !in_picture || !out.rgba) return;
	const int x0 = mb_col * 16 + (b & 1) * 8, y0 = mb_row * 16 + (b >> 1) * 8;  // this block's top-left sample
	const int cx0 = local * 8 + (b & 1) * 4, cy0 = (b >> 1) * 4;                  // its chroma samples in the CTA's tile
	const int xlim = (out.width >> 1) * 2, ylim = (out.height >> 1) * 2;
	if (x0 >= xlim || y0 >= ylim) return;
	const bool whole = x0 + 8 <= xlim && (out.width & 3) == 0;  // 16-byte stores need aligned rows
#pragma unroll
	for (int r = 0; r < 8; r++) {
		if (y0 + r >= ylim) break;
		const uint32_t cb4 = *reinterpret_cast<const uint32_t *>(&chroma[0][cy0 + (r >> 1)][cx0]);
		const uint32_t cr4 = *reinterpret_cast<const uint32_t *>(&chroma[1][cy0 + (r >> 1)][cx0]);
		uint32_t px[8];
#pragma unroll
		for (int i = 0; i < 8; i++) {
			const int cb = (int)((cb4 >> (8 * (i >> 1))) & 255u), cr = (int)((cr4 >> (8 * (i >> 1))) & 255u);
			const int rr = (cr + ((cr * 103) >> 8)) - 179;
			const int gg = ((cb * 88) >> 8) - 44 + ((cr * 183) >> 8) - 91;
			const int bb = (cb + ((cb * 198) >> 8)) - 227;
			const int yy = (int)(((i < 4 ? rows[r].x : rows[r].y) >> (8 * (i & 3))) & 255u);
			px[i] = rgba_px(yy, rr, gg, bb);
		}
		uint32_t *dstp = reinterpret_cast<uint32_t *>(out.rgba) + (size_t)(y0 + r) * out.width + x0;
		if (whole) {
			reinterpret_cast<uint4 *>(dstp)[0] = make_uint4(px[0], px[1], px[2], px[3]);
			reinterpret_cast<uint4 *>(dstp)[1] = make_uint4(px[4], px[5], px[6], px[7]);
		} else {
#pragma unroll
			for (int i = 0; i < 8; i++)
				if (x0 + i < xlim) dstp[i] = px[i];
		}
	}
}

#endif

}  // namespace
