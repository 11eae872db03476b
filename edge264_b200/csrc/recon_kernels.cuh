/* recon_kernels.cuh — what the sm_100a kernels of the pixel-reconstruction path share: the picture job, the per-warp
 * shared-memory tile, mbarrier / cp.async.bulk helpers, the inverse transforms (reference edge264_residual.c:108-538)
 * and the intra predictors (edge264_intra.c:291-765).  The kernels themselves:
 *   inter_kernels.cuh    e264_inter4_kernel      inter macroblocks: inverse transform + motion compensation + weighting
 *   intra_kernels.cuh    e264_intra_kernel       intra macroblocks of P/B pictures, in dependency order (flags)
 *                        e264_intra_rows_kernel  intra pictures: band wavefront
 *   deblock_kernels.cuh  e264_deblock_kernel     boundary strengths + the in-loop filter: band wavefront
 * Up to three launches per picture.  Arithmetic is restated from ITU-T H.264 with the reference's observable integer
 * widths; results are bit-exact with the reference decoder (tests/test_gpu_parity.py). */
#pragma once
#include <cstddef>
#include <cuda_runtime.h>
#include <stdint.h>
#include "records.h"
#include "h264_tables.h"

struct PicJob {
	const E264MbRec *recs; const int16_t *coefs; const E264SliceRec *slices;
	uint8_t *frames;
	int frame_bytes, w_mbs, h_mbs, stride_y, stride_c, plane_y, dst_slot, n_slots;
	unsigned *flags;      /* [nmb] "reconstructed" == epoch, then [3][h_mbs] row progress (epoch * 2048 + macroblocks done): deblocking luma, deblocking chroma, intra pictures */
	unsigned epoch;
	unsigned *tickets;    /* [4] this picture's ticket words: 1 deblock bands, 2 intra list / intra bands */
	unsigned *tickets_next;   /* [4] the next picture's: every kernel clears them on entry (pictures alternate between two sets, so no memset and no extra launch separates two pictures) */
	unsigned *err;
	int rows_mode;
	struct E264DbkMb *dbk;        /* [nmb] deblocking digests written by e264_prepass_kernel; NULL = picture is not deblocked */
	const uint32_t *intra_list;   /* addresses of the intra macroblocks in raster order */
	int n_intra;
	unsigned long long *trace;   /* measurement only (e264b_replay): [trace_base + kind] = {first block start, last block end} in globaltimer ns; kinds: 1 inter, 2 intra, 3 deblock */
	int trace_base;
	const unsigned *trace_rep;   /* graph replay: device counter of the repetition under way; its slots start trace_rep_stride further on */
	int trace_rep_stride;
	int diag;                    /* measurement only: count block placement per SM (g_diag_*) */
};

#define WARPS_PER_BLOCK 4
#define YT_STRIDE 48     /* luma tile row: [15]=left neighbour, [16..31]=samples, [32..39]=top-right */
#define CT_STRIDE 16     /* chroma tile row: [7]=left neighbour, [8..15]=samples */
struct __align__(16) WarpSmem {
	uint4 rec4[12];                 /* the macroblock record */
	int16_t res[384];               /* residual: luma y*16+x, then Cb, Cr 8x8 */
	uint8_t ytile[17 * YT_STRIDE];  /* row 0 = samples above the macroblock */
	uint8_t ctile[2][9 * CT_STRIDE];
	int dc[24];                     /* scaled DC: 16 luma (raster over blocks), 4 Cb, 4 Cr */
	union {
		int16_t t8[4 * 64];         /* 8x8 transform transpose buffer */
		int edge[2][28];            /* intra 8x8 filtered reference samples */
	} u;
};

__device__ __forceinline__ int clip255(int v) { return min(max(v, 0), 255); }
__device__ __forceinline__ int sat16(int v) { return min(max(v, -32768), 32767); }
__device__ __forceinline__ int blk_x(int b) { return (b & 1) | ((b >> 1) & 2); }
__device__ __forceinline__ int blk_y(int b) { return ((b >> 1) & 1) | ((b >> 2) & 2); }
__device__ __forceinline__ int blk_z(int x, int y) { return (x & 1) | ((y & 1) << 1) | ((x & 2) << 1) | ((y & 2) << 2); }
__device__ __forceinline__ int norm4(int m, int i, int j) { return h264_norm4x4[m][((i & 1) && (j & 1)) ? 1 : (!(i & 1) && !(j & 1)) ? 0 : 2]; }
__device__ __forceinline__ int norm8(int m, int i, int j) {
	int k;
	if (!(i & 3) && !(j & 3)) k = 0;
	else if ((i & 1) && (j & 1)) k = 1;
	else if ((i & 3) == 2 && (j & 3) == 2) k = 2;
	else if ((!(i & 3) && (j & 1)) || ((i & 1) && !(j & 3))) k = 3;
	else if ((!(i & 3) && (j & 3) == 2) || ((i & 3) == 2 && !(j & 3))) k = 4;
	else k = 5;
	return h264_norm8x8[m][k];
}

__device__ __forceinline__ void reset_next_tickets(const PicJob &J) { if (blockIdx.x == 0 && threadIdx.x < 4) J.tickets_next[threadIdx.x] = 0; }

/* measurement only (replay with E264B_DIAG=1): how the blocks of each kernel kind land on the SMs —
 * [kind][sm]: blocks started, blocks of this kind resident right now, the maximum of that */
__device__ unsigned g_diag_cnt[4][160], g_diag_cur[4][160], g_diag_max[4][160];
/* -DE264_ROWS_TIMING / -DE264_INTER_TIMING (make variants): SM cycles the warps of e264_intra_rows_kernel spend per part
 * of a macroblock step, or those of e264_inter4_kernel per part of a chunk */
__device__ unsigned long long g_diag_phase[16];
#ifdef E264_ROWS_TIMING
#define RT_DECL unsigned rt_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}; unsigned rt_t = (unsigned)clock64();
#define RT_MARK(k) { const unsigned rt_n = (unsigned)clock64(); rt_acc[k] += rt_n - rt_t; rt_t = rt_n; }
#define RT_FLUSH(base) if (lane == 0) { for (int rt_k = 0; rt_k < 8; rt_k++) atomicAdd(&g_diag_phase[(base) + rt_k], (unsigned long long)rt_acc[rt_k]); }
#else
#define RT_DECL
#define RT_MARK(k)
#define RT_FLUSH(base)
#endif
/* -DE264_INTER_TIMING (make variants): SM cycles the warps of e264_inter4_kernel spend per part of a chunk, all warps
 * summed: 0 records + binning, 1 interpolation, 2 digest, 3 residual, 4 combine + store (a barrier's wait counts to the
 * part in front of it) */
#ifdef E264_INTER_TIMING
#define IT_DECL unsigned long long it_acc[5] = {0, 0, 0, 0, 0}; long long it_t = clock64();
#define IT_MARK(k) { const long long it_n = clock64(); it_acc[k] += (unsigned long long)(it_n - it_t); it_t = it_n; }
#define IT_FLUSH if (lane == 0) { for (int it_k = 0; it_k < 5; it_k++) atomicAdd(&g_diag_phase[it_k], it_acc[it_k]); }
#else
#define IT_DECL
#define IT_MARK(k)
#define IT_FLUSH
#endif
/* measurement only: first-start / last-end timestamps of a launch, see e264b_replay */
struct TraceScope {
	unsigned long long *t; int dk; unsigned sm;
	__device__ __forceinline__ static unsigned long long now() { unsigned long long v; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v)); return v; }
	/* one thread per block: two atomics per block keep the timed replay undisturbed (a block's first warp starts it, its exit is within one macroblock of the block's end) */
	__device__ __forceinline__ TraceScope(const PicJob &J, int kind) { t = J.trace ? J.trace + 2 * ((size_t)J.trace_base + kind + (J.trace_rep ? (size_t)*J.trace_rep * J.trace_rep_stride : 0)) : nullptr; if (t && threadIdx.x == 0) atomicMin(t, now());
		dk = -1;
		if (J.diag && threadIdx.x == 0) { dk = kind; asm volatile("mov.u32 %0, %%smid;" : "=r"(sm)); sm = sm < 160 ? sm : 159; atomicAdd(&g_diag_cnt[kind][sm], 1u); unsigned c = atomicAdd(&g_diag_cur[kind][sm], 1u) + 1; atomicMax(&g_diag_max[kind][sm], c); } }
	__device__ __forceinline__ ~TraceScope() { if (t && threadIdx.x == 0) atomicMax(t + 1, now()); if (dk >= 0 && threadIdx.x == 0) atomicSub(&g_diag_cur[dk][sm], 1u); }
};

/* Dependency waits are bounded so that a bug cannot hang the GPU: they give up after ~0.2 s of SM clocks, or at once when
 * another warp has already raised the error flag. */
/* spin until flags[idx] == epoch, with acquire loads (no fence behind it): several lanes of a warp may each wait for their
 * own flag, so the round trips to L2 overlap instead of adding up; a __syncwarp() behind the waits orders the other lanes' loads */
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) { unsigned v; asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ bool wait_flag_acquire(const unsigned *flags, int idx, unsigned epoch, unsigned *err) {
	const unsigned *f = flags + idx;
	unsigned spins = 0;
	long long t0 = 0;
	bool ok = true;
	while (ok && ld_acquire_u32(f) != epoch) {
		__nanosleep(64);
		if ((++spins & 63) == 0) {
			if (*(const volatile unsigned *)err) ok = false;
			else if (t0 == 0) t0 = clock64();
			else if (clock64() - t0 > 400000000ll) { atomicExch(err, 1u); ok = false; }
		}
	}
	return ok;
}
/* ---- shared-memory barrier + TMA helpers (sm_90+ PTX; SASS: SYNCS.*, UBLKCP, UTMALDG) ---- */
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(void *bar, unsigned count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, unsigned bytes, void *bar) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
	             :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
/* wait for the phase with the given parity; gives up after ~10 ms of SM clocks (a window arrives in
 * microseconds), false = gave up (the caller raises the error flag).  One loop, one exit: ptxas reconverges the
 * warp behind it, which the __syncwarp()s that follow rely on (they compile to NOPs where the compiler has proved
 * convergence). */
__device__ __forceinline__ bool mbar_wait(void *bar, unsigned parity) {
	unsigned done = 0;
	const long long t0 = clock64();
	do {
		asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
		             : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
	} while (!done && clock64() - t0 < 20000000ll);
	return done != 0;
}

/* ------------------------------------------------------------------------------------------ */
/* residual                                                                                     */
/* ------------------------------------------------------------------------------------------ */
/* 4x4 inverse transform of 16 levels at c (16-byte aligned) -> residual o[y*4+x] in registers, saturated to int16 */
static_assert(offsetof(E264SliceRec, scaling4x4) % 8 == 0 && sizeof(E264SliceRec) % 8 == 0, "idct4x4 loads a 4x4 scaling list as two 8-byte words");
__device__ __forceinline__ void idct4x4_core(const int16_t *c, bool have_levels, const uint8_t *scaling, int qp, bool dc_override, int dc, int o[16]) {
	int d[16];
	if (have_levels) {
		uint4 a = *(const uint4 *)c, b = *((const uint4 *)c + 1);   /* c points into the TMA-staged shared copy */
		int16_t lv[16];
		*(uint4 *)lv = a; *(uint4 *)(lv + 8) = b;
		int sh = qp / 6, m = qp - sh * 6;
		/* the 16 weights arrive as two 8-byte loads (the lists sit at offset 904 + 16 k of 1128-byte slice records: 8-byte
		 * aligned), the three normalisation values of this qp % 6 once */
		const uint2 s01 = __ldg((const uint2 *)scaling), s23 = __ldg((const uint2 *)scaling + 1);
		const uint32_t sw[4] = {s01.x, s01.y, s23.x, s23.y};
		const int n0 = h264_norm4x4[m][0], n1 = h264_norm4x4[m][1], n2 = h264_norm4x4[m][2];
#pragma unroll
		for (int i = 0; i < 4; i++)
#pragma unroll
			for (int j = 0; j < 4; j++) {
				const int nrm = ((i & 1) && (j & 1)) ? n1 : (!(i & 1) && !(j & 1)) ? n0 : n2;
				int ls = (int)((sw[i] >> (8 * j)) & 255u) * nrm;
				d[i * 4 + j] = (int)(((unsigned)(lv[i * 4 + j] * ls) << sh) + 8u) >> 4;
			}
	} else {
#pragma unroll
		for (int i = 0; i < 16; i++) d[i] = 0;
	}
	if (dc_override) d[0] = dc;
	int f[16];
#pragma unroll
	for (int i = 0; i < 4; i++) {
		int e0 = d[i * 4] + d[i * 4 + 2], e1 = d[i * 4] - d[i * 4 + 2];
		int e2 = (d[i * 4 + 1] >> 1) - d[i * 4 + 3], e3 = d[i * 4 + 1] + (d[i * 4 + 3] >> 1);
		f[i * 4] = e0 + e3; f[i * 4 + 1] = e1 + e2; f[i * 4 + 2] = e1 - e2; f[i * 4 + 3] = e0 - e3;
	}
#pragma unroll
	for (int j = 0; j < 4; j++) {
		int g0 = f[j] + f[8 + j], g1 = f[j] - f[8 + j];
		int g2 = (f[4 + j] >> 1) - f[12 + j], g3 = f[4 + j] + (f[12 + j] >> 1);
		o[j] = sat16((g0 + g3 + 32) >> 6);
		o[4 + j] = sat16((g1 + g2 + 32) >> 6);
		o[8 + j] = sat16((g1 - g2 + 32) >> 6);
		o[12 + j] = sat16((g0 - g3 + 32) >> 6);
	}
}
/* the same, residual written to dst[y*dstride+x] */
__device__ __noinline__ void idct4x4(const int16_t *c, bool have_levels, const uint8_t *scaling, int qp, bool dc_override, int dc, int16_t *dst, int dstride) {
	int o[16];
	idct4x4_core(c, have_levels, scaling, qp, dc_override, dc, o);
#pragma unroll
	for (int y = 0; y < 4; y++)
#pragma unroll
		for (int x = 0; x < 4; x++) dst[y * dstride + x] = (int16_t)o[y * 4 + x];
}

/* one 8-point pass in the reference's int16 arithmetic (edge264_residual.c:250-296) */
__device__ __forceinline__ void idct8_1d(short a[8]) {
	short e0 = (short)(a[0] + a[4]), e1 = (short)(a[5] - a[3] - (short)((a[7] >> 1) + a[7])), e2 = (short)(a[0] - a[4]);
	short e3 = (short)(a[1] + a[7] - (short)((a[3] >> 1) + a[3])), e4 = (short)((a[2] >> 1) - a[6]);
	short e5 = (short)(a[7] - a[1] + (short)((a[5] >> 1) + a[5])), e6 = (short)((a[6] >> 1) + a[2]);
	short e7 = (short)(a[3] + a[5] + (short)((a[1] >> 1) + a[1]));
	short f0 = (short)(e0 + e6), f1 = (short)((e7 >> 2) + e1), f2 = (short)(e2 + e4), f3 = (short)((e5 >> 2) + e3);
	short f4 = (short)(e2 - e4), f5 = (short)((e3 >> 2) - e5), f6 = (short)(e0 - e6), f7 = (short)(e7 - (e1 >> 2));
	a[0] = (short)(f0 + f7); a[1] = (short)(f2 + f5); a[2] = (short)(f4 + f3); a[3] = (short)(f6 + f1);
	a[4] = (short)(f6 - f1); a[5] = (short)(f4 - f3); a[6] = (short)(f2 - f5); a[7] = (short)(f0 - f7);
}

/* luma of a macroblock with the 8x8 transform: lane (blk, k) = (lane >> 3, lane & 7) runs row k then column k of 8x8 block
 * blk through the two passes; the residual of every coded 8x8 block goes to ws->res (luma y*16+x), the others are not
 * written.  cf_luma: the macroblock's first luma level in the staged coefficient run. */
__device__ __forceinline__ void residual_luma8x8(WarpSmem *ws, const E264MbRec *r, const E264SliceRec *sr, const int16_t *cf_luma, int lane) {
	const unsigned coded = r->coded;
	const int inter = r->kind == MBK_INTER, qpy = r->qp[0];
	int blk = lane >> 3, k = lane & 7;
	bool on = (coded >> (blk * 4)) & 1;
	short a[8];
	if (on) {
		int idx = __popc(coded & 0x1111 & ((1u << (blk * 4)) - 1));
		uint4 q = *(const uint4 *)(cf_luma + idx * 64 + k * 8);
		short lv[8]; *(uint4 *)lv = q;
		int div = qpy / 6, m = qpy - div * 6;
		const uint8_t *sc = sr->scaling8x8[inter] + k * 8;
#pragma unroll
		for (int j = 0; j < 8; j++) {
			int ls = sc[j] * norm8(m, k, j);
			a[j] = div < 6 ? (short)sat16((lv[j] * ls + (1 << (5 - div))) >> (6 - div)) : (short)(lv[j] * (short)(ls << (div - 6)));
		}
		idct8_1d(a);
#pragma unroll
		for (int j = 0; j < 8; j++) ws->u.t8[blk * 64 + k * 8 + j] = a[j];
	}
	__syncwarp();
	if (on) {
#pragma unroll
		for (int j = 0; j < 8; j++) a[j] = ws->u.t8[blk * 64 + j * 8 + k];
		a[0] = (short)(a[0] + 32);
		idct8_1d(a);
		int x = (blk & 1) * 8 + k, y0 = (blk >> 1) * 8;
#pragma unroll
		for (int j = 0; j < 8; j++) ws->res[(y0 + j) * 16 + x] = (short)(a[j] >> 6);
	}
	__syncwarp();
}

/* scaled DC of chroma 4x4 block i of plane pl: the 2x2 transform of the plane's four DC levels at cdc (8.5.11) */
__device__ __forceinline__ int chroma_dc(const int16_t *cdc, const E264MbRec *r, const E264SliceRec *sr, int inter, int pl, int i) {
	const int a = cdc[4 * pl], b = cdc[4 * pl + 1], c = cdc[4 * pl + 2], d = cdc[4 * pl + 3];
	const int f = i == 0 ? a + b + c + d : i == 1 ? a - b + c - d : i == 2 ? a + b - c - d : a - b - c + d;
	const int qpc = r->qp[1 + pl];
	const int ls = (sr->scaling4x4[1 + pl + inter * 3][0] * h264_norm4x4[qpc % 6][0]) << (qpc / 6);
	return (f * ls) >> 5;
}

/* cf: this macroblock's coefficient run, staged in shared memory by the caller (cp.async.bulk) */
__device__ __noinline__ void residual_stage(WarpSmem *ws, const E264MbRec *r, const E264SliceRec *sr, const int16_t *cf, int lane) {
	/* clear */
	uint4 z = make_uint4(0, 0, 0, 0);
	((uint4 *)ws->res)[lane] = z;
	if (lane < 16) ((uint4 *)ws->res)[32 + lane] = z;
	const unsigned coded = r->coded;
	const int inter = r->kind == MBK_INTER, i16 = r->kind == MBK_I16x16;
	const int qpy = r->qp[0];
	/* --- DC transforms first --- */
	if (coded & CODED_Y_DC) {
		if (lane < 16) {
			int i = lane >> 2, j = lane & 3, u = 0;
			const unsigned neg[4] = {0x0, 0xC, 0x6, 0xA};
#pragma unroll
			for (int k = 0; k < 4; k++)
#pragma unroll
				for (int l = 0; l < 4; l++) {
					int v = cf[k * 4 + l];
					int s = ((neg[i] >> k) ^ (neg[j] >> l)) & 1;
					u += s ? -v : v;
				}
			int ls = (sr->scaling4x4[0][0] * h264_norm4x4[qpy % 6][0]) << (qpy / 6);
			ws->dc[lane] = (u * ls + 32) >> 6;
		}
		cf += 16;
	} else if (lane < 16) ws->dc[lane] = 0;
	const int n_luma = (r->flags & MBF_T8x8) ? 64 * __popc(coded & 0x1111) : 16 * __popc(coded & 0xffff);
	const int16_t *cf_luma = cf;
	cf += n_luma;
	const bool any_cdc = (coded & (CODED_CB_DC | CODED_CR_DC)) != 0;
	if (lane >= 16 && lane < 24) {
		const int pl = (lane - 16) >> 2, i = lane & 3;
		ws->dc[16 + pl * 4 + i] = any_cdc ? chroma_dc(cf, r, sr, inter, pl, i) : 0;
	}
	if (any_cdc) cf += 8;
	__syncwarp();
	if (r->flags & MBF_T8x8) residual_luma8x8(ws, r, sr, cf_luma, lane);
	/* --- 4x4 blocks: luma on lanes 0..15 (unless the macroblock uses the 8x8 transform) and chroma AC (+DC) on lanes
	 * 16..23 go through ONE call of the transform --- */
	{
		bool act = false, on = false, dcov = false;
		const int16_t *src = cf; const uint8_t *scal = sr->scaling4x4[0]; int qp = qpy, dc = 0, stride = 16; int16_t *dst = ws->res;
		if (lane < 16) {
			if (!(r->flags & MBF_T8x8)) {
				const int b = lane, bx = blk_x(b), by = blk_y(b);
				on = (coded >> b) & 1; dcov = i16 && (coded & CODED_Y_DC); act = on || dcov;
				src = cf_luma + __popc(coded & ((1u << b) - 1)) * 16; scal = sr->scaling4x4[inter * 3]; dcov = i16; dc = ws->dc[by * 4 + bx];
				dst = ws->res + by * 4 * 16 + bx * 4;
			}
		} else if (lane < 24) {
			const int j = lane - 16, pl = j >> 2, i = j & 3;
			on = (coded >> (16 + j)) & 1; act = on || any_cdc; dcov = true;
			src = cf + __popc((coded >> 16) & ((1u << j) - 1) & 0xff) * 16; scal = sr->scaling4x4[1 + pl + inter * 3]; qp = r->qp[1 + pl]; dc = ws->dc[16 + pl * 4 + i];
			dst = ws->res + 256 + pl * 64 + (i >> 1) * 4 * 8 + (i & 1) * 4; stride = 8;
		}
		if (act) idct4x4(src, on, scal, qp, dcov, dc, dst, stride);
	}
	__syncwarp();
}

/* ------------------------------------------------------------------------------------------ */
/* intra prediction                                                                             */
/* ------------------------------------------------------------------------------------------ */
#define YT(x, y) ws->ytile[((y) + 1) * YT_STRIDE + 16 + (x)]     /* x in -1..23, y in -1..15 */
#define CT(pl, x, y) ws->ctile[pl][((y) + 1) * CT_STRIDE + 8 + (x)]

/* ---- Intra 4x4 / 8x8 prediction: one edge vector in registers, a table of taps, three shuffles ----
 * Every directional predictor of 8.3.1.2 / 8.3.2.2 is a copy, a 2-tap or a 3-tap average of ADJACENT entries of one
 * vector  E = [L(N-1) L(N-1) .. L0  TL  T0 .. T(2N-1)  T(2N-1)]  (the duplicated ends absorb the "3*last" cases), so a
 * lane holds one entry of E, a 64-bit constant per sample holds (index, kind) for the 9 modes, and a block costs one
 * shared-memory load, three shuffles and a handful of integer instructions instead of a per-sample walk over the tile.
 * (reference formulation: the shuffle-table predictors of edge264_intra.c:13-420; same arithmetic, other machinery). */
struct IntraTap { int idx, kind; };   /* kind 0: E[idx]; 1: (E[idx] + E[idx+1] + 1) >> 1; 2: (E[idx] + 2 E[idx+1] + E[idx+2] + 2) >> 2 */
constexpr IntraTap intra_tap(int N, int mode, int x, int y) {
	const int bT = N + 2, bL = N;        /* T(i) = E[bT + i], L(i) = E[bL - i], TL = E[N + 1] */
	switch (mode) {
	case 0: return {bT + x, 0};
	case 1: return {bL - y, 0};
	case 3: return {bT + x + y, 2};
	case 4: return {x > y ? bT + x - y - 2 : x < y ? bL - (y - x) : bL, 2};
	case 5: { const int z = 2 * x - y;
		if (z >= 0 && !(z & 1)) return {bT + x - (y >> 1) - 1, 1};
		if (z > 0) return {bT + x - (y >> 1) - 2, 2};
		if (z == -1) return {bL, 2};
		return {bL - (y - 2 * x - 1), 2}; }
	case 6: { const int z = 2 * y - x;
		if (z >= 0 && !(z & 1)) return {bL - (y - (x >> 1)), 1};
		if (z > 0) return {bL - (y - (x >> 1)), 2};
		if (z == -1) return {bL, 2};
		return {bT + x - 2 * y - 3, 2}; }
	case 7: return {bT + x + (y >> 1), (y & 1) ? 2 : 1};
	case 8: { const int z = x + 2 * y, k = y + (x >> 1);
		if (z > 2 * N - 3) return {1, 0};
		if (z == 2 * N - 3) return {0, 2};
		if (!(z & 1)) return {bL - (k + 1), 1};
		return {bL - (k + 2), 2}; }
	default: return {0, 0};
	}
}
struct I4Taps { uint64_t v[16];
	constexpr I4Taps() : v{} { for (int p = 0; p < 16; p++) { uint64_t w = 0; for (int m = 0; m < 9; m++) { const IntraTap t = intra_tap(4, m, p & 3, p >> 2); w |= (uint64_t)(t.idx | t.kind << 4) << (6 * m); } v[p] = w; } } };
struct I8Taps { uint64_t v[64];
	constexpr I8Taps() : v{} { for (int p = 0; p < 64; p++) { uint64_t w = 0; for (int m = 0; m < 9; m++) { const IntraTap t = intra_tap(8, m, p & 7, p >> 3); w |= (uint64_t)(t.idx | t.kind << 5) << (7 * m); } v[p] = w; } } };
__device__ const I4Taps e264_i4taps = I4Taps();
__device__ const I8Taps e264_i8taps = I8Taps();

__device__ __forceinline__ int intra_tap_apply(int E, int idx, int kind) {
	const int a = __shfl_sync(0xffffffffu, E, idx), b = __shfl_sync(0xffffffffu, E, idx + 1), c = __shfl_sync(0xffffffffu, E, idx + 2);
	return kind == 2 ? (a + 2 * b + c + 2) >> 2 : kind == 1 ? (a + b + 1) >> 1 : a;
}

/* one 4x4 block at tile coordinate (X0, Y0) per HALF-WARP: lane hl = lane & 15 of half `half` returns its predicted sample
 * (x = hl & 3, y = hl >> 2); the two halves work on different blocks with different modes, so nothing here branches on
 * the mode — the DC sum and the tap shuffles are both computed (a shuffle inside diverged code can hang) */
__device__ __forceinline__ int pred4x4_half(const WarpSmem *ws, int X0, int Y0, int imode, uint64_t taps, int hl, int half) {
	const int mode = imode & 15, un = imode >> 4;
	const bool hasA = !(un & 1), hasB = !(un & 2);
	const int e = min(hl, 14);
	int i = min(e - 6, 7); if ((un & 4) && i > 3) i = 3;          /* top-right unavailable: T4..T7 = T3 */
	const int E = YT(X0 + (e <= 5 ? -1 : i), Y0 + (e <= 4 ? min(4 - e, 3) : -1));
	int s = (hl < 15 && ((e >= 6 && e <= 9 && hasB) || (e >= 1 && e <= 4 && hasA))) ? E : 0;
	s += __shfl_xor_sync(0xffffffffu, s, 1); s += __shfl_xor_sync(0xffffffffu, s, 2); s += __shfl_xor_sync(0xffffffffu, s, 4); s += __shfl_xor_sync(0xffffffffu, s, 8);
	const int dc = (hasA && hasB) ? (s + 4) >> 3 : (hasA || hasB) ? (s + 2) >> 2 : 128;
	const int ent = (int)(taps >> (6 * mode)) & 63;
	const int idx = (ent & 15) + half * 16, kind = ent >> 4;
	const int a = __shfl_sync(0xffffffffu, E, idx), b = __shfl_sync(0xffffffffu, E, (idx + 1) & 31), c = __shfl_sync(0xffffffffu, E, (idx + 2) & 31);
	const int dir = kind == 2 ? (a + 2 * b + c + 2) >> 2 : kind == 1 ? (a + b + 1) >> 1 : a;
	return mode == 2 ? dc : dir;
}

/* one 8x8 block: reference samples filtered in registers (8.3.2.2.1), then two samples per lane (rows y and y + 4) */
__device__ __forceinline__ void pred8x8_warp(const WarpSmem *ws, int X0, int Y0, int imode, uint64_t taps0, uint64_t taps1, int lane, int &v0, int &v1) {
	const int mode = imode & 15, un = imode >> 4;
	const bool hasA = !(un & 1), hasB = !(un & 2), hasD = !(un & 8);
	const int e = min(lane, 26);
	int i = min(e - 10, 15); if ((un & 4) && i > 7) i = 7;
	const int raw = YT(X0 + (e <= 9 ? -1 : i), Y0 + (e <= 8 ? min(8 - e, 7) : -1));
	int lo = __shfl_up_sync(0xffffffffu, raw, 1), hi = __shfl_down_sync(0xffffffffu, raw, 1);
	if ((e == 9 && !hasA) || (e == 10 && !hasD)) lo = raw;
	if ((e == 9 && !hasB) || (e == 8 && !hasD)) hi = raw;
	int E = (lo + 2 * raw + hi + 2) >> 2;
	if ((e >= 10 && !hasB) || (e <= 8 && !hasA) || (e == 9 && !hasD)) E = 128;
	E = __shfl_sync(0xffffffffu, E, min(max(e, 1), 25));     /* the duplicated ends */
	if (mode == 2) {
		int s = ((e >= 10 && e <= 17 && hasB) || (e >= 1 && e <= 8 && hasA)) ? E : 0;
		s += __shfl_xor_sync(0xffffffffu, s, 1); s += __shfl_xor_sync(0xffffffffu, s, 2); s += __shfl_xor_sync(0xffffffffu, s, 4);
		s += __shfl_xor_sync(0xffffffffu, s, 8); s += __shfl_xor_sync(0xffffffffu, s, 16);
		v0 = v1 = (hasA && hasB) ? (s + 8) >> 4 : (hasA || hasB) ? (s + 4) >> 3 : 128;
		return;
	}
	const int e0 = (int)(taps0 >> (7 * mode)) & 127, e1 = (int)(taps1 >> (7 * mode)) & 127;
	v0 = intra_tap_apply(E, e0 & 31, e0 >> 5);
	v1 = intra_tap_apply(E, e1 & 31, e1 >> 5);
}

/* four predicted samples (bytes of p) plus four int16 residuals (r01 = first two, r23 = last two), clipped to 8 bits;
 * the sum wraps in 16 bits first like the reference's saturating 16-bit adds never see it: v + res fits unless res is garbage */
__device__ __forceinline__ uint32_t intra_add_res4(uint32_t p, uint32_t r01, uint32_t r23) {
	const int v0 = clip255((short)((int)(p & 255u) + (short)(r01 & 0xffffu))), v1 = clip255((short)((int)((p >> 8) & 255u) + (short)(r01 >> 16)));
	const int v2 = clip255((short)((int)((p >> 16) & 255u) + (short)(r23 & 0xffffu))), v3 = clip255((short)((int)(p >> 24) + (short)(r23 >> 16)));
	return (uint32_t)v0 | (uint32_t)v1 << 8 | (uint32_t)v2 << 16 | (uint32_t)v3 << 24;
}

__device__ __noinline__ void intra_luma(WarpSmem *ws, const E264MbRec *r, int lane) {
	if (r->kind == MBK_I4x4) {
		/* the 16 blocks along anti-diagonals: block (x, y) in step x + 2 y, so its left, top, top-left and top-right
		 * neighbours are finished (8.3.1.2: top-right counts only where it precedes in decoding order — the record's
		 * availability bits say so); two blocks per step in the two half-warps, 10 steps instead of 16 */
		const int hl = lane & 15, half = lane >> 4, x = hl & 3, y = hl >> 2;
		const uint64_t taps = __ldg(&e264_i4taps.v[hl]);
#pragma unroll 1
		for (int st = 0; st < 10; st++) {
			const int by = (st < 2 ? 0 : (st - 2) >> 1) + half, bx = st - 2 * by;
			const bool on = bx >= 0 && bx < 4 && by < 4;
			const int X0 = on ? bx * 4 : 0, Y0 = on ? by * 4 : 0;
			int v = pred4x4_half(ws, X0, Y0, r->modes[on ? blk_z(bx, by) : 0], taps, hl, half);
			v = clip255((short)(v + ws->res[(Y0 + y) * 16 + X0 + x]));
			if (on) YT(X0 + x, Y0 + y) = (uint8_t)v;   /* the reads above touch only samples outside the two blocks of this step */
			__syncwarp();
		}
	} else if (r->kind == MBK_I8x8) {
		const uint64_t taps0 = __ldg(&e264_i8taps.v[lane]), taps1 = __ldg(&e264_i8taps.v[lane + 32]);
#pragma unroll 1
		for (int i = 0; i < 4; i++) {
			const int X0 = (i & 1) * 8, Y0 = (i >> 1) * 8, x = lane & 7, y = lane >> 3;
			int v0, v1;
			pred8x8_warp(ws, X0, Y0, r->modes[i], taps0, taps1, lane, v0, v1);
			v0 = clip255((short)(v0 + ws->res[(Y0 + y) * 16 + X0 + x]));
			v1 = clip255((short)(v1 + ws->res[(Y0 + y + 4) * 16 + X0 + x]));
			YT(X0 + x, Y0 + y) = (uint8_t)v0; YT(X0 + x, Y0 + y + 4) = (uint8_t)v1;
			__syncwarp();
		}
	} else {   /* Intra16x16: lanes 0-15 hold the row above, 16-31 the column to the left; a lane predicts 8 samples of one row */
		const int mode = r->i16_mode & 15, un = r->i16_mode >> 4;
		const bool hasA = !(un & 1), hasB = !(un & 2);
		const int ei = lane & 15, y = lane >> 1, x0 = (lane & 1) * 8;
		const int ev = lane < 16 ? YT(ei, -1) : YT(-1, ei);
		uint32_t p0, p1;
		if (mode == 0) { const uint2 t = hasB ? *(const uint2 *)&YT(x0, -1) : make_uint2(0x80808080u, 0x80808080u); p0 = t.x; p1 = t.y; }
		else if (mode == 1) { const int v = __shfl_sync(0xffffffffu, ev, 16 + y); p0 = p1 = (hasA ? (uint32_t)v : 128u) * 0x01010101u; }
		else if (mode == 2) {
			int sdc = ev;
			sdc += __shfl_xor_sync(0xffffffffu, sdc, 1); sdc += __shfl_xor_sync(0xffffffffu, sdc, 2); sdc += __shfl_xor_sync(0xffffffffu, sdc, 4); sdc += __shfl_xor_sync(0xffffffffu, sdc, 8);
			const int st = __shfl_sync(0xffffffffu, sdc, 0), sl = __shfl_sync(0xffffffffu, sdc, 16);
			const int dc = (hasA && hasB) ? (st + sl + 16) >> 5 : hasA ? (sl + 8) >> 4 : hasB ? (st + 8) >> 4 : 128;
			p0 = p1 = (uint32_t)dc * 0x01010101u;
		} else {   /* plane: H = sum (i - 7) T(i) - 8 TL over i = 0..15, likewise V */
			int t = (ei - 7) * ev;
			t += __shfl_xor_sync(0xffffffffu, t, 1); t += __shfl_xor_sync(0xffffffffu, t, 2); t += __shfl_xor_sync(0xffffffffu, t, 4); t += __shfl_xor_sync(0xffffffffu, t, 8);
			const int corner = YT(-1, -1);
			const int Hs = __shfl_sync(0xffffffffu, t, 0) - 8 * corner, Vs = __shfl_sync(0xffffffffu, t, 16) - 8 * corner;
			const int a = 16 * (__shfl_sync(0xffffffffu, ev, 31) + __shfl_sync(0xffffffffu, ev, 15)), b = (5 * Hs + 32) >> 6, c = (5 * Vs + 32) >> 6;
			const int base = a + c * (y - 7) + 16 + b * (x0 - 7);
			p0 = p1 = 0;
#pragma unroll
			for (int k = 0; k < 4; k++) { p0 |= (uint32_t)clip255((base + b * k) >> 5) << (8 * k); p1 |= (uint32_t)clip255((base + b * (k + 4)) >> 5) << (8 * k); }
		}
		const uint4 rs = *(const uint4 *)&ws->res[y * 16 + x0];
		*(uint2 *)&YT(x0, y) = make_uint2(intra_add_res4(p0, rs.x, rs.y), intra_add_res4(p1, rs.z, rs.w));   /* the reads above touch only samples outside the macroblock */
		__syncwarp();
	}
}

/* both chroma planes: lanes 0-15 hold the rows above (plane, x), 16-31 the columns to the left (plane, y); a lane predicts 4
 * samples of one row (plane = lane >> 4, y = (lane >> 1) & 7, x0 = 4 (lane & 1)), i.e. one quadrant's DC for all four */
__device__ __noinline__ void intra_chroma(WarpSmem *ws, const E264MbRec *r, int lane) {
	const int mode = r->chroma_mode & 15, un = r->chroma_mode >> 4;
	const bool hasA = !(un & 1), hasB = !(un & 2);
	const int ep = (lane >> 3) & 1, ei = lane & 7;
	const int pl = lane >> 4, y = (lane >> 1) & 7, x0 = (lane & 1) * 4;
	const int ev = lane < 16 ? CT(ep, ei, -1) : CT(ep, -1, ei);
	uint32_t p;
	if (mode == 0) {
		int s4 = ev + __shfl_xor_sync(0xffffffffu, ev, 1); s4 += __shfl_xor_sync(0xffffffffu, s4, 2);
		const int bx = x0 >> 2, by = y >> 2;
		const int st = __shfl_sync(0xffffffffu, s4, pl * 8 + bx * 4), sl = __shfl_sync(0xffffffffu, s4, 16 + pl * 8 + by * 4);
		int v;
		if (bx == by) v = (hasA && hasB) ? (st + sl + 4) >> 3 : hasA ? (sl + 2) >> 2 : hasB ? (st + 2) >> 2 : 128;
		else if (bx == 1) v = hasB ? (st + 2) >> 2 : hasA ? (sl + 2) >> 2 : 128;
		else v = hasA ? (sl + 2) >> 2 : hasB ? (st + 2) >> 2 : 128;
		p = (uint32_t)v * 0x01010101u;
	} else if (mode == 1) { const int v = __shfl_sync(0xffffffffu, ev, 16 + pl * 8 + y); p = (hasA ? (uint32_t)v : 128u) * 0x01010101u; }
	else if (mode == 2) p = hasB ? *(const uint32_t *)&CT(pl, x0, -1) : 0x80808080u;
	else {   /* plane: H = sum (i - 3) T(i) - 4 TL over i = 0..7, likewise V */
		int t = (ei - 3) * ev;
		t += __shfl_xor_sync(0xffffffffu, t, 1); t += __shfl_xor_sync(0xffffffffu, t, 2); t += __shfl_xor_sync(0xffffffffu, t, 4);
		const int corner = CT(pl, -1, -1);
		const int Hs = __shfl_sync(0xffffffffu, t, pl * 8) - 4 * corner, Vs = __shfl_sync(0xffffffffu, t, 16 + pl * 8) - 4 * corner;
		const int a = 16 * (__shfl_sync(0xffffffffu, ev, 16 + pl * 8 + 7) + __shfl_sync(0xffffffffu, ev, pl * 8 + 7)), b = (34 * Hs + 32) >> 6, c = (34 * Vs + 32) >> 6;
		const int base = a + c * (y - 3) + 16 + b * (x0 - 3);
		p = 0;
#pragma unroll
		for (int k = 0; k < 4; k++) p |= (uint32_t)clip255((base + b * k) >> 5) << (8 * k);
	}
	const uint2 rs = *(const uint2 *)&ws->res[256 + pl * 64 + y * 8 + x0];
	*(uint32_t *)&CT(pl, x0, y) = intra_add_res4(p, rs.x, rs.y);   /* the reads above touch only the row above / column left of the block */
	__syncwarp();
}

/* ------------------------------------------------------------------------------------------ */
/* shared by the reconstruction kernels                                                         */
/* ------------------------------------------------------------------------------------------ */
__device__ __forceinline__ void store_mb(WarpSmem *ws, const PicJob &J, uint8_t *Y, uint8_t *C, int lane) {
	const int cpl = J.stride_c >> 1;
	if (lane < 16) *(uint4 *)(Y + (size_t)lane * J.stride_y) = *(const uint4 *)&YT(0, lane);
	else { int j = lane - 16, pl = j >> 3, row = j & 7; *(uint2 *)(C + pl * cpl + (size_t)row * J.stride_c) = *(const uint2 *)&CT(pl, 0, row); }
}

#define RES_COEF_MAX 416   /* 16 + 256 + 8 + 128 levels, rounded up */

/* number of int16 levels a record owns in the pool (same layout rule as sx_pool_take on the host) */
__device__ __forceinline__ int rec_coef_count(const E264MbRec *r) {
	const unsigned coded = r->coded;
	int n = (coded & CODED_Y_DC) ? 16 : 0;
	n += (r->flags & MBF_T8x8) ? 64 * __popc(coded & 0x1111) : 16 * __popc(coded & 0xffff);
	if (coded & (CODED_CB_DC | CODED_CR_DC)) n += 8;
	n += 16 * __popc((coded >> 16) & 0xff);
	return n;
}

