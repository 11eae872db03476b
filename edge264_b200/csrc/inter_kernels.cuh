/* inter_kernels.cuh — inter macroblocks: inverse transform + motion compensation + weighting + residual in ONE kernel.
 *
 * The unit of prediction is always the 4x4 luma block and reference list (that is what the record carries a vector for —
 * partition shapes never reach the device): an ITEM.  A thread handles one item: it loads the item's 9x9 luma window and
 * two 3x3 chroma windows of the reference picture straight into registers (aligned 32-bit loads + funnel shifts; the
 * windows of neighbouring blocks overlap in L1/L2) and interpolates 4x4 + 2x2 + 2x2 samples with the register arithmetic of
 * mc_math.cuh (dp4a tap sums).  Items are binned by interpolation class so that a warp runs ONE class body on 32 items
 * (reference edge264_inter.c:416-1251: per-partition SIMD interpolation + five weighting schemes).
 * The macroblock's coefficient run (16..816 bytes) arrives by cp.async.bulk on an mbarrier one macroblock ahead; each 4x4
 * block is inverse-transformed by the lane that also weights and stores it, so the residual stays in registers (only the
 * 8x8 transform passes through shared memory).
 * History: round 1's kernel (rectangles regrouped on the device, windows by cp.async.bulk.tensor into shared memory, one
 * output sample per lane and loop iteration) needed ~3600 warp instructions per macroblock and 77 us per 1080p picture;
 * this one 1630 and 39 us, and 35 k pictures/s with 32 streams in flight since its blocks are 16 warps in lock-step phases
 * (DESIGN.md section 4, profiles/r2_inter_geometry.txt). */
#pragma once
#include "recon_kernels.cuh"
#include "deblock_kernels.cuh"
#include "mc_math.cuh"

struct __align__(16) InterStage {
	uint4 rec4[12];
	int16_t coef[RES_COEF_MAX];
};

__device__ __forceinline__ uint32_t ldg32(const uint8_t *p) { return __ldg((const uint32_t *)p); }

/* the thread's 9x9 luma window at (X0, Y0) = top-left of the window (block position + integer vector - 2) */
__device__ __forceinline__ void mc_load_luma(const uint8_t *ref, int stride, int W, int H, int X0, int Y0, uint32_t w[9][3]) {
	if (X0 >= 0 && X0 + 9 <= W) {
		const int al = X0 & ~3, sh = (X0 & 3) * 8;
#pragma unroll
		for (int r = 0; r < 9; r++) {
			const int yy = min(max(Y0 + r, 0), H - 1);
			const uint8_t *p = ref + (size_t)yy * stride + al;
			const uint32_t a0 = ldg32(p), a1 = ldg32(p + 4), a2 = ldg32(p + 8);
			w[r][0] = __funnelshift_r(a0, a1, sh); w[r][1] = __funnelshift_r(a1, a2, sh); w[r][2] = a2 >> sh;
		}
	} else {   /* the window reaches over the left or right picture edge: samples are replicated (8.4.2.2.1) */
#pragma unroll
		for (int r = 0; r < 9; r++) {
			const int yy = min(max(Y0 + r, 0), H - 1);
			const uint8_t *p = ref + (size_t)yy * stride;
			uint32_t v[3] = {0, 0, 0};
#pragma unroll
			for (int k = 0; k < 9; k++) v[k >> 2] |= (uint32_t)__ldg(p + min(max(X0 + k, 0), W - 1)) << (8 * (k & 3));
			w[r][0] = v[0]; w[r][1] = v[1]; w[r][2] = v[2];
		}
	}
}
/* the thread's 3x3 window of one chroma plane (rows alternate Cb | Cr inside stride_c; `plane` points at the plane's column 0) */
__device__ __forceinline__ void mc_load_chroma(const uint8_t *plane, int stride, int Wc, int Hc, int X0, int Y0, uint32_t c[3]) {
	if (X0 >= 0 && X0 + 3 <= Wc) {
		const int al = X0 & ~3, sh = (X0 & 3) * 8;
#pragma unroll
		for (int r = 0; r < 3; r++) {
			const uint8_t *p = plane + (size_t)min(max(Y0 + r, 0), Hc - 1) * stride + al;
			c[r] = __funnelshift_r(ldg32(p), ldg32(p + 4), sh);
		}
	} else {
#pragma unroll
		for (int r = 0; r < 3; r++) {
			const uint8_t *p = plane + (size_t)min(max(Y0 + r, 0), Hc - 1) * stride;
			c[r] = (uint32_t)__ldg(p + min(max(X0, 0), Wc - 1)) | (uint32_t)__ldg(p + min(max(X0 + 1, 0), Wc - 1)) << 8 | (uint32_t)__ldg(p + min(max(X0 + 2, 0), Wc - 1)) << 16;
		}
	}
}

/* 8.4.2.3 on four packed samples in ONE form: ((a * wa + b * wb + rnd) >> sh) + o, clipped.  Explicit or implicit
 * bi-prediction: wa = w0, wb = w1, rnd = 2^logWD, sh = logWD + 1; explicit weighting of a single prediction: wa = w, wb = 0,
 * rnd = 2^(logWD-1) (0 when logWD = 0), sh = logWD (reference edge264_inter.c:1140-1180 keeps five variants). */
__device__ __forceinline__ uint32_t wp_word(uint32_t a, uint32_t b, int wa, int wb, int rnd, int sh, int o) {
	uint32_t r = 0;
#pragma unroll
	for (int k = 0; k < 4; k++) {
		const int pa = (a >> (8 * k)) & 255, pb = (b >> (8 * k)) & 255;
		const int v = ((pa * wa + pb * wb + rnd) >> sh) + o;
		r |= (uint32_t)min(max(v, 0), 255) << (8 * k);
	}
	return r;
}
/* prediction + residual of four packed samples; res: four int16 residuals */
__device__ __forceinline__ uint32_t add_res4(uint32_t p, const int res[4]) {
	return mc_pack4(clip255((short)((int)(p & 255) + res[0])), clip255((short)((int)((p >> 8) & 255) + res[1])),
	                clip255((short)((int)((p >> 16) & 255) + res[2])), clip255((short)((int)(p >> 24) + res[3])));
}
/* the four prediction rows of one list for the lane's 4x4 block of samples (see phase 3): a luma lane's block as it was
 * stored; chroma lane 16 + 4 pl + i joins the 2x2 predictions of plane pl of luma blocks 4i..4i+3 (a 2x2 word holds row 0
 * in its low, row 1 in its high half) */
__device__ __forceinline__ void inter_pred_words(const uint32_t (*pred)[8], int lane, uint32_t w[4]) {
	if (lane < 16) {
		const uint4 a = *(const uint4 *)pred[lane];
		w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
	} else {
		const int j = lane - 16, z = (j & 3) * 4, e = 4 + (j >> 2);
		const uint32_t a = pred[z][e], b = pred[z + 1][e], c = pred[z + 2][e], d = pred[z + 3][e];
		w[0] = __byte_perm(a, b, 0x5410); w[1] = __byte_perm(a, b, 0x7632); w[2] = __byte_perm(c, d, 0x5410); w[3] = __byte_perm(c, d, 0x7632);
	}
}

/* ---- the kernel ----
 * A block takes chunks of INTER_CHUNK consecutive macroblocks.  Per chunk:
 *   1. records into shared memory; every (macroblock, list, 4x4 block) that is predicted becomes an ITEM and is queued by
 *      interpolation class (mc_class: full, horizontal, vertical, diagonal, centre h-first, centre v-first) — warp
 *      votes give the queue positions;
 *   2. the warps take 32 items of ONE class at a time: the same instruction stream for all lanes, every lane busy —
 *      window loads, interpolation, predictions (24 bytes) into shared memory;
 *   3. a warp per macroblock: inverse transform of its coefficient run (cp.async.bulk one macroblock ahead), list-0 /
 *      list-1 combination with the slice's weighting, residual, 128-bit row stores.
 * A thread-per-block version without the binning ran every class present in a macroblock one after the other (about
 * 2000 warp instructions per macroblock on random vectors, no faster than round 1's). */
/* Block geometry: INTER_WARPS warps take INTER_CHUNK macroblocks at a time (4 per warp).  The kernel's three phases are
 * separated by block barriers, so all warps of a block execute the same part of the code: the bigger the block, the fewer
 * different parts of the kernel (12 400 instructions when this was measured, 5 600 now) the SM's instruction cache has to hold at a time — and a
 * 16-warp block at 128 registers per thread fills the SM's register file, so no block of another kernel shares the SM. */
#ifndef INTER_WARPS
#define INTER_WARPS 16      /* measured (profiles/r2_inter_geometry.txt), 32 streams: 4 warps 9.7 k, 8 warps 13.2 k, 16 warps 17.8 k frames/s */
#endif
#ifndef INTER_CHUNK
#define INTER_CHUNK (4 * INTER_WARPS)
#endif
#define INTER_MINB0 (16 / INTER_WARPS)      /* blocks per SM at 128 registers per thread */
struct __align__(16) InterSmem {
	uint4 rec4[INTER_CHUNK][12];
	uint32_t pred[INTER_CHUNK][2][16][8];          /* [macroblock][list][luma4x4BlkIdx]: four luma rows, 2x2 Cb, 2x2 Cr, (pad: 16-byte aligned entries) */
	uint16_t queue[6][INTER_CHUNK * 32];           /* item = macroblock << 5 | list << 4 | luma4x4BlkIdx */
	int qn[6];
	WarpSmem ws[INTER_WARPS];
	uint4 drecs[INTER_WARPS][3][12];               /* deblocking digests: records of neighbours outside the chunk (left, top) per warp */
	E264DbkMb ddg[INTER_WARPS];
	int16_t coef[INTER_WARPS][2][RES_COEF_MAX];
	unsigned long long bars[INTER_WARPS][2];
};

/* One item: the window loads are the same for every interpolation class and exist ONCE in the kernel (the six class bodies
 * used to carry their own copies: 3 000 of the kernel's 12 000 instructions, and with blocks of several pictures in
 * different phases on an SM the instruction cache, 32 KB in its first shared level, is what the warps wait for);
 * `cls` is uniform over the warp, so the switch is one resolved branch per pass. */
__device__ __forceinline__ void inter_item(const PicJob &J, InterSmem &sm, int cls, int item, int mb0, int W, int H) {
	const int m = item >> 5, l = (item >> 4) & 1, z = item & 15, bx = blk_x(z), by = blk_y(z);
	const E264MbRec *r = (const E264MbRec *)sm.rec4[m];
	const int mb = mb0 + m, mbx = mb % J.w_mbs, mby = mb / J.w_mbs;
	int slot = r->ref_pic[l][z >> 2];
	if (slot < 0 || slot >= J.n_slots) slot = J.dst_slot;
	const uint8_t *ref = J.frames + (size_t)slot * J.frame_bytes;
	const int mvx = r->mv[l][z][0], mvy = r->mv[l][z][1];
	const int fx = mvx & 3, fy = mvy & 3;
	uint32_t win[9][3], py[4];
	mc_load_luma(ref, J.stride_y, W, H, mbx * 16 + bx * 4 + (mvx >> 2) - 2, mby * 16 + by * 4 + (mvy >> 2) - 2, win);
	uint32_t cb[3], cr[3];
	const uint8_t *cplane = ref + J.plane_y;
	const int cx = mbx * 8 + bx * 2 + (mvx >> 3), cy = mby * 8 + by * 2 + (mvy >> 3);
	mc_load_chroma(cplane, J.stride_c, W >> 1, H >> 1, cx, cy, cb);
	mc_load_chroma(cplane + (J.stride_c >> 1), J.stride_c, W >> 1, H >> 1, cx, cy, cr);
	switch (cls) {
	case 0:
#pragma unroll
		for (int y = 0; y < 4; y++) py[y] = mc_fsr(win[y + 2][0], win[y + 2][1], 16);
		break;
	case 1: mc_luma_h(win, fx, py); break;
	case 2: mc_luma_v(win, fy, py); break;
	case 3: mc_luma_diag(win, fx, fy, py); break;
	case 4: mc_luma_center(win, fy, py); break;
	default: mc_luma_center_v(win, fx, py); break;
	}
	uint32_t *o = sm.pred[m][l][z];
	*(uint4 *)o = make_uint4(py[0], py[1], py[2], py[3]);
	*(uint2 *)(o + 4) = make_uint2(mc_chroma2x2(cb[0], cb[1], cb[2], mvx & 7, mvy & 7), mc_chroma2x2(cr[0], cr[1], cr[2], mvx & 7, mvy & 7));
}

template <int MINB>
__global__ void __launch_bounds__(INTER_WARPS * 32, MINB) e264_inter4_kernel(PicJob J) {
	TraceScope trace_(J, 1);
	reset_next_tickets(J);
	extern __shared__ __align__(16) unsigned char inter_smem_raw[];
	InterSmem &sm = *(InterSmem *)inter_smem_raw;
	const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
	WarpSmem *ws = &sm.ws[w];
	const int nmb = J.w_mbs * J.h_mbs;
	const int W = J.w_mbs * 16, H = J.h_mbs * 16;
	uint8_t *dst = J.frames + (size_t)J.dst_slot * J.frame_bytes;
	if (lane == 0) {
		mbar_init(&sm.bars[w][0], 1); mbar_init(&sm.bars[w][1], 1);
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
	}
	unsigned parity = 0;      /* bit b: phase parity of bars[w][b] (a bit mask, not an array: b is not a constant) */
	const int nchunks = (nmb + INTER_CHUNK - 1) / INTER_CHUNK;
	IT_DECL
	for (int chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
		const int mb0 = chunk * INTER_CHUNK, cnt = min(INTER_CHUNK, nmb - mb0);
		__syncthreads();                               /* the previous chunk's predictions and records are no longer read */
		IT_MARK(4)
		/* ---- 1. records, queues ---- */
		for (int i = tid; i < cnt * 12; i += INTER_WARPS * 32) sm.rec4[i / 12][i % 12] = __ldg((const uint4 *)(J.recs + mb0) + i);
		if (tid < 6) sm.qn[tid] = 0;
		__syncthreads();
		/* the macroblocks this warp finishes in step 3 are w, w + 4, ...: get the first coefficient run under way */
		auto coef_issue = [&](int m, int b) -> int {     /* 0 not inter, 1 inter, 2 inter with coefficients (copy in flight) */
			if (m >= cnt) return 0;
			const E264MbRec *r = (const E264MbRec *)sm.rec4[m];
			if (r->kind != MBK_INTER) return 0;
			if (r->coded == 0) return 1;
			if (lane == 0) tma_bulk_g2s(sm.coef[w][b], J.coefs + r->coef_off, (unsigned)rec_coef_count(r) * 2u, &sm.bars[w][b]);
			return 2;
		};
		int what = coef_issue(w, 0);
#pragma unroll 1
		for (int i0 = 0; i0 < cnt * 32; i0 += INTER_WARPS * 32) {
			const int item = i0 + tid, m = item >> 5, l = (item >> 4) & 1, z = item & 15;
			int cls = -1;
			if (m < cnt) {
				const E264MbRec *r = (const E264MbRec *)sm.rec4[m];
				if (r->kind == MBK_INTER && r->ref_idx[l][z >> 2] >= 0) cls = mc_class(r->mv[l][z][0] & 3, r->mv[l][z][1] & 3);
			}
			/* queue position: the lanes of one class find each other with one match instruction, their first lane reserves the
			 * run in the class queue */
			const unsigned peers = __match_any_sync(0xffffffffu, cls);
			const int leader = __ffs(peers) - 1;
			int base = 0;
			if (cls >= 0 && lane == leader) base = atomicAdd(&sm.qn[cls], __popc(peers));
			base = __shfl_sync(0xffffffffu, base, leader);
			if (cls >= 0) sm.queue[cls][base + __popc(peers & ((1u << lane) - 1))] = (uint16_t)item;
		}
		__syncthreads();
		IT_MARK(0)
		/* ---- 2. one class at a time, 32 items per warp pass: the groups of all classes form one list ---- */
		{
			int total = 0;
#pragma unroll
			for (int j = 0; j < 6; j++) total += (sm.qn[j] + 31) >> 5;
#pragma unroll 1
			for (int g = w; g < total; g += INTER_WARPS) {
				int c = 0, gb = 0, acc = 0;
#pragma unroll
				for (int j = 0; j < 6; j++) { const int gj = (sm.qn[j] + 31) >> 5; if (g >= acc) { c = j; gb = acc; } acc += gj; }
				const int k = (g - gb) * 32 + lane;
				if (k < sm.qn[c]) inter_item(J, sm, c, sm.queue[c][k], mb0, W, H);
			}
		}
		__syncthreads();
		IT_MARK(1)
		/* ---- 3. a warp per macroblock: inverse transform, weighting, residual, store ---- */
		int b = 0;
		bool failed = false;
#pragma unroll 1
		for (int m = w; m < cnt; m += INTER_WARPS, b ^= 1) {
			const int what2 = coef_issue(m + INTER_WARPS, b ^ 1);
			/* the macroblock's deblocking digest (every macroblock, intra ones too): record-only work whose load of the
			 * record above is in flight together with the coefficient run requested above; the current and left records
			 * (and the one above in pictures narrower than a chunk) are the chunk's */
			if (J.dbk != nullptr)
				dbk_digest_mb(J, sm.drecs[w], &sm.ddg[w], mb0 + m, lane, (const E264MbRec *)sm.rec4[m], m > 0 ? (const E264MbRec *)sm.rec4[m - 1] : nullptr,
				              m >= J.w_mbs ? (const E264MbRec *)sm.rec4[m - J.w_mbs] : nullptr);
			IT_MARK(2)
			if (what) {
				const int mb = mb0 + m, mbx = mb % J.w_mbs, mby = mb / J.w_mbs;
				const E264MbRec *r = (const E264MbRec *)sm.rec4[m];
				const E264SliceRec *sr = J.slices + r->slice_idx;
				const unsigned coded = r->coded;
				const bool t8 = r->flags & MBF_T8x8;
				const int16_t *cf = sm.coef[w][b];
				if (what == 2) {
					if (!mbar_wait(&sm.bars[w][b], (parity >> b) & 1)) { if (lane == 0) atomicExch(J.err, 4u); failed = true; }
					parity ^= 1u << b;
					if (coded & CODED_Y_DC) cf += 16;     /* Intra16x16 only: not in an inter macroblock's run */
					if (!failed && t8 && (coded & 0x1111)) residual_luma8x8(ws, r, sr, cf, lane);
				}
				IT_MARK(3)
				/* a lane per 4x4 block of samples: lanes 0-15 luma block z = lane, lane 16 + 4 pl + i chroma block i of plane
				 * pl (the 2x2 predictions of luma blocks 4i..4i+3); prediction, weighting, residual in registers, store */
				if (lane < 24 && !failed) {
					const bool luma = lane < 16;
					const int j = lane - 16, pl = (j >> 2) & 1, i8 = luma ? lane >> 2 : j & 3;
					const int r0 = r->ref_idx[0][i8], r1 = r->ref_idx[1][i8];
					uint32_t p[4] = {0, 0, 0, 0}, q[4] = {0, 0, 0, 0};
					if (r0 >= 0) inter_pred_words(sm.pred[m][0], lane, p);
					if (r1 >= 0) inter_pred_words(sm.pred[m][1], lane, q);
					const int wpm = sr->wp_mode;
					const bool bi = r0 >= 0 && r1 >= 0;
					if (!bi && r0 < 0) {
#pragma unroll
						for (int k = 0; k < 4; k++) p[k] = q[k];
					}
					if (bi && wpm == WP_DEFAULT) {
#pragma unroll
						for (int k = 0; k < 4; k++) p[k] = mc_avg4(p[k], q[k]);
					} else if ((bi && wpm != WP_DEFAULT) || (wpm == WP_EXPLICIT && (r0 >= 0 || r1 >= 0))) {
						/* one weighting body for every scheme, with the parameters of the lane's plane */
						const int c = luma ? 0 : 1 + pl, lw = c ? sr->chroma_log2_wd : sr->luma_log2_wd;
						const int ll = r0 >= 0 ? 0 : 1, ri = (ll ? r1 : r0) & 15;
						int wa, wb, o, sh, rnd;
						if (bi && wpm == WP_EXPLICIT) { wa = sr->wp_w[0][r0 & 15][c]; wb = sr->wp_w[1][r1 & 15][c]; o = (sr->wp_o[0][r0 & 15][c] + sr->wp_o[1][r1 & 15][c] + 1) >> 1; sh = lw + 1; rnd = 1 << lw; }
						else if (bi) { wb = sr->implicit_w1[r0 & 15][r1 & 15]; wa = 64 - wb; o = 0; sh = 6; rnd = 32; }
						else { wa = sr->wp_w[ll][ri][c]; wb = 0; o = sr->wp_o[ll][ri][c]; sh = lw; rnd = lw >= 1 ? 1 << (lw - 1) : 0; }
#pragma unroll
						for (int k = 0; k < 4; k++) p[k] = wp_word(p[k], q[k], wa, wb, rnd, sh, o);
					}
					if (what == 2) {
						int res[16];
						bool act = false;
						if (luma && t8) {     /* the 8x8 transform's residual, written above for coded 8x8 blocks only */
							act = (coded >> lane) & 1;
							if (act) {
								const int16_t *rs = ws->res + blk_y(lane) * 64 + blk_x(lane) * 4;
#pragma unroll
								for (int k = 0; k < 4; k++) {
									const uint2 v = *(const uint2 *)(rs + k * 16);
									res[4 * k] = (short)(v.x & 0xffff); res[4 * k + 1] = (short)(v.x >> 16); res[4 * k + 2] = (short)(v.y & 0xffff); res[4 * k + 3] = (short)(v.y >> 16);
								}
							}
						} else {
							const int16_t *cfc = cf + (t8 ? 64 * __popc(coded & 0x1111) : 16 * __popc(coded & 0xffff));   /* chroma DC, then AC */
							const bool any_cdc = (coded & (CODED_CB_DC | CODED_CR_DC)) != 0;
							bool on;
							const int16_t *src; const uint8_t *scal; int qp, dc = 0;
							if (luma) {
								on = (coded >> lane) & 1; act = on;
								src = cf + __popc(coded & ((1u << lane) - 1)) * 16; scal = sr->scaling4x4[3]; qp = r->qp[0];
							} else {
								on = (coded >> lane) & 1; act = on || any_cdc;
								if (any_cdc) dc = chroma_dc(cfc, r, sr, 1, pl, j & 3);
								src = cfc + (any_cdc ? 8 : 0) + __popc((coded >> 16) & ((1u << j) - 1) & 0xff) * 16; scal = sr->scaling4x4[4 + pl]; qp = r->qp[1 + pl];
							}
							if (act) idct4x4_core(src, on, scal, qp, !luma, dc, res);
						}
						IT_MARK(3)
						if (act) {
#pragma unroll
							for (int k = 0; k < 4; k++) p[k] = add_res4(p[k], res + 4 * k);
						}
					}
					if (luma) {
#pragma unroll
						for (int k = 0; k < 4; k++) *(uint32_t *)&YT(blk_x(lane) * 4, blk_y(lane) * 4 + k) = p[k];
					} else {
#pragma unroll
						for (int k = 0; k < 4; k++) *(uint32_t *)&CT(pl, (j & 1) * 4, (j & 2) * 2 + k) = p[k];
					}
				}
				__syncwarp();
				if (!failed) {
					store_mb(ws, J, dst + (size_t)(mby * 16) * J.stride_y + mbx * 16, dst + J.plane_y + (size_t)(mby * 8) * J.stride_c + mbx * 8, lane);
					if (lane == 0) J.flags[mb] = J.epoch;     /* visible to the intra kernel through the kernel boundary */
				}
				__syncwarp();
			}
			IT_MARK(4)
			what = what2;
		}
	}
	IT_FLUSH
}
