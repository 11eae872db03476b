/* deblock_kernels.cuh — the in-loop filter (8.7).
 *
 *   dbk_digest_mb         a 64-byte E264DbkMb per macroblock: 32 boundary strengths (one lane per edge segment), alpha /
 *                         beta / tC0 of the 9 plane x edge-kind combinations (reference: deblock_mb's bS derivation
 *                         and table look-ups, edge264_deblock.c:530-1123) — record-only work without dependencies, a
 *                         warp per macroblock.  It runs inside the reconstruction kernels (the inter kernel derives
 *                         the digests of its chunk, the intra-picture kernel those of its rows): hundreds of warps
 *                         share it and no separate launch is needed.
 *   e264_deblock_kernel   the sample filter as a wavefront over macroblock ROW PAIRS.  The standard fixes the order
 *                         (raster macroblocks, vertical edges left to right, then horizontal edges top to bottom;
 *                         reference order edge264_deblock.c:537-891): macroblock (x, y) needs (x-1, y) complete,
 *                         (x, y-1) complete and the left edge of (x+1, y-1) done.  One warp walks two rows at once,
 *                         lanes 0-15 on row 2k at macroblock x, lanes 16-31 on row 2k+1 at macroblock x-1 (the rows above are
 *                         needed by the horizontal pass only, and the vertical pass of x+1 above is what finalises x) — the same
 *                         instruction stream, no divergence — and hands the four bottom sample rows from the upper to
 *                         the lower row through a shared-memory ring.  Inside an iteration a lane owns a whole sample
 *                         ROW for the four vertical edges (registers only, no exchange between edges), the tile is
 *                         transposed through shared memory, and a lane owns a whole COLUMN for the four horizontal
 *                         edges.  Luma and the two chroma planes are independent and run as separate warps.
 *                         Only the hand-over between warps goes through global memory: a progress counter per row,
 *                         published one macroblock late so that the fence never waits for stores just issued.
 */
#pragma once
#include "recon_kernels.cuh"

struct __align__(16) E264DbkMb {
	uint32_t bs[4];          /* [0..1] vertical edges, [2..3] horizontal edges: nibble (edge * 4 + segment) = bS 0..4 */
	uint8_t alpha[9];        /* [plane * 3 + kind], kind 0 internal, 1 left macroblock edge, 2 top macroblock edge */
	uint8_t beta[9];
	uint8_t tc0[27];         /* [(plane * 3 + kind) * 3 + bS - 1] */
	uint8_t pad[3];
};                           /* 64 bytes */

__device__ __forceinline__ int dbk_iabs(int v) { return v < 0 ? -v : v; }

/* bS of one edge segment between 4x4 block bp of p and bq of q (8.7.2.1), every condition evaluated and the answer
 * selected: the lanes of a warp reach different answers, and early returns made the warp run them one after another */
__device__ __forceinline__ int dbk_bs_pair(const E264MbRec *p, int bp, const E264MbRec *q, int bq, bool mb_edge) {
	const bool intra = p->kind != MBK_INTER || q->kind != MBK_INTER;
	const bool coef = ((p->coded >> bp) & 1) || ((q->coded >> bq) & 1);
	const int p0 = p->ref_idx[0][bp >> 2] < 0 ? -1 : p->ref_pic[0][bp >> 2], p1 = p->ref_idx[1][bp >> 2] < 0 ? -1 : p->ref_pic[1][bp >> 2];
	const int q0 = q->ref_idx[0][bq >> 2] < 0 ? -1 : q->ref_pic[0][bq >> 2], q1 = q->ref_idx[1][bq >> 2] < 0 ? -1 : q->ref_pic[1][bq >> 2];
	const bool same = (p0 == q0 && p1 == q1) || (p0 == q1 && p1 == q0);
#define FAR(lp, lq) (dbk_iabs(p->mv[lp][bp][0] - q->mv[lq][bq][0]) >= 4 || dbk_iabs(p->mv[lp][bp][1] - q->mv[lq][bq][1]) >= 4)
	const bool f00 = FAR(0, 0), f11 = FAR(1, 1), f01 = FAR(0, 1), f10 = FAR(1, 0);
#undef FAR
	const bool bi = p0 >= 0 && p1 >= 0;
	const bool two = p0 != p1 ? (p0 == q0 ? f00 || f11 : f01 || f10) : (f00 || f11) && (f01 || f10);
	const bool one = p0 >= 0 ? (q0 >= 0 ? f00 : f01) : (q0 >= 0 ? f10 : f11);
	const int mvbs = (bi ? two : one) ? 1 : 0;
	return intra ? (mb_edge ? 4 : 3) : coef ? 2 : !same ? 1 : mvbs;
}

/* digest of one macroblock by one warp: 32 boundary strengths (one lane per edge segment), thresholds of the nine plane x
 * edge-kind combinations.  recs: 3 x 12 uint4 of shared memory for the warp, dg: 64 bytes of shared memory.  cur, left,
 * top: the records of the macroblock and its neighbours where the caller already holds them in shared memory, else
 * nullptr (they are then fetched into recs). */
__device__ __forceinline__ void dbk_digest_mb(const PicJob &J, uint4 (*recs)[12], E264DbkMb *dg, int mb, int lane,
                                              const E264MbRec *cur = nullptr, const E264MbRec *left = nullptr, const E264MbRec *top = nullptr) {
	const int W = J.w_mbs, mbx = mb % W, mby = mb / W;
	const E264MbRec *q = cur ? cur : (const E264MbRec *)recs[0], *pL = left ? left : (const E264MbRec *)recs[1], *pT = top ? top : (const E264MbRec *)recs[2];
	if (lane < 12) { if (!cur) recs[0][lane] = __ldg((const uint4 *)(J.recs + mb) + lane); }
	else if (lane < 24) { if (!left && mbx > 0) recs[1][lane - 12] = __ldg((const uint4 *)(J.recs + mb - 1) + lane - 12); }
	if (lane < 12 && !top && mby > 0) recs[2][lane] = __ldg((const uint4 *)(J.recs + mb - W) + lane);
	__syncwarp();
	const int qflags = q->flags;
	const bool on_mb = qflags & MBF_DEBLOCK, fl = qflags & MBF_EDGE_L, ft = qflags & MBF_EDGE_T, t8 = qflags & MBF_T8x8;
	int bs = 0;
	{
		const int dir = lane >> 4, e = (lane >> 2) & 3, k = lane & 3;
		const E264MbRec *p = q;
		bool on = on_mb && !(t8 && (e & 1));
		if (e == 0) { on = on && (dir ? ft : fl); p = dir ? pT : pL; }
		if (q->kind != MBK_INTER) bs = on ? (e == 0 ? 4 : 3) : 0;     /* intra macroblock: no per-lane work */
		else if (on) {
			const int qx = dir ? k : e, qy = dir ? e : k;
			const int px_ = dir ? k : (e ? e - 1 : 3), py_ = dir ? (e ? e - 1 : 3) : k;
			bs = dbk_bs_pair(p, blk_z(px_, py_), q, blk_z(qx, qy), e == 0);
		}
	}
	unsigned v = (unsigned)bs << ((lane & 7) * 4);
	v |= __shfl_xor_sync(0xffffffffu, v, 1); v |= __shfl_xor_sync(0xffffffffu, v, 2); v |= __shfl_xor_sync(0xffffffffu, v, 4);
	if ((lane & 7) == 0) dg->bs[lane >> 3] = v;
	if (lane < 9) {
		const int pl = lane / 3, kind = lane % 3;
		const E264MbRec *p = kind == 0 ? q : kind == 1 ? pL : pT;
		if ((kind == 1 && !fl) || (kind == 2 && !ft) || !on_mb) p = q;
		const E264SliceRec *sr = J.slices + q->slice_idx;
		const int qpav = (p->qp[pl] + q->qp[pl] + 1) >> 1;
		const int ia = min(max(qpav + sr->filter_offset_a, 0), 51), ib = min(max(qpav + sr->filter_offset_b, 0), 51);
		dg->alpha[lane] = h264_alpha[ia]; dg->beta[lane] = h264_beta[ib];
		dg->tc0[lane * 3] = h264_tc0[ia][0]; dg->tc0[lane * 3 + 1] = h264_tc0[ia][1]; dg->tc0[lane * 3 + 2] = h264_tc0[ia][2];
	}
	if (lane == 9) { dg->pad[0] = dg->pad[1] = dg->pad[2] = 0; }
	__syncwarp();
	if (lane < 4) ((uint4 *)(J.dbk + mb))[lane] = ((const uint4 *)dg)[lane];
	__syncwarp();
}

/* ---- sample filters on one line across an edge, samples as ints ----
 * Branch-free: a line that is not filtered runs the same arithmetic with its clipping bounds set to zero (a lone
 * warp pays ~10 cycles for every branch it resolves). */
template <bool STRONG>
__device__ __forceinline__ void dbk_line_luma(int &p3, int &p2, int &p1, int &p0, int &q0, int &q1, int &q2, int &q3, int bs, int alpha, int beta, int tc0, bool any4) {
	const int ad = __sad(p0, q0, 0);
	const bool f = bs != 0 && ad < alpha && __sad(p1, p0, 0) < beta && __sad(q1, q0, 0) < beta;
	const bool ap = __sad(p2, p0, 0) < beta, aq = __sad(q2, q0, 0) < beta;
	const int tcp = f && ap ? tc0 : 0, tcq = f && aq ? tc0 : 0;
	const int tc = f ? tc0 + (int)ap + (int)aq : 0;
	const int d = min(max((((q0 - p0) << 2) + (p1 - q1) + 4) >> 3, -tc), tc);
	const int avg = (p0 + q0 + 1) >> 1;
	int n_p1 = p1 + min(max((p2 + avg - (p1 << 1)) >> 1, -tcp), tcp);
	int n_q1 = q1 + min(max((q2 + avg - (q1 << 1)) >> 1, -tcq), tcq);
	int n_p0 = min(max(p0 + d, 0), 255), n_q0 = min(max(q0 - d, 0), 255);
	if (STRONG && any4) {   /* bS 4 exists only on macroblock edges; `any4` is uniform over the warp */
		const bool s4 = f && bs == 4;
		const bool small = ad < ((alpha >> 2) + 2);
		const bool sp = ap && small, sq = aq && small;
		const int s_p0 = sp ? (p2 + 2 * p1 + 2 * p0 + 2 * q0 + q1 + 4) >> 3 : (2 * p1 + p0 + q1 + 2) >> 2;
		const int s_p1 = sp ? (p2 + p1 + p0 + q0 + 2) >> 2 : p1;
		const int s_p2 = sp ? (2 * p3 + 3 * p2 + p1 + p0 + q0 + 4) >> 3 : p2;
		const int s_q0 = sq ? (p1 + 2 * p0 + 2 * q0 + 2 * q1 + q2 + 4) >> 3 : (2 * q1 + q0 + p1 + 2) >> 2;
		const int s_q1 = sq ? (p0 + q0 + q1 + q2 + 2) >> 2 : q1;
		const int s_q2 = sq ? (2 * q3 + 3 * q2 + q1 + q0 + p0 + 4) >> 3 : q2;
		n_p0 = s4 ? s_p0 : n_p0; n_p1 = s4 ? s_p1 : n_p1; p2 = s4 ? s_p2 : p2;
		n_q0 = s4 ? s_q0 : n_q0; n_q1 = s4 ? s_q1 : n_q1; q2 = s4 ? s_q2 : q2;
	}
	p0 = n_p0; p1 = n_p1; q0 = n_q0; q1 = n_q1;
}
__device__ __forceinline__ void dbk_line_chroma(int p1, int &p0, int &q0, int q1, int bs, int alpha, int beta, int tc0) {
	const bool f = bs != 0 && __sad(p0, q0, 0) < alpha && __sad(p1, p0, 0) < beta && __sad(q1, q0, 0) < beta;
	const int tc = f ? tc0 + 1 : 0;
	const int d = min(max((((q0 - p0) << 2) + (p1 - q1) + 4) >> 3, -tc), tc);
	const bool s4 = f && bs == 4;
	const int n_p0 = s4 ? (2 * p1 + p0 + q1 + 2) >> 2 : min(max(p0 + d, 0), 255);
	const int n_q0 = s4 ? (2 * q1 + q0 + p1 + 2) >> 2 : min(max(q0 - d, 0), 255);
	p0 = n_p0; q0 = n_q0;
}

#define DBK_TS 5      /* tile row stride in words: odd, so the 32 rows of the two halves fall into 32 different banks */
#define DBK_PAIRS 8   /* row pairs (warps) per block: a block owns a band of 16 macroblock rows of one kind of plane */
#define DBK_RING 8    /* macroblocks a row may run ahead of the row below it */
#define DBK_CHUNK 8   /* macroblocks between two publications of a band's last row to the next block */
struct __align__(16) DbkSmem {
	uint32_t tile[DBK_PAIRS][32][DBK_TS];            /* [half * 16 + sample row][word]: the macroblock between the vertical and the horizontal pass */
	uint32_t top[DBK_PAIRS][2][4][4];                /* [half][row][word]: luma rows -4..-1; chroma [plane * 2 + row -2..-1][2 words] */
	E264DbkMb dg[DBK_PAIRS][2];
	uint32_t ring[2 * DBK_PAIRS][DBK_RING][4][4];    /* per row of the band: bottom sample rows of its finished macroblocks [x % RING], layout of top */
	int done[2 * DBK_PAIRS];                         /* macroblocks a row has put into its ring */
	int taken[2 * DBK_PAIRS];                        /* macroblocks a row has taken from the ring of the row above */
	int band;
};

__device__ __forceinline__ int dbk_byte(uint32_t w, int k) { return (int)((w >> (8 * k)) & 0xffu); }
__device__ __forceinline__ uint32_t dbk_pack(int a, int b, int c, int d) { return (uint32_t)a | (uint32_t)b << 8 | (uint32_t)c << 16 | (uint32_t)d << 24; }

/* One warp = one pair of macroblock rows of the band, one kind of plane.  Hand-over of the bottom sample rows:
 *   upper row -> lower row of the warp: shared-memory ring, fixed lag of one iteration (written before, read behind the
 *     barrier between the two passes), no counters;
 *   lower row -> upper row of the next warp: the same ring with done/taken counters in shared memory (block-scope fences);
 *   last row of the band -> first row of the next band (another block): global memory, a progress counter per row
 *   published every DBK_CHUNK macroblocks (the only gpu-scope fences of the kernel, off the per-macroblock path). */
template <bool CH>
__device__ __forceinline__ void dbk_walk(const PicJob &J, DbkSmem *sm, int band, int wid, int lane) {
	constexpr int NW = CH ? 2 : 4;            /* words per sample row of a macroblock */
	constexpr int MBW = CH ? 8 : 16;          /* bytes per sample row, rows per plane */
	const int half = lane >> 4, hl = lane & 15;
	const int W = J.w_mbs, H = J.h_mbs;
	const int lrow = wid * 2 + half, mby = band * (2 * DBK_PAIRS) + lrow;
	const bool row_ok = mby < H;
	const bool from_global = lrow == 0;                                   /* rows above come from another block (or do not exist) */
	const bool to_ring = lrow + 1 < 2 * DBK_PAIRS && mby + 1 < H;          /* the row below is in this block */
	const bool to_global = row_ok && lrow + 1 == 2 * DBK_PAIRS && mby + 1 < H;   /* the row below belongs to the next band */
	const int pl = CH ? hl >> 3 : 0, r = CH ? hl & 7 : hl;      /* row ownership: plane and sample row of this lane */
	const int cpl = J.stride_c >> 1;
	const size_t stride = CH ? (size_t)J.stride_c : (size_t)J.stride_y;
	uint8_t *frame = J.frames + (size_t)J.dst_slot * J.frame_bytes + (CH ? J.plane_y : 0);
	uint8_t *rowp = frame + (size_t)(mby * MBW + r) * stride + pl * cpl;
	/* lanes hl < 4 also own one sample row above the macroblock row: luma -4..-1, chroma (plane hl >> 1, row -2 + (hl & 1)) */
	const int tpl = CH ? hl >> 1 : 0, tr = CH ? (hl & 1) - 2 : hl - 4;
	uint8_t *topp = frame + (ptrdiff_t)(mby * MBW + tr) * (ptrdiff_t)stride + tpl * cpl;
	const bool top_lane = hl < 4 && mby > 0 && row_ok;
	const bool wb_lane = top_lane && (CH ? (hl & 1) != 0 : hl >= 1);    /* rows the top edge may change: luma -3..-1, chroma -1 */
	volatile unsigned *prog = J.flags + W * H + (CH ? H : 0);
	const volatile unsigned *errp = J.err;
	const unsigned base = J.epoch * 2048u;
	const E264DbkMb *dgp = J.dbk + (size_t)mby * W;
	const int pi = CH ? 1 + pl : 0;           /* plane index of alpha/beta/tc0 in row ownership */
	uint32_t (*tile)[DBK_TS] = sm->tile[wid];
	uint32_t (*top)[4][4] = sm->top[wid];
	E264DbkMb *dgs = sm->dg[wid];
	uint32_t (*ring_in)[4][4] = sm->ring[lrow > 0 ? lrow - 1 : 0];
	uint32_t (*ring_out)[4][4] = sm->ring[lrow];
	volatile int *done_in = sm->done + (lrow > 0 ? lrow - 1 : 0), *done_out = sm->done + lrow;
	volatile int *taken_me = sm->taken + lrow;
	const bool cross_in = half == 0 && wid > 0;      /* upper row fed by another warp: wait on its counter */
	const bool cross_out = half == 1 && to_ring;     /* lower row feeding another warp: respect the ring's depth */

	uint32_t prev[NW], nxt[NW], ntop[NW];
	uint4 ndg = make_uint4(0, 0, 0, 0);
#pragma unroll
	for (int k = 0; k < NW; k++) { prev[k] = 0; nxt[k] = 0; ntop[k] = 0; }
	bool have_top = false;
	int avail = 0;       /* warp-uniform: macroblocks of the row above the band known to be stored (global hand-over) */
	/* prologue: what iteration 0 consumes (upper row, macroblock 0) */
	if (half == 0 && row_ok && W > 0) {
		if (CH) { uint2 v = *(const uint2 *)rowp; nxt[0] = v.x; nxt[1] = v.y; }
		else { uint4 v = *(const uint4 *)rowp; nxt[0] = v.x; nxt[1] = v.y; nxt[2 % NW] = v.z; nxt[3 % NW] = v.w; }
		if (hl < 4) ndg = *((const uint4 *)dgp + hl);
	}

#pragma unroll 1
	for (int i = 0; i <= W + 1; i++) {
		const int x = i - half;
		const bool act = row_ok && x >= 0 && x < W;       /* a macroblock to filter */
		const bool fin = row_ok && x >= 1 && x <= W;      /* macroblock x-1 receives its last change (our left edge) and is stored */
		uint32_t cur[NW];
#pragma unroll
		for (int k = 0; k < NW; k++) cur[k] = nxt[k];
		/* ---- digest into shared memory; room in the lower row's ring ---- */
		if (act && hl < 4) ((uint4 *)&dgs[half])[hl] = ndg;
		if (lane == 0) {	/* the lower row (local row lrow + 1) stores macroblock i - 2 into its ring in this iteration */
			const int xl = i - 1;
			const bool l_out = lrow + 2 < 2 * DBK_PAIRS && mby + 2 < H;
			if (l_out && xl >= 1 && xl <= W) {
				unsigned spins = 0; bool bad = false;
				volatile int *tk = sm->taken + lrow + 2;
				while (*tk < xl - DBK_RING && !bad) { if ((++spins & 1023) == 0) bad = *errp != 0 || spins > (1u << 26); }
				if (bad) atomicExch(J.err, 1u);
			}
		}
		/* ---- requests for the next iteration ---- */
		const bool had_top = have_top;        /* ntop holds the rows above macroblock x */
		uint32_t ctop[NW];
#pragma unroll
		for (int k = 0; k < NW; k++) ctop[k] = ntop[k];
		{
			const int xn = x + 1;
			const bool nact = row_ok && xn >= 0 && xn < W;
			if (nact) {
				if (CH) { uint2 v = *(const uint2 *)(rowp + xn * MBW); nxt[0] = v.x; nxt[1] = v.y; }
				else { uint4 v = *(const uint4 *)(rowp + xn * MBW); nxt[0] = v.x; nxt[1] = v.y; nxt[2 % NW] = v.z; nxt[3 % NW] = v.w; }
				if (hl < 4) ndg = *((const uint4 *)(dgp + xn) + hl);
			}
			have_top = from_global && nact && avail >= xn + 1;     /* already known to be stored: no flag access */
			if (have_top && top_lane) {
				if (CH) { uint2 v = __ldcg((const uint2 *)(topp + xn * MBW)); ntop[0] = v.x; ntop[1] = v.y; }
				else { uint4 v = __ldcg((const uint4 *)(topp + xn * MBW)); ntop[0] = v.x; ntop[1] = v.y; ntop[2 % NW] = v.z; ntop[3 % NW] = v.w; }
			}
		}
		__syncwarp();
		/* ---- vertical edges: this lane's sample row, left to right, in registers ---- */
		uint32_t carry = prev[NW - 1];
		/* the bS 4 vote is taken by the whole warp, outside the predicated region (a vote inside diverged code can hang) */
		const int seg4 = (CH ? r >> 1 : hl >> 2) * 4;
		uint32_t bs0 = 0, bs1 = 0;
		if (act) { bs0 = dgs[half].bs[0]; bs1 = dgs[half].bs[1]; }
		const bool any4 = CH ? false : __any_sync(0xffffffffu, ((bs0 >> seg4) & 15) == 4);
		if (act) {
			const E264DbkMb *dg = &dgs[half];
			const int a_in = dg->alpha[pi * 3], b_in = dg->beta[pi * 3], a_mb = dg->alpha[pi * 3 + 1], b_mb = dg->beta[pi * 3 + 1];
			const uint8_t *tc_in = dg->tc0 + pi * 9, *tc_mb = dg->tc0 + pi * 9 + 3;
			if (CH) {
				int c2 = dbk_byte(carry, 2), c3 = dbk_byte(carry, 3);
				int s0 = dbk_byte(cur[0], 0), s1 = dbk_byte(cur[0], 1), s2 = dbk_byte(cur[0], 2), s3 = dbk_byte(cur[0], 3);
				int s4 = dbk_byte(cur[1], 0), s5 = dbk_byte(cur[1], 1), s6 = dbk_byte(cur[1], 2), s7 = dbk_byte(cur[1], 3);
				const int b0 = (bs0 >> seg4) & 15, b2 = (bs1 >> seg4) & 15;      /* chroma edges 0, 1 take the bS of luma edges 0, 2 */
				dbk_line_chroma(c2, c3, s0, s1, b0, a_mb, b_mb, tc_mb[(b0 - 1) & 3]);
				dbk_line_chroma(s2, s3, s4, s5, b2, a_in, b_in, tc_in[(b2 - 1) & 3]);
				carry = (carry & 0x00ffffffu) | (uint32_t)c3 << 24;
				cur[0] = dbk_pack(s0, s1, s2, s3); cur[1] = dbk_pack(s4, s5, s6, s7);
			} else {
				int s[20];
#pragma unroll
				for (int k = 0; k < 4; k++) s[k] = dbk_byte(carry, k);
#pragma unroll
				for (int k = 0; k < 16; k++) s[4 + k] = dbk_byte(cur[(k >> 2) % NW], k & 3);
				const int b0 = (bs0 >> seg4) & 15, b1 = (bs0 >> (16 + seg4)) & 15, b2 = (bs1 >> seg4) & 15, b3 = (bs1 >> (16 + seg4)) & 15;
				dbk_line_luma<true>(s[0], s[1], s[2], s[3], s[4], s[5], s[6], s[7], b0, a_mb, b_mb, tc_mb[(b0 - 1) & 3], any4);
				dbk_line_luma<false>(s[4], s[5], s[6], s[7], s[8], s[9], s[10], s[11], b1, a_in, b_in, tc_in[(b1 - 1) & 3], false);
				dbk_line_luma<false>(s[8], s[9], s[10], s[11], s[12], s[13], s[14], s[15], b2, a_in, b_in, tc_in[(b2 - 1) & 3], false);
				dbk_line_luma<false>(s[12], s[13], s[14], s[15], s[16], s[17], s[18], s[19], b3, a_in, b_in, tc_in[(b3 - 1) & 3], false);
				carry = dbk_pack(s[0], s[1], s[2], s[3]);
#pragma unroll
				for (int k = 0; k < 4; k++) cur[k % NW] = dbk_pack(s[4 + 4 * k], s[5 + 4 * k], s[6 + 4 * k], s[7 + 4 * k]);
			}
		}
		/* ---- macroblock x-1 is final for this row ---- */
		if (to_global && fin && hl == 0 && x >= 2 && (x - 1) % DBK_CHUNK == 0) { __threadfence(); prog[mby] = base + (unsigned)(x - 1); }   /* covers the stores of earlier iterations only */
		if (fin) {
			uint8_t *d = rowp + (x - 1) * MBW;
			if (CH) *(uint2 *)d = make_uint2(prev[0], carry);
			else *(uint4 *)d = make_uint4(prev[0], prev[1 % NW], prev[2 % NW], carry);
			if (to_ring) {      /* its bottom rows are the top rows of the row below */
				uint32_t (*slot)[4] = ring_out[(x - 1) % DBK_RING];
				if (CH) { if (r >= 6) { slot[pl * 2 + r - 6][0] = prev[0]; slot[pl * 2 + r - 6][1] = carry; } }
				else if (hl >= 12) { slot[hl - 12][0] = prev[0]; slot[hl - 12][1] = prev[1 % NW]; slot[hl - 12][2] = prev[2 % NW]; slot[hl - 12][3] = carry; }
			}
		}
		if (act) {
#pragma unroll
			for (int k = 0; k < NW; k++) tile[lane][k] = cur[k];
		}
		__syncwarp();
		if (cross_out && fin && hl == 0) { __threadfence_block(); *done_out = x; }     /* macroblocks 0..x-1 are in the ring */
		/* ---- the rows above: needed by the horizontal pass only, so the row above has to be just ONE macroblock ahead
		 * (its vertical pass of x + 1 finalises x).  Lower row of the warp: the upper row wrote the ring slot before the
		 * barrier above.  Upper row: lane 0 waits (single-exit loops, the warp reconverges behind them) for the warp above
		 * (shared-memory counter) or the previous band (global progress counter). */
		if (lane == 0 && act && mby > 0) {      /* lane 0 belongs to the upper row: act, mby, x are the upper row's */
			unsigned spins = 0; bool bad = false;
			if (wid > 0) {
				while (*done_in < x + 1 && !bad) { if ((++spins & 1023) == 0) bad = *errp != 0 || spins > (1u << 26); }
				__threadfence_block();
			} else if (avail < x + 1) {
				const unsigned need = base + (unsigned)x + 1u;
				unsigned v = prog[mby - 1];
				while ((int)(v - need) < 0 && !bad) { __nanosleep(40); if ((++spins & 255) == 0) bad = *errp != 0 || spins > (1u << 22); v = prog[mby - 1]; }
				__threadfence();
				avail = bad ? W : (int)(v - base);
			}
			if (bad) atomicExch(J.err, 1u);
		}
		__syncwarp();
		avail = __shfl_sync(0xffffffffu, avail, 0);
		if (act && top_lane) {
			uint32_t tw[NW];
#pragma unroll
			for (int k = 0; k < NW; k++) tw[k] = from_global ? ctop[k] : ring_in[x % DBK_RING][hl][k];
			if (from_global && !had_top) {       /* rare: the row above was not known to be ready one iteration ago */
				if (CH) { uint2 v = __ldcg((const uint2 *)(topp + x * MBW)); tw[0] = v.x; tw[1] = v.y; }
				else { uint4 v = __ldcg((const uint4 *)(topp + x * MBW)); tw[0] = v.x; tw[1] = v.y; tw[2 % NW] = v.z; tw[3 % NW] = v.w; }
			}
#pragma unroll
			for (int k = 0; k < NW; k++) top[half][hl][k] = tw[k];
		}
		__syncwarp();
		if (cross_in && act && hl == 0) *taken_me = x + 1;      /* the ring slot has been copied */
		/* ---- horizontal edges: this lane's sample column, top to bottom ---- */
		const int c = CH ? hl & 7 : hl;
		const int hseg4 = (CH ? c >> 1 : c >> 2) * 4;
		uint32_t bs2 = 0, bs3 = 0;
		if (act) { bs2 = dgs[half].bs[2]; bs3 = dgs[half].bs[3]; }
		const bool hany4 = CH ? false : __any_sync(0xffffffffu, ((bs2 >> hseg4) & 15) == 4);
		if (act) {
			const E264DbkMb *dg = &dgs[half];
			const int a_in = dg->alpha[pi * 3], b_in = dg->beta[pi * 3], a_mb = dg->alpha[pi * 3 + 2], b_mb = dg->beta[pi * 3 + 2];
			const uint8_t *tc_in = dg->tc0 + pi * 9, *tc_mb = dg->tc0 + pi * 9 + 6;
			const uint8_t *tcol = (const uint8_t *)tile[half * 16 + (CH ? pl * 8 : 0)] + c;
			uint8_t *topc = (uint8_t *)top[half][CH ? pl * 2 : 0] + c;
			if (CH) {
				int t0 = 0, t1 = 0, s[8];
				if (mby > 0) { t0 = topc[0]; t1 = topc[16]; }
#pragma unroll
				for (int k = 0; k < 8; k++) s[k] = tcol[k * DBK_TS * 4];
				const int b0 = (bs2 >> hseg4) & 15, b2 = (bs3 >> hseg4) & 15;
				dbk_line_chroma(t0, t1, s[0], s[1], b0, a_mb, b_mb, tc_mb[(b0 - 1) & 3]);
				dbk_line_chroma(s[2], s[3], s[4], s[5], b2, a_in, b_in, tc_in[(b2 - 1) & 3]);
				uint8_t *wcol = (uint8_t *)tcol;
				if (mby > 0) topc[16] = (uint8_t)t1;
				wcol[0] = (uint8_t)s[0]; wcol[3 * DBK_TS * 4] = (uint8_t)s[3]; wcol[4 * DBK_TS * 4] = (uint8_t)s[4];
			} else {
				int s[20];
#pragma unroll
				for (int k = 0; k < 4; k++) s[k] = mby > 0 ? (int)topc[k * 16] : 0;
#pragma unroll
				for (int k = 0; k < 16; k++) s[4 + k] = tcol[k * DBK_TS * 4];
				const int b0 = (bs2 >> hseg4) & 15, b1 = (bs2 >> (16 + hseg4)) & 15, b2 = (bs3 >> hseg4) & 15, b3 = (bs3 >> (16 + hseg4)) & 15;
				dbk_line_luma<true>(s[0], s[1], s[2], s[3], s[4], s[5], s[6], s[7], b0, a_mb, b_mb, tc_mb[(b0 - 1) & 3], hany4);
				dbk_line_luma<false>(s[4], s[5], s[6], s[7], s[8], s[9], s[10], s[11], b1, a_in, b_in, tc_in[(b1 - 1) & 3], false);
				dbk_line_luma<false>(s[8], s[9], s[10], s[11], s[12], s[13], s[14], s[15], b2, a_in, b_in, tc_in[(b2 - 1) & 3], false);
				dbk_line_luma<false>(s[12], s[13], s[14], s[15], s[16], s[17], s[18], s[19], b3, a_in, b_in, tc_in[(b3 - 1) & 3], false);
				uint8_t *wcol = (uint8_t *)tcol;
				if (mby > 0) { topc[16] = (uint8_t)s[1]; topc[32] = (uint8_t)s[2]; topc[48] = (uint8_t)s[3]; }
#pragma unroll
				for (int k = 0; k < 15; k++) wcol[k * DBK_TS * 4] = (uint8_t)s[4 + k];
			}
		}
		__syncwarp();
		/* ---- back to rows: keep the macroblock for its last change, write the rows above back ---- */
		if (act) {
#pragma unroll
			for (int k = 0; k < NW; k++) prev[k] = tile[lane][k];
			if (wb_lane) {
				uint8_t *d = topp + x * MBW;
				if (CH) *(uint2 *)d = make_uint2(top[half][hl][0], top[half][hl][1]);
				else *(uint4 *)d = make_uint4(top[half][hl][0], top[half][hl][1], top[half][hl][2 % NW], top[half][hl][3 % NW]);
			}
		}
		__syncwarp();
	}
	/* the band's last row is stored: let the next band finish */
	__syncwarp();
	if (to_global && hl == 0) { __threadfence(); prog[mby] = base + (unsigned)W; }
}

/* MINB blocks per SM = the register budget: the kernel is a chain of dependent steps (a lone warp per scheduler issues
 * about one instruction in five cycles) and holds its registers for the whole picture, so with many pictures in flight
 * the registers of waiting deblocking warps are what the other kernels lack */
template <int MINB>
__global__ void __launch_bounds__(DBK_PAIRS * 32, MINB) e264_deblock_kernel(PicJob J) {
	TraceScope trace_(J, 3);
	reset_next_tickets(J);
	__shared__ DbkSmem sm;
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
	const int bands = (J.h_mbs + 2 * DBK_PAIRS - 1) / (2 * DBK_PAIRS);
	/* bands x {luma, chroma}; tickets in dispatch order: a band only waits for bands drawn before it */
	for (;;) {
		__syncthreads();
		if (threadIdx.x < 2 * DBK_PAIRS) { sm.done[threadIdx.x] = 0; sm.taken[threadIdx.x] = 0; }
		if (threadIdx.x == 0) sm.band = (int)atomicAdd(J.tickets + 1, 1u);
		__syncthreads();
		const int t = sm.band;
		if (t >= 2 * bands) break;
		if (t & 1) dbk_walk<true>(J, &sm, t >> 1, wid, lane);
		else dbk_walk<false>(J, &sm, t >> 1, wid, lane);
	}
}

