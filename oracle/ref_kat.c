/* oracle/ref_kat.c — TEST INFRASTRUCTURE (build container only).  Includes the reference's intra and inter
 * sources the way its own edge264_check.c:20-22 does, and
 *   ref_kat fuzz     differential fuzz of the reference's decode_inter_luma / decode_inter_chroma against
 *                    the plain-C restatement (oracle/port_recon.c), all 48 luma modes, random + extreme sources
 *   ref_kat residual differential fuzz of the reference's add_idct4x4 / add_idct8x8 / transform_dc4x4 / transform_dc2x2
 *                    (edge264_residual.c:108-538) against port_idct4x4 / port_idct8x8 / port_luma_dc / port_chroma_dc:
 *                    random QP 0..51, random and flat scaling lists, intra/inter lists, conformant-range and extreme levels
 *   ref_kat deblock  differential fuzz of the reference's deblock_Y_8bit + deblock_CbCr_8bit (edge264_deblock.c:284-895) on one
 *                    macroblock with its left and top neighbours against the restatement's line filters: random alpha/beta,
 *                    tC0 per 4-sample (2-sample chroma) segment incl. -1 = bS 0, HARD edges when a neighbour is intra,
 *                    transform_size_8x8_flag, smooth and noisy pictures
 *   ref_kat dump     prints the known-answer inputs/outputs of the reference's KAT setup as JSON
 *                    (tests/golden/kat_*.json are generated from this)
 *   ref_kat <fuzz|residual|deblock> --digests FILE   also writes one FNV-1a digest of the reference's outputs per trial
 *                    (uint32, little-endian) to FILE: tests/golden/kat_fuzz_*.bin, which tests/native/kat_fuzz_check.c
 *                    replays against the restatement where the reference is not available
 * Nothing from the reference is copied: the sources are compiled from $(REF)/src at build time. */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "edge264_internal.h"
#include "edge264_intra.c"
#include "edge264_inter.c"
#include "edge264_residual.c"
#include "edge264_deblock.c"

typedef struct { const uint8_t *p; int stride, w, h; } Plane;
int port_mc_luma_sample(const Plane *r, int x, int y, int fx, int fy);
int port_mc_chroma_sample(const Plane *r, int x, int y, int fx, int fy);
void port_intra4x4(uint8_t *p, int stride, int imode);
void port_intra8x8(uint8_t *p, int stride, int imode);
void port_intra16x16(uint8_t *p, int stride, int imode);
void port_intra_chroma(uint8_t *p, int stride, int imode);
void port_idct4x4(const int16_t *c, const uint8_t *scaling, int qp, int has_dc_override, int dc, int16_t *r);
void port_idct8x8(const int16_t *c, const uint8_t *scaling, int qp, int16_t *r);
void port_luma_dc(const int16_t *c, const uint8_t *scaling_y_intra, int qp, int *dc);
void port_chroma_dc(const int16_t *c, int scale0, int qpc, int *dc);
void port_deblock_luma_line(uint8_t *pix, int step, int bs, int alpha, int beta, int tc0);
void port_deblock_chroma_line(uint8_t *pix, int step, int bs, int alpha, int beta, int tc0);

static uint64_t rs = 88172645463325252ull;
static unsigned rnd(void) { rs ^= rs << 13; rs ^= rs >> 7; rs ^= rs << 17; return (unsigned)(rs >> 11); }

static FILE *digests;
static uint32_t fnv(uint32_t h, const void *p, size_t n) { const uint8_t *b = (const uint8_t *)p; for (size_t i = 0; i < n; i++) h = (h ^ b[i]) * 16777619u; return h; }
static void put_digest(uint32_t d) { if (digests) fwrite(&d, 4, 1, digests); }

static int fuzz_inter(void) {
	static uint8_t src[64 * 64] __attribute__((aligned(16))), dst[16 * 16] __attribute__((aligned(16)));
	int bad = 0;
	for (int trial = 0; trial < 3000 && bad < 10; trial++) {
		int kind = trial % 4;
		int px = 1 + rnd() % 3, py = 1 + rnd() % 3, ph = rnd();
		uint32_t d = 2166136261u;
		for (int i = 0; i < 64 * 64; i++) src[i] = kind == 0 ? rnd() : kind == 1 ? ((rnd() & 1) ? 255 : 0) : kind == 2 ? (uint8_t)((((i % 64) / px + (i / 64) / py + ph) & 1) ? 255 - rnd() % 3 : rnd() % 3) : ((rnd() % 5) ? 255 : rnd());
		for (int mode = 0; mode < 48; mode++) {
			int w = 4 << (mode >> 4), fx = mode & 3, fy = (mode >> 2) & 3;
			for (int hh = 0; hh < 3; hh++) {
				int h = 4 << hh;
				if ((w == 4 && h == 16) || (w == 16 && h == 4)) continue;
				memset(dst, 0, sizeof(dst));
				decode_inter_luma(mode, h, 64, src + 20 * 64 + 20, 16, dst, (i8x16){0, 1});
				for (int y = 0; y < h; y++) d = fnv(d, dst + y * 16, w);
				Plane P = {src, 64, 64, 64};
				for (int y = 0; y < h; y++) for (int x = 0; x < w; x++) {
					int v = port_mc_luma_sample(&P, 20 + x, 20 + y, fx, fy);
					if (v != dst[y * 16 + x] && bad < 10) { printf("LUMA MISMATCH trial %d mode %d (w%d h%d fx%d fy%d) at (%d,%d): ref %d port %d\n", trial, mode, w, h, fx, fy, x, y, dst[y * 16 + x], v); bad++; }
				}
			}
		}
		put_digest(d);
	}
	printf("inter luma fuzz: %s\n", bad ? "MISMATCHES" : "ok");
	return bad;
}


/* ---- residual: the reference works on ctx->c[] (int32, column-major: c[x*4+y], SURVEY §0.5) and adds into the picture;
 * the restatement works on raster int16 levels and returns the residual.  Scaling lists are stored by the reference in
 * the same column-major order as c[] (they multiply element-wise, residual.c:114-121), ours are raster. */
static int clip8(int v) { return v < 0 ? 0 : v > 255 ? 255 : v; }
static int fuzz_residual(void) {
	static Edge264Context ctx __attribute__((aligned(64)));
	static Edge264Macroblock mbs __attribute__((aligned(64)));
	static uint8_t pix[32 * 16] __attribute__((aligned(16))), want[32 * 16];
	int bad = 0;
	memset(&ctx, 0, sizeof(ctx)); memset(&mbs, 0, sizeof(mbs));
	ctx._mb = &mbs;
	for (int k = 0; k < 3; k++) { ctx.t.stride[k] = 32; ctx.t.samples_clip[k][0] = 255; }
	for (int trial = 0; trial < 20000 && bad < 10; trial++) {
		const int iY = rnd() % 3, inter = rnd() & 1, qp = rnd() % 52, extreme = (trial % 5) == 4, flat = (trial % 3) == 0;
		ctx.t.QP[0] = ctx.t.QP[1] = ctx.t.QP[2] = qp; mbs.mbIsInterFlag = inter;
		for (int i = 0; i < 32 * 16; i++) pix[i] = rnd();
		memcpy(want, pix, sizeof(pix));
		/* --- 4x4 --- */
		uint8_t sc[16]; int16_t lv[16], res[16];
		for (int i = 0; i < 16; i++) sc[i] = flat ? 16 : 1 + rnd() % 255;
		const int range = extreme ? 32768 : (rnd() % 3 ? 64 : 2048);
		for (int i = 0; i < 16; i++) lv[i] = (rnd() % 3) ? 0 : (int)(rnd() % (2 * range)) - range;
		const int dcidx = (rnd() % 3 == 0) ? (int)(rnd() % 8) : -1, dcv = (int)(rnd() % 65536) - 32768;
		for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) {
			ctx.c[j * 4 + i] = lv[i * 4 + j];
			((uint8_t *)&ctx.t.pps.weightScale4x4_v[iY + inter * 3])[j * 4 + i] = sc[i * 4 + j];
		}
		if (dcidx >= 0) ctx.c[16 + dcidx] = dcv;
		add_idct4x4(&ctx, iY, dcidx, pix + 32 * 4 + 8);
		uint32_t d = fnv(2166136261u, pix, sizeof(pix));
		port_idct4x4(lv, sc, qp, dcidx >= 0, dcv, res);
		for (int y = 0; y < 4; y++) for (int x = 0; x < 4; x++) want[32 * (4 + y) + 8 + x] = (uint8_t)clip8((int16_t)(want[32 * (4 + y) + 8 + x] + res[y * 4 + x]));
		if (memcmp(want, pix, sizeof(pix))) { if (bad++ < 5) printf("IDCT4x4 MISMATCH trial %d qp %d plane %d inter %d dcidx %d\n", trial, qp, iY, inter, dcidx); memcpy(want, pix, sizeof(pix)); }
		for (int i = 0; i < 16; i++) if (ctx.c[i]) { if (bad++ < 5) printf("IDCT4x4 did not clear c[]\n"); break; }
		/* --- 8x8 (luma lists only in 4:2:0: index (iYCbCr*2+inter)*4 with iYCbCr = 0, residual.c:203) --- */
		uint8_t sc8[64]; int16_t lv8[64], res8[64];
		for (int i = 0; i < 64; i++) { sc8[i] = flat ? 16 : 1 + rnd() % 255; lv8[i] = (rnd() % 4) ? 0 : (int)(rnd() % (2 * range)) - range; }
		for (int i = 0; i < 8; i++) for (int j = 0; j < 8; j++) {
			ctx.c[j * 8 + i] = lv8[i * 8 + j];
			((uint8_t *)(ctx.t.pps.weightScale8x8_v + inter * 4))[j * 8 + i] = sc8[i * 8 + j];
		}
		add_idct8x8(&ctx, 0, pix + 32 * 6 + 16);
		d = fnv(d, pix, sizeof(pix));
		port_idct8x8(lv8, sc8, qp, res8);
		for (int y = 0; y < 8; y++) for (int x = 0; x < 8; x++) want[32 * (6 + y) + 16 + x] = (uint8_t)clip8((int16_t)(want[32 * (6 + y) + 16 + x] + res8[y * 8 + x]));
		if (memcmp(want, pix, sizeof(pix))) { if (bad++ < 5) printf("IDCT8x8 MISMATCH trial %d qp %d inter %d extreme %d\n", trial, qp, inter, extreme); memcpy(want, pix, sizeof(pix)); }
		memset(ctx.c, 0, sizeof(ctx.c));
		/* --- Intra16x16 luma DC (results kept for the AC pass: mb->bits[0] bit 5, residual.c:395-399) --- */
		int16_t dl[16]; int dcs[16];
		for (int i = 0; i < 16; i++) dl[i] = (int)(rnd() % (2 * (extreme ? 32768 : 512))) - (extreme ? 32768 : 512);
		for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) ctx.c[j * 4 + i] = dl[i * 4 + j];
		((uint8_t *)&ctx.t.pps.weightScale4x4_v[0])[0] = sc[0]; ((uint8_t *)ctx.t.pps.weightScale4x4[0])[0] = sc[0];
		mbs.bits[0] |= 1 << 5;
		transform_dc4x4(&ctx, 0);
		port_luma_dc(dl, sc, qp, dcs);
		{	/* the reference stores the 16 DCs in luma4x4BlkIdx order (ziplo64/ziphi64 pairs, residual.c:396-399) */
			static const uint8_t zr[16] = {0, 1, 4, 5, 2, 3, 6, 7, 8, 9, 12, 13, 10, 11, 14, 15};
			int ok = 1;
			for (int b = 0; b < 16; b++) if (ctx.c[16 + b] != dcs[zr[b]]) ok = 0;
			for (int b = 0; b < 16; b++) { int32_t v = ctx.c[16 + b]; d = fnv(d, &v, 4); }
			if (!ok && bad++ < 5) { printf("LUMA DC MISMATCH trial %d qp %d:", trial, qp); for (int b = 0; b < 16; b++) printf(" %d/%d", ctx.c[16 + b], dcs[zr[b]]); printf("\n"); }
		}
		memset(ctx.c, 0, sizeof(ctx.c));
		/* --- chroma DC 2x2, both planes at once (Cb at c[{0,4,2,6}], Cr at c[{1,5,3,7}], slice.c:448-462) --- */
		int16_t cb[4], cr[4]; int dcb[4], dcr[4];
		for (int i = 0; i < 4; i++) { cb[i] = (int)(rnd() % 2048) - 1024; cr[i] = (int)(rnd() % 2048) - 1024; }
		static const uint8_t posb[4] = {0, 4, 2, 6}, posr[4] = {1, 5, 3, 7};
		for (int i = 0; i < 4; i++) { ctx.c[posb[i]] = cb[i]; ctx.c[posr[i]] = cr[i]; }
		const int qb = rnd() % 52, qr = rnd() % 52, sb = flat ? 16 : 1 + rnd() % 255, sr_ = flat ? 16 : 1 + rnd() % 255;
		ctx.t.QP[1] = qb; ctx.t.QP[2] = qr;
		((uint8_t *)ctx.t.pps.weightScale4x4[1 + inter * 3])[0] = sb; ((uint8_t *)ctx.t.pps.weightScale4x4[2 + inter * 3])[0] = sr_;
		mbs.f.CodedBlockPatternChromaAC = 1;
		transform_dc2x2(&ctx);
		port_chroma_dc(cb, sb, qb, dcb); port_chroma_dc(cr, sr_, qr, dcr);
		{
			int ok = 1;
			for (int i = 0; i < 4; i++) if (ctx.c[16 + i] != dcb[i] || ctx.c[20 + i] != dcr[i]) ok = 0;
			for (int i = 0; i < 8; i++) { int32_t v = ctx.c[16 + i]; d = fnv(d, &v, 4); }
			put_digest(d);
			if (!ok && bad++ < 5) { printf("CHROMA DC MISMATCH trial %d:", trial); for (int i = 0; i < 4; i++) printf(" %d/%d %d/%d", ctx.c[16 + i], dcb[i], ctx.c[20 + i], dcr[i]); printf("\n"); }
		}
		memset(ctx.c, 0, sizeof(ctx.c));
	}
	printf("residual fuzz: %s\n", bad ? "MISMATCHES" : "ok");
	return bad;
}

/* ---- deblocking: the reference filters a whole macroblock from ctx->alpha/beta/tC0 (layout edge264_internal.h:323-325:
 * alpha/beta {internal Y,Cb,Cr,-,...,left Y,Cb,Cr @8,-,top Y,Cb,Cr @12}; tC0: 4 bytes per edge, 8 luma edges (4 vertical
 * left to right, 4 horizontal top to bottom) then Cb/Cr alternating for left, internal vertical, top, internal horizontal).
 * The expected picture applies the restatement's one-line filters in the same edge order (vertical edges first). */
static int fuzz_deblock(void) {
	static Edge264Context ctx __attribute__((aligned(64)));
	static Edge264Macroblock mbs[3] __attribute__((aligned(64)));
	enum { ST = 64 };
	static uint8_t y[ST * 48] __attribute__((aligned(16))), c[ST * 32] __attribute__((aligned(16))), wy[ST * 48], wc[ST * 32];
	int bad = 0;
	memset(&ctx, 0, sizeof(ctx)); memset(mbs, 0, sizeof(mbs));
	ctx._mb = &mbs[0]; ctx._mbA = &mbs[1]; ctx._mbB = &mbs[2];
	ctx.t.stride[0] = ST; ctx.t.stride[1] = ST;
	for (int trial = 0; trial < 30000 && bad < 10; trial++) {
		const int smooth = trial % 3 != 0;
		int v = rnd() % 256;
		for (int i = 0; i < ST * 48; i++) { if (smooth) { v += (int)(rnd() % 9) - 4; v = v < 0 ? 0 : v > 255 ? 255 : v; if (rnd() % 23 == 0) v = rnd() % 256; y[i] = (uint8_t)v; } else y[i] = rnd(); }
		for (int i = 0; i < ST * 32; i++) { if (smooth) { v += (int)(rnd() % 7) - 3; v = v < 0 ? 0 : v > 255 ? 255 : v; if (rnd() % 19 == 0) v = rnd() % 256; c[i] = (uint8_t)v; } else c[i] = rnd(); }
		memcpy(wy, y, sizeof(y)); memcpy(wc, c, sizeof(c));
		const int fe = trial % 7 == 0 ? rnd() & 3 : 3, t8 = rnd() & 1;
		mbs[0].filter_edges = fe; mbs[0].f.transform_size_8x8_flag = t8;
		mbs[0].mbIsInterFlag = rnd() % 4 != 0; mbs[1].mbIsInterFlag = rnd() % 3 != 0; mbs[2].mbIsInterFlag = rnd() % 3 != 0;
		for (int i = 0; i < 16; i++) { ctx.alpha[i] = (rnd() % 5 == 0) ? 0 : (smooth ? 4 + rnd() % 60 : rnd() % 256); ctx.beta[i] = (rnd() % 7 == 0) ? 0 : 2 + rnd() % 17; }
		int8_t *tc = (int8_t *)ctx.tC0_s;
		for (int i = 0; i < 64; i++) tc[i] = (rnd() % 3 == 0) ? -1 : (int8_t)(rnd() % 14);
		if (rnd() % 5 == 0) for (int e = 0; e < 16; e++) if (rnd() & 1) for (int k = 0; k < 4; k++) tc[e * 4 + k] = -1;
		ctx.samples_mb[0] = y + ST * 16 + 16; ctx.samples_mb[1] = c + ST * 8 + 8; ctx.samples_mb[2] = ctx.samples_mb[1] + ST / 2;
		/* expected */
		uint8_t *Y = wy + ST * 16 + 16;
		for (int dir = 0; dir < 2; dir++) for (int e = 0; e < 4; e++) {
			if (e == 0 && !(fe & (dir ? 2 : 1))) continue;
			if (e && t8 && (e & 1)) continue;
			const int hard = e == 0 && !(mbs[0].mbIsInterFlag & (dir ? mbs[2].mbIsInterFlag : mbs[1].mbIsInterFlag));
			const int ai = e ? 0 : dir ? 12 : 8;
			if (hard && ctx.alpha[ai] == 0) continue;
			for (int k = 0; k < 16; k++) {
				const int t0 = tc[(dir * 4 + e) * 4 + (k >> 2)];
				if (!hard && t0 < 0) continue;
				uint8_t *pix = dir ? Y + e * 4 * ST + k : Y + k * ST + e * 4;
				port_deblock_luma_line(pix, dir ? ST : 1, hard ? 4 : 1, ctx.alpha[ai], ctx.beta[ai], hard ? 0 : t0);
			}
		}
		for (int pl = 0; pl < 2; pl++) {
			uint8_t *C = wc + ST * 8 + 8 + pl * (ST / 2);
			for (int dir = 0; dir < 2; dir++) for (int e = 0; e < 2; e++) {
				if (e == 0 && !(fe & (dir ? 2 : 1))) continue;
				const int hard = e == 0 && !(mbs[0].mbIsInterFlag & (dir ? mbs[2].mbIsInterFlag : mbs[1].mbIsInterFlag));
				const int ai = (e ? 0 : dir ? 12 : 8) + 1 + pl;
				for (int k = 0; k < 8; k++) {
					const int t0 = tc[32 + ((dir * 2 + e) * 2 + pl) * 4 + (k >> 1)];
					if (!hard && t0 < 0) continue;
					uint8_t *pix = dir ? C + e * 4 * ST + k : C + k * ST + e * 4;
					port_deblock_chroma_line(pix, dir ? ST : 1, hard ? 4 : 1, ctx.alpha[ai], ctx.beta[ai], hard ? 0 : t0);
				}
			}
		}
		deblock_Y_8bit(&ctx);
		put_digest(fnv(fnv(2166136261u, y, sizeof(y)), c, sizeof(c)));
		if (memcmp(wy, y, sizeof(y)) || memcmp(wc, c, sizeof(c))) {
			if (bad++ < 6) {
				int py = -1, pc = -1;
				for (int i = 0; i < ST * 48 && py < 0; i++) if (wy[i] != y[i]) py = i;
				for (int i = 0; i < ST * 32 && pc < 0; i++) if (wc[i] != c[i]) pc = i;
				printf("DEBLOCK MISMATCH trial %d fe %d t8 %d inter %d/%d/%d: first luma diff at (%d,%d) ref %d port %d, first chroma diff at (%d,%d)\n", trial, fe, t8, mbs[0].mbIsInterFlag, mbs[1].mbIsInterFlag, mbs[2].mbIsInterFlag,
				       py < 0 ? -1 : py % ST - 16, py < 0 ? -1 : py / ST - 16, py < 0 ? 0 : y[py], py < 0 ? 0 : wy[py], pc < 0 ? -1 : pc % ST - 8, pc < 0 ? -1 : pc / ST - 8);
			}
		}
	}
	printf("deblock fuzz: %s\n", bad ? "MISMATCHES" : "ok");
	return bad;
}

/* Known-answer dump: the inputs of the reference's own KATs (edge264_check.c:173-180 border ramp, :286-290
 * luma source) run through the reference's functions; one JSON object on stdout. */
static void dump_block(const char *name, int mode, const uint8_t *p, int stride, int w, int h, int last) {
	printf("  {\"fn\": \"%s\", \"mode\": %d, \"w\": %d, \"h\": %d, \"out\": [", name, mode, w, h);
	for (int y = 0; y < h; y++) for (int x = 0; x < w; x++) printf("%d%s", p[y * stride + x], (y == h - 1 && x == w - 1) ? "" : ",");
	printf("]}%s\n", last ? "" : ",");
}
static int dump_kat(void) {
	uint8_t buf[32 * 18] __attribute__((aligned(16)));
	uint8_t *p = buf + 80;
	i16x8 clip = {255, 255, 255, 255, 255, 255, 255, 255};
	printf("{\"intra\": [\n");
#define RESET_BORDER() do { memset(buf, 0, sizeof(buf)); for (int x = -1; x < 16; x++) { p[x - 32] = 194 + x * 4; p[x - 64] = 198 + x * 4; } for (int y = 0; y < 16; y++) p[y * 32 - 1] = 186 - y * 4; } while (0)
	for (int m = 0; m <= I4x4_HU_8; m++) { RESET_BORDER(); decode_intra4x4(p, 32, m, clip); dump_block("intra4x4", m, p, 32, 4, 4, 0); }
	for (int m = 0; m <= I8x8_HU_D_8; m++) { RESET_BORDER(); decode_intra8x8(p, 32, m, clip); dump_block("intra8x8", m, p, 32, 8, 8, 0); }
	for (int m = 0; m <= I16x16_P_8; m++) { RESET_BORDER(); decode_intra16x16(p, 32, m, clip); dump_block("intra16x16", m, p, 32, 16, 16, 0); }
	for (int m = 0; m <= IC8x8_P_8; m++) { RESET_BORDER(); decode_intraChroma(p, 32, m, clip); dump_block("intraChroma", m, p, 32, 8, 16, m == IC8x8_P_8); }
	printf("], \"inter_luma\": [\n");
	uint8_t src[444], dst[256] __attribute__((aligned(16)));
	for (int i = 0; i < 441; i++) src[i] = (uint8_t)(i * 37);
	for (int mode = 0; mode < 48; mode++) {
		memset(dst, 0, sizeof(dst));
		int h = mode < 16 ? 8 : 16, w = 4 << (mode >> 4);
		decode_inter_luma(mode, h, 21, src + 44, 16, dst, (i8x16){0, 1});
		dump_block("inter_luma", mode, dst, 16, w, h, mode == 47);
	}
	printf("]}\n");
	return 0;
}

int main(int argc, char **argv) {
	if (argc > 3 && !strcmp(argv[2], "--digests") && !(digests = fopen(argv[3], "wb"))) { perror(argv[3]); return 2; }
	if (argc > 1 && !strcmp(argv[1], "fuzz")) return fuzz_inter() != 0;
	if (argc > 1 && !strcmp(argv[1], "residual")) return fuzz_residual() != 0;
	if (argc > 1 && !strcmp(argv[1], "deblock")) return fuzz_deblock() != 0;
	if (argc > 1 && !strcmp(argv[1], "dump")) return dump_kat();
	fprintf(stderr, "usage: ref_kat fuzz | residual | deblock [--digests FILE] | dump\n");
	return 2;
}
