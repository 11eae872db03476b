/* The differential fuzz of oracle/ref_kat.c without the reference: the same seeded inputs (same generator, same draw
 * order) through the restatement (oracle/port_recon.c) only, one FNV-1a digest per trial over the outputs in the layout
 * the reference's functions leave them in, compared with the digests `ref_kat <fuzz|residual|deblock> --digests` recorded
 * from the reference (tests/golden/kat_fuzz_*.bin).
 *   kat_fuzz_check fuzz|residual|deblock GOLDEN   prints "<what> fuzz: ok" when every trial matches */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

typedef struct { const uint8_t *p; int stride, w, h; } Plane;
int port_mc_luma_sample(const Plane *r, int x, int y, int fx, int fy);
void port_idct4x4(const int16_t *c, const uint8_t *scaling, int qp, int has_dc_override, int dc, int16_t *r);
void port_idct8x8(const int16_t *c, const uint8_t *scaling, int qp, int16_t *r);
void port_luma_dc(const int16_t *c, const uint8_t *scaling_y_intra, int qp, int *dc);
void port_chroma_dc(const int16_t *c, int scale0, int qpc, int *dc);
void port_deblock_luma_line(uint8_t *pix, int step, int bs, int alpha, int beta, int tc0);
void port_deblock_chroma_line(uint8_t *pix, int step, int bs, int alpha, int beta, int tc0);

static uint64_t rs = 88172645463325252ull;
static unsigned rnd(void) { rs ^= rs << 13; rs ^= rs >> 7; rs ^= rs << 17; return (unsigned)(rs >> 11); }
static uint32_t fnv(uint32_t h, const void *p, size_t n) { const uint8_t *b = (const uint8_t *)p; for (size_t i = 0; i < n; i++) h = (h ^ b[i]) * 16777619u; return h; }

static const uint32_t *gold; static long n_gold; static int bad;
static void check(const char *what, int trial, uint32_t d) {
	if (trial >= n_gold || gold[trial] != d) { if (bad < 5) printf("%s MISMATCH trial %d\n", what, trial); bad++; }
}

static void fuzz_inter(void) {
	static uint8_t src[64 * 64], row[16];
	for (int trial = 0; trial < 3000; trial++) {
		int kind = trial % 4;
		int px = 1 + rnd() % 3, py = 1 + rnd() % 3, ph = rnd();
		uint32_t d = 2166136261u;
		for (int i = 0; i < 64 * 64; i++) src[i] = kind == 0 ? rnd() : kind == 1 ? ((rnd() & 1) ? 255 : 0) : kind == 2 ? (uint8_t)((((i % 64) / px + (i / 64) / py + ph) & 1) ? 255 - rnd() % 3 : rnd() % 3) : ((rnd() % 5) ? 255 : rnd());
		for (int mode = 0; mode < 48; mode++) {
			int w = 4 << (mode >> 4), fx = mode & 3, fy = (mode >> 2) & 3;
			for (int hh = 0; hh < 3; hh++) {
				int h = 4 << hh;
				if ((w == 4 && h == 16) || (w == 16 && h == 4)) continue;
				Plane P = {src, 64, 64, 64};
				for (int y = 0; y < h; y++) {
					for (int x = 0; x < w; x++) row[x] = (uint8_t)port_mc_luma_sample(&P, 20 + x, 20 + y, fx, fy);
					d = fnv(d, row, w);
				}
			}
		}
		check("LUMA", trial, d);
	}
	printf("inter luma fuzz: %s\n", bad ? "MISMATCHES" : "ok");
}

static int clip8(int v) { return v < 0 ? 0 : v > 255 ? 255 : v; }
static void fuzz_residual(void) {
	static uint8_t want[32 * 16];
	static const uint8_t zr[16] = {0, 1, 4, 5, 2, 3, 6, 7, 8, 9, 12, 13, 10, 11, 14, 15};
	for (int trial = 0; trial < 20000; trial++) {
		const int iY = rnd() % 3, inter = rnd() & 1, qp = rnd() % 52, extreme = (trial % 5) == 4, flat = (trial % 3) == 0;
		(void)iY; (void)inter;    /* they select the reference's scaling list; the restatement takes the list itself */
		for (int i = 0; i < 32 * 16; i++) want[i] = rnd();
		/* --- 4x4 --- */
		uint8_t sc[16]; int16_t lv[16], res[16];
		for (int i = 0; i < 16; i++) sc[i] = flat ? 16 : 1 + rnd() % 255;
		const int range = extreme ? 32768 : (rnd() % 3 ? 64 : 2048);
		for (int i = 0; i < 16; i++) lv[i] = (rnd() % 3) ? 0 : (int)(rnd() % (2 * range)) - range;
		const int dcidx = (rnd() % 3 == 0) ? (int)(rnd() % 8) : -1, dcv = (int)(rnd() % 65536) - 32768;
		port_idct4x4(lv, sc, qp, dcidx >= 0, dcv, res);
		for (int y = 0; y < 4; y++) for (int x = 0; x < 4; x++) want[32 * (4 + y) + 8 + x] = (uint8_t)clip8((int16_t)(want[32 * (4 + y) + 8 + x] + res[y * 4 + x]));
		uint32_t d = fnv(2166136261u, want, sizeof(want));
		/* --- 8x8 --- */
		uint8_t sc8[64]; int16_t lv8[64], res8[64];
		for (int i = 0; i < 64; i++) { sc8[i] = flat ? 16 : 1 + rnd() % 255; lv8[i] = (rnd() % 4) ? 0 : (int)(rnd() % (2 * range)) - range; }
		port_idct8x8(lv8, sc8, qp, res8);
		for (int y = 0; y < 8; y++) for (int x = 0; x < 8; x++) want[32 * (6 + y) + 16 + x] = (uint8_t)clip8((int16_t)(want[32 * (6 + y) + 16 + x] + res8[y * 8 + x]));
		d = fnv(d, want, sizeof(want));
		/* --- Intra16x16 luma DC, in the reference's luma4x4BlkIdx order --- */
		int16_t dl[16]; int dcs[16];
		for (int i = 0; i < 16; i++) dl[i] = (int)(rnd() % (2 * (extreme ? 32768 : 512))) - (extreme ? 32768 : 512);
		port_luma_dc(dl, sc, qp, dcs);
		for (int b = 0; b < 16; b++) { int32_t v = dcs[zr[b]]; d = fnv(d, &v, 4); }
		/* --- chroma DC 2x2, Cb then Cr --- */
		int16_t cb[4], cr[4]; int dcb[4], dcr[4];
		for (int i = 0; i < 4; i++) { cb[i] = (int)(rnd() % 2048) - 1024; cr[i] = (int)(rnd() % 2048) - 1024; }
		const int qb = rnd() % 52, qr = rnd() % 52, sb = flat ? 16 : 1 + rnd() % 255, sr_ = flat ? 16 : 1 + rnd() % 255;
		port_chroma_dc(cb, sb, qb, dcb); port_chroma_dc(cr, sr_, qr, dcr);
		for (int i = 0; i < 8; i++) { int32_t v = i < 4 ? dcb[i] : dcr[i - 4]; d = fnv(d, &v, 4); }
		check("RESIDUAL", trial, d);
	}
	printf("residual fuzz: %s\n", bad ? "MISMATCHES" : "ok");
}

static void fuzz_deblock(void) {
	enum { ST = 64 };
	static uint8_t wy[ST * 48], wc[ST * 32];
	uint8_t alpha[16], beta[16]; int8_t tc[64]; int inter[3];
	for (int trial = 0; trial < 30000; trial++) {
		const int smooth = trial % 3 != 0;
		int v = rnd() % 256;
		for (int i = 0; i < ST * 48; i++) { if (smooth) { v += (int)(rnd() % 9) - 4; v = v < 0 ? 0 : v > 255 ? 255 : v; if (rnd() % 23 == 0) v = rnd() % 256; wy[i] = (uint8_t)v; } else wy[i] = rnd(); }
		for (int i = 0; i < ST * 32; i++) { if (smooth) { v += (int)(rnd() % 7) - 3; v = v < 0 ? 0 : v > 255 ? 255 : v; if (rnd() % 19 == 0) v = rnd() % 256; wc[i] = (uint8_t)v; } else wc[i] = rnd(); }
		const int fe = trial % 7 == 0 ? rnd() & 3 : 3, t8 = rnd() & 1;
		inter[0] = rnd() % 4 != 0; inter[1] = rnd() % 3 != 0; inter[2] = rnd() % 3 != 0;
		for (int i = 0; i < 16; i++) { alpha[i] = (rnd() % 5 == 0) ? 0 : (smooth ? 4 + rnd() % 60 : rnd() % 256); beta[i] = (rnd() % 7 == 0) ? 0 : 2 + rnd() % 17; }
		for (int i = 0; i < 64; i++) tc[i] = (rnd() % 3 == 0) ? -1 : (int8_t)(rnd() % 14);
		if (rnd() % 5 == 0) for (int e = 0; e < 16; e++) if (rnd() & 1) for (int k = 0; k < 4; k++) tc[e * 4 + k] = -1;
		uint8_t *Y = wy + ST * 16 + 16;
		for (int dir = 0; dir < 2; dir++) for (int e = 0; e < 4; e++) {
			if (e == 0 && !(fe & (dir ? 2 : 1))) continue;
			if (e && t8 && (e & 1)) continue;
			const int hard = e == 0 && !(inter[0] & (dir ? inter[2] : inter[1]));
			const int ai = e ? 0 : dir ? 12 : 8;
			if (hard && alpha[ai] == 0) continue;
			for (int k = 0; k < 16; k++) {
				const int t0 = tc[(dir * 4 + e) * 4 + (k >> 2)];
				if (!hard && t0 < 0) continue;
				uint8_t *pix = dir ? Y + e * 4 * ST + k : Y + k * ST + e * 4;
				port_deblock_luma_line(pix, dir ? ST : 1, hard ? 4 : 1, alpha[ai], beta[ai], hard ? 0 : t0);
			}
		}
		for (int pl = 0; pl < 2; pl++) {
			uint8_t *C = wc + ST * 8 + 8 + pl * (ST / 2);
			for (int dir = 0; dir < 2; dir++) for (int e = 0; e < 2; e++) {
				if (e == 0 && !(fe & (dir ? 2 : 1))) continue;
				const int hard = e == 0 && !(inter[0] & (dir ? inter[2] : inter[1]));
				const int ai = (e ? 0 : dir ? 12 : 8) + 1 + pl;
				for (int k = 0; k < 8; k++) {
					const int t0 = tc[32 + ((dir * 2 + e) * 2 + pl) * 4 + (k >> 1)];
					if (!hard && t0 < 0) continue;
					uint8_t *pix = dir ? C + e * 4 * ST + k : C + k * ST + e * 4;
					port_deblock_chroma_line(pix, dir ? ST : 1, hard ? 4 : 1, alpha[ai], beta[ai], hard ? 0 : t0);
				}
			}
		}
		check("DEBLOCK", trial, fnv(fnv(2166136261u, wy, sizeof(wy)), wc, sizeof(wc)));
	}
	printf("deblock fuzz: %s\n", bad ? "MISMATCHES" : "ok");
}

int main(int argc, char **argv) {
	if (argc != 3) { fprintf(stderr, "usage: kat_fuzz_check fuzz|residual|deblock GOLDEN\n"); return 2; }
	FILE *f = fopen(argv[2], "rb");
	if (!f) { perror(argv[2]); return 2; }
	fseek(f, 0, SEEK_END); n_gold = ftell(f) / 4; fseek(f, 0, SEEK_SET);
	uint32_t *g = (uint32_t *)malloc((size_t)n_gold * 4 + 4);
	if (fread(g, 4, (size_t)n_gold, f) != (size_t)n_gold) { fprintf(stderr, "%s: short read\n", argv[2]); return 2; }
	fclose(f); gold = g;
	long want = !strcmp(argv[1], "fuzz") ? 3000 : !strcmp(argv[1], "residual") ? 20000 : !strcmp(argv[1], "deblock") ? 30000 : -1;
	if (want < 0) { fprintf(stderr, "unknown fuzz %s\n", argv[1]); return 2; }
	if (n_gold != want) { printf("%s holds %ld digests, %ld trials expected\n", argv[2], n_gold, want); return 1; }
	if (want == 3000) fuzz_inter(); else if (want == 20000) fuzz_residual(); else fuzz_deblock();
	return bad != 0;
}
