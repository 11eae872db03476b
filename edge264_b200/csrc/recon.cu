/* recon.cu — CUDA runtime of the reconstruction backend + its C-ABI shim (include/e264b_recon.h).
 *
 * Replaces the reference's in-process contract between the slice parser and the pixel functions
 * (reference: prototypes edge264_internal.h:1349-1374, call sites edge264_slice.c:466-664,881,1816,
 * edge264_mvpred.c:73-513, edge264_headers.c:510,551) by: pinned staging filled by the parser ->
 * cudaMemcpyAsync -> two kernels per picture on the decoder's stream -> cudaMemcpyAsync of the
 * finished frame into a pinned host mirror.  Frames live in HBM in the reference's own layout
 * (edge264_headers.c:2027-2046) so the mirror is what edge264_get_frame hands out.
 * There is NO CPU fallback: without a CUDA device e264b_create() fails and edge264_alloc() returns NULL.
 */
#include <cuda_runtime.h>
#include <stdio.h>
#include <time.h>
#include <unistd.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include <mutex>
#include "recon_kernels.cuh"
#include "deblock_kernels.cuh"
#include "inter_kernels.cuh"
#include "intra_kernels.cuh"
extern "C" {
#include "dec.h"
}
#include "../../include/e264b_recon.h"

#define NSTAGE 8            /* staging areas allocated at most; a decoder uses n_stage of them */
#define NTICK 64
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "edge264_b200: CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); return -1; } } while (0)

struct Staging {
	E264MbRec *d_recs; int16_t *d_coefs, *h_coefs; E264SliceRec *d_slices, *h_slices;
	E264DbkMb *d_dbk;            /* deblocking digests of the picture in flight */
	uint32_t *d_intra, *h_intra; /* intra macroblock list */
	cudaEvent_t done; bool busy;
};
struct KeptPic { E264PicDesc pd; E264MbRec *d_recs; int16_t *d_coefs; E264SliceRec *d_slices; uint32_t *d_intra; };

struct E264bDevice {
	int dev; cudaStream_t stream;
	E264PicDesc g; int n_slots; size_t nmb; uint32_t coef_cap;
	uint8_t *d_frames;
	E264MbRec *h_recs[E264_MAX_SLOTS]; cudaEvent_t rec_up[E264_MAX_SLOTS]; bool rec_busy[E264_MAX_SLOTS];
	Staging st[NSTAGE]; int stage, n_stage;
	unsigned *d_sync;            /* [0..7] tickets (0 inter, 1 deblock, 2 intra), [8] err, [16..) flags[nmb] + row progress[3 * h_mbs] */
	size_t sync_words;
	unsigned epoch;
	cudaEvent_t tick_ev[NTICK]; uint64_t tick_seq;
	unsigned *h_err;             /* pinned [NTICK]: the device error word as it stood when ticket t % NTICK completed */
	bool keep; std::vector<KeptPic> kept;
	uint64_t launches, h2d_bytes, d2h_bytes;
	int sm_count;
	std::vector<std::pair<void *, size_t>> host_free_list;   /* pinned buffers returned by the decoder, reused by the next one */
	std::vector<std::pair<void *, size_t>> host_live;        /* pinned buffers handed out, with their sizes */
};

/* Device contexts are pooled per process: creating pinned staging and the frame pool costs tens of
 * milliseconds, a decoder for the next clip of the same geometry reuses everything. */
static std::mutex g_pool_mu;
static std::vector<E264bDevice *> g_pool;

static void free_mirror(void *p) {
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) == cudaSuccess && a.type == cudaMemoryTypeDevice) cudaFree(p); else { cudaGetLastError(); cudaFreeHost(p); }
}
static void free_geometry(E264bDevice *c) {
	cudaStreamSynchronize(c->stream);
	if (c->d_frames) cudaFree(c->d_frames);
	c->d_frames = NULL;
	for (int i = 0; i < E264_MAX_SLOTS; i++) { if (c->h_recs[i]) cudaFreeHost(c->h_recs[i]); c->h_recs[i] = NULL; c->rec_busy[i] = false; }
	for (int i = 0; i < NSTAGE; i++) {
		Staging *s = &c->st[i];
		if (s->d_recs) cudaFree(s->d_recs); if (s->d_coefs) cudaFree(s->d_coefs); if (s->d_slices) cudaFree(s->d_slices);
		if (s->d_dbk) cudaFree(s->d_dbk); if (s->d_intra) cudaFree(s->d_intra); if (s->h_intra) cudaFreeHost(s->h_intra); s->d_dbk = NULL; s->d_intra = NULL; s->h_intra = NULL;
		if (s->h_coefs) cudaFreeHost(s->h_coefs); if (s->h_slices) cudaFreeHost(s->h_slices);
		s->d_recs = NULL; s->d_coefs = NULL; s->d_slices = NULL; s->h_coefs = NULL; s->h_slices = NULL; s->busy = false;
	}
	if (c->d_sync) cudaFree(c->d_sync);
	c->d_sync = NULL;
	for (auto &k : c->kept) { cudaFree(k.d_recs); cudaFree(k.d_coefs); cudaFree(k.d_slices); cudaFree(k.d_intra); }
	c->kept.clear();
}

extern "C" int e264b_create(E264bDevice **out) {
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
		fprintf(stderr, "edge264_b200: no CUDA device — the reconstruction backend has no CPU fallback\n");
		return -1;
	}
	const char *e = getenv("E264B_DEVICE");
	int dev = e ? atoi(e) : 0;
	if (dev < 0 || dev >= n) dev = 0;
	CK(cudaSetDevice(dev));
	{
		std::lock_guard<std::mutex> lk(g_pool_mu);
		for (size_t i = 0; i < g_pool.size(); i++) if (g_pool[i]->dev == dev) {
			E264bDevice *c = g_pool[i]; g_pool.erase(g_pool.begin() + i);
			const char *k = getenv("E264B_KEEP"); c->keep = k && atoi(k) != 0;
			c->launches = c->h2d_bytes = c->d2h_bytes = 0;
			*out = c; return 0;
		}
	}
	E264bDevice *c = new E264bDevice();
	c->dev = 0; c->stream = 0; memset(&c->g, 0, sizeof(c->g)); c->n_slots = 0; c->nmb = 0; c->coef_cap = 0; c->d_frames = NULL;
	memset(c->h_recs, 0, sizeof(c->h_recs)); memset(c->rec_busy, 0, sizeof(c->rec_busy)); memset(c->st, 0, sizeof(c->st)); c->stage = 0; c->d_sync = NULL; c->epoch = 0; c->tick_seq = 0;
	c->launches = c->h2d_bytes = c->d2h_bytes = 0;
	c->dev = dev;
	CK(cudaFuncSetAttribute(e264_intra_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IntraRowsSmem)));
	CK(cudaFuncSetAttribute(e264_inter4_kernel<INTER_MINB0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(InterSmem)));
	CK(cudaFuncSetAttribute(e264_intra_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IntraTkSmem)));
#if INTER_WARPS == 4
	CK(cudaFuncSetAttribute(e264_inter4_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(InterSmem)));
	CK(cudaFuncSetAttribute(e264_inter4_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(InterSmem)));
#endif
	CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
	for (int i = 0; i < E264_MAX_SLOTS; i++) CK(cudaEventCreateWithFlags(&c->rec_up[i], cudaEventDisableTiming | cudaEventBlockingSync));
	for (int i = 0; i < NSTAGE; i++) CK(cudaEventCreateWithFlags(&c->st[i].done, cudaEventDisableTiming | cudaEventBlockingSync));
	for (int i = 0; i < NTICK; i++) CK(cudaEventCreateWithFlags(&c->tick_ev[i], cudaEventDisableTiming | cudaEventBlockingSync));   /* waiting threads sleep: host CPUs are the scarce resource */
	cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, dev);
	c->h_err = NULL; CK(cudaHostAlloc(&c->h_err, NTICK * sizeof(unsigned), cudaHostAllocDefault)); memset(c->h_err, 0, NTICK * sizeof(unsigned));
	const char *k = getenv("E264B_KEEP");
	c->keep = k && atoi(k) != 0;
	*out = c;
	return 0;
}

static void drop_kept(E264bDevice *c) { for (auto &k : c->kept) { cudaFree(k.d_recs); cudaFree(k.d_coefs); cudaFree(k.d_slices); cudaFree(k.d_intra); } c->kept.clear(); }

extern "C" void e264b_destroy(E264bDevice *c) {
	if (!c) return;
	cudaSetDevice(c->dev);
	cudaStreamSynchronize(c->stream);
	drop_kept(c);
	{
		std::lock_guard<std::mutex> lk(g_pool_mu);
		if (g_pool.size() < 256) { g_pool.push_back(c); return; }
	}
	free_geometry(c);
	for (auto &h : c->host_free_list) free_mirror(h.first);
	c->host_free_list.clear();
	for (int i = 0; i < E264_MAX_SLOTS; i++) cudaEventDestroy(c->rec_up[i]);
	for (int i = 0; i < NSTAGE; i++) cudaEventDestroy(c->st[i].done);
	for (int i = 0; i < NTICK; i++) cudaEventDestroy(c->tick_ev[i]);
	if (c->h_err) cudaFreeHost(c->h_err);
	cudaStreamDestroy(c->stream);
	delete c;
}


extern "C" int e264b_configure(E264bDevice *c, const E264PicDesc *g, int n_slots) {
	CK(cudaSetDevice(c->dev));
	if (c->d_frames && c->n_slots == n_slots && !memcmp(&c->g, g, sizeof(*g))) {   /* pooled context of the same geometry */
		CK(cudaStreamSynchronize(c->stream));
		drop_kept(c);
		CK(cudaMemsetAsync(c->d_sync, 0, c->sync_words * sizeof(unsigned), c->stream));
		for (int i = 0; i < NSTAGE; i++) c->st[i].busy = false;
		for (int i = 0; i < E264_MAX_SLOTS; i++) c->rec_busy[i] = false;
		c->epoch = 0; c->stage = 0;
		return 0;
	}
	free_geometry(c);
	for (auto &h : c->host_free_list) free_mirror(h.first);
	c->host_free_list.clear();
	c->g = *g; c->n_slots = n_slots; c->nmb = (size_t)g->width_mbs * g->height_mbs;
	c->n_stage = g->staging > 0 ? (g->staging < NSTAGE ? g->staging : NSTAGE) : 4;   /* 4 for a synchronous parser; more when pictures are parsed ahead */
	c->coef_cap = (uint32_t)(c->nmb * 408);
	size_t pool = (size_t)g->frame_bytes * n_slots;
	CK(cudaMalloc(&c->d_frames, pool + 256));
	CK(cudaMemsetAsync(c->d_frames, 128, pool + 256, c->stream));
	for (int i = 0; i < n_slots; i++) CK(cudaHostAlloc(&c->h_recs[i], c->nmb * sizeof(E264MbRec), cudaHostAllocDefault));
	for (int i = 0; i < c->n_stage; i++) {
		Staging *s = &c->st[i];
		CK(cudaMalloc(&s->d_recs, c->nmb * sizeof(E264MbRec)));
		CK(cudaMalloc(&s->d_coefs, (size_t)c->coef_cap * 2 + 64));
		CK(cudaMalloc(&s->d_slices, E264_MAX_SLICES * sizeof(E264SliceRec)));
		CK(cudaHostAlloc(&s->h_coefs, (size_t)c->coef_cap * 2 + 64, cudaHostAllocDefault));
		CK(cudaHostAlloc(&s->h_slices, E264_MAX_SLICES * sizeof(E264SliceRec), cudaHostAllocDefault));
		CK(cudaMalloc(&s->d_dbk, c->nmb * sizeof(E264DbkMb)));
		CK(cudaMalloc(&s->d_intra, c->nmb * sizeof(uint32_t)));
		CK(cudaHostAlloc(&s->h_intra, c->nmb * sizeof(uint32_t), cudaHostAllocDefault));
	}
	c->sync_words = 16 + c->nmb + 3 * (size_t)g->height_mbs + 16;
	CK(cudaMalloc(&c->d_sync, c->sync_words * sizeof(unsigned)));
	CK(cudaMemsetAsync(c->d_sync, 0, c->sync_words * sizeof(unsigned), c->stream));
	c->epoch = 0; c->stage = 0;
	CK(cudaStreamSynchronize(c->stream));
	return 0;
}

extern "C" void *e264b_host_alloc(E264bDevice *c, size_t bytes) {
	void *p = NULL;
	cudaSetDevice(c->dev);
	for (size_t i = 0; i < c->host_free_list.size(); i++) if (c->host_free_list[i].second == bytes) {
		p = c->host_free_list[i].first; c->host_free_list.erase(c->host_free_list.begin() + i);
		c->host_live.push_back(std::make_pair(p, bytes));
		return p;
	}
	static int dev_out = -1;
	if (dev_out < 0) { const char *e = getenv("E264B_OUTPUT"); dev_out = e && !strcmp(e, "device"); }
	if ((dev_out ? cudaMalloc(&p, bytes) : cudaHostAlloc(&p, bytes, cudaHostAllocDefault)) != cudaSuccess) return NULL;
	c->host_live.push_back(std::make_pair(p, bytes));
	return p;
}
extern "C" void e264b_host_free(E264bDevice *c, void *p) {
	/* decoder mirrors of one geometry have the same size: keep them (with the size they were allocated with) for the next decoder */
	for (size_t i = 0; i < c->host_live.size(); i++) if (c->host_live[i].first == p) {
		c->host_free_list.push_back(c->host_live[i]);
		c->host_live.erase(c->host_live.begin() + i);
		return;
	}
	cudaSetDevice(c->dev); free_mirror(p);   /* not ours to pool */
}

extern "C" int e264b_acquire_staging(E264bDevice *c, int slot, E264Staging *out) {
	CK(cudaSetDevice(c->dev));
	c->stage = (c->stage + 1) % c->n_stage;
	Staging *s = &c->st[c->stage];
	if (s->busy) { CK(cudaEventSynchronize(s->done)); s->busy = false; }
	if (c->rec_busy[slot]) { CK(cudaEventSynchronize(c->rec_up[slot])); c->rec_busy[slot] = false; }
	out->handle = c->stage; out->recs = c->h_recs[slot]; out->coefs = s->h_coefs; out->coef_capacity = c->coef_cap; out->slices = s->h_slices; out->intra_list = s->h_intra;
	return 0;
}

static PicJob make_job(E264bDevice *c, const E264PicDesc *pd, int stage, const E264MbRec *recs, const int16_t *coefs, const E264SliceRec *slices, const uint32_t *intra) {
	PicJob J;
	J.recs = recs; J.coefs = coefs; J.slices = slices; J.frames = c->d_frames;
	J.frame_bytes = pd->frame_bytes; J.w_mbs = pd->width_mbs; J.h_mbs = pd->height_mbs;
	J.stride_y = pd->stride_y; J.stride_c = pd->stride_c; J.plane_y = pd->plane_y; J.dst_slot = pd->dst_slot; J.n_slots = c->n_slots;
	J.err = c->d_sync + 8; J.flags = c->d_sync + 16;
	J.dbk = pd->any_deblock ? c->st[stage].d_dbk : NULL;
	J.intra_list = intra; J.n_intra = pd->n_intra;
	J.rows_mode = pd->n_intra * 2 > pd->width_mbs * pd->height_mbs;   /* intra pictures: wavefront of row warps */
	J.trace = NULL; J.trace_base = 0; J.trace_rep = NULL; J.trace_rep_stride = 0; J.diag = 0;
	if (c->epoch >= (1u << 20)) {   /* row progress counters encode epoch * 2048 + count: restart before it wraps */
		cudaStreamSynchronize(c->stream);
		cudaMemsetAsync(c->d_sync, 0, c->sync_words * sizeof(unsigned), c->stream);
		c->epoch = 0;
	}
	J.epoch = ++c->epoch;
	J.tickets = c->d_sync + (J.epoch & 1) * 4; J.tickets_next = c->d_sync + ((J.epoch + 1) & 1) * 4;    /* two sets, pictures alternate; every kernel clears the next picture's */
	return J;
}
static int launch_picture(E264bDevice *c, const PicJob &J, const E264PicDesc *pd, int with_deblock) {
	const int nmb = J.w_mbs * J.h_mbs;
	const int cap = c->sm_count * 8;
	static int minb = -1, dm = -1;
	if (minb < 0) { const char *e = getenv("E264B_MINB"); minb = e ? atoi(e) : 4; }
	if (dm < 0) { const char *e = getenv("E264B_DBK_MINB"); dm = e ? atoi(e) : 2; }
	/* experiments (replay only): E264B_REPLAY_ONLY = mask of kernel kinds to launch (1 inter, 2 intra, 4 deblocking; J.trace
	 * marks a replay), E264B_DBK_SMEM = extra dynamic shared memory of the deblocking blocks (limits blocks per SM) */
	static int only = -1, dbk_smem = -1;
	if (only < 0) { const char *e = getenv("E264B_REPLAY_ONLY"); only = e && atoi(e) > 0 ? atoi(e) : 7; }
	if (dbk_smem < 0) {
		const char *e = getenv("E264B_DBK_SMEM"); dbk_smem = e ? atoi(e) : 0;
		if (dbk_smem > 0) { cudaFuncSetAttribute(e264_deblock_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, dbk_smem); cudaFuncSetAttribute(e264_deblock_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, dbk_smem); cudaFuncSetAttribute(e264_deblock_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, dbk_smem); }
	}
	const int mask = J.trace ? only : 7;
	/* up to three launches per picture, nothing in between: inter macroblocks (inverse transform + prediction), intra
	 * macroblocks (flags order them behind their neighbours), deblocking (its blocks derive the boundary strengths first) */
	if (pd->n_intra < nmb && (mask & 1)) {
		int ib = (nmb + INTER_CHUNK - 1) / INTER_CHUNK;
		if (ib > cap) ib = cap;
#if INTER_WARPS == 4
		if (minb >= 8) e264_inter4_kernel<8><<<ib, INTER_WARPS * 32, sizeof(InterSmem), c->stream>>>(J);
		else if (minb >= 6) e264_inter4_kernel<6><<<ib, INTER_WARPS * 32, sizeof(InterSmem), c->stream>>>(J);
		else
#endif
		e264_inter4_kernel<INTER_MINB0><<<ib, INTER_WARPS * 32, sizeof(InterSmem), c->stream>>>(J);
		c->launches++;
	}
	if (pd->n_intra > 0 && (mask & 2)) {
		if (J.rows_mode) {   /* intra pictures: bands of rows, hand-over through shared memory */
			e264_intra_rows_kernel<<<(J.h_mbs + IR_ROWS - 1) / IR_ROWS, IR_ROWS * 64, sizeof(IntraRowsSmem), c->stream>>>(J);
		} else {
			/* a warp takes several list entries (E264B_INTRA_DIV, default 2): see INTRA_WARPS */
			static int idiv = -1;
			if (idiv < 0) { const char *e = getenv("E264B_INTRA_DIV"); idiv = e && atoi(e) > 0 ? atoi(e) : 2; }
			int ib = (pd->n_intra + INTRA_WARPS * idiv - 1) / (INTRA_WARPS * idiv);
			if (ib > cap) ib = cap;
			e264_intra_kernel<<<ib, INTRA_WARPS * 32, sizeof(IntraTkSmem), c->stream>>>(J);
		}
		c->launches++;
	}
	if (with_deblock && (mask & 4)) {      /* one block per band of 16 rows and kind of plane */
		const int bands = (J.h_mbs + 2 * DBK_PAIRS - 1) / (2 * DBK_PAIRS);
		if (dm >= 5) e264_deblock_kernel<5><<<2 * bands, DBK_PAIRS * 32, dbk_smem, c->stream>>>(J);
		else if (dm == 4) e264_deblock_kernel<4><<<2 * bands, DBK_PAIRS * 32, dbk_smem, c->stream>>>(J);
		else e264_deblock_kernel<2><<<2 * bands, DBK_PAIRS * 32, dbk_smem, c->stream>>>(J);
		c->launches++;
	}
	CK(cudaGetLastError());
	return 0;
}

extern "C" int e264b_submit(E264bDevice *c, const E264PicDesc *pd, uint8_t *host_out, uint64_t *ticket) {
	CK(cudaSetDevice(c->dev));
	if (pd->staging < 0 || pd->staging >= c->n_stage) return -1;
	Staging *s = &c->st[pd->staging];
	size_t rec_bytes = c->nmb * sizeof(E264MbRec), coef_bytes = ((size_t)pd->n_coefs * 2 + 15) & ~(size_t)15, sl_bytes = (size_t)pd->n_slices * sizeof(E264SliceRec);
	CK(cudaMemcpyAsync(s->d_recs, c->h_recs[pd->dst_slot], rec_bytes, cudaMemcpyHostToDevice, c->stream));
	CK(cudaEventRecord(c->rec_up[pd->dst_slot], c->stream)); c->rec_busy[pd->dst_slot] = true;
	if (coef_bytes) CK(cudaMemcpyAsync(s->d_coefs, s->h_coefs, coef_bytes, cudaMemcpyHostToDevice, c->stream));
	if (sl_bytes) CK(cudaMemcpyAsync(s->d_slices, s->h_slices, sl_bytes, cudaMemcpyHostToDevice, c->stream));
	size_t in_bytes = (size_t)pd->n_intra * sizeof(uint32_t);
	if (in_bytes) CK(cudaMemcpyAsync(s->d_intra, s->h_intra, in_bytes, cudaMemcpyHostToDevice, c->stream));
	c->h2d_bytes += rec_bytes + coef_bytes + sl_bytes + in_bytes;
	PicJob J = make_job(c, pd, pd->staging, s->d_recs, s->d_coefs, s->d_slices, s->d_intra);
	if (launch_picture(c, J, pd, pd->any_deblock)) return -1;
	{	/* E264B_DEBUG_SYNC=1: synchronise after every picture and report the device error word (debugging aid) */
		static int dbg = -1; if (dbg < 0) { const char *e = getenv("E264B_DEBUG_SYNC"); dbg = e ? atoi(e) : 0; }
		if (dbg) {
			fprintf(stderr, "e264b: picture slot %d epoch %u (intra %d of %d, coefs %u) launched, waiting...\n", pd->dst_slot, J.epoch, pd->n_intra, J.w_mbs * J.h_mbs, pd->n_coefs);
			cudaError_t e = cudaStreamSynchronize(c->stream); unsigned v = 0; cudaMemcpy(&v, c->d_sync + 8, sizeof(v), cudaMemcpyDeviceToHost);
			fprintf(stderr, "e264b:   -> %s, device error word %u\n", cudaGetErrorString(e), v);
		}
	}
	/* the output mirror: pinned host memory by default (D2H copy); memory the application's alloc_cb handed out may as well
	 * be DEVICE memory — unified addressing picks the direction, the frame then reaches the application as device pointers
	 * without ever crossing PCIe (zero-copy output, SURVEY section 8 f2); E264B_OUTPUT=device makes the decoder's own mirrors device memory */
	if (host_out) { CK(cudaMemcpyAsync(host_out, c->d_frames + (size_t)pd->dst_slot * pd->frame_bytes, (size_t)pd->frame_bytes - 16, cudaMemcpyDefault, c->stream)); c->d2h_bytes += (size_t)pd->frame_bytes - 16; }
	if (c->keep) {
		KeptPic k; k.pd = *pd;
		CK(cudaMalloc(&k.d_recs, rec_bytes)); CK(cudaMalloc(&k.d_coefs, coef_bytes + 64)); CK(cudaMalloc(&k.d_slices, sl_bytes + 64)); CK(cudaMalloc(&k.d_intra, in_bytes + 64));
		if (in_bytes) CK(cudaMemcpyAsync(k.d_intra, s->d_intra, in_bytes, cudaMemcpyDeviceToDevice, c->stream));
		CK(cudaMemcpyAsync(k.d_recs, s->d_recs, rec_bytes, cudaMemcpyDeviceToDevice, c->stream));
		if (coef_bytes) CK(cudaMemcpyAsync(k.d_coefs, s->d_coefs, coef_bytes, cudaMemcpyDeviceToDevice, c->stream));
		if (sl_bytes) CK(cudaMemcpyAsync(k.d_slices, s->d_slices, sl_bytes, cudaMemcpyDeviceToDevice, c->stream));
		c->kept.push_back(k);
	}
	CK(cudaEventRecord(s->done, c->stream)); s->busy = true;
	uint64_t t = ++c->tick_seq;
	if (c->d_sync) CK(cudaMemcpyAsync(&c->h_err[t % NTICK], c->d_sync + 8, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
	CK(cudaEventRecord(c->tick_ev[t % NTICK], c->stream));
	*ticket = t;
	return 0;
}

static_assert(sizeof(IntraRowsSmem) <= 227 * 1024 && sizeof(InterSmem) <= 227 * 1024, "dynamic shared memory of a block");
extern "C" int e264b_wait(E264bDevice *c, uint64_t ticket) {
	if (ticket == 0) return 0;
	/* the ring slot holds this ticket or a later one of the same stream: either way it implies completion */
	CK(cudaSetDevice(c->dev));
	CK(cudaEventSynchronize(c->tick_ev[ticket % NTICK]));
	if (c->h_err[ticket % NTICK]) {   /* a kernel gave up on a dependency or a TMA transfer: the picture is not trustworthy */
		fprintf(stderr, "edge264_b200: the device raised error word %u while reconstructing (ticket %llu)\n", c->h_err[ticket % NTICK], (unsigned long long)ticket);
		return -1;
	}
	return 0;
}

/* non-blocking: 0 = complete, EAGAIN = the picture (or a later one that took its ring slot) is still on the device */
extern "C" int e264b_poll(E264bDevice *c, uint64_t ticket) {
	if (ticket == 0) return 0;
	CK(cudaSetDevice(c->dev));
	cudaError_t q = cudaEventQuery(c->tick_ev[ticket % NTICK]);
	if (q == cudaErrorNotReady) return EAGAIN;
	if (q != cudaSuccess) { fprintf(stderr, "edge264_b200: cudaEventQuery: %s\n", cudaGetErrorString(q)); return -1; }
	return c->h_err[ticket % NTICK] ? -1 : 0;
}

extern "C" int e264b_fill_slot(E264bDevice *c, int slot, int y, int cc) {
	CK(cudaSetDevice(c->dev));
	uint8_t *f = c->d_frames + (size_t)slot * c->g.frame_bytes;
	CK(cudaMemsetAsync(f, y, (size_t)c->g.plane_y, c->stream));
	CK(cudaMemsetAsync(f + c->g.plane_y, cc, (size_t)c->g.frame_bytes - c->g.plane_y, c->stream));
	return 0;
}

extern "C" int e264b_error_flag(E264bDevice *c) {
	unsigned v = 0;
	cudaSetDevice(c->dev);
	cudaStreamSynchronize(c->stream);
	cudaMemcpy(&v, c->d_sync + 8, sizeof(v), cudaMemcpyDeviceToHost);
	return (int)v;
}
extern "C" void e264b_stats(E264bDevice *c, uint64_t *launches, uint64_t *h2d, uint64_t *d2h) { if (launches) *launches = c->launches; if (h2d) *h2d = c->h2d_bytes; if (d2h) *d2h = c->d2h_bytes; }
extern "C" int e264b_kept_count(E264bDevice *c) { return (int)c->kept.size(); }

/* algorithmic bytes of the kept pictures per SURVEY.md §8(d): Rec + 384*(1+L) + 768*D per macroblock */
extern "C" double e264b_kept_algorithmic_bytes(E264bDevice *c, double *recon_bytes, double *deblock_bytes, uint64_t *mbs) {
	cudaSetDevice(c->dev); cudaStreamSynchronize(c->stream);
	double rec = 0, db = 0; uint64_t n = 0;
	std::vector<E264MbRec> h(c->nmb);
	for (auto &k : c->kept) {
		cudaMemcpy(h.data(), k.d_recs, c->nmb * sizeof(E264MbRec), cudaMemcpyDeviceToHost);
		rec += (double)k.pd.n_coefs * 2 + (double)c->nmb * sizeof(E264MbRec);
		for (size_t i = 0; i < c->nmb; i++) {
			int L = 0;
			if (h[i].kind == MBK_INTER) { int l0 = 0, l1 = 0; for (int j = 0; j < 4; j++) { l0 |= h[i].ref_idx[0][j] >= 0; l1 |= h[i].ref_idx[1][j] >= 0; } L = l0 + l1; }
			rec += 384.0 * (1 + L);
			if (h[i].flags & MBF_DEBLOCK) db += 768.0;
		}
		n += c->nmb;
	}
	if (recon_bytes) *recon_bytes = rec; if (deblock_bytes) *deblock_bytes = db; if (mbs) *mbs = n;
	return rec + db;
}

/* Replay the kept pictures of several decoders concurrently (one CUDA stream each), `reps` times, and return the
 * elapsed device time between a start event and the last stream's end.  `threads` host threads issue the launches
 * (each owns a share of the streams): one thread alone tops out near 40-50 thousand launches per second and would
 * make the result a CPU number.  Every kernel stamps its first block's start and last block's end (%globaltimer)
 * into a trace array during the timed pass; stats->kernel_ms[k] is the sum over launches of that span per kernel
 * kind (1 inter, 2 intra, 3 deblock; 0 and 4 unused since the inverse transform and the boundary-strength pass were folded into them) — spans of concurrent launches overlap, so their sum may
 * exceed the elapsed time.  E264B_TRACE=<file> also dumps the spans. */
#include <thread>
__global__ void e264_replay_rep_kernel(unsigned *rep) { if (threadIdx.x == 0) *rep += 1; }
extern "C" int e264b_replay(E264bDevice **cs, int n, int reps, int threads, E264bReplayStats *stats) {
	if (n <= 0 || !stats) return -1;
	memset(stats, 0, sizeof(*stats));
	CK(cudaSetDevice(cs[0]->dev));
	cudaEvent_t start, stop; std::vector<cudaEvent_t> ends(n);
	CK(cudaEventCreate(&start)); CK(cudaEventCreate(&stop));
	for (int i = 0; i < n; i++) { CK(cudaEventCreateWithFlags(&ends[i], cudaEventDisableTiming)); CK(cudaStreamSynchronize(cs[i]->stream)); }
	size_t npic = cs[0]->kept.size();
	for (int i = 1; i < n; i++) if (cs[i]->kept.size() < npic) npic = cs[i]->kept.size();
	uint64_t l0 = 0; for (int i = 0; i < n; i++) l0 += cs[i]->launches;
	const int NK = 5;
	size_t n_trace = (size_t)reps * npic * n * NK;
	unsigned long long *d_trace = NULL;
	{
		std::vector<unsigned long long> init(n_trace * 2);
		for (size_t i = 0; i < n_trace; i++) { init[2 * i] = ~0ull; init[2 * i + 1] = 0; }
		CK(cudaMalloc(&d_trace, n_trace * 16 + 128)); CK(cudaMemcpy(d_trace, init.data(), n_trace * 16, cudaMemcpyHostToDevice)); CK(cudaMemset(d_trace + n_trace * 2, 0, 128));
	}
	if (threads < 1) threads = 1;
	if (threads > n) threads = n;
	/* Default: every stream's pictures of one repetition are captured into ONE CUDA graph (its kernels stay the same
	 * launches, in the same order, on the same stream) and a repetition is one graph launch per stream — the issue rate
	 * of individual launches (tens of thousands per second for the whole process, less with several threads contending
	 * for the driver) would otherwise bound the result.  The synchronisation words restart at every repetition
	 * (two memset nodes) because the captured epochs repeat.  E264B_REPLAY_GRAPH=0 issues plain launches instead. */
	const int diag = getenv("E264B_DIAG") && atoi(getenv("E264B_DIAG")) ? 1 : 0;
	if (diag) { static unsigned long long zp[16]; cudaMemcpyToSymbol(g_diag_phase, zp, sizeof zp); }
	if (diag) { static unsigned z[3][4][160]; cudaMemcpyToSymbol(g_diag_cnt, z[0], sizeof z[0]); cudaMemcpyToSymbol(g_diag_cur, z[1], sizeof z[1]); cudaMemcpyToSymbol(g_diag_max, z[2], sizeof z[2]); }
	const char *ge = getenv("E264B_REPLAY_GRAPH");
	const bool use_graph = !(ge && atoi(ge) == 0);
	std::vector<cudaGraphExec_t> execs(n, nullptr);
	unsigned *d_rep = NULL;
	uint64_t per_rep_launches = 0;
	if (use_graph) {
		CK(cudaMalloc(&d_rep, n * sizeof(unsigned))); CK(cudaMemset(d_rep, 0, n * sizeof(unsigned)));
		for (int i = 0; i < n; i++) {
			E264bDevice *c = cs[i];
			c->epoch = 0;
			const uint64_t lbefore = c->launches;
			cudaGraph_t g = nullptr;
			CK(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeRelaxed));
			CK(cudaMemsetAsync(c->d_sync, 0, 8 * sizeof(unsigned), c->stream));
			CK(cudaMemsetAsync(c->d_sync + 16, 0, (c->sync_words - 16) * sizeof(unsigned), c->stream));
			int bad = 0;
			for (size_t k = 0; k < npic && !bad; k++) {
				KeptPic &kp = c->kept[k];
				PicJob J = make_job(c, &kp.pd, kp.pd.staging, kp.d_recs, kp.d_coefs, kp.d_slices, kp.d_intra);
				J.trace = d_trace; J.trace_base = (int)((k * n + i) * NK); J.trace_rep = d_rep + i; J.trace_rep_stride = (int)(npic * n * NK); J.diag = diag;
				bad = launch_picture(c, J, &kp.pd, kp.pd.any_deblock);
			}
			e264_replay_rep_kernel<<<1, 32, 0, c->stream>>>(d_rep + i);
			cudaError_t ce = cudaStreamEndCapture(c->stream, &g);
			if (bad || ce != cudaSuccess) { fprintf(stderr, "edge264_b200: replay graph capture failed: %s\n", cudaGetErrorString(ce)); return -1; }
			CK(cudaGraphInstantiate(&execs[i], g, 0));
			CK(cudaGraphDestroy(g));
			CK(cudaGraphUpload(execs[i], c->stream));
			per_rep_launches += c->launches - lbefore;
			c->launches += (c->launches - lbefore) * (uint64_t)(reps - 1);
		}
		for (int i = 0; i < n; i++) CK(cudaStreamSynchronize(cs[i]->stream));
	}
	CK(cudaEventRecord(start, cs[0]->stream));
	for (int i = 1; i < n; i++) CK(cudaStreamWaitEvent(cs[i]->stream, start, 0));
	std::vector<int> rc(threads, 0);
	if (use_graph) {
		/* at most `inflight` streams have pictures on the GPU at a time (stream i starts a repetition when stream
		 * i - inflight has finished its own).  With 4-warp inter blocks more than 12-16 streams in flight only took each
		 * other's instruction cache; with the 16-warp blocks the curve is flat from 16 on (16: 17.9 k, 24: 17.8 k, 32: 18.9 k
		 * frames/s, profiles/r2_inflight.txt), so the default is the bench's batch */
		const char *fe = getenv("E264B_REPLAY_INFLIGHT");
		const int inflight = fe && atoi(fe) > 0 ? atoi(fe) : 32;
		std::vector<cudaEvent_t> done(n);
		for (int i = 0; i < n; i++) CK(cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming));
		for (int r = 0; r < reps; r++) for (int i = 0; i < n; i++) {
			if (i >= inflight) CK(cudaStreamWaitEvent(cs[i]->stream, done[i - inflight], 0));
			CK(cudaGraphLaunch(execs[i], cs[i]->stream));
			CK(cudaEventRecord(done[i], cs[i]->stream));
		}
		for (int i = 0; i < n; i++) cudaEventDestroy(done[i]);
		threads = 0;
		stats->inflight = inflight < n ? inflight : n;
	}
	auto issue = [&](int t) {
		cudaSetDevice(cs[0]->dev);
		for (int r = 0; r < reps; r++)
			for (size_t k = 0; k < npic; k++)
				for (int i = t; i < n; i += threads) {
					KeptPic &kp = cs[i]->kept[k];
					PicJob J = make_job(cs[i], &kp.pd, kp.pd.staging, kp.d_recs, kp.d_coefs, kp.d_slices, kp.d_intra);
					J.trace = d_trace; J.trace_base = (int)((((size_t)r * npic + k) * n + i) * NK);
					if (launch_picture(cs[i], J, &kp.pd, kp.pd.any_deblock)) { rc[t] = -1; return; }
				}
	};
	if (threads == 0) {}
	else if (threads == 1) issue(0);
	else { std::vector<std::thread> th; for (int t = 0; t < threads; t++) th.emplace_back(issue, t); for (auto &x : th) x.join(); }
	for (int t = 0; t < threads; t++) if (rc[t]) return -1;
	for (int i = 1; i < n; i++) { CK(cudaEventRecord(ends[i], cs[i]->stream)); CK(cudaStreamWaitEvent(cs[0]->stream, ends[i], 0)); }
	CK(cudaEventRecord(stop, cs[0]->stream));
	CK(cudaEventSynchronize(stop));
	CK(cudaEventElapsedTime(&stats->ms_total, start, stop));
	{ uint64_t l1 = 0; for (int i = 0; i < n; i++) l1 += cs[i]->launches; stats->launches = l1 - l0; }
	stats->threads = threads;      /* 0: graph replay */
	for (int i = 0; i < n; i++) if (execs[i]) cudaGraphExecDestroy(execs[i]);
	if (d_rep) cudaFree(d_rep);
	if (use_graph) for (int i = 0; i < n; i++) { cs[i]->epoch = (unsigned)npic; }     /* the words hold the last repetition's epochs */
	std::vector<unsigned long long> h(n_trace * 2 + 16);
	CK(cudaMemcpy(h.data(), d_trace, n_trace * 16 + 128, cudaMemcpyDeviceToHost)); cudaFree(d_trace);
	for (size_t j = 0; j < n_trace; j++) if (h[2 * j + 1] && h[2 * j] != ~0ull) { stats->kernel_ms[j % NK] += 1e-6 * (double)(h[2 * j + 1] - h[2 * j]); stats->kernel_launches[j % NK]++; }
	if (diag) {     /* block placement: per kernel kind, how many SMs saw blocks, the spread of blocks per SM, the most blocks resident at once */
		static unsigned cnt[4][160], mx[4][160];
		cudaMemcpyFromSymbol(cnt, g_diag_cnt, sizeof cnt); cudaMemcpyFromSymbol(mx, g_diag_max, sizeof mx);
		for (int k = 1; k < 4; k++) {
			unsigned used = 0, lo = ~0u, hi = 0, m = 0; unsigned long long tot = 0; unsigned hist[9] = {0};
			for (int s_ = 0; s_ < 160; s_++) if (cnt[k][s_]) { used++; tot += cnt[k][s_]; lo = cnt[k][s_] < lo ? cnt[k][s_] : lo; hi = cnt[k][s_] > hi ? cnt[k][s_] : hi; m = mx[k][s_] > m ? mx[k][s_] : m; hist[mx[k][s_] > 8 ? 8 : mx[k][s_]]++; }
			fprintf(stderr, "diag kind %d: %llu blocks on %u SMs (per SM min %u max %u), max resident on one SM %u; SMs by max resident 1..8+:", k, tot, used, used ? lo : 0, hi, m);
			for (int j = 1; j < 9; j++) fprintf(stderr, " %u", hist[j]);
			fprintf(stderr, "\n");
		}
	}
#ifdef E264_INTER_TIMING
	if (diag) {     /* -DE264_INTER_TIMING builds: cycles per part of a chunk in the inter kernel, all warps summed */
		unsigned long long ph[16]; cudaMemcpyFromSymbol(ph, g_diag_phase, sizeof ph);
		unsigned long long tt = 0; for (int k = 0; k < 5; k++) tt += ph[k];
		const double pics = (double)reps * (double)npic * n;
		const char *in[5] = {"records+binning", "interpolation", "digest", "residual", "combine+store"};
		fprintf(stderr, "inter kernel, all warps, %.0f pictures: %.3f Mcycles per picture:", pics, tt / pics * 1e-6);
		for (int k = 0; k < 5; k++) fprintf(stderr, " %s %.3f (%.1f%%)", in[k], ph[k] / pics * 1e-6, 100.0 * ph[k] / (double)(tt ? tt : 1));
		fprintf(stderr, "\n");
	}
#endif
#ifdef E264_ROWS_TIMING
	if (diag) {     /* -DE264_ROWS_TIMING builds: cycles per part of a macroblock step in the intra-picture kernel, all warps summed */
		unsigned long long ph[16]; cudaMemcpyFromSymbol(ph, g_diag_phase, sizeof ph);
		unsigned long long tt = 0, tp = 0; for (int k = 0; k < 8; k++) { tt += ph[k]; tp += ph[8 + k]; }
		if (tt + tp) {
			const char *tn[8] = {"wait slot", "records+issue", "wait coefficients", "transforms", "digest", "-", "-", "-"};
			const char *pn[8] = {"wait residual", "wait row above", "ring+hand-shake+tile", "luma", "chroma", "stores", "publish+column", "-"};
			fprintf(stderr, "rows kernel, transform warps:"); for (int k = 0; k < 5; k++) fprintf(stderr, " %s %.1f%%", tn[k], 100.0 * ph[k] / (double)tt); fprintf(stderr, "\n");
			fprintf(stderr, "rows kernel, prediction warps:"); for (int k = 0; k < 7; k++) fprintf(stderr, " %s %.1f%%", pn[k], 100.0 * ph[8 + k] / (double)tp); fprintf(stderr, "\n");
		}
	}
#endif
	const char *trace_path = getenv("E264B_TRACE");
	if (trace_path) {
		FILE *f = fopen(trace_path, "w");
		if (f) {
			fprintf(f, "rep,pic,stream,kind,start_ns,end_ns\n");
			for (size_t j = 0; j < n_trace; j++) if (h[2 * j + 1]) fprintf(f, "%zu,%zu,%zu,%zu,%llu,%llu\n", j / NK / n / npic, j / NK / n % npic, j / NK % n, j % NK, h[2 * j], h[2 * j + 1]);
			fclose(f);
		}
	}
	cudaEventDestroy(start); cudaEventDestroy(stop); for (int i = 0; i < n; i++) cudaEventDestroy(ends[i]);
	return 0;
}

/* checksum of a frame slot (FNV-1a over the whole slot), for replay-vs-decode comparisons */
extern "C" uint64_t e264b_slot_hash(E264bDevice *c, int slot) {
	cudaSetDevice(c->dev); cudaStreamSynchronize(c->stream);
	std::vector<uint8_t> h((size_t)c->g.frame_bytes);
	cudaMemcpy(h.data(), c->d_frames + (size_t)slot * c->g.frame_bytes, h.size(), cudaMemcpyDeviceToHost);
	uint64_t x = 0xcbf29ce484222325ull;
	for (size_t i = 0; i + 16 < h.size(); i++) x = (x ^ h[i]) * 0x100000001b3ull;
	return x;
}

/* ---- known-answer entry point (tests/test_kat.py -m gpu): the reference's own KAT inputs through the DEVICE functions ----
 * fn 0 intra4x4, 1 intra8x8, 2 intra16x16, 3 chroma: `in` is the 32-byte-stride border buffer of edge264_check.c:173-180
 * (sample (0,0) at in + 80), mode = prediction mode | unavailable bits << 4; the block is predicted into the same layout.
 * fn 4 inter luma: `in` is the 21x21 source of edge264_check.c:286-290, mode = xFrac | yFrac << 2, w x h output samples. */
__global__ void e264_kat_kernel(int fn, int imode, const uint8_t *in, uint8_t *out, int w, int h) {
	__shared__ WarpSmem wsm;
	__shared__ E264MbRec rec;
	WarpSmem *ws = &wsm;
	const int lane = threadIdx.x;
	if (fn == 4) {
		const int fx = imode & 3, fy = (imode >> 2) & 3, bw = w >> 2, nb = bw * (h >> 2);
		if (lane < nb) {
			const int bx = lane % bw, by = lane / bw;
			uint32_t win[9][3], o[4];
#pragma unroll
			for (int r = 0; r < 9; r++) {
				uint32_t v[3] = {0, 0, 0};
#pragma unroll
				for (int k = 0; k < 9; k++) v[k >> 2] |= (uint32_t)in[(by * 4 + r) * 21 + bx * 4 + k] << (8 * (k & 3));      /* block origin (2,2): window from (0,0) */
				win[r][0] = v[0]; win[r][1] = v[1]; win[r][2] = v[2];
			}
			mc_luma4x4(win, fx, fy, o);
			for (int y = 0; y < 4; y++) for (int x = 0; x < 4; x++) out[(by * 4 + y) * w + bx * 4 + x] = (uint8_t)(o[y] >> (8 * x));
		}
		return;
	}
	const uint8_t *p = in + 80;
	for (int i = lane; i < 384; i += 32) ws->res[i] = 0;
	if (lane == 0) { memset(&rec, 0, sizeof(rec)); rec.kind = fn == 0 ? MBK_I4x4 : fn == 1 ? MBK_I8x8 : MBK_I16x16; for (int b = 0; b < 16; b++) rec.modes[b] = IMODE(2, 0); rec.modes[0] = (uint8_t)imode; rec.i16_mode = (uint8_t)imode; rec.chroma_mode = (uint8_t)imode; }
	__syncwarp();
	if (fn < 3) {
		for (int x = lane - 1; x < 24; x += 32) YT(x, -1) = x < 16 ? p[x - 32] : p[15 - 32];
		if (lane < 16) YT(-1, lane) = p[lane * 32 - 1];
		__syncwarp();
		intra_luma(ws, &rec, lane);
		__syncwarp();
		for (int i = lane; i < w * h; i += 32) out[i] = YT(i % w, i / w);
	} else {   /* Cb = even rows, Cr = odd rows of the reference's interleaved chroma plane */
		if (lane < 18) { const int pl = lane / 9, x = lane % 9 - 1; CT(pl, x, -1) = p[x + (pl ? -32 : -64)]; }
		if (lane < 16) { const int pl = lane >> 3, y = lane & 7; CT(pl, -1, y) = p[(2 * y + pl) * 32 - 1]; }
		__syncwarp();
		intra_chroma(ws, &rec, lane);
		__syncwarp();
		for (int i = lane; i < 128; i += 32) { const int row = i >> 3, x = i & 7; out[i] = CT(row & 1, x, row >> 1); }
	}
}
extern "C" int e264b_kat(int fn, int mode, const uint8_t *in, int in_bytes, uint8_t *out, int w, int h) {
	uint8_t *d_in = NULL, *d_out = NULL;
	CK(cudaMalloc(&d_in, in_bytes + 64)); CK(cudaMalloc(&d_out, 1024));
	CK(cudaMemset(d_in, 0, in_bytes + 64)); CK(cudaMemcpy(d_in, in, in_bytes, cudaMemcpyHostToDevice)); CK(cudaMemset(d_out, 0, 1024));
	e264_kat_kernel<<<1, 32>>>(fn, mode, d_in, d_out, w, h);
	CK(cudaGetLastError()); CK(cudaDeviceSynchronize());
	CK(cudaMemcpy(out, d_out, (size_t)w * h, cudaMemcpyDeviceToHost));
	cudaFree(d_in); cudaFree(d_out);
	return 0;
}

/* ---- backend vtable for decoder.c ---- */
static int be_create(void **ctx) { return e264b_create((E264bDevice **)ctx); }
static void be_destroy(void *ctx) { e264b_destroy((E264bDevice *)ctx); }
static int be_configure(void *ctx, const E264PicDesc *g, int n) { return e264b_configure((E264bDevice *)ctx, g, n); }
static void *be_host_alloc(void *ctx, size_t b) { return e264b_host_alloc((E264bDevice *)ctx, b); }
static void be_host_free(void *ctx, void *p) { e264b_host_free((E264bDevice *)ctx, p); }
static int be_acquire(void *ctx, int slot, E264Staging *out) { return e264b_acquire_staging((E264bDevice *)ctx, slot, out); }
static int be_submit(void *ctx, const E264PicDesc *pd, uint8_t *out, uint64_t *t) { return e264b_submit((E264bDevice *)ctx, pd, out, t); }
static int be_wait(void *ctx, uint64_t t) { return e264b_wait((E264bDevice *)ctx, t); }
static int be_fill(void *ctx, int slot, int y, int c) { return e264b_fill_slot((E264bDevice *)ctx, slot, y, c); }
static int be_poll(void *ctx, uint64_t t) { return e264b_poll((E264bDevice *)ctx, t); }
static const E264Backend cuda_backend = {"cuda-sm_100a", be_create, be_destroy, be_configure, be_host_alloc, be_host_free, be_acquire, be_submit, be_wait, be_fill, be_poll};
extern "C" const E264Backend *e264_default_backend(void) { return &cuda_backend; }
extern "C" E264bDevice *e264b_of_decoder(Edge264Decoder *d) { return d ? (E264bDevice *)d->be_ctx : NULL; }
