/* e264_bench — multi-stream decode driver over the edge264 C API (bench/test infrastructure).
 * Compiled twice from this one source: against libedge264_b200.so (tools/libe264bench.so) and against
 * the compiled reference (oracle/_ref/libe264bench_ref.so), so both arms of bench.py run the SAME
 * application loop (reference README.md:117-156) with one decoder instance per stream and one POSIX
 * thread per decoder.  Every output frame is read back on the host (64-bit word sum of the cropped
 * planes) so that the GPU arm's device->host copies are inside the timed region. */
#define _GNU_SOURCE
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include "edge264.h"

typedef struct Job {
	int stream; const uint8_t *buf; size_t size;
	long frames; uint64_t sum; int last_ret;
	Edge264Decoder *dec; int keep;
} Job;
typedef struct Pool { Job *jobs; int n, next; pthread_mutex_t mu; pthread_barrier_t *bar; } Pool;

static uint64_t frame_sum(const Edge264Frame *f) {
	uint64_t s = 0;
	for (int pl = 0; pl < 3; pl++) {
		int w = pl ? f->width_C : f->width_Y, h = pl ? f->height_C : f->height_Y, st = pl ? f->stride_C : f->stride_Y;
		for (int y = 0; y < h; y++) {
			const uint8_t *r = f->samples[pl] + (size_t)y * st;
			int x = 0; uint64_t a = 0;
			for (; x + 8 <= w; x += 8) { uint64_t v; memcpy(&v, r + x, 8); a += v; }
			for (; x < w; x++) a += r[x];
			s = s * 1000003u + a;
		}
	}
	return s;
}

/* frames copied out during e264bench_run (bench.py --dump-outputs), set by e264bench_capture */
static struct { int n; const int *stream; const long *index; uint8_t **dst; size_t cap; int *info; } capture;

static void capture_frame(const Job *j, long index, const Edge264Frame *f) {
	for (int k = 0; k < capture.n; k++) {
		if (capture.stream[k] != j->stream || capture.index[k] != index) continue;
		uint8_t *d = capture.dst[k], *e = d + capture.cap;
		for (int pl = 0; pl < 3; pl++) {
			int w = pl ? f->width_C : f->width_Y, h = pl ? f->height_C : f->height_Y, st = pl ? f->stride_C : f->stride_Y;
			for (int y = 0; y < h && d + w <= e; y++, d += w) memcpy(d, f->samples[pl] + (size_t)y * st, (size_t)w);
		}
		int *info = capture.info + 5 * k;
		info[0] = f->FrameId; info[1] = f->width_Y; info[2] = f->height_Y; info[3] = f->width_C; info[4] = f->height_C;
	}
}

static void decode_stream(Job *j) {
	const uint8_t *buf = j->buf, *end = buf + j->size;
	const uint8_t *nal = buf + 3 + (buf[2] == 0);
	/* E264_BENCH_DEC_THREADS: n_threads of every decoder (0 = parse inside decode_NAL; the GPU library parses pictures ahead on
	 * worker threads otherwise; the reference's threaded mode hangs here, SURVEY section 0.7, so its arm stays at 0) */
	const char *nt = getenv("E264_BENCH_DEC_THREADS");
	Edge264Decoder *dec = edge264_alloc(nt ? atoi(nt) : 0, NULL, NULL, 0, NULL, NULL, NULL);
	Edge264Frame f; int res, drained = 0; long frames = 0; uint64_t sum = 0;
	if (!dec) { j->last_ret = -1; return; }
	for (;;) {
		const uint8_t *sc = nal < end ? edge264_find_start_code(nal, end, 0) : end;
		long before = frames;
		res = edge264_decode_NAL(dec, nal, sc, NULL, NULL);
		if (nal >= end) drained = 1;
		while (!edge264_get_frame(dec, &f, 0)) {
			sum = sum * 31 + frame_sum(&f);
			if (capture.n) capture_frame(j, frames, &f);
			frames++;
		}
		if (res == ENOBUFS) { if (frames == before) break; continue; }
		if (res == ENOTSUP || res == EBADMSG) res = 0;
		nal = sc + 3 < end ? sc + 3 : end;
		if (res != 0 || drained) break;
	}
	j->frames = frames; j->sum = sum; j->last_ret = res;
	if (j->keep) j->dec = dec; else edge264_free(&dec);
}

static void *worker(void *arg) {
	Pool *p = (Pool *)arg;
	pthread_barrier_wait(p->bar);
	for (;;) {
		pthread_mutex_lock(&p->mu);
		int i = p->next < p->n ? p->next++ : -1;
		pthread_mutex_unlock(&p->mu);
		if (i < 0) break;
		decode_stream(&p->jobs[i]);
	}
	return NULL;
}

/* Decode n_streams buffers with n_threads threads.  Returns wall seconds of the decode region.
 * frames[i], sums[i] per stream; decoders[i] kept alive when keep != 0 (caller frees with e264bench_free). */
double e264bench_run(const uint8_t **bufs, const size_t *sizes, int n_streams, int n_threads, int keep,
                     long *frames, uint64_t *sums, void **decoders) {
	Job *jobs = (Job *)calloc((size_t)n_streams, sizeof(Job));
	for (int i = 0; i < n_streams; i++) { jobs[i].stream = i; jobs[i].buf = bufs[i]; jobs[i].size = sizes[i]; jobs[i].keep = keep; }
	if (n_threads > n_streams) n_threads = n_streams;
	if (n_threads < 1) n_threads = 1;
	pthread_barrier_t bar; pthread_barrier_init(&bar, NULL, (unsigned)n_threads + 1);
	Pool p = {jobs, n_streams, 0, PTHREAD_MUTEX_INITIALIZER, &bar};
	pthread_t *th = (pthread_t *)calloc((size_t)n_threads, sizeof(pthread_t));
	for (int i = 0; i < n_threads; i++) pthread_create(&th[i], NULL, worker, &p);
	struct timespec t0, t1;
	pthread_barrier_wait(&bar);
	clock_gettime(CLOCK_MONOTONIC, &t0);
	for (int i = 0; i < n_threads; i++) pthread_join(th[i], NULL);
	clock_gettime(CLOCK_MONOTONIC, &t1);
	for (int i = 0; i < n_streams; i++) { if (frames) frames[i] = jobs[i].frames; if (sums) sums[i] = jobs[i].sum; if (decoders) decoders[i] = jobs[i].dec; }
	free(th); free(jobs); pthread_barrier_destroy(&bar);
	return (t1.tv_sec - t0.tv_sec) + 1e-9 * (t1.tv_nsec - t0.tv_nsec);
}
/* Output frames to copy during the following e264bench_run calls: frame index[k] (in output order) of stream stream[k]
 * goes to dst[k] (at most cap bytes: the cropped Y, Cb and Cr planes one after the other), its FrameId, width_Y,
 * height_Y, width_C and height_C to info[5k..5k+4].  n = 0 ends the capture. */
void e264bench_capture(int n, const int *stream, const long *index, uint8_t **dst, size_t cap, int *info) {
	capture.stream = stream; capture.index = index; capture.dst = dst; capture.cap = cap; capture.info = info; capture.n = n;
}
void e264bench_free(void **decoders, int n) { for (int i = 0; i < n; i++) { Edge264Decoder *d = (Edge264Decoder *)decoders[i]; edge264_free(&d); decoders[i] = NULL; } }
