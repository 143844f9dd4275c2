/*
 * qs_cuda.cu - host side of the CUDA back end: context, device memory, launch sequencing
 * and the C ABI declared in include/jpegqs_cuda.h.
 *
 * The sequencing restates the reference driver do_quantsmooth (reference
 * quantsmooth.h:2404-2878) as a schedule of kernel launches; the arithmetic itself lives in
 * qs_kernels.cu.  Independent components (and, in the batch entry point, independent
 * images) share launches; the luma -> chroma dependency of JOINT_YUV / UPSAMPLE_UV
 * (quantsmooth.h:2495, 2691-2815) splits a run into two phases.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <memory>
#include <unordered_map>
#include <vector>
#include "qs_common.h"
#include "qs_kernels.h"
#include "qs_hostio.h"
#include "../../include/jpegqs_cuda.h"

/* ------------------------------------------------------------------------------------------
 * weight tables: quantsmooth_init, reference quantsmooth.h:251-301, built from the float
 * LL&M IDCT of reference idct.h:565-604.  Host code; this TU is compiled without FMA
 * contraction so the values are the reference's bits (DESIGN.md 3.4; tests compare them
 * against the reference's own table builder).
 * ------------------------------------------------------------------------------------------ */
static void tab_idct_1d(const float *in, int is, float *out, int os, bool scale) {
	float t0, t1, t2, t3, t4, t5, t6, t7, z1, z2, z3, z4, z5, r[8];
	z2 = in[2 * is]; z3 = in[6 * is];
	z1 = (z2 + z3) * 0.541196100f;
	t2 = z1 - z3 * 1.847759065f;
	t3 = z1 + z2 * 0.765366865f;
	z2 = in[0]; z3 = in[4 * is];
	t0 = z2 + z3; t1 = z2 - z3;
	t4 = t0 + t3; t7 = t0 - t3; t5 = t1 + t2; t6 = t1 - t2;
	t0 = in[7 * is]; t1 = in[5 * is]; t2 = in[3 * is]; t3 = in[1 * is];
	z1 = t0 + t3; z2 = t1 + t2; z3 = t0 + t2; z4 = t1 + t3;
	z5 = (z3 + z4) * 1.175875602f;
	t0 *= 0.298631336f; t1 *= 2.053119869f; t2 *= 3.072711026f; t3 *= 1.501321110f;
	z1 *= 0.899976223f; z2 *= 2.562915447f; z3 *= 1.961570560f; z4 *= 0.390180644f;
	z3 -= z5; t0 -= z1 + z3; t2 -= z2 + z3;
	z4 -= z5; t1 -= z2 + z4; t3 -= z1 + z4;
	r[0] = t4 + t3; r[7] = t4 - t3; r[1] = t5 + t2; r[6] = t5 - t2;
	r[2] = t6 + t1; r[5] = t6 - t1; r[3] = t7 + t0; r[4] = t7 - t0;
	for (int k = 0; k < 8; k++) out[k * os] = scale ? r[k] * 0.125f : r[k];
}

static int build_tables(int flags, float *out, float prescale) {
	const int size = (flags & QS_DIAGONALS) ? QS_TAB_DIAG : QS_TAB_PLAIN;
	const float bcoef = (flags & QS_DIAGONALS) ? 4.0f : 2.0f;
	for (int i = 0; i < 64; i++) {
		float e[64], ws[64], B[64], *t = out + i * size;
		memset(e, 0, sizeof(e)); e[i] = 1.0f;
		for (int x = 0; x < 8; x++) tab_idct_1d(e + x, 8, ws + x, 8, false);
		for (int y = 0; y < 8; y++) tab_idct_1d(ws + y * 8, 1, B + y * 8, 1, true);
		for (int y = 0; y < 8; y++) for (int x = 0; x < 8; x++) {
			t[y * 8 + x] = x < 7 ? B[y * 8 + x] - B[y * 8 + x + 1] : 0.0f;
			t[96 + y * 8 + x] = y < 7 ? B[y * 8 + x] - B[y * 8 + 8 + x] : 0.0f;
		}
		for (int x = 0; x < 8; x++) {
			t[64 + x] = B[x] * bcoef; t[72 + x] = B[56 + x] * bcoef;
			t[80 + x] = B[x * 8] * bcoef; t[88 + x] = B[x * 8 + 7] * bcoef;
		}
		if (flags & QS_DIAGONALS) for (int y = 0; y < 7; y++) {
			float *d = t + 160 + y * 16;
			for (int x = 0; x < 7; x++) {
				d[x] = B[y * 8 + x] - B[y * 8 + 9 + x];
				d[8 + x] = B[y * 8 + x + 1] - B[y * 8 + 8 + x];
			}
			d[7] = d[15] = 0.0f;
		}
		if (prescale != 1.0f) for (int k = 0; k < size; k++) t[k] *= prescale;   /* power of two: exact */
	}
	return size;
}

/* chunk schedule of one quant table: anti-diagonals s = 14..1 of the 8x8 coefficient grid in the
 * reference's visiting order (reverse zig-zag, quantsmooth.h:1403 + zigzag_refresh 313-322).
 * Inside an anti-diagonal the coefficients are independent, so they may be regrouped: runs of
 * equal quant value become "uniform" chunks (type 2) that share t and d*t per term. */
static int build_chunks(QsChunk *ch, int maxn, const uint16_t *q, int uniform, int merge = 0) {
	int n = 0;
	for (int s = 14; s >= 1; s--) {
		int full[8], nf = 0; bool first = true;
		for (int u = 0; u < 8; u++) {
			int v = s - u;
			if (v < 0 || v > 7 || u == 0 || v == 0) continue;
			full[nf++] = v * 8 + u;
		}
		bool used[8] = { false };
		if (s <= 7) {
			/* merge: the diagonal's two edge coefficients ride along with (up to) two of its full
			 * coefficients in one "mixed" chunk (type 3) instead of forming a chunk of their own
			 * with single-coefficient horizontal / vertical passes.  Not when those full
			 * coefficients would otherwise share their threshold work in a uniform chunk. */
			int take = 0;
			if (merge && maxn >= 4 && nf >= 1) {
				take = nf < 2 ? nf : 2;
				if (nf - take == 1) take = 1;              /* do not leave one full coefficient on its own */
				if (uniform && q) {
					/* keep uniform runs whole: only coefficients whose quant value is unique on this diagonal */
					int pick[2], np = 0;
					for (int a = 0; a < nf && np < take; a++) {
						bool tie = false;
						for (int b = 0; b < nf; b++) tie = tie || (b != a && q[full[b]] == q[full[a]]);
						if (!tie) pick[np++] = a;
					}
					if (np < take) take = 0;
					else for (int k = 0; k < take; k++) used[pick[k]] = true;
				} else for (int k = 0; k < take; k++) used[k] = true;
			}
			QsChunk c; memset(&c, 0, sizeof(c));
			c.first = 1; first = false;
			if (take) {
				int k = 0;
				c.type = 3; c.n = (uint8_t)take;
				for (int a = 0; a < nf; a++) if (used[a]) c.idx[k++] = (uint8_t)full[a];
				c.idx[k++] = (uint8_t)s; c.idx[k++] = (uint8_t)(s * 8);
			} else {
				c.type = 1; c.n = 2;
				c.idx[0] = (uint8_t)s;          /* row 0:    horizontal + border (+diag) */
				c.idx[1] = (uint8_t)(s * 8);    /* column 0: border + vertical   (+diag) */
			}
			ch[n++] = c;
		}
		int rest[8], nr = 0;
		if (uniform && q && maxn >= 2) {
			for (int a = 0; a < nf; a++) {
				if (used[a]) continue;
				int run[8], rl = 0;
				for (int b = a; b < nf; b++) if (!used[b] && q[full[b]] == q[full[a]]) run[rl++] = b;
				if (rl < 2) continue;
				for (int pos = 0; pos < rl; ) {
					int len = rl - pos > maxn ? maxn : rl - pos;
					if (rl - pos - len == 1) len--;            /* never leave a run member alone */
					if (len < 2) break;
					QsChunk c; memset(&c, 0, sizeof(c));
					c.type = 2; c.n = (uint8_t)len; c.first = first; first = false;
					for (int k = 0; k < len; k++) { c.idx[k] = (uint8_t)full[run[pos + k]]; used[run[pos + k]] = true; }
					pos += len;
					ch[n++] = c;
				}
			}
		}
		for (int a = 0; a < nf; a++) if (!used[a]) rest[nr++] = full[a];
		int parts = (nr + maxn - 1) / maxn, pos = 0;
		for (int p = 0; p < parts; p++) {
			int len = (nr - pos + (parts - p) - 1) / (parts - p);
			QsChunk c; memset(&c, 0, sizeof(c));
			c.type = 0; c.n = (uint8_t)len; c.first = first; first = false;
			for (int k = 0; k < len; k++) c.idx[k] = (uint8_t)rest[pos + k];
			pos += len;
			ch[n++] = c;
		}
	}
	return n;
}

#ifdef QS_EXPERIMENTS
/* pair schedule + interleaved pair tables of the packed FP32x2 path (qs_common.h QsChunk2):
 * per anti-diagonal the two edge coefficients form one pair, the others pair up in order, a
 * left-over coefficient gets a dummy lane.  out_tab: [nslots][size][2] floats. */
static int build_pairs(QsChunk2 *ch, int *nslots_out, int maxpairs, uint8_t lanes[][2]) {
	int n = 0, ns = 0;
	for (int s = 14; s >= 1; s--) {
		int list[8], nl = 0;
		if (s <= 7) { list[nl++] = s; list[nl++] = s * 8; }       /* row-0 and column-0 coefficient */
		for (int u = 1; u < 8; u++) { int v = s - u; if (v >= 1 && v <= 7) list[nl++] = v * 8 + u; }
		int npairs = (nl + 1) / 2; bool first = true;
		for (int p0 = 0; p0 < npairs; p0 += maxpairs) {
			QsChunk2 c; memset(&c, 0xFF, sizeof(c));
			c.np = (uint8_t)((npairs - p0) < maxpairs ? (npairs - p0) : maxpairs);
			c.first = first; first = false;
			for (int k = 0; k < c.np; k++) {
				int a = list[2 * (p0 + k)], b = 2 * (p0 + k) + 1 < nl ? list[2 * (p0 + k) + 1] : 0xFF;
				c.slot[k] = (uint8_t)ns; c.idx[2 * k] = (uint8_t)a; c.idx[2 * k + 1] = (uint8_t)b;
				lanes[ns][0] = (uint8_t)a; lanes[ns][1] = (uint8_t)b; ns++;
			}
			ch[n++] = c;
		}
	}
	*nslots_out = ns;
	return n;
}

static void build_pair_tables(int flags, const uint8_t lanes[][2], int nslots, float prescale, float *out) {
	const int size = (flags & QS_DIAGONALS) ? QS_TAB_DIAG : QS_TAB_PLAIN;
	std::vector<float> t(64 * size);
	build_tables(flags, t.data(), prescale);
	for (int sl = 0; sl < nslots; sl++) for (int h = 0; h < 2; h++) {
		int i = lanes[sl][h];
		for (int p = 0; p < size; p++) {
			float v = i < 64 ? t[i * size + p] : 0.0f;
			/* the reference skips these sections (quantsmooth.h:1527, 1531); a zero weight makes
			 * the term an exact no-op (adds +-0 to a2 and +0 to a3) */
			if (i < 64 && (i & 7) == 0 && p < 64) v = 0.0f;
			if (i < 64 && i <= 7 && p >= 96 && p < 160) v = 0.0f;
			out[((size_t)sl * size + p) * 2 + h] = v;
		}
	}
}

#endif

/* ------------------------------------------------------------------------------------------ */
struct jpegqs_cuda_ctx {
	int device, num_sms;
	char devname[256];
	cudaStream_t stream;
	cudaStream_t up_stream, down_stream;   /* H2D / D2H of the host entry points, overlapped with compute */
	/* host I/O of the host entry points (qs_hostio.h): pinned staging (grow-only), the gather /
	 * scatter pool and the two queues that keep uploads and downloads going */
	char *stage; size_t stage_cap;
	int io_threads;
	QsPool *pool; QsWorker *up, *down;
	std::vector<cudaEvent_t> io_ev; size_t io_ev_used;
	std::vector<cudaEvent_t> sync_ev;      /* per group: coefficients uploaded / group finished */
	std::vector<cudaEvent_t> slab_ev;      /* per slab of a pipelined group: uploaded / smoothed */
	float *tab_plain, *tab_diag;
	float *tab2_plain, *tab2_diag; int nslots2;   /* pair tables of the FP32x2 path */
	QsQuantDev *quant_dev; int quant_cap;
	QsJob *jobs_dev;                       /* two slots of QS_MAX_JOBS */
	std::vector<QsJob> jobs_cache[2];
	int *flags_dev;                        /* [QS_MAX_JOBS] bad flags + [1] tile counter */
	int *flags_host;                       /* pinned */
	char *arena; size_t arena_cap, arena_pos;
	cudaEvent_t ev0, ev1;
	float last_ms; int launches;
	/* optional per-kernel timing (bench.py's roofline line): event pairs around launches */
	int profiling;
	int tune_sync, tune_maxn, tune_wpg, tune_gs, tune_x2, tune_uni, tune_slabs, tune_wave, tune_merge;              /* kernel variant knobs (jpegqs_cuda_set_tuning) */
	std::vector<cudaEvent_t> ev_pool; size_t ev_used;
	std::vector<int> ev_kind;              /* 0 = idct pass, 1 = smoothing pass, per pair */
	float kernel_ms[2]; int kernel_launches[2];
	char err[512];
};

static char g_err[512] = "";

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
	snprintf(ctx ? ctx->err : g_err, 512, "%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
	return JPEGQS_ERR_CUDA; } } while (0)

extern "C" const char *jpegqs_cuda_last_error(const jpegqs_cuda_ctx *ctx) { return ctx ? ctx->err : g_err; }
extern "C" const char *jpegqs_cuda_device_name(const jpegqs_cuda_ctx *ctx) { return ctx->devname; }
extern "C" float jpegqs_cuda_last_device_ms(const jpegqs_cuda_ctx *ctx) { return ctx->last_ms; }
extern "C" int jpegqs_cuda_last_launches(const jpegqs_cuda_ctx *ctx) { return ctx->launches; }
extern "C" size_t jpegqs_cuda_plane_bytes(uint32_t wblk, uint32_t hblk) { return QS_PLANE_BYTES(wblk, hblk); }
extern "C" int jpegqs_cuda_plane_stride(uint32_t wblk) { return QS_PLANE_STRIDE(wblk); }
extern "C" int jpegqs_cuda_plane_pad(void) { return QS_PLANE_PAD; }
extern "C" int jpegqs_cuda_tables(int flags, float *out) { return build_tables(flags, out, 1.0f); }
extern "C" int jpegqs_cuda_orig_coef(int coef, int q) { return qs_host_orig_coef(coef, q); }

extern "C" void *jpegqs_cuda_host_alloc(size_t bytes) {
	void *p = NULL;
	if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return NULL;
	return p;
}
extern "C" void jpegqs_cuda_host_free(void *p) { if (p) cudaFreeHost(p); }

extern "C" void jpegqs_cuda_destroy(jpegqs_cuda_ctx *ctx) {
	if (!ctx) return;
	cudaSetDevice(ctx->device);
	if (ctx->stream) { cudaStreamSynchronize(ctx->stream); cudaStreamDestroy(ctx->stream); }
	delete ctx->up; delete ctx->down; delete ctx->pool;      /* joins the threads */
	if (ctx->up_stream) { cudaStreamSynchronize(ctx->up_stream); cudaStreamDestroy(ctx->up_stream); }
	if (ctx->down_stream) { cudaStreamSynchronize(ctx->down_stream); cudaStreamDestroy(ctx->down_stream); }
	for (cudaEvent_t e : ctx->io_ev) cudaEventDestroy(e);
	if (ctx->stage) cudaFreeHost(ctx->stage);
	for (cudaEvent_t e : ctx->sync_ev) cudaEventDestroy(e);
	for (cudaEvent_t e : ctx->slab_ev) cudaEventDestroy(e);
	cudaFree(ctx->tab_plain); cudaFree(ctx->tab_diag); cudaFree(ctx->tab2_plain); cudaFree(ctx->tab2_diag); cudaFree(ctx->quant_dev);
	cudaFree(ctx->jobs_dev); cudaFree(ctx->flags_dev); cudaFree(ctx->arena);
	if (ctx->flags_host) cudaFreeHost(ctx->flags_host);
	if (ctx->ev0) cudaEventDestroy(ctx->ev0);
	if (ctx->ev1) cudaEventDestroy(ctx->ev1);
	for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
	delete ctx;
}

extern "C" int jpegqs_cuda_create(int device, jpegqs_cuda_ctx **out) {
	jpegqs_cuda_ctx *ctx = NULL;
	if (!out) return JPEGQS_ERR_ARG;
	*out = NULL;
	int ndev = 0;
	CK(cudaGetDeviceCount(&ndev));
	if (ndev <= 0) { snprintf(g_err, sizeof(g_err), "no CUDA device"); return JPEGQS_ERR_CUDA; }
	if (device < 0) CK(cudaGetDevice(&device));
	CK(cudaSetDevice(device));
	cudaDeviceProp prop;
	CK(cudaGetDeviceProperties(&prop, device));
	if (prop.major < 10) {
		snprintf(g_err, sizeof(g_err), "device %d (%s, sm_%d%d) is not a Blackwell sm_100 part; "
				"this library carries sm_100a code only and has no fallback", device, prop.name, prop.major, prop.minor);
		return JPEGQS_ERR_CUDA;
	}
	ctx = new jpegqs_cuda_ctx();
	memset(ctx->err, 0, sizeof(ctx->err));
	ctx->device = device; ctx->num_sms = prop.multiProcessorCount;
	snprintf(ctx->devname, sizeof(ctx->devname), "%s", prop.name);
	ctx->tab2_plain = ctx->tab2_diag = NULL; ctx->nslots2 = 0;
	ctx->stream = NULL; ctx->up_stream = ctx->down_stream = NULL;
	ctx->stage = NULL; ctx->stage_cap = 0; ctx->pool = NULL; ctx->up = ctx->down = NULL; ctx->io_ev_used = 0;
	{
		const char *e = getenv("JPEGQS_IO_THREADS");
		int hw = (int)std::thread::hardware_concurrency();
		ctx->io_threads = e ? atoi(e) : (hw >= 16 ? 8 : hw >= 4 ? hw / 2 : 1);
		if (ctx->io_threads < 1) ctx->io_threads = 1;
		if (ctx->io_threads > 64) ctx->io_threads = 64;
	}
	ctx->tab_plain = ctx->tab_diag = NULL; ctx->quant_dev = NULL; ctx->quant_cap = 0;
	ctx->jobs_dev = NULL; ctx->flags_dev = NULL; ctx->flags_host = NULL;
	ctx->arena = NULL; ctx->arena_cap = ctx->arena_pos = 0; ctx->ev0 = ctx->ev1 = NULL;
	ctx->last_ms = 0; ctx->launches = 0;
	ctx->profiling = 0; ctx->ev_used = 0; ctx->tune_sync = 2; ctx->tune_maxn = 4; ctx->tune_wpg = 4; ctx->tune_gs = 1; ctx->tune_uni = 1; ctx->tune_merge = 1; ctx->tune_slabs = 1; ctx->tune_wave = 0; ctx->tune_x2 = 0;   /* packed FP32x2 measured slower: profiles/README.md */
	ctx->kernel_ms[0] = ctx->kernel_ms[1] = 0; ctx->kernel_launches[0] = ctx->kernel_launches[1] = 0;
	int rc = [&]() -> int {
		CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
		CK(cudaStreamCreateWithFlags(&ctx->up_stream, cudaStreamNonBlocking));
		CK(cudaStreamCreateWithFlags(&ctx->down_stream, cudaStreamNonBlocking));
		CK(cudaEventCreate(&ctx->ev0)); CK(cudaEventCreate(&ctx->ev1));
		std::vector<float> t(64 * QS_TAB_DIAG);
		const float pre = 1073741824.0f;               /* 2^(2*QS_SCALE_BITS) */
		build_tables(0, t.data(), pre);
		CK(cudaMalloc(&ctx->tab_plain, 64 * QS_TAB_PLAIN * sizeof(float)));
		CK(cudaMemcpy(ctx->tab_plain, t.data(), 64 * QS_TAB_PLAIN * sizeof(float), cudaMemcpyHostToDevice));
		build_tables(QS_DIAGONALS, t.data(), pre);
		CK(cudaMalloc(&ctx->tab_diag, 64 * QS_TAB_DIAG * sizeof(float)));
		CK(cudaMemcpy(ctx->tab_diag, t.data(), 64 * QS_TAB_DIAG * sizeof(float), cudaMemcpyHostToDevice));
		{
			QsChunk ch[QS_MAX_CHUNKS * 2];
			int n = build_chunks(ch, ctx->tune_maxn, NULL, 0, ctx->tune_merge);
			CK(qs_set_chunks(ch, n));
		}
#ifdef QS_EXPERIMENTS
		{
			QsChunk2 ch2[QS_MAX_CHUNKS]; uint8_t lanes[QS_MAX_SLOTS][2]; int ns = 0;
			int n2 = build_pairs(ch2, &ns, 2, lanes);
			CK(qs_set_chunks2(ch2, n2, ns));
			ctx->nslots2 = ns;
			std::vector<float> t2((size_t)ns * QS_TAB_DIAG * 2);
			build_pair_tables(0, lanes, ns, pre, t2.data());
			CK(cudaMalloc(&ctx->tab2_plain, (size_t)ns * QS_TAB_PLAIN * 2 * sizeof(float)));
			CK(cudaMemcpy(ctx->tab2_plain, t2.data(), (size_t)ns * QS_TAB_PLAIN * 2 * sizeof(float), cudaMemcpyHostToDevice));
			build_pair_tables(QS_DIAGONALS, lanes, ns, pre, t2.data());
			CK(cudaMalloc(&ctx->tab2_diag, (size_t)ns * QS_TAB_DIAG * 2 * sizeof(float)));
			CK(cudaMemcpy(ctx->tab2_diag, t2.data(), (size_t)ns * QS_TAB_DIAG * 2 * sizeof(float), cudaMemcpyHostToDevice));
		}
#endif
		CK(qs_smooth_configure());
		CK(cudaMalloc(&ctx->jobs_dev, 2 * QS_MAX_JOBS * sizeof(QsJob)));
		CK(cudaMalloc(&ctx->flags_dev, (QS_MAX_JOBS + 1) * sizeof(int)));
		CK(cudaMallocHost(&ctx->flags_host, QS_MAX_JOBS * sizeof(int)));
		return 0;
	}();
	if (rc) { snprintf(g_err, sizeof(g_err), "%s", ctx->err); jpegqs_cuda_destroy(ctx); return rc; }
	*out = ctx;
	return 0;
}

static int arena_reserve(jpegqs_cuda_ctx *ctx, size_t bytes) {
	if (bytes > ctx->arena_cap) {
		CK(cudaStreamSynchronize(ctx->stream));
		if (ctx->arena) CK(cudaFree(ctx->arena));
		ctx->arena = NULL; ctx->arena_cap = 0;
		size_t cap = bytes + bytes / 8 + (1 << 20);
		CK(cudaMalloc(&ctx->arena, cap));
		ctx->arena_cap = cap;
	}
	ctx->arena_pos = 0;
	return 0;
}
static void *arena_take(jpegqs_cuda_ctx *ctx, size_t bytes) {
	size_t p = (ctx->arena_pos + 255) & ~(size_t)255;
	ctx->arena_pos = p + bytes;
	return ctx->arena + p;
}
static size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

/* pinned staging of the host entry points: grow-only, so a caller that smooths image after image
 * pays cudaHostAlloc once (round 1 allocated and freed 100-300 MB of pinned memory per call) */
static int stage_reserve(jpegqs_cuda_ctx *ctx, size_t bytes) {
	if (bytes <= ctx->stage_cap) return 0;
	if (ctx->stage) { CK(cudaFreeHost(ctx->stage)); ctx->stage = NULL; ctx->stage_cap = 0; }
	size_t cap = bytes + bytes / 8 + (1 << 20);
	CK(cudaHostAlloc((void **)&ctx->stage, cap, cudaHostAllocPortable));
	ctx->stage_cap = cap;
	return 0;
}
static int io_start(jpegqs_cuda_ctx *ctx) {
	if (!ctx->pool) ctx->pool = new QsPool(ctx->io_threads - 1);   /* the caller of parallel_for works too */
	if (!ctx->up) ctx->up = new QsWorker();
	if (!ctx->down) ctx->down = new QsWorker();
	return 0;
}
static int io_event(jpegqs_cuda_ctx *ctx, cudaEvent_t *e) {
	if (ctx->io_ev_used == ctx->io_ev.size()) {
		cudaEvent_t n; CK(cudaEventCreateWithFlags(&n, cudaEventDisableTiming | cudaEventBlockingSync));
		ctx->io_ev.push_back(n);
	}
	*e = ctx->io_ev[ctx->io_ev_used++];
	return 0;
}
/* is p memory the copy engines can read directly (cudaHostAlloc / cudaHostRegister)? */
static bool is_pinned(const void *p) {
	cudaPointerAttributes at;
	if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
	return at.type == cudaMemoryTypeHost;
}

/* One contiguous run of block rows of one coefficient array moving between the host and the
 * device.  rows != NULL: the host side is a table of separately allocated block rows (libjpeg's
 * virtual arrays, or a flat pageable array cut into rows) that is gathered into / scattered from
 * the pinned memory at `pin`; rows == NULL: `pin` is the caller's own pinned flat array. */
struct IoSeg {
	int16_t *dev, *pin; int16_t *const *rows;
	int wblk, r0, r1;
};
/* gather (dir 0: rows -> pin) or scatter (dir 1: pin -> rows) the segments on the pool */
static void io_rows_copy(QsPool *pool, const std::vector<IoSeg> &segs, int dir) {
	struct Task { const IoSeg *s; int r0, r1; };
	std::vector<Task> tasks;
	for (const IoSeg &sg : segs) {
		if (!sg.rows || sg.r1 <= sg.r0) continue;
		size_t rowb = (size_t)sg.wblk * 128;
		int step = (int)std::max<size_t>(1, (512 << 10) / std::max<size_t>(rowb, 1));    /* ~512 KB per task */
		for (int r = sg.r0; r < sg.r1; r += step) tasks.push_back({ &sg, r, std::min(sg.r1, r + step) });
	}
	if (tasks.empty()) return;
	auto run = [&](int i) {
		const Task &t = tasks[i]; size_t rowb = (size_t)t.s->wblk * 128;
		for (int r = t.r0; r < t.r1; r++) {
			char *pin = (char *)t.s->pin + (size_t)r * rowb;
			if (dir == 0) memcpy(pin, t.s->rows[r], rowb); else memcpy(t.s->rows[r], pin, rowb);
		}
	};
	if (pool) pool->parallel_for((int)tasks.size(), run);
	else for (int i = 0; i < (int)tasks.size(); i++) run(i);
}

/* The host side of one run of a host entry point.
 * Uploads are a list of units (one slab of one phase, or a whole phase): gather the unit's block
 * rows into pinned memory (pool threads), H2D on the upload stream, record the unit's event.  With
 * anything to gather the list runs on the context's upload thread, so that the calling thread
 * can go on enqueueing kernels; wait(unit, st) makes stream st wait for a unit (after its event
 * has actually been recorded).  Downloads: D2H on the download stream behind an event of the
 * compute stream; block-row tables are scattered by the download thread + pool once the copy
 * has landed in pinned memory.  The destructor drains both threads: no return path may leave a
 * worker running on the caller's frame. */
struct HostIo {
	struct Unit { std::vector<IoSeg> segs; cudaEvent_t ev; };
	jpegqs_cuda_ctx *ctx;
	std::vector<Unit> units;
	std::atomic<int> recorded, failed;
	char err[256];
	explicit HostIo(jpegqs_cuda_ctx *c) : ctx(c), recorded(0), failed(0) { err[0] = 0; }
	~HostIo() { if (ctx->up) ctx->up->drain(); if (ctx->down) ctx->down->drain(); }
	int add_unit(std::vector<IoSeg> segs, cudaEvent_t ev) {
		Unit u; u.segs = std::move(segs); u.ev = ev;
		units.push_back(std::move(u));
		return (int)units.size() - 1;
	}
	int start() {                                        /* all units are known: go */
		bool gather = false;
		for (const Unit &u : units) for (const IoSeg &sg : u.segs) gather = gather || sg.rows != NULL;
		if (gather && io_start(ctx)) return JPEGQS_ERR_CUDA;
		if (gather) ctx->up->post([this] { run_units(); }); else run_units();
		return 0;
	}
	void run_units() {
		cudaStream_t cup = ctx->up_stream;
		cudaError_t e = cudaSetDevice(ctx->device);
		for (size_t i = 0; i < units.size() && e == cudaSuccess; i++) {
			io_rows_copy(ctx->pool, units[i].segs, 0);
			for (const IoSeg &sg : units[i].segs) {
				size_t off = (size_t)sg.r0 * sg.wblk * 64, cnt = (size_t)(sg.r1 - sg.r0) * sg.wblk * 64;
				if (cnt && e == cudaSuccess)
					e = cudaMemcpyAsync(sg.dev + off, sg.pin + off, cnt * 2, cudaMemcpyHostToDevice, cup);
			}
			if (e == cudaSuccess) e = cudaEventRecord(units[i].ev, cup);
			if (e == cudaSuccess) recorded.store((int)i + 1, std::memory_order_release);
		}
		if (e != cudaSuccess) {
			snprintf(err, sizeof(err), "upload: %s", cudaGetErrorString(e));
			failed.store(1, std::memory_order_release);
		}
	}
	int wait(int unit, cudaStream_t st) {
		if (unit < 0) return 0;
		while (recorded.load(std::memory_order_acquire) <= unit && !failed.load(std::memory_order_acquire))
			std::this_thread::yield();
		if (failed.load()) { snprintf(ctx->err, sizeof(ctx->err), "%s", err); return JPEGQS_ERR_CUDA; }
		CK(cudaStreamWaitEvent(st, units[unit].ev, 0));
		return 0;
	}
	int download(std::vector<IoSeg> segs, cudaEvent_t after) {
		cudaStream_t cdn = ctx->down_stream;
		CK(cudaStreamWaitEvent(cdn, after, 0));
		bool scatter = false;
		for (const IoSeg &sg : segs) {
			size_t off = (size_t)sg.r0 * sg.wblk * 64, cnt = (size_t)(sg.r1 - sg.r0) * sg.wblk * 64;
			if (cnt) CK(cudaMemcpyAsync(sg.pin + off, sg.dev + off, cnt * 2, cudaMemcpyDeviceToHost, cdn));
			scatter = scatter || sg.rows != NULL;
		}
		if (scatter) {
			cudaEvent_t e;
			if (io_event(ctx, &e) || io_start(ctx)) return JPEGQS_ERR_CUDA;
			CK(cudaEventRecord(e, cdn));
			QsPool *pool = ctx->pool; int devno = ctx->device;
			ctx->down->post([segs, e, pool, devno]() {
				cudaSetDevice(devno);
				if (cudaEventSynchronize(e) == cudaSuccess) io_rows_copy(pool, segs, 1);
			});
		}
		return 0;
	}
	int finish() {                                       /* everything has landed in the caller's memory */
		CK(cudaStreamSynchronize(ctx->down_stream));
		if (ctx->up) ctx->up->drain();
		if (ctx->down) ctx->down->drain();
		return 0;
	}
};

static void quant_prepare(const uint16_t *raw, QsQuantDev *q, int *val_out, int maxn = 4, int uniform = 1, int merge = 0) {
	int val = 0;
	for (int i = 0; i < 64; i++) {
		int v = raw[i]; val |= v;
		int qq = v ? v : 1;                            /* quantsmooth.h:2508-2511 */
		q->qraw[i] = (uint16_t)v; q->q[i] = (uint16_t)qq;
		q->Rs[i] = (float)(2 * qq) * (1.0f / (float)(1 << QS_SCALE_BITS));
		q->m31[i] = (uint32_t)(((1ull << 31) + (uint32_t)qq - 1) / (uint32_t)qq);
	}
	{
		QsChunk tmp[QS_MAX_CHUNKS * 2];
		int n = build_chunks(tmp, maxn, q->q, uniform, merge);
		if (n > QS_MAX_CHUNKS) n = build_chunks(tmp, maxn, NULL, 0);   /* cannot happen for maxn 1..4 */
		memset(q->chunks, 0, sizeof(q->chunks));
		memcpy(q->chunks, tmp, (size_t)n * sizeof(QsChunk));
		q->nchunks = n;
	}
	q->sched_slot = 0;      /* callers that smooth run assign_sched_slots over the upload */
	*val_out = val;
}

static int quant_reserve(jpegqs_cuda_ctx *ctx, int n) {
	if (n > ctx->quant_cap) {
		CK(cudaStreamSynchronize(ctx->stream));
		if (ctx->quant_dev) CK(cudaFree(ctx->quant_dev));
		ctx->quant_dev = NULL; ctx->quant_cap = 0;
		CK(cudaMalloc(&ctx->quant_dev, (size_t)(n + 16) * sizeof(QsQuantDev)));
		ctx->quant_cap = n + 16;
	}
	return 0;
}

/* sched_slot: tables with identical chunk schedules get the same id, so the kernel can tell
 * whether the warps of a lock-step group may follow their own table's schedule */
static void assign_sched_slots(QsQuantDev *q, int n) {
	std::unordered_map<uint64_t, std::vector<int> > seen;
	for (int i = 0; i < n; i++) {
		uint64_t h = 1469598103934665603ull;
		const uint8_t *b = (const uint8_t *)q[i].chunks;
		size_t len = (size_t)q[i].nchunks * sizeof(QsChunk);
		for (size_t k = 0; k < len; k++) h = (h ^ b[k]) * 1099511628211ull;
		h ^= (uint64_t)q[i].nchunks << 56;
		int slot = i;
		for (int j : seen[h])
			if (q[j].nchunks == q[i].nchunks && !memcmp(q[j].chunks, q[i].chunks, len)) { slot = j; break; }
		if (slot == i) seen[h].push_back(i);
		q[i].sched_slot = slot;
	}
}

/* upload a job list into one of the two device slots unless it is already there */
static int upload_jobs(jpegqs_cuda_ctx *ctx, int slot, std::vector<QsJob> &jobs, cudaStream_t st,
		const QsJob **dev, int *total_tiles, bool keep_bad_slots = false) {
	int tiles = 0;
	for (size_t i = 0; i < jobs.size(); i++) {
		jobs[i].tile_begin = tiles;
		if (!keep_bad_slots) jobs[i].bad_slot = (int)i;
		tiles += (jobs[i].nblocks + 31) / 32;
	}
	*total_tiles = tiles;
	*dev = ctx->jobs_dev + (size_t)slot * QS_MAX_JOBS;
	std::vector<QsJob> &c = ctx->jobs_cache[slot];
	if (c.size() == jobs.size() && (jobs.empty() || !memcmp(c.data(), jobs.data(), jobs.size() * sizeof(QsJob))))
		return 0;
	if (jobs.size() > QS_MAX_JOBS) { snprintf(ctx->err, sizeof(ctx->err), "too many jobs in one launch"); return JPEGQS_ERR_ARG; }
	/* travels as kernel parameters: an H2D copy would queue behind the bulk coefficient uploads */
	if (!jobs.empty()) CK(qs_store_jobs((QsJob *)*dev, jobs.data(), (int)jobs.size(), st));
	c = jobs;
	return 0;
}

/* per-kernel timing helpers: prof_begin/prof_end bracket one launch with an event pair */
static int prof_begin(jpegqs_cuda_ctx *ctx, int kind, cudaStream_t st) {
	if (!ctx->profiling) return 0;
	while (ctx->ev_pool.size() < ctx->ev_used + 2) {
		cudaEvent_t e; CK(cudaEventCreate(&e)); ctx->ev_pool.push_back(e);
	}
	ctx->ev_kind.push_back(kind);
	CK(cudaEventRecord(ctx->ev_pool[ctx->ev_used], st));
	return 0;
}
static int prof_end(jpegqs_cuda_ctx *ctx, cudaStream_t st) {
	if (!ctx->profiling) return 0;
	CK(cudaEventRecord(ctx->ev_pool[ctx->ev_used + 1], st));
	ctx->ev_used += 2;
	return 0;
}
static int prof_collect(jpegqs_cuda_ctx *ctx) {
	ctx->kernel_ms[0] = ctx->kernel_ms[1] = 0; ctx->kernel_launches[0] = ctx->kernel_launches[1] = 0;
	for (size_t i = 0; i < ctx->ev_kind.size(); i++) {
		float ms = 0; int k = ctx->ev_kind[i];
		CK(cudaEventElapsedTime(&ms, ctx->ev_pool[2 * i], ctx->ev_pool[2 * i + 1]));
		ctx->kernel_ms[k] += ms; ctx->kernel_launches[k]++;
	}
	ctx->ev_kind.clear(); ctx->ev_used = 0;
	return 0;
}

extern "C" void jpegqs_cuda_set_profiling(jpegqs_cuda_ctx *ctx, int on) { ctx->profiling = on; }

/* kernel-variant knobs for tuning runs (tools/tune.py); results are identical for every
 * setting.  key 0: lock-step sub-partition groups (0/1); key 1: max coefficients per chunk (1..4) */
extern "C" int jpegqs_cuda_set_tuning(jpegqs_cuda_ctx *ctx, int key, int value) {
	if (!ctx) return JPEGQS_ERR_ARG;
#ifdef QS_EXPERIMENTS
	if (key == 0) { ctx->tune_sync = value < 0 || value > 2 ? 2 : value; return 0; }
#else
	if (key == 0) return value == 2 ? 0 : JPEGQS_ERR_UNSUPPORTED;                              /* experiments build only */
#endif
#ifdef QS_EXPERIMENTS
	if (key == 4) { ctx->tune_x2 = value ? 1 : 0; return 0; }
	if (key == 2) { ctx->tune_wpg = value == 6 ? 6 : 4; return 0; }
#else
	if (key == 4 || key == 2) return value == (key == 4 ? 0 : 4) ? 0 : JPEGQS_ERR_UNSUPPORTED;   /* experiments build only */
#endif
	if (key == 3) return 0;                            /* retired */
	if (key == 1) {
		if (value < 1 || value > 4) return JPEGQS_ERR_ARG;
		CK(cudaSetDevice(ctx->device));
		CK(cudaStreamSynchronize(ctx->stream));
		CK(cudaDeviceSynchronize());
		QsChunk ch[QS_MAX_CHUNKS * 2];
		int n = build_chunks(ch, value, NULL, 0, ctx->tune_merge);
		if (n > QS_MAX_CHUNKS) return JPEGQS_ERR_ARG;
		CK(qs_set_chunks(ch, n));                  /* the table-independent schedule */
		ctx->tune_maxn = value;                    /* per-table schedules follow with the next upload */
		return 0;
	}
	if (key == 5) { ctx->tune_uni = value ? 1 : 0; return 0; }
	if (key == 8) {                                    /* edge coefficients merged into mixed chunks */
		CK(cudaSetDevice(ctx->device));
		CK(cudaStreamSynchronize(ctx->stream));
		CK(cudaDeviceSynchronize());
		ctx->tune_merge = value ? 1 : 0;
		QsChunk ch[QS_MAX_CHUNKS * 2];
		int n = build_chunks(ch, ctx->tune_maxn, NULL, 0, ctx->tune_merge);
		CK(qs_set_chunks(ch, n));
		return 0;
	}
	if (key == 6) { ctx->tune_slabs = value ? 1 : 0; return 0; }
	if (key == 7) { if (value < 0) return JPEGQS_ERR_ARG; ctx->tune_wave = value; return 0; }
	return JPEGQS_ERR_ARG;
}
extern "C" int jpegqs_cuda_chunk_schedule(const uint16_t *quant, int max_coefs, int uniform, uint8_t *out) {
	if (max_coefs < 1 || max_coefs > 4 || !out) return JPEGQS_ERR_ARG;
	uint16_t q[64];
	if (quant) for (int i = 0; i < 64; i++) q[i] = quant[i] ? quant[i] : 1;       /* as quant_prepare */
	QsChunk tmp[QS_MAX_CHUNKS * 2];
	int n = build_chunks(tmp, max_coefs, quant ? q : NULL, quant ? (uniform & 1) : 0, (uniform >> 1) & 1);
	if (n > QS_MAX_CHUNKS) return JPEGQS_ERR_ARG;
	memcpy(out, tmp, (size_t)n * sizeof(QsChunk));
	return n;
}
extern "C" void jpegqs_cuda_kernel_stats(const jpegqs_cuda_ctx *ctx, float *idct_ms, int *idct_launches,
		float *smooth_ms, int *smooth_launches) {
	if (idct_ms) *idct_ms = ctx->kernel_ms[0];
	if (idct_launches) *idct_launches = ctx->kernel_launches[0];
	if (smooth_ms) *smooth_ms = ctx->kernel_ms[1];
	if (smooth_launches) *smooth_launches = ctx->kernel_launches[1];
}

/* ------------------------------------------------------------------------------------------
 * The two drivers, both restating the reference driver do_quantsmooth (quantsmooth.h:2404-2878):
 * run_images (whole images; the host decides `stop`) and run_slab (one slab of an image sharded
 * by MCU rows; the device decides `stop`).  Each has its own iteration loop; everything else they
 * share is below.
 * ------------------------------------------------------------------------------------------ */
struct CompWork {
	int img, ci;
	jpegqs_cuda_comp *c;
	int16_t *coef_dev; uint8_t *plane;
	int W, H, luma, qslot;
	int qval;              /* OR of the raw quant values (2501-2504) */
	int niter2, extra;
	bool iterate;          /* takes part in the IDCT / smoothing iterations */
	bool done_clamp;
	bool downloaded;       /* the slab pipeline already sent the coefficients back */
	/* host side (host entry points only): pinned memory the copy engines use, and the block-row
	 * table it is gathered from / scattered to (NULL: pin is the caller's own pinned array) */
	int16_t *pin; int16_t *const *rows;
	int16_t *pin_up; int16_t *const *rows_up;
};

struct ImgState {
	jpegqs_cuda_image *im;
	bool skip;             /* early return of quantsmooth.h:2458: image untouched */
	int need_downsample, stop;
	int stop_ci;           /* component at which `stop` was raised (components run in order) */
	uint8_t *image1, *image2;    /* full-res luma plane / down-sampled luma plane */
	uint8_t *image2_buf, *mem_buf[2];
	int16_t *coef_up_dev[2];
	int ngroups;
};

#define QS_MAX_SLABS 16    /* upload / download units of one group of a host entry point */

/* start of a run: counters, niter clamp (quantsmooth.h:2455-2456), and nothing of an earlier
 * (failed) call may linger in the I/O threads */
static int run_start(jpegqs_cuda_ctx *ctx, int *niter) {
	CK(cudaSetDevice(ctx->device));
	ctx->launches = 0; ctx->last_ms = 0;
	ctx->ev_kind.clear(); ctx->ev_used = 0;
	*niter = std::min(std::max(*niter, 0), 100);
	if (ctx->up) ctx->up->drain();
	if (ctx->down) ctx->down->drain();
	ctx->io_ev_used = 0;
	return 0;
}

/* start of one image: need_downsample (2447-2453) and the early return of 2458 (s.skip) */
static int image_start(ImgState &s, jpegqs_cuda_image *im, int flags, int niter) {
	memset(&s, 0, sizeof(s)); s.im = im; s.stop_ci = 1 << 30;
	im->upsampled = 0;
	if (im->ncomp < 1 || im->ncomp > JPEGQS_CUDA_MAX_COMP) return JPEGQS_ERR_ARG;
	s.need_downsample = (flags & (QS_JOINT_YUV | QS_UPSAMPLE_UV)) && im->is_ycbcr && im->ncomp >= 3 &&
			im->comp[1].h_samp == 1 && im->comp[1].v_samp == 1 &&
			im->comp[2].h_samp == 1 && im->comp[2].v_samp == 1;
	s.skip = niter <= 0 && !((flags & QS_UPSAMPLE_UV) && s.need_downsample);
	if (!s.skip && s.need_downsample && (im->comp[1].wblk != im->comp[2].wblk || im->comp[1].hblk != im->comp[2].hblk))
		return JPEGQS_ERR_ARG;
	return 0;
}

/* Device arena and pinned staging of a run.  image_layout walks the images twice with the same
 * code: the first sweep only counts bytes, the second (after reserve) hands out pointers and
 * prepares the quant constants. */
struct Layout {
	jpegqs_cuda_ctx *ctx;
	bool on_device, carve;
	size_t bytes, stage_bytes, stage_pos;
	int nquant;
	std::vector<QsQuantDev> qhost;
	std::vector<std::unique_ptr<int16_t *[]> > rowstore;    /* block-row tables made up for flat pageable arrays */
	Layout(jpegqs_cuda_ctx *c, bool dev) : ctx(c), on_device(dev), carve(false), bytes(0), stage_bytes(0), stage_pos(0), nquant(0) {}
	void *take(size_t b) {
		if (carve) return arena_take(ctx, b);
		bytes += align256(b);
		return NULL;
	}
	int16_t *stage(size_t b) {
		char *p = carve ? ctx->stage + stage_pos : NULL;
		(carve ? stage_pos : stage_bytes) += align256(b);
		return (int16_t *)p;
	}
	/* one coefficient array [hblk][wblk][64]: its device copy, and where the copy engines meet its
	 * host side - a block-row table gathered into staging, the caller's own pinned array, or a
	 * flat pageable array cut into rows and staged like a table */
	int16_t *coef(int16_t *host, int16_t *const *rows, uint32_t wblk, uint32_t hblk, int16_t **pin, int16_t *const **prows) {
		if (on_device) return host;
		size_t cb = (size_t)wblk * hblk * 128;
		int16_t *dev = (int16_t *)take(cb);
		if (rows) { *prows = rows; *pin = stage(cb); }
		else if (is_pinned(host)) { *prows = NULL; *pin = host; }
		else {
			if (carve) {
				rowstore.emplace_back(new int16_t *[hblk ? hblk : 1]);
				int16_t **t = rowstore.back().get();
				for (uint32_t y = 0; y < hblk; y++) t[y] = host + (size_t)y * wblk * 64;
				*prows = t;
			}
			*pin = stage(cb);
		}
		return dev;
	}
	int quant(const uint16_t *raw, int *val) {
		if (!carve) { nquant++; return -1; }
		QsQuantDev q; quant_prepare(raw, &q, val, ctx->tune_maxn, ctx->tune_uni, ctx->tune_merge);
		qhost.push_back(q);
		return (int)qhost.size() - 1;
	}
	int reserve() {
		if (arena_reserve(ctx, bytes + 4096)) return JPEGQS_ERR_CUDA;
		if (quant_reserve(ctx, nquant)) return JPEGQS_ERR_CUDA;
		if (stage_bytes && stage_reserve(ctx, stage_bytes)) return JPEGQS_ERR_CUDA;
		qhost.reserve(nquant);
		carve = true;
		return 0;
	}
};

/* memory of one image: per component its coefficients, plane and quant slot; the down-sampled
 * luma plane and, for UPSAMPLE_UV, the up-sampled chroma pixels and coefficients */
static int image_layout(Layout &ly, ImgState &s, std::vector<CompWork> &W, int img, int flags) {
	jpegqs_cuda_image *im = s.im;
	W.resize(im->ncomp);
	for (int ci = 0; ci < im->ncomp; ci++) {
		jpegqs_cuda_comp *c = &im->comp[ci]; CompWork &w = W[ci];
		if (!c->coef && !(!ly.on_device && c->rows) && c->wblk && c->hblk) return JPEGQS_ERR_ARG;
		memset(&w, 0, sizeof(w));
		w.img = img; w.ci = ci; w.c = c; w.W = c->wblk; w.H = c->hblk;
		w.luma = !ci || !im->is_ycbcr;                                    /* 2639 */
		w.coef_dev = ly.coef(c->coef, c->rows, c->wblk, c->hblk, &w.pin, &w.rows);
		w.plane = (uint8_t *)ly.take(QS_PLANE_BYTES(c->wblk, c->hblk));
		w.qslot = ly.quant(c->quant, &w.qval);
	}
	if (!s.need_downsample || (im->comp[0].h_samp == 1 && im->comp[0].v_samp == 1)) return 0;
	s.image2_buf = (uint8_t *)ly.take(QS_PLANE_BYTES(im->comp[1].wblk, im->comp[1].hblk));
	if (flags & QS_UPSAMPLE_UV) for (int j = 0; j < 2; j++) {
		jpegqs_cuda_comp *c = &im->comp[1 + j]; CompWork &w = W[1 + j];
		uint32_t W0 = im->comp[0].wblk, H0 = im->comp[0].hblk;
		if (!c->coef_up && !(!ly.on_device && c->rows_up)) return JPEGQS_ERR_ARG;
		s.mem_buf[j] = (uint8_t *)ly.take((size_t)W0 * H0 * 64);       /* up-sampled pixel plane */
		s.coef_up_dev[j] = ly.coef(c->coef_up, c->rows_up, W0, H0, &w.pin_up, &w.rows_up);
	}
	return 0;
}

/* memory of a run: count, reserve, carve; then the quant constants go up */
static int run_layout(Layout &ly, ImgState *S, std::vector<CompWork> *W, int nimg, int flags, cudaStream_t st) {
	jpegqs_cuda_ctx *ctx = ly.ctx;
	for (int sweep = 0; sweep < 2; sweep++) {
		if (sweep && ly.reserve()) return JPEGQS_ERR_CUDA;
		for (int n = 0; n < nimg; n++) {
			if (S[n].skip) continue;
			int rc = image_layout(ly, S[n], W[n], n, flags);
			if (rc) return rc;
		}
	}
	assign_sched_slots(ly.qhost.data(), (int)ly.qhost.size());
	if (!ly.qhost.empty())
		CK(cudaMemcpyAsync(ctx->quant_dev, ly.qhost.data(), ly.qhost.size() * sizeof(QsQuantDev), cudaMemcpyHostToDevice, st));
	ctx->jobs_cache[0].clear(); ctx->jobs_cache[1].clear();
	return 0;
}

/* grow-only event pools: per group uploaded / finished (sync_ev) and per slab or band (slab_ev) */
static int group_events(jpegqs_cuda_ctx *ctx, int ngroups) {
	while ((int)ctx->sync_ev.size() < 2 * ngroups) {
		cudaEvent_t e; CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); ctx->sync_ev.push_back(e);
	}
	while ((int)ctx->slab_ev.size() < 2 * ngroups * QS_MAX_SLABS) {
		cudaEvent_t e; CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); ctx->slab_ev.push_back(e);
	}
	return 0;
}

/* block rows [r0, r1) of a component's coefficients / of its up-sampled coefficients (luma geometry) */
static IoSeg coef_seg(const CompWork &w, int r0, int r1) {
	IoSeg sg; sg.dev = w.coef_dev; sg.pin = w.pin; sg.rows = w.rows; sg.wblk = w.W; sg.r0 = r0; sg.r1 = r1;
	return sg;
}
static IoSeg up_seg(const ImgState &s, const CompWork &w, int r0, int r1) {
	IoSeg sg; sg.dev = s.coef_up_dev[w.ci - 1]; sg.pin = w.pin_up; sg.rows = w.rows_up;
	sg.wblk = s.im->comp[0].wblk; sg.r0 = r0; sg.r1 = r1;
	return sg;
}

/* one component's job; top / bottom: it touches the image's top / bottom edge */
static QsJob make_job(const jpegqs_cuda_ctx *ctx, const CompWork &w, const uint8_t *plane2, int top, int bottom) {
	QsJob j; memset(&j, 0, sizeof(j));
	j.coef = w.coef_dev; j.plane = w.plane; j.plane2 = plane2;
	j.quant = ctx->quant_dev + w.qslot;
	j.wblk = w.W; j.hblk = w.H; j.stride = QS_PLANE_STRIDE(w.W); j.nblocks = w.W * w.H;
	j.luma = w.luma; j.top_edge = top; j.bottom_edge = bottom;
	return j;
}

/* the down-sampled luma plane a chroma component is predicted from (JOINT_YUV, 2639) */
static const uint8_t *plane2_of(const ImgState &s, const CompWork &w, int flags) {
	return (s.image2 && (flags & QS_JOINT_YUV) && w.ci > 0) ? s.image2 : NULL;
}

/* IDCT pass (2589-2620) over jobs.  stop_aware: the jobs carry their own bad_slot (run_slab) */
static int launch_idct(jpegqs_cuda_ctx *ctx, std::vector<QsJob> &jobs, int mode, bool stop_aware, cudaStream_t st) {
	const QsJob *jd; int tiles;
	if (upload_jobs(ctx, 0, jobs, st, &jd, &tiles, stop_aware)) return JPEGQS_ERR_CUDA;
	if (prof_begin(ctx, 0, st)) return JPEGQS_ERR_CUDA;
	CK(qs_launch_idct_pass(jd, (int)jobs.size(), tiles, mode, ctx->flags_dev, st));
	if (prof_end(ctx, st)) return JPEGQS_ERR_CUDA;
	ctx->launches++;
	return 0;
}

/* smoothing pass (2627-2640) over jobs: LOW_QUALITY, the packed FP32x2 experiment or the
 * default kernel.  stop_aware: the kernels consult the run's out-of-range flags (run_slab) */
static int launch_smooth(jpegqs_cuda_ctx *ctx, std::vector<QsJob> &jobs, int flags, int clampv, bool stop_aware,
		cudaStream_t st) {
	const QsJob *jd; int tiles;
	if (upload_jobs(ctx, 1, jobs, st, &jd, &tiles, stop_aware)) return JPEGQS_ERR_CUDA;
	const int nj = (int)jobs.size();
	const int *bad = stop_aware ? ctx->flags_dev : NULL;
	int *tile_counter = ctx->flags_dev + QS_MAX_JOBS;
	if (prof_begin(ctx, 1, st)) return JPEGQS_ERR_CUDA;
	if (flags & QS_LOW_QUALITY) CK(qs_launch_lowq(jd, nj, tiles, flags, clampv, bad, st));
#ifdef QS_EXPERIMENTS
	else if (ctx->tune_x2 && !bad) CK(qs_launch_smooth_x2(jd, nj, tiles,
			(flags & QS_DIAGONALS) ? ctx->tab2_diag : ctx->tab2_plain, ctx->nslots2, tile_counter, flags, clampv,
			ctx->num_sms, ctx->tune_sync, st));
#endif
	else CK(qs_launch_smooth(jd, nj, tiles, (flags & QS_DIAGONALS) ? ctx->tab_diag : ctx->tab_plain, tile_counter,
			flags, clampv, ctx->num_sms, ctx->tune_sync, ctx->tune_wpg, bad, st));
	if (prof_end(ctx, st)) return JPEGQS_ERR_CUDA;
	ctx->launches++;
	return 0;
}

/* de-quantize only (2551-2566) or clamp only (2670-2689) a whole component */
static int launch_scale_clamp(jpegqs_cuda_ctx *ctx, const CompWork &w, int dequant, int clamp, cudaStream_t st) {
	CK(qs_launch_scale_clamp(w.coef_dev, (size_t)w.W * w.H * 64, ctx->quant_dev + w.qslot, dequant, clamp, st));
	ctx->launches++;
	return 0;
}

/* per-component prelude of 2484-2566: the passes component w takes (niter2 smoothing iterations
 * + the extra render pass); once `stop` is set it is de-quantized only.  Returns 1 when w
 * iterates, 0 when not, or an error. */
static int comp_prelude(jpegqs_cuda_ctx *ctx, ImgState &s, CompWork &w, int niter, cudaStream_t st) {
	if (!w.c->has_qtbl) return 0;                                      /* 2494 */
	w.extra = (s.image1 || (!w.ci && s.need_downsample)) ? 1 : 0;      /* 2495 */
	w.niter2 = w.qval <= 1 ? 0 : niter;                                /* 2501 */
	if (w.qval >= 0x800 && !s.stop) { s.stop = 1; s.stop_ci = w.ci; }  /* 2504 */
	if (w.niter2 + w.extra == 0) return 0;                             /* 2542 */
	if (s.stop) return launch_scale_clamp(ctx, w, 1, 0, st);           /* 2551-2566 */
	if (!(w.W * w.H)) return 0;
	w.iterate = true;
	return 1;
}

/* post step of chroma component w: upsample_row + FDCT (2691-2752) into its luma-sized
 * coefficients.  y_row0_px: first luma pixel row of the slab inside the image */
static int post_upsample(jpegqs_cuda_ctx *ctx, const ImgState &s, const CompWork &w, int y_row0_px, cudaStream_t st) {
	const jpegqs_cuda_image *im = s.im;
	int ws = im->comp[0].h_samp, hs = im->comp[0].v_samp;
	int w1 = ((int)im->image_width + ws - 1) / ws, h1 = ((int)im->image_height + hs - 1) / hs;
	int W0 = im->comp[0].wblk, H0 = im->comp[0].hblk;
	uint8_t *mem = s.mem_buf[w.ci - 1];
	CK(qs_launch_upsample(w.plane, s.image2, QS_PLANE_STRIDE(w.W), s.image1, QS_PLANE_STRIDE(W0),
			mem, W0 * 8, w1, h1, ws, hs, W0 * 8, H0 * 8, y_row0_px, st));
	CK(qs_launch_fdct_plane(mem, W0 * 8, s.coef_up_dev[w.ci - 1], W0, H0, st));
	ctx->launches += 2;
	return 0;
}

/* post step of the luma component w: the down-sampled luma plane of 2753-2815 into s.image2_buf,
 * for the chroma block rows this slab holds.  Rows are addressed inside the whole components:
 * y_row0 / c_row0 = first luma / chroma block row of the slab, *_hblk_total = block rows of the
 * whole component.  At an image edge (top / bottom) the replicated border row is written too;
 * interior halo rows come from the neighbours. */
static int post_downsample(jpegqs_cuda_ctx *ctx, const ImgState &s, const CompWork &w, int y_row0, int y_hblk_total,
		int c_row0, int c_hblk_total, bool top, bool bottom, cudaStream_t st) {
	const jpegqs_cuda_comp *cc = &s.im->comp[1];
	int ws = w.c->h_samp, hs = w.c->v_samp;
	int h = y_hblk_total * 8, h2 = c_hblk_total * 8, h1_total = (h + hs - 1) / hs;
	int first = top ? -1 : c_row0 * 8;
	int last = bottom ? h2 : (c_row0 + (int)cc->hblk) * 8 - 1;
	int dstride = QS_PLANE_STRIDE(cc->wblk);
	if (last < first) return 0;
	CK(qs_launch_downsample(w.plane, QS_PLANE_STRIDE(w.W), w.W * 8, h,
			s.image2_buf + (size_t)(first - c_row0 * 8 + 1) * dstride, dstride, (int)cc->wblk * 8, h2,
			ws, hs, y_row0 * 8, first, last - first + 1, h1_total, st));
	ctx->launches++;
	return 0;
}

/* end of an image (2834-2859): quant tables := 1, chroma replaced by the up-sampled arrays */
static void image_finish(jpegqs_cuda_image *im, bool upsampled) {
	for (int ci = 0; ci < im->ncomp; ci++)
		if (im->comp[ci].has_qtbl) for (int k = 0; k < 64; k++) im->comp[ci].quant[k] = 1;
	im->upsampled = upsampled ? 1 : 0;
}

/* end of a run (ev1 recorded): everything has landed in the caller's memory; device time and
 * per-kernel timing */
static int run_end(jpegqs_cuda_ctx *ctx, HostIo &io, bool on_device, cudaStream_t st) {
	CK(cudaStreamSynchronize(st));
	if (!on_device && io.finish()) return JPEGQS_ERR_CUDA;       /* the last scatter has finished */
	CK(cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
	if (prof_collect(ctx)) return JPEGQS_ERR_CUDA;
	return 0;
}

/* ------------------------------------------------------------------------------------------
 * whole-image driver
 * ------------------------------------------------------------------------------------------ */
/* Host entry points, one large image: a group's block rows are cut into slabs of about one
 * wave of the persistent smoothing kernel.  Iteration 0 then follows the upload slab by slab
 * (IDCT pass of slab k, smoothing of slab k-1 - which needs the first pixel row of slab k), and
 * the last iteration hands its slabs to the download as they finish, so that only the first
 * slab's upload and the last slab's download are not hidden behind kernels.  Results do not
 * depend on this: a pass reads only start-of-pass neighbour pixels (quantsmooth.h:1396-1401). */
struct SlabPlan { int K; int r[QS_MAX_SLABS + 1]; };

static int run_images(jpegqs_cuda_ctx *ctx, int nimg, jpegqs_cuda_image *imgs, int flags, int niter,
		int progprec, jpegqs_cuda_progress_fn progress, void *userdata, bool on_device, int *ret,
		cudaStream_t st) {
	if (!ctx || nimg < 0 || (nimg && !imgs)) return JPEGQS_ERR_ARG;
	if (progress && nimg != 1) return JPEGQS_ERR_ARG;
	if (run_start(ctx, &niter)) return JPEGQS_ERR_CUDA;

	std::vector<ImgState> S(nimg);
	std::vector<std::vector<CompWork> > W(nimg);
	int max_groups = 0;
	for (int n = 0; n < nimg; n++) {
		ImgState &s = S[n];
		if (ret) ret[n] = 0;
		int rc = image_start(s, &imgs[n], flags, niter);
		if (rc) return rc;
		if (s.skip) continue;
		/* host buffers: luma and chroma are separate phases even when independent, so that the
		 * chroma upload and the luma download overlap with compute (copy stream + events) */
		s.ngroups = progress ? s.im->ncomp : ((s.need_downsample || (!on_device && s.im->ncomp > 1)) ? 2 : 1);
		if (s.ngroups > max_groups) max_groups = s.ngroups;
	}
	/* carve device memory, upload quant constants */
	Layout ly(ctx, on_device);
	{ int rc = run_layout(ly, S.data(), W.data(), nimg, flags, st); if (rc) return rc; }

	auto group_range = [&](const ImgState &s, int g, int *c0, int *c1) {
		if (progress) { *c0 = g; *c1 = g + 1; }
		else if (s.ngroups == 2) { *c0 = g ? 1 : 0; *c1 = g ? s.im->ncomp : 1; }
		else { *c0 = 0; *c1 = s.im->ncomp; }
	};
	std::vector<SlabPlan> plan(max_groups > 0 ? max_groups : 1);
	for (SlabPlan &pl : plan) pl.K = 0;

	/* ---- uploads / downloads: HostIo above ---- */
	HostIo io(ctx);
	std::vector<int> unit_of_group(max_groups > 0 ? max_groups : 1, -1);
	std::vector<std::vector<int> > unit_of_slab(max_groups > 0 ? max_groups : 1);
	if (!on_device) {
		if (group_events(ctx, max_groups)) return JPEGQS_ERR_CUDA;
		for (int g = 0; g < max_groups; g++) {
			if (nimg == 1 && !progress && ctx->tune_slabs && !ctx->tune_x2 && !(flags & QS_LOW_QUALITY) &&
					!S[0].skip && g < S[0].ngroups && niter >= 1) {
				/* slab plan of this group: all its components alike and certain to iterate */
				ImgState &s = S[0];
				int c0, c1; group_range(s, g, &c0, &c1);
				bool ok = c1 > c0;
				for (int ci = c0; ci < c1 && ok; ci++) {
					CompWork &w = W[0][ci];
					ok = w.c->has_qtbl && w.qval > 1 && w.qval < 0x800 && w.W > 0 && w.H > 0 &&
							w.W == W[0][c0].W && w.H == W[0][c0].H;
				}
				if (ok) {
					int Wb = W[0][c0].W, Hb = W[0][c0].H, nc = c1 - c0;
					long wave = (long)ctx->num_sms * ctx->tune_wpg * 4 * 32;     /* blocks in flight */
					if (ctx->tune_wave) wave = ctx->tune_wave;
					int rpw = (int)(wave / ((long)nc * Wb));
					if (rpw >= 1) {
						int waves = (Hb + rpw - 1) / rpw;
						int m = (waves + QS_MAX_SLABS - 1) / QS_MAX_SLABS;
						int K = (Hb + m * rpw - 1) / (m * rpw);
						if (K >= 2) {
							plan[g].K = K;
							for (int k = 0; k <= K; k++) plan[g].r[k] = (int)((long)k * Hb / K);
						}
					}
				}
			}
			if (plan[g].K) {
				int c0, c1; group_range(S[0], g, &c0, &c1);
				for (int k = 0; k < plan[g].K; k++) {
					std::vector<IoSeg> segs;
					for (int ci = c0; ci < c1; ci++) segs.push_back(coef_seg(W[0][ci], plan[g].r[k], plan[g].r[k + 1]));
					unit_of_slab[g].push_back(io.add_unit(std::move(segs), ctx->slab_ev[(2 * g) * QS_MAX_SLABS + k]));
				}
				unit_of_group[g] = unit_of_slab[g].back();
				continue;
			}
			std::vector<IoSeg> segs;
			for (int n = 0; n < nimg; n++) {
				ImgState &s = S[n];
				if (s.skip || g >= s.ngroups) continue;
				int c0, c1; group_range(s, g, &c0, &c1);
				for (int ci = c0; ci < c1; ci++) if (W[n][ci].W && W[n][ci].H) segs.push_back(coef_seg(W[n][ci], 0, W[n][ci].H));
			}
			unit_of_group[g] = io.add_unit(std::move(segs), ctx->sync_ev[2 * g]);
		}
		if (io.start()) return JPEGQS_ERR_CUDA;
	}

	int *bad_dev = ctx->flags_dev;
	CK(cudaEventRecord(ctx->ev0, st));

	/* progress bookkeeping, quantsmooth.h:2474-2482 (single image only) */
	int prog_next = 0, prog_max = 0, prog_thr = 0;
	if (progress && !S[0].skip) {
		jpegqs_cuda_image *im = S[0].im;
		for (int ci = 0; ci < im->ncomp; ci++) prog_max += im->comp[ci].hblk * im->comp[ci].v_samp * niter;
		if (progprec == 0) progprec = 20;
		if (progprec < 0) progprec = prog_max;
		prog_thr = progprec ? (int)((unsigned)(prog_max + progprec - 1) / (unsigned)progprec) : 0;
	}

	auto slab_job = [&](const CompWork &w, const uint8_t *plane2, int r0, int r1) {
		QsJob j = make_job(ctx, w, plane2, r0 == 0, r1 == w.H);
		size_t poff = (size_t)r0 * 8 * j.stride;
		j.coef += (size_t)r0 * w.W * 64; j.plane += poff;
		if (plane2) j.plane2 += poff;
		j.hblk = r1 - r0; j.nblocks = w.W * (r1 - r0);
		return j;
	};

	for (int g = 0; g < max_groups; g++) {
		bool slab_in = !on_device && plan[g].K > 0 && !S[0].stop;
		if (!on_device && !slab_in && io.wait(unit_of_group[g], st)) return JPEGQS_ERR_CUDA;
		/* ---- which components belong to this phase; per-component prelude 2484-2566 ---- */
		std::vector<CompWork *> works;
		int prog_cur = 0, prog_inc = 0;
		for (int n = 0; n < nimg; n++) {
			ImgState &s = S[n];
			if (s.skip || g >= s.ngroups) continue;
			int c0, c1; group_range(s, g, &c0, &c1);
			for (int ci = c0; ci < c1; ci++) {
				CompWork &w = W[n][ci];
				if (progress) { prog_cur = prog_next; prog_inc = w.c->v_samp; prog_next += w.H * prog_inc * niter; }
				int rc = comp_prelude(ctx, s, w, niter, st);
				if (rc < 0) return rc;
				if (rc) works.push_back(&w);
			}
		}

		int max_pass = 0;
		for (CompWork *w : works) if (w->niter2 + w->extra > max_pass) max_pass = w->niter2 + w->extra;
		if (slab_in) {
			int c0, c1; group_range(S[0], g, &c0, &c1);
			bool ok = (int)works.size() == c1 - c0;
			for (CompWork *w : works) ok = ok && w->niter2 == works[0]->niter2 && w->extra == works[0]->extra && w->niter2 >= 1;
			if (!ok) { slab_in = false; if (io.wait(unit_of_group[g], st)) return JPEGQS_ERR_CUDA; }
		}
		/* the download pipeline needs the slab plan but not the upload pipeline, and vice versa:
		 * a middle group's transfers hide behind its neighbours' kernels anyway */
		bool slab_out = slab_in && works[0]->niter2 >= 2 && !works[0]->extra && g == S[0].ngroups - 1;
		if (slab_in && g > 0) { slab_in = false; if (io.wait(unit_of_group[g], st)) return JPEGQS_ERR_CUDA; }
		for (int iter = 0; iter < max_pass; iter++) {
			if (iter == 0 && slab_in) {
				/* ---- iteration 0 behind the upload, slab by slab ---- */
				const SlabPlan &pl = plan[g];
				int cl = (works[0]->niter2 == 1 && !works[0]->extra) ? 1 : 0;
				CK(cudaMemsetAsync(bad_dev, 0, works.size() * sizeof(int), st));
				for (int k = 0; k <= pl.K; k++) {
					if (k < pl.K) {
						if (io.wait(unit_of_slab[g][k], st)) return JPEGQS_ERR_CUDA;
						std::vector<QsJob> jobs;
						for (CompWork *w : works) jobs.push_back(slab_job(*w, NULL, pl.r[k], pl.r[k + 1]));
						if (launch_idct(ctx, jobs, QS_IDCT_DEQUANT, false, st)) return JPEGQS_ERR_CUDA;
					}
					if (k >= 1) {
						std::vector<QsJob> jobs;
						for (CompWork *w : works) jobs.push_back(slab_job(*w, plane2_of(S[0], *w, flags), pl.r[k - 1], pl.r[k]));
						if (launch_smooth(ctx, jobs, flags, cl, false, st)) return JPEGQS_ERR_CUDA;
					}
				}
				CK(qs_copy_flags(bad_dev, ctx->flags_host, (int)works.size(), st));
				CK(cudaStreamSynchronize(st));
				bool bad = false;
				for (size_t k = 0; k < works.size(); k++) bad = bad || ctx->flags_host[k];
				if (!bad) {
					if (cl) for (CompWork *w : works) w->done_clamp = true;
					continue;
				}
				/* a coefficient left the legal range (quantsmooth.h:2602): the reference stops
				 * before smoothing anything of that component.  The host copy is still intact:
				 * fetch the group again and take the plain path, which implements the stop. */
				for (CompWork *w : works) {
					size_t cb = (size_t)w->W * w->H * 128;
					CK(cudaMemcpyAsync(w->coef_dev, w->pin, cb, cudaMemcpyHostToDevice, st));
				}
				slab_in = slab_out = false;
			}
			/* ---- IDCT pass, 2589-2620.  The extra (render-only) pass also applies the
			 *      final +-1023 clamp of 2670-2689 after rendering from unclamped values. */
			for (int clampv = 0; clampv < 2; clampv++) {
				std::vector<QsJob> jobs; std::vector<CompWork *> who;
				for (CompWork *w : works) {
					if (!w->iterate || iter >= w->niter2 + w->extra) continue;
					int cl = (iter == w->niter2) ? 1 : 0;
					if (cl != clampv) continue;
					jobs.push_back(make_job(ctx, *w, NULL, 1, 1)); who.push_back(w);
				}
				if (jobs.empty()) continue;
				int mode = (iter == 0 ? QS_IDCT_DEQUANT : 0) | (clampv ? QS_IDCT_CLAMP : 0);
				if (iter == 0) CK(cudaMemsetAsync(bad_dev, 0, jobs.size() * sizeof(int), st));
				if (launch_idct(ctx, jobs, mode, false, st)) return JPEGQS_ERR_CUDA;
				if (clampv) for (CompWork *w : who) w->done_clamp = true;
				if (iter == 0) {                                           /* bad_coef, 2602-2610 */
					CK(qs_copy_flags(bad_dev, ctx->flags_host, (int)jobs.size(), st));
					CK(cudaStreamSynchronize(st));
					for (size_t k = 0; k < who.size(); k++) {
						CompWork *w = who[k]; ImgState &s = S[w->img];
						if (s.stop && w->ci > s.stop_ci) {
							/* an earlier component of this image already failed: the reference
							 * would only have de-quantized this one - which the pass just did */
							w->iterate = false; w->done_clamp = true;
						} else if (ctx->flags_host[k]) {
							/* components run in order in the reference: this one stops here (it
							 * falls to the clamp below), earlier ones are unaffected */
							s.stop = 1; s.stop_ci = w->ci; w->iterate = false;
						}
					}
				}
			}
			/* ---- smoothing pass, 2627-2640 ---- */
			if (slab_out) for (CompWork *w : works) if (!w->iterate) slab_out = false;   /* a component stopped */
			if (slab_out && iter == works[0]->niter2 - 1) {
				/* last iteration: each finished slab goes straight to the download */
				const SlabPlan &pl = plan[g];
				for (int k = 0; k < pl.K; k++) {
					std::vector<QsJob> jobs;
					for (CompWork *w : works) jobs.push_back(slab_job(*w, plane2_of(S[0], *w, flags), pl.r[k], pl.r[k + 1]));
					if (launch_smooth(ctx, jobs, flags, 1, false, st)) return JPEGQS_ERR_CUDA;
					cudaEvent_t e = ctx->slab_ev[(2 * g + 1) * QS_MAX_SLABS + k];
					CK(cudaEventRecord(e, st));
					std::vector<IoSeg> segs;
					for (CompWork *w : works) segs.push_back(coef_seg(*w, pl.r[k], pl.r[k + 1]));
					if (io.download(std::move(segs), e)) return JPEGQS_ERR_CUDA;
				}
				for (CompWork *w : works) { w->done_clamp = true; w->downloaded = true; }
				continue;
			}
			for (int clampv = 0; clampv < 2; clampv++) {
				std::vector<QsJob> jobs; std::vector<CompWork *> who;
				for (CompWork *w : works) {
					if (!w->iterate || iter >= w->niter2) continue;
					int cl = (iter == w->niter2 - 1 && !w->extra) ? 1 : 0;
					if (cl != clampv) continue;
					jobs.push_back(make_job(ctx, *w, plane2_of(S[w->img], *w, flags), 1, 1)); who.push_back(w);
				}
				if (jobs.empty()) continue;
				if (launch_smooth(ctx, jobs, flags, clampv, false, st)) return JPEGQS_ERR_CUDA;
				if (clampv) for (CompWork *w : who) w->done_clamp = true;
			}
			if (progress && works.size() == 1 && works[0]->iterate && iter < works[0]->niter2) {   /* 2656-2664 */
				CompWork *w = works[0]; ImgState &s = S[0];
				int cur = prog_cur += w->H * prog_inc;
				if (cur >= prog_thr) {
					CK(cudaStreamSynchronize(st));
					cur = (int)((int64_t)progprec * cur / prog_max);
					prog_thr = (int)(((int64_t)(cur + 1) * prog_max + progprec - 1) / progprec);
					s.stop = progress(userdata, cur, progprec);
					if (s.stop) s.stop_ci = w->ci;
				}
				if (s.stop) w->iterate = false;
			}
		}
		/* ---- components that left the loop early still get the clamp of 2670-2689 ---- */
		for (CompWork *w : works) if (!w->done_clamp) {
			if (launch_scale_clamp(ctx, *w, 0, 1, st)) return JPEGQS_ERR_CUDA;
			w->done_clamp = true;
		}
		/* ---- post steps: chroma up-sampling (2691-2752), luma planes (2753-2815) ---- */
		for (CompWork *w : works) {
			ImgState &s = S[w->img];
			if (s.stop) continue;
			if (w->ci > 0 && s.image1 && w->ci <= 2) {
				if (post_upsample(ctx, s, *w, 0, st)) return JPEGQS_ERR_CUDA;
			} else if (w->ci == 0 && s.need_downsample) {
				if (w->c->h_samp == 1 && w->c->v_samp == 1) s.image2 = w->plane;
				else {
					if (flags & QS_UPSAMPLE_UV) s.image1 = w->plane;
					if (post_downsample(ctx, s, *w, 0, w->H, 0, (int)s.im->comp[1].hblk, true, true, st)) return JPEGQS_ERR_CUDA;
					s.image2 = s.image2_buf;
				}
			}
		}
		/* ---- downloads of this phase, on the copy stream, behind the phase's last kernel ---- */
		if (!on_device) {
			CK(cudaEventRecord(ctx->sync_ev[2 * g + 1], st));
			std::vector<IoSeg> segs;
			for (int n = 0; n < nimg; n++) {
				ImgState &s = S[n];
				if (s.skip || g >= s.ngroups) continue;
				int c0, c1; group_range(s, g, &c0, &c1);
				for (int ci = c0; ci < c1; ci++) {
					CompWork &w = W[n][ci];
					if (w.W && w.H && !w.downloaded) segs.push_back(coef_seg(w, 0, w.H));
					if (s.image1 && !s.stop && ci >= 1 && ci <= 2) segs.push_back(up_seg(s, w, 0, s.im->comp[0].hblk));
				}
			}
			if (io.download(std::move(segs), ctx->sync_ev[2 * g + 1])) return JPEGQS_ERR_CUDA;
		}
	}
	CK(cudaEventRecord(ctx->ev1, st));
	for (int n = 0; n < nimg; n++) {
		ImgState &s = S[n];
		if (s.skip) continue;
		image_finish(s.im, s.image1 && !s.stop);
		if (ret) ret[n] = s.stop;
	}
	return run_end(ctx, io, on_device, st);
}

extern "C" int jpegqs_cuda_run_host(jpegqs_cuda_ctx *ctx, jpegqs_cuda_image *img, int flags, int niter,
		int progprec, jpegqs_cuda_progress_fn progress, void *userdata) {
	int ret = 0;
	if (!ctx) return JPEGQS_ERR_ARG;
	int rc = run_images(ctx, 1, img, flags, niter, progprec, progress, userdata, false, &ret, ctx->stream);
	return rc < 0 ? rc : ret;
}

extern "C" int jpegqs_cuda_run_device(jpegqs_cuda_ctx *ctx, jpegqs_cuda_image *img, int flags, int niter,
		int progprec, jpegqs_cuda_progress_fn progress, void *userdata, void *stream) {
	int ret = 0;
	if (!ctx) return JPEGQS_ERR_ARG;
	int rc = run_images(ctx, 1, img, flags, niter, progprec, progress, userdata, true, &ret,
			stream ? (cudaStream_t)stream : ctx->stream);
	return rc < 0 ? rc : ret;
}

extern "C" int jpegqs_cuda_run_batch(jpegqs_cuda_ctx *ctx, int nimages, jpegqs_cuda_image *imgs, int flags,
		int niter, int on_device, int *ret, void *stream) {
	if (!ctx || nimages < 0) return JPEGQS_ERR_ARG;
	/* a launch carries at most QS_MAX_JOBS components: larger batches run as several sub-batches */
	for (int i = 0; i < nimages; ) {
		int n = 0, jobs = 0;
		while (i + n < nimages && imgs[i + n].ncomp > 0 && jobs + imgs[i + n].ncomp <= QS_MAX_JOBS) jobs += imgs[i + n++].ncomp;
		if (!n) return JPEGQS_ERR_ARG;
		int rc = run_images(ctx, n, imgs + i, flags, niter, 0, NULL, NULL, on_device != 0, ret ? ret + i : NULL,
				stream ? (cudaStream_t)stream : ctx->stream);
		if (rc) return rc;
		i += n;
	}
	return 0;
}

/* ------------------------------------------------------------------------------------------
 * One image sharded by MCU rows over several GPUs (SURVEY.md 8e): links + run_slab.
 *
 * Every rank (a device of this process, or another process on the box) owns a mailbox in its
 * device memory and maps the mailboxes of all ranks: cudaDeviceEnablePeerAccess inside a
 * process, CUDA IPC handles between processes - NVLink / NVSwitch peer memory either way.  The
 * exchange kernels (qs_kernels.cu qs_xchg_*) store pixel rows and the out-of-range masks
 * straight into the peers' mailboxes and hand over by sequence numbers, so between the IDCT pass
 * and the smoothing pass of an iteration there is neither a host round trip nor a library call.
 * ------------------------------------------------------------------------------------------ */
#define QS_BOX_HALO_FLAG 0            /* uint32[2]: rows from the upper / lower neighbour have arrived */
#define QS_BOX_BAD_FLAG 64            /* uint32[QS_MAX_RANKS]: mask message of rank r has arrived */
#define QS_BOX_BAD_MASK 128           /* uint32[QS_MAX_RANKS][16] */
#define QS_BOX_ROWS 2048              /* uint8 [2 parity][2 side][QS_XCHG_SLOTS][row_bytes] */

struct jpegqs_cuda_link {
	jpegqs_cuda_ctx *ctx;
	int rank, world;
	size_t row_bytes, box_bytes;
	char *box;                           /* this rank's mailbox */
	char *peer[QS_MAX_RANKS];            /* every rank's mailbox in this rank's address space */
	bool ipc_open[QS_MAX_RANKS];
	bool connected;
	uint32_t seq;                        /* exchanges so far: every rank counts the same */
	int *timeout_host;                   /* mapped: set by a pull kernel whose peer never signalled */
};

extern "C" int jpegqs_cuda_link_create(jpegqs_cuda_ctx *ctx, int rank, int world, uint32_t max_wblk,
		jpegqs_cuda_link **out) {
	if (!ctx || !out || world < 1 || world > QS_MAX_RANKS || rank < 0 || rank >= world || !max_wblk) return JPEGQS_ERR_ARG;
	CK(cudaSetDevice(ctx->device));
	jpegqs_cuda_link *l = new jpegqs_cuda_link();
	memset(l, 0, sizeof(*l));
	l->ctx = ctx; l->rank = rank; l->world = world;
	l->row_bytes = align256((size_t)QS_PLANE_STRIDE(max_wblk));
	l->box_bytes = QS_BOX_ROWS + (size_t)2 * 2 * QS_XCHG_SLOTS * l->row_bytes;
	cudaError_t e = cudaMalloc((void **)&l->box, l->box_bytes);
	if (e == cudaSuccess) e = cudaMemset(l->box, 0, l->box_bytes);
	if (e == cudaSuccess) e = cudaHostAlloc((void **)&l->timeout_host, 4 * sizeof(int), cudaHostAllocMapped);
	if (e != cudaSuccess) {
		snprintf(ctx->err, sizeof(ctx->err), "link_create: %s", cudaGetErrorString(e));
		cudaFree(l->box); delete l; return JPEGQS_ERR_CUDA;
	}
	memset(l->timeout_host, 0, 4 * sizeof(int));
	l->peer[rank] = l->box;
	l->connected = world == 1;
	*out = l;
	return 0;
}

extern "C" void jpegqs_cuda_link_destroy(jpegqs_cuda_link *l) {
	if (!l) return;
	cudaSetDevice(l->ctx->device);
	cudaStreamSynchronize(l->ctx->stream);
	for (int r = 0; r < l->world; r++) if (l->ipc_open[r]) cudaIpcCloseMemHandle(l->peer[r]);
	cudaFree(l->box);
	if (l->timeout_host) cudaFreeHost(l->timeout_host);
	delete l;
}

extern "C" int jpegqs_cuda_link_handle_bytes(void) { return (int)sizeof(cudaIpcMemHandle_t); }

/* this rank's mailbox as a CUDA IPC handle (jpegqs_cuda_link_handle_bytes() bytes) */
extern "C" int jpegqs_cuda_link_export(jpegqs_cuda_link *l, void *handle) {
	if (!l || !handle) return JPEGQS_ERR_ARG;
	jpegqs_cuda_ctx *ctx = l->ctx;
	CK(cudaSetDevice(ctx->device));
	cudaIpcMemHandle_t h;
	CK(cudaIpcGetMemHandle(&h, l->box));
	memcpy(handle, &h, sizeof(h));
	return 0;
}

/* ranks in different processes: handles = world x jpegqs_cuda_link_handle_bytes(), in rank order
 * (gathered by whatever the caller uses to talk between processes) */
extern "C" int jpegqs_cuda_link_connect_ipc(jpegqs_cuda_link *l, const void *handles) {
	if (!l || !handles) return JPEGQS_ERR_ARG;
	jpegqs_cuda_ctx *ctx = l->ctx;
	CK(cudaSetDevice(ctx->device));
	for (int r = 0; r < l->world; r++) {
		if (r == l->rank || l->peer[r]) continue;
		cudaIpcMemHandle_t h;
		memcpy(&h, (const char *)handles + (size_t)r * sizeof(h), sizeof(h));
		void *p = NULL;
		CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
		l->peer[r] = (char *)p; l->ipc_open[r] = true;
	}
	l->connected = true;
	return 0;
}

/* ranks on several devices of THIS process: peer access + plain pointers */
extern "C" int jpegqs_cuda_link_connect_local(jpegqs_cuda_link **links, int world) {
	if (!links || world < 1 || world > QS_MAX_RANKS) return JPEGQS_ERR_ARG;
	for (int a = 0; a < world; a++) {
		jpegqs_cuda_link *l = links[a];
		if (!l || l->world != world || l->rank != a) return JPEGQS_ERR_ARG;
		jpegqs_cuda_ctx *ctx = l->ctx;
		CK(cudaSetDevice(ctx->device));
		for (int b = 0; b < world; b++) {
			if (b == a) continue;
			int can = 0;
			if (links[b]->ctx->device != ctx->device) {
				CK(cudaDeviceCanAccessPeer(&can, ctx->device, links[b]->ctx->device));
				if (!can) {
					snprintf(ctx->err, sizeof(ctx->err), "device %d cannot access device %d's memory (no P2P path)",
							ctx->device, links[b]->ctx->device);
					return JPEGQS_ERR_CUDA;
				}
				cudaError_t e = cudaDeviceEnablePeerAccess(links[b]->ctx->device, 0);
				if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
				cudaGetLastError();
			}
			l->peer[b] = links[b]->box;
		}
		l->connected = true;
	}
	return 0;
}

static char *box_rows(const jpegqs_cuda_link *l, char *box, int parity, int side, int slot) {
	return box + QS_BOX_ROWS + (((size_t)parity * 2 + side) * QS_XCHG_SLOTS + slot) * l->row_bytes;
}

struct XchgPlane { uint8_t *plane; int wblk, rows; };

/* one exchange on stream st: first / last pixel row of every plane to the neighbours, theirs into
 * the halo rows; with bad_n > 0 also the OR of bad_dev[0..bad_n) over all ranks */
static int slab_exchange(jpegqs_cuda_ctx *ctx, jpegqs_cuda_link *l, const std::vector<XchgPlane> &planes,
		int *bad_dev, int bad_n, cudaStream_t st) {
	if (!l || l->world == 1) return 0;
	if (planes.size() > QS_XCHG_SLOTS || bad_n > 16) return JPEGQS_ERR_ARG;
	uint32_t seq = ++l->seq; int parity = (int)(seq & 1), rank = l->rank, world = l->world;
	QsXchgPush ps; QsXchgPull pl;
	memset(&ps, 0, sizeof(ps)); memset(&pl, 0, sizeof(pl));
	ps.seq = pl.seq = seq;
	for (size_t k = 0; k < planes.size(); k++) {
		const XchgPlane &p = planes[k];
		uint32_t stride = (uint32_t)QS_PLANE_STRIDE(p.wblk); int h = p.rows * 8;
		if (p.rows < 1 || stride > l->row_bytes) {
			snprintf(ctx->err, sizeof(ctx->err), "sharded run: a rank holds no block row of a component, or the link is too narrow");
			return JPEGQS_ERR_ARG;
		}
		if (rank > 0) {          /* my first pixel row is the upper neighbour's bottom halo (side 1 there) */
			ps.rows[ps.nrows++] = { p.plane + (size_t)1 * stride, (uint8_t *)box_rows(l, l->peer[rank - 1], parity, 1, (int)k), stride, 0 };
			pl.rows[pl.nrows++] = { (const uint8_t *)box_rows(l, l->box, parity, 0, (int)k), p.plane, stride, 0 };
		}
		if (rank < world - 1) {
			ps.rows[ps.nrows++] = { p.plane + (size_t)h * stride, (uint8_t *)box_rows(l, l->peer[rank + 1], parity, 0, (int)k), stride, 0 };
			pl.rows[pl.nrows++] = { (const uint8_t *)box_rows(l, l->box, parity, 1, (int)k), p.plane + (size_t)(h + 1) * stride, stride, 0 };
		}
	}
	if (rank > 0) {
		ps.flag[0] = (uint32_t *)(l->peer[rank - 1] + QS_BOX_HALO_FLAG) + 1;
		pl.flag[0] = (const uint32_t *)(l->box + QS_BOX_HALO_FLAG) + 0;
	}
	if (rank < world - 1) {
		ps.flag[1] = (uint32_t *)(l->peer[rank + 1] + QS_BOX_HALO_FLAG) + 0;
		pl.flag[1] = (const uint32_t *)(l->box + QS_BOX_HALO_FLAG) + 1;
	}
	if (bad_n > 0) {
		ps.bad_src = bad_dev; ps.bad_n = bad_n; pl.bad_io = bad_dev; pl.bad_n = bad_n;
		for (int r = 0; r < world; r++) {
			if (r == rank) continue;
			ps.bad_dst[ps.npeers] = (uint32_t *)(l->peer[r] + QS_BOX_BAD_MASK) + (size_t)rank * 16;
			ps.bad_flag[ps.npeers] = (uint32_t *)(l->peer[r] + QS_BOX_BAD_FLAG) + rank;
			ps.npeers++;
			pl.bad_in[pl.npeers] = (const uint32_t *)(l->box + QS_BOX_BAD_MASK) + (size_t)r * 16;
			pl.bad_flag[pl.npeers] = (const uint32_t *)(l->box + QS_BOX_BAD_FLAG) + r;
			pl.npeers++;
		}
	}
	CK(cudaHostGetDevicePointer((void **)&pl.timeout_flag, l->timeout_host, 0));
	CK(qs_launch_xchg(&ps, &pl, st));
	ctx->launches += 2;
	return 0;
}

/* do_quantsmooth on ONE SLAB of an image: img describes the slab (comp[].hblk = block rows held
 * by this rank, coef / rows = those rows), geom where it sits.  Unlike run_images the schedule is
 * unconditional - what the reference decides with `stop` is decided on the device from the
 * run's out-of-range flags (QsJob.stop_aware), which the ranks OR-combine in the first exchange
 * of a phase - so every rank issues the same exchanges whatever its data look like. */
static int run_slab(jpegqs_cuda_ctx *ctx, jpegqs_cuda_link *link, jpegqs_cuda_image *im, const jpegqs_cuda_slab *geom,
		int flags, int niter, bool on_device, int *ret, cudaStream_t st) {
	if (!ctx || !im || !geom) return JPEGQS_ERR_ARG;
	const int rank = link ? link->rank : 0, world = link ? link->world : 1;
	if (link && (link->ctx != ctx || !link->connected)) return JPEGQS_ERR_ARG;
	if (geom->rank != rank || geom->world != world) return JPEGQS_ERR_ARG;
	if (run_start(ctx, &niter)) return JPEGQS_ERR_CUDA;
	const bool top = rank == 0, bottom = rank == world - 1;
	if (ret) *ret = 0;
	ImgState s;
	{ int rc = image_start(s, im, flags, niter); if (rc) return rc; }
	if (s.skip) return 0;
	const int nc = im->ncomp;
	for (int ci = 0; ci < nc && world > 1; ci++) if (!im->comp[ci].hblk || !im->comp[ci].wblk) {
		snprintf(ctx->err, sizeof(ctx->err), "sharded run: rank %d holds no block row of component %d", rank, ci);
		return JPEGQS_ERR_ARG;
	}
	Layout ly(ctx, on_device);
	std::vector<CompWork> W;
	{ int rc = run_layout(ly, &s, &W, 1, flags, st); if (rc) return rc; }

	/* ---- phases (luma | chroma when the chroma needs the finished luma, or to overlap the
	 *      transfers of host buffers), uploads ---- */
	const int ngroups = (s.need_downsample || (!on_device && nc > 1)) ? 2 : 1;
	auto group_range = [&](int g, int *c0, int *c1) {
		if (ngroups == 2) { *c0 = g ? 1 : 0; *c1 = g ? nc : 1; } else { *c0 = 0; *c1 = nc; }
	};
	HostIo io(ctx);
	int unit_of_group[2] = { -1, -1 }, nbands[2] = { 1, 1 };
	if (!on_device) {
		/* a phase travels in bands of ~8 MB: the H2D copy of band k runs while band k+1 is being
		 * gathered (and, on the way back, band k is scattered while band k+1 is still in flight) */
		if (group_events(ctx, ngroups)) return JPEGQS_ERR_CUDA;
		for (int g = 0; g < ngroups; g++) {
			int c0, c1; group_range(g, &c0, &c1);
			size_t gb = 0;
			for (int ci = c0; ci < c1; ci++) gb += (size_t)W[ci].W * W[ci].H * 128;
			nbands[g] = (int)std::min<size_t>(QS_MAX_SLABS, std::max<size_t>(1, gb >> 23));
			for (int k = 0; k < nbands[g]; k++) {
				std::vector<IoSeg> segs;
				for (int ci = c0; ci < c1; ci++) {
					int r0 = (int)((long)k * W[ci].H / nbands[g]), r1 = (int)((long)(k + 1) * W[ci].H / nbands[g]);
					if (W[ci].W && r1 > r0) segs.push_back(coef_seg(W[ci], r0, r1));
				}
				unit_of_group[g] = io.add_unit(std::move(segs), k == nbands[g] - 1 ? ctx->sync_ev[2 * g] : ctx->slab_ev[(2 * g) * QS_MAX_SLABS + k]);
			}
		}
		if (io.start()) return JPEGQS_ERR_CUDA;
	}

	int *bad_dev = ctx->flags_dev;
	CK(cudaMemsetAsync(bad_dev, 0, 16 * sizeof(int), st));
	CK(cudaEventRecord(ctx->ev0, st));
	auto slab_job = [&](const CompWork &w, const uint8_t *plane2) {
		QsJob j = make_job(ctx, w, plane2, top, bottom);
		j.bad_slot = w.ci; j.bad_first = 0; j.stop_aware = 1;
		return j;
	};

	for (int g = 0; g < ngroups; g++) {
		if (!on_device && io.wait(unit_of_group[g], st)) return JPEGQS_ERR_CUDA;
		int c0, c1; group_range(g, &c0, &c1);
		std::vector<CompWork *> works;
		for (int ci = c0; ci < c1; ci++) {              /* only the static stop of 2504 is known on the host */
			int rc = comp_prelude(ctx, s, W[ci], niter, st);
			if (rc < 0) return rc;
			if (rc) works.push_back(&W[ci]);
		}
		int max_pass = 0;
		for (CompWork *w : works) max_pass = std::max(max_pass, w->niter2 + w->extra);
		for (int iter = 0; iter < max_pass; iter++) {
			std::vector<XchgPlane> xp;
			for (int clampv = 0; clampv < 2; clampv++) {                   /* IDCT pass, 2589-2620 (+ final clamp) */
				std::vector<QsJob> jobs;
				for (CompWork *w : works) {
					if (iter >= w->niter2 + w->extra) continue;
					if (((iter == w->niter2) ? 1 : 0) != clampv) continue;
					jobs.push_back(slab_job(*w, NULL));
					xp.push_back({ w->plane, w->W, w->H });
				}
				if (jobs.empty()) continue;
				int mode = (iter == 0 ? QS_IDCT_DEQUANT : 0) | (clampv ? QS_IDCT_CLAMP : 0);
				if (launch_idct(ctx, jobs, mode, true, st)) return JPEGQS_ERR_CUDA;
			}
			/* halo rows from the neighbours; the first exchange of a phase also ORs the flags */
			if ((!xp.empty() || iter == 0) && slab_exchange(ctx, link, xp, bad_dev, iter == 0 ? nc : 0, st)) return JPEGQS_ERR_CUDA;
			for (int clampv = 0; clampv < 2; clampv++) {                   /* smoothing pass, 2627-2640 */
				std::vector<QsJob> jobs;
				for (CompWork *w : works) {
					if (iter >= w->niter2) continue;
					if (((iter == w->niter2 - 1 && !w->extra) ? 1 : 0) != clampv) continue;
					jobs.push_back(slab_job(*w, plane2_of(s, *w, flags)));
				}
				if (jobs.empty()) continue;
				if (launch_smooth(ctx, jobs, flags, clampv, true, st)) return JPEGQS_ERR_CUDA;
			}
		}
		{	/* the component that overflowed is clamped only (2602-2610, 2670-2689); on the device */
			std::vector<QsJob> jobs;
			for (CompWork *w : works) jobs.push_back(slab_job(*w, NULL));
			if (!jobs.empty()) {
				const QsJob *jd; int tiles;
				if (upload_jobs(ctx, 0, jobs, st, &jd, &tiles, true)) return JPEGQS_ERR_CUDA;
				CK(qs_launch_stop_fixup(jd, (int)jobs.size(), bad_dev, st));
				ctx->launches++;
			}
		}
		/* post steps: chroma up-sampling (2691-2752), luma planes (2753-2815); results are dropped
		 * at the end if the run stopped */
		for (CompWork *w : works) {
			if (w->ci > 0 && s.image1 && w->ci <= 2) {
				if (post_upsample(ctx, s, *w, (int)geom->row0[0] * 8, st)) return JPEGQS_ERR_CUDA;
			} else if (w->ci == 0 && s.need_downsample) {
				if (w->c->h_samp == 1 && w->c->v_samp == 1) s.image2 = w->plane;
				else {
					if (flags & QS_UPSAMPLE_UV) s.image1 = w->plane;
					if (post_downsample(ctx, s, *w, (int)geom->row0[0], (int)geom->hblk_total[0], (int)geom->row0[1],
							(int)geom->hblk_total[1], top, bottom, st)) return JPEGQS_ERR_CUDA;
					s.image2 = s.image2_buf;
					std::vector<XchgPlane> xp; xp.push_back({ s.image2_buf, (int)im->comp[1].wblk, (int)im->comp[1].hblk });
					if (slab_exchange(ctx, link, xp, bad_dev, 0, st)) return JPEGQS_ERR_CUDA;
				}
			}
		}
		if (!on_device) {                                                  /* downloads of this phase, band by band */
			CK(cudaEventRecord(ctx->sync_ev[2 * g + 1], st));
			const int H0 = (int)im->comp[0].hblk;
			for (int k = 0; k < nbands[g]; k++) {
				std::vector<IoSeg> segs;
				for (int ci = c0; ci < c1; ci++) {
					CompWork &w = W[ci];
					int r0 = (int)((long)k * w.H / nbands[g]), r1 = (int)((long)(k + 1) * w.H / nbands[g]);
					if (w.W && r1 > r0) segs.push_back(coef_seg(w, r0, r1));
					r0 = (int)((long)k * H0 / nbands[g]); r1 = (int)((long)(k + 1) * H0 / nbands[g]);
					if (s.image1 && ci >= 1 && ci <= 2 && r1 > r0) segs.push_back(up_seg(s, w, r0, r1));
				}
				if (io.download(std::move(segs), ctx->sync_ev[2 * g + 1])) return JPEGQS_ERR_CUDA;
			}
		}
	}
	CK(cudaEventRecord(ctx->ev1, st));
	CK(qs_copy_flags(bad_dev, ctx->flags_host, nc, st));
	if (run_end(ctx, io, on_device, st)) return JPEGQS_ERR_CUDA;
	if (link && *link->timeout_host) {
		int *t = link->timeout_host;
		snprintf(ctx->err, sizeof(ctx->err), "sharded run: rank %d of %d waited 10 s for %s %d: sequence %d expected, %d found "
				"(its own count: %u)", rank, world, t[1] > 32 ? "the mask message of peer" : "the halo rows of neighbour",
				t[1] > 32 ? t[1] - 33 : t[1] - 1, t[2], t[3], link->seq);
		memset(t, 0, 4 * sizeof(int));
		return JPEGQS_ERR_TIMEOUT;
	}
	int stop = s.stop;
	for (int ci = 0; ci < nc; ci++) if (W[ci].iterate && ctx->flags_host[ci]) stop = 1;
	/* NOTE on upsampled chroma when the run stopped: coef_up holds data nobody will look at */
	image_finish(im, s.image1 && !stop);
	if (ret) *ret = stop;
	return 0;
}

extern "C" int jpegqs_cuda_run_slab(jpegqs_cuda_ctx *ctx, jpegqs_cuda_link *link, jpegqs_cuda_image *slab,
		const jpegqs_cuda_slab *geom, int flags, int niter, int on_device, void *stream) {
	int ret = 0;
	if (!ctx) return JPEGQS_ERR_ARG;
	int rc = run_slab(ctx, link, slab, geom, flags, niter, on_device != 0, &ret, stream ? (cudaStream_t)stream : ctx->stream);
	return rc < 0 ? rc : ret;
}

/* ---- the devices of one process behind one call ------------------------------------------- */
struct jpegqs_cuda_multi {
	std::vector<jpegqs_cuda_ctx *> ctx;
	std::vector<jpegqs_cuda_link *> link;
	uint32_t max_wblk;
	long min_blocks;                      /* luma blocks a device must get before another one is added */
	char err[512];
};

static void multi_drop_links(jpegqs_cuda_multi *m) {
	for (jpegqs_cuda_link *l : m->link) jpegqs_cuda_link_destroy(l);
	m->link.clear(); m->max_wblk = 0;
}

extern "C" void jpegqs_cuda_multi_destroy(jpegqs_cuda_multi *m) {
	if (!m) return;
	multi_drop_links(m);
	for (jpegqs_cuda_ctx *c : m->ctx) jpegqs_cuda_destroy(c);
	delete m;
}

extern "C" int jpegqs_cuda_multi_create(int ndev, const int *devices, jpegqs_cuda_multi **out) {
	jpegqs_cuda_ctx *ctx = NULL;
	if (!out) return JPEGQS_ERR_ARG;
	*out = NULL;
	int have = 0;
	CK(cudaGetDeviceCount(&have));
	if (ndev <= 0) ndev = have;                          /* all devices */
	if (ndev < 1 || ndev > QS_MAX_RANKS || (!devices && ndev > have)) {
		snprintf(g_err, sizeof(g_err), "multi_create: %d device(s) asked for, %d present", ndev, have);
		return JPEGQS_ERR_ARG;
	}
	jpegqs_cuda_multi *m = new jpegqs_cuda_multi();
	m->max_wblk = 0; m->err[0] = 0;
	const char *e = getenv("JPEGQS_MIN_BLOCKS_PER_GPU");
	m->min_blocks = e ? atol(e) : 148L * 16 * 32;        /* one wave of the persistent smoothing kernel */
	for (int i = 0; i < ndev; i++) {
		jpegqs_cuda_ctx *c = NULL;
		int rc = jpegqs_cuda_create(devices ? devices[i] : i, &c);
		if (rc) { jpegqs_cuda_multi_destroy(m); return rc; }
		m->ctx.push_back(c);
	}
	*out = m;
	return 0;
}

extern "C" int jpegqs_cuda_multi_devices(const jpegqs_cuda_multi *m) { return m ? (int)m->ctx.size() : 0; }
extern "C" jpegqs_cuda_ctx *jpegqs_cuda_multi_ctx(jpegqs_cuda_multi *m, int i) {
	return m && i >= 0 && i < (int)m->ctx.size() ? m->ctx[i] : NULL;
}
extern "C" const char *jpegqs_cuda_multi_last_error(const jpegqs_cuda_multi *m) { return m ? m->err : g_err; }

/* MCU-row ranges, sizes differing by at most one (SURVEY.md 8e: slabs are MCU aligned, so the
 * chroma / luma / down-sampled planes of a slab line up) */
static void split_mcu_rows(int total, int world, int r, int *m0, int *m1) {
	int base = total / world, rem = total % world;
	*m0 = r * base + std::min(r, rem);
	*m1 = *m0 + base + (r < rem ? 1 : 0);
}

/* how many devices an image of this geometry is worth (the north star's "only when the
 * component is large enough to shard") */
extern "C" int jpegqs_cuda_multi_plan(const jpegqs_cuda_multi *m, const jpegqs_cuda_image *img) {
	if (!m || !img || img->ncomp < 1) return 0;
	int maxv = 1;
	for (int c = 0; c < img->ncomp; c++) maxv = std::max(maxv, (int)img->comp[c].v_samp);
	int mcu_rows = ((int)img->image_height + 8 * maxv - 1) / (8 * maxv);
	long blocks = (long)img->comp[0].wblk * img->comp[0].hblk;
	int use = (int)std::min<long>((long)m->ctx.size(), std::max<long>(1, blocks / std::max<long>(1, m->min_blocks)));
	use = std::min(use, mcu_rows);
	/* every rank needs at least one block row of every component (libjpeg geometry is not MCU padded) */
	while (use > 1) {
		bool ok = true;
		for (int r = 0; r < use && ok; r++) {
			int m0, m1; split_mcu_rows(mcu_rows, use, r, &m0, &m1);
			for (int c = 0; c < img->ncomp && ok; c++) {
				int v = img->comp[c].v_samp, H = (int)img->comp[c].hblk;
				ok = std::min(m1 * v, H) - std::min(m0 * v, H) >= 1;
			}
		}
		if (ok) break;
		use--;
	}
	return use;
}

extern "C" int jpegqs_cuda_run_host_multi(jpegqs_cuda_multi *m, jpegqs_cuda_image *img, int flags, int niter) {
	if (!m || !img || img->ncomp < 1 || img->ncomp > JPEGQS_CUDA_MAX_COMP) return JPEGQS_ERR_ARG;
	const int use = jpegqs_cuda_multi_plan(m, img);
	if (use <= 1) {
		int rc = jpegqs_cuda_run_host(m->ctx[0], img, flags, niter, 0, NULL, NULL);
		if (rc < 0) snprintf(m->err, sizeof(m->err), "%s", jpegqs_cuda_last_error(m->ctx[0]));
		return rc;
	}
	uint32_t maxw = 0; int maxv = 1;
	for (int c = 0; c < img->ncomp; c++) { maxw = std::max(maxw, img->comp[c].wblk); maxv = std::max(maxv, (int)img->comp[c].v_samp); }
	if ((int)m->link.size() != use || maxw > m->max_wblk) {
		multi_drop_links(m);
		for (int r = 0; r < use; r++) {
			jpegqs_cuda_link *l = NULL;
			int rc = jpegqs_cuda_link_create(m->ctx[r], r, use, maxw, &l);
			if (rc) { snprintf(m->err, sizeof(m->err), "%s", jpegqs_cuda_last_error(m->ctx[r])); multi_drop_links(m); return rc; }
			m->link.push_back(l);
		}
		int rc = jpegqs_cuda_link_connect_local(m->link.data(), use);
		if (rc) { snprintf(m->err, sizeof(m->err), "%s", jpegqs_cuda_last_error(m->ctx[0])); multi_drop_links(m); return rc; }
		m->max_wblk = maxw;
	}
	const int mcu_rows = ((int)img->image_height + 8 * maxv - 1) / (8 * maxv);
	std::vector<jpegqs_cuda_image> slab(use, *img);
	std::vector<jpegqs_cuda_slab> geom(use);
	for (int r = 0; r < use; r++) {
		int m0, m1; split_mcu_rows(mcu_rows, use, r, &m0, &m1);
		memset(&geom[r], 0, sizeof(geom[r]));
		geom[r].rank = r; geom[r].world = use;
		for (int c = 0; c < img->ncomp; c++) {
			const jpegqs_cuda_comp *src = &img->comp[c]; jpegqs_cuda_comp *d = &slab[r].comp[c];
			int v = src->v_samp, H = (int)src->hblk;
			int r0 = std::min(m0 * v, H), r1 = std::min(m1 * v, H);
			geom[r].row0[c] = (uint32_t)r0; geom[r].hblk_total[c] = src->hblk;
			d->hblk = (uint32_t)(r1 - r0);
			if (src->rows) d->rows = src->rows + r0;
			if (src->coef) d->coef = src->coef + (size_t)r0 * src->wblk * 64;
		}
		for (int c = 1; c <= 2 && c < img->ncomp; c++) {            /* luma-sized outputs of UPSAMPLE_UV */
			const jpegqs_cuda_comp *src = &img->comp[c]; jpegqs_cuda_comp *d = &slab[r].comp[c];
			if (src->rows_up) d->rows_up = src->rows_up + geom[r].row0[0];
			if (src->coef_up) d->coef_up = src->coef_up + (size_t)geom[r].row0[0] * img->comp[0].wblk * 64;
		}
	}
	/* one host thread per device: a rank's pull kernel waits for its neighbours' push kernels,
	 * which only get enqueued if their host threads run */
	std::vector<int> rc(use, 0);
	std::vector<std::thread> th;
	for (int r = 1; r < use; r++)
		th.emplace_back([&, r] { rc[r] = jpegqs_cuda_run_slab(m->ctx[r], m->link[r], &slab[r], &geom[r], flags, niter, 0, NULL); });
	rc[0] = jpegqs_cuda_run_slab(m->ctx[0], m->link[0], &slab[0], &geom[0], flags, niter, 0, NULL);
	for (std::thread &t : th) t.join();
	int out = 0;
	for (int pass = 0; pass < 2 && out >= 0; pass++)            /* a timeout is usually the echo of another rank's error */
		for (int r = 0; r < use; r++)
			if (rc[r] < 0 && out >= 0 && (pass == 1 || rc[r] != JPEGQS_ERR_TIMEOUT)) {
				out = rc[r]; snprintf(m->err, sizeof(m->err), "rank %d: %s", r, jpegqs_cuda_last_error(m->ctx[r]));
			}
	for (int r = 0; r < use && out >= 0; r++) if (rc[r] > out) out = rc[r];
	if (out < 0) { multi_drop_links(m); return out; }               /* sequence numbers may be out of step */
	for (int c = 0; c < img->ncomp; c++) memcpy(img->comp[c].quant, slab[0].comp[c].quant, sizeof(img->comp[c].quant));
	img->upsampled = slab[0].upsampled;
	return out;
}

/* ---- decode to RGB (SURVEY.md 8f row f2) --------------------------------------------------- */
extern "C" int jpegqs_cuda_render_rgb(jpegqs_cuda_ctx *ctx, const jpegqs_cuda_image *img, int on_device,
		uint8_t *rgb, void *stream) {
	if (!ctx || !img || !rgb) return JPEGQS_ERR_ARG;
	int nc = img->ncomp;
	if (nc != 1 && nc != 3) {
		snprintf(ctx->err, sizeof(ctx->err), "render_rgb supports 1 or 3 components (got %d)", nc);
		return JPEGQS_ERR_UNSUPPORTED;
	}
	CK(cudaSetDevice(ctx->device));
	cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
	int maxh = 1, maxv = 1;
	for (int c = 0; c < nc; c++) {
		if (img->comp[c].h_samp < 1 || img->comp[c].v_samp < 1 || !img->comp[c].coef) return JPEGQS_ERR_ARG;
		if (img->comp[c].h_samp > maxh) maxh = img->comp[c].h_samp;
		if (img->comp[c].v_samp > maxv) maxv = img->comp[c].v_samp;
	}
	size_t bytes = 0, rgb_bytes = (size_t)img->image_width * img->image_height * 3;
	for (int c = 0; c < nc; c++) {
		size_t cb = (size_t)img->comp[c].wblk * img->comp[c].hblk * 128;
		if (!on_device) bytes += align256(cb);
		bytes += align256(QS_PLANE_BYTES(img->comp[c].wblk, img->comp[c].hblk));
	}
	if (!on_device) bytes += align256(rgb_bytes);
	if (arena_reserve(ctx, bytes + 4096)) return JPEGQS_ERR_CUDA;
	if (quant_reserve(ctx, nc)) return JPEGQS_ERR_CUDA;
	std::vector<QsJob> jobs[2]; std::vector<QsQuantDev> q(nc);
	const uint8_t *planes[3]; int strides[3], cw[3], ch[3], hs[3], vs[3];
	for (int c = 0; c < nc; c++) {
		const jpegqs_cuda_comp *cc = &img->comp[c];
		size_t cb = (size_t)cc->wblk * cc->hblk * 128; int val;
		int16_t *cd = cc->coef;
		if (!on_device) {
			cd = (int16_t *)arena_take(ctx, cb);
			if (cb) CK(cudaMemcpyAsync(cd, cc->coef, cb, cudaMemcpyHostToDevice, st));
		}
		uint8_t *pl = (uint8_t *)arena_take(ctx, QS_PLANE_BYTES(cc->wblk, cc->hblk));
		quant_prepare(cc->quant, &q[c], &val);
		QsJob j; memset(&j, 0, sizeof(j));
		j.coef = cd; j.plane = pl; j.quant = ctx->quant_dev + c;
		j.wblk = cc->wblk; j.hblk = cc->hblk; j.stride = QS_PLANE_STRIDE(cc->wblk); j.nblocks = cc->wblk * cc->hblk;
		j.top_edge = j.bottom_edge = 1;
		/* tables that are not all ones: the coefficients are still quantized (plain decode).
		 * NOTE: on_device coefficients are de-quantized in place in that case. */
		jobs[cc->has_qtbl && val > 1 ? 1 : 0].push_back(j);
		planes[c] = pl; strides[c] = j.stride;
		cw[c] = (int)((img->image_width * (unsigned)cc->h_samp + maxh - 1) / maxh);
		ch[c] = (int)((img->image_height * (unsigned)cc->v_samp + maxv - 1) / maxv);
		hs[c] = maxh / cc->h_samp; vs[c] = maxv / cc->v_samp;
	}
	CK(cudaMemcpyAsync(ctx->quant_dev, q.data(), nc * sizeof(QsQuantDev), cudaMemcpyHostToDevice, st));
	ctx->jobs_cache[0].clear(); ctx->jobs_cache[1].clear();
	for (int m = 0; m < 2; m++) {
		if (jobs[m].empty()) continue;
		const QsJob *jd; int tiles;
		if (upload_jobs(ctx, m, jobs[m], st, &jd, &tiles)) return JPEGQS_ERR_CUDA;
		CK(cudaMemsetAsync(ctx->flags_dev, 0, jobs[m].size() * sizeof(int), st));
		CK(qs_launch_idct_pass(jd, (int)jobs[m].size(), tiles, m ? QS_IDCT_DEQUANT : 0, ctx->flags_dev, st));
	}
	uint8_t *out = on_device ? rgb : (uint8_t *)arena_take(ctx, rgb_bytes);
	CK(qs_launch_render_rgb(planes, strides, cw, ch, hs, vs, nc, (int)img->image_width, (int)img->image_height,
			img->is_ycbcr, out, st));
	if (!on_device) CK(cudaMemcpyAsync(rgb, out, rgb_bytes, cudaMemcpyDeviceToHost, st));
	CK(cudaStreamSynchronize(st));
	return 0;
}
