/*
 * qs_oracle.c - TEST INFRASTRUCTURE, not part of the product.
 *
 * A plain-C, scalar restatement of the reference's coefficient-smoothing hot
 * path (the -DNO_SIMD build of reference quantsmooth.h + idct.h), operating on
 * flat arrays instead of libjpeg structures.  It is the parity oracle that
 * travels to the GPU box; it is itself pinned against the real reference
 * (oracle/_ref/libqsref_scalar.so, built from /root/reference by
 * oracle/Makefile) by tests/test_oracle_vs_reference.py and against the golden
 * vectors under tests/golden/ (generated from the real reference by
 * tests/golden/make_golden.py).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may load this object.  The product never does.
 *
 * Arithmetic contract (SURVEY.md appendix A): all floats are IEEE binary32,
 * every + - * / individually rounded, no FMA contraction (build with
 * -ffp-contract=off, x86-64 SSE math); float->int conversions follow x86
 * cvttss2si (NaN / out of range -> INT_MIN).
 *
 * Every function cites the reference lines it restates.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <limits.h>
#include <stddef.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define QSO_DIAGONALS 1
#define QSO_JOINT_YUV 2
#define QSO_UPSAMPLE_UV 4
#define QSO_LOW_QUALITY 8
#define QSO_NO_REBALANCE 16
#define QSO_NO_REBALANCE_UV 32

/* zig-zag scan position -> natural (row-major) index; reference idct.h:24-33 */
static const unsigned char zz_to_natural[64] = {
	 0,  1,  8, 16,  9,  2,  3, 10, 17, 24, 32, 25, 18, 11,  4,  5,
	12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13,  6,  7, 14, 21, 28,
	35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
	58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63
};

/* x86 cvttss2si: truncation; NaN and |x| >= 2^31 give INT_MIN.
 * (reference relies on this implicitly at quantsmooth.h:1549, 557, 2380-2386, 2748) */
static int cvtt(float x) {
	if (!(x > -2147483904.0f && x < 2147483648.0f)) return INT_MIN;
	return (int)x;
}

/* ---- integer "islow" IDCT, reference idct.h:39-89 (constants, butterfly M3),
 *      469-538 (scalar passes, descale and clamp).  The reference's zero-AC
 *      shortcuts (idct.h:487-499, 520-532) are value-identical and omitted. */
enum { C0298 = 2446, C0390 = 3196, C0541 = 4433, C0765 = 6270, C0899 = 7373, C1175 = 9633,
	C1501 = 12299, C1847 = 15137, C1961 = 16069, C2053 = 16819, C2562 = 20995, C3072 = 25172 };

static void islow_1d(const int32_t in[8], int32_t out[8]) {
	int32_t z1, z2, z3, z4, z5, e0, e1, e2, e3, t0, t1, t2, t3, a, b;
	z2 = in[2]; z3 = in[6];
	z1 = (z2 + z3) * C0541;
	a = z1 - z3 * C1847; b = z1 + z2 * C0765;
	t0 = (in[0] + in[4]) * 8192; t1 = (in[0] - in[4]) * 8192;   /* << CONST_BITS */
	e0 = t0 + b; e3 = t0 - b; e1 = t1 + a; e2 = t1 - a;
	t0 = in[7]; t1 = in[5]; t2 = in[3]; t3 = in[1];
	z1 = t0 + t3; z2 = t1 + t2; z3 = t0 + t2; z4 = t1 + t3;
	z5 = (z3 + z4) * C1175;
	t0 *= C0298; t1 *= C2053; t2 *= C3072; t3 *= C1501;
	z1 *= C0899; z2 *= C2562; z3 *= C1961; z4 *= C0390;
	z3 = z5 - z3; z4 = z5 - z4;
	t0 += z3 - z1; t1 += z4 - z2; t2 += z3 - z2; t3 += z4 - z1;
	out[0] = e0 + t3; out[7] = e0 - t3; out[1] = e1 + t2; out[6] = e1 - t2;
	out[2] = e2 + t1; out[5] = e2 - t1; out[3] = e3 + t0; out[4] = e3 - t0;
}

void qso_idct_islow(const int16_t *coef, uint8_t *out, int stride) {
	int32_t ws[64], in[8], o[8]; int x, y, k;
	for (x = 0; x < 8; x++) {                       /* pass 1: columns, idct.h:483-502 */
		for (k = 0; k < 8; k++) in[k] = coef[k * 8 + x];
		islow_1d(in, o);
		for (k = 0; k < 8; k++) ws[k * 8 + x] = (o[k] + 1024) >> 11;   /* DESCALE(.,13-2) */
	}
	for (y = 0; y < 8; y++) {                       /* pass 2: rows, idct.h:506-537 */
		islow_1d(ws + y * 8, o);
		for (k = 0; k < 8; k++) {
			int32_t v = (o[k] + (257 << 17)) >> 18;       /* (x + ((256+1) << 17)) >> 18 */
			out[y * stride + k] = v < 0 ? 0 : v > 255 ? 255 : v;
		}
	}
}

/* ---- float LL&M IDCT used only to build the weight tables; reference idct.h:565-604 */
static void idctf_1d(const float *in, int is, float *out, int os, float scale, int use_scale) {
	float t0, t1, t2, t3, t4, t5, t6, t7, z1, z2, z3, z4, z5, r[8]; int k;
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
	for (k = 0; k < 8; k++) out[k * os] = use_scale ? r[k] * scale : r[k];
}

void qso_idct_float(const float *in, float *out) {
	float ws[64]; int i;
	for (i = 0; i < 8; i++) idctf_1d(in + i, 8, ws + i, 8, 0, 0);       /* columns, unscaled */
	for (i = 0; i < 8; i++) idctf_1d(ws + i * 8, 1, out + i * 8, 1, 0.125f, 1);  /* rows, x0.125 */
}

/* ---- float LL&M FDCT; reference idct.h:606-628 (op order M3), 896-915 (scalar passes) */
static void fdctf_1d(const float *in, int is, float *out, int os, int scale) {
	float t0, t1, t2, t3, t4, t5, t6, t7, z1, z2, z3, z4, z5, r[8]; int k;
	z1 = in[0]; z2 = in[7 * is]; t0 = z1 + z2; t7 = z1 - z2;
	z1 = in[1 * is]; z2 = in[6 * is]; t1 = z1 + z2; t6 = z1 - z2;
	z1 = in[2 * is]; z2 = in[5 * is]; t2 = z1 + z2; t5 = z1 - z2;
	z1 = in[3 * is]; z2 = in[4 * is]; t3 = z1 + z2; t4 = z1 - z2;
	z1 = t0 + t3; z4 = t0 - t3; z2 = t1 + t2; z3 = t1 - t2;
	r[0] = z1 + z2; r[4] = z1 - z2;
	z1 = (z3 + z4) * 0.541196100f;
	r[2] = z1 + z4 * 0.765366865f;
	r[6] = z1 - z3 * 1.847759065f;
	z1 = t4 + t7; z2 = t5 + t6; z3 = t4 + t6; z4 = t5 + t7;
	z5 = (z3 + z4) * 1.175875602f;
	t4 = t4 * 0.298631336f; t5 = t5 * 2.053119869f;
	t6 = t6 * 3.072711026f; t7 = t7 * 1.501321110f;
	z1 = z1 * 0.899976223f; z2 = z2 * 2.562915447f;
	z3 = z3 * 1.961570560f - z5;
	z4 = z4 * 0.390180644f - z5;
	r[7] = t4 - (z1 + z3); r[5] = t5 - (z2 + z4);
	r[3] = t6 - (z2 + z3); r[1] = t7 - (z1 + z4);
	for (k = 0; k < 8; k++) out[k * os] = scale ? r[k] * 0.125f : r[k];
}

void qso_fdct_float(const float *in, float *out) {
	float ws[64]; int i;
	for (i = 0; i < 8; i++) fdctf_1d(in + i, 8, ws + i, 8, 0);
	for (i = 0; i < 8; i++) fdctf_1d(ws + i * 8, 1, out + i * 8, 1, 1);
}

/* ---- weight tables, reference quantsmooth.h:251-301.  out[i*size ..] for natural
 *      coefficient index i; size = 160, or 272 with DIAGONALS.  Layout per coefficient:
 *      [0,64) horizontal pair diffs, [64,96) top/bottom/left/right edge * bcoef,
 *      [96,160) vertical pair diffs, [160,272) 7 rows x {8 "\" diffs, 8 "/" diffs}. */
int qso_table_size(int flags) { return flags & QSO_DIAGONALS ? 272 : 160; }

void qso_tables(int flags, float *out) {
	int i, x, y, size = qso_table_size(flags);
	float bcoef = flags & QSO_DIAGONALS ? 4.0f : 2.0f;
	for (i = 0; i < 64; i++) {
		float e[64], B[64], *t = out + i * size;
		memset(e, 0, sizeof(e)); e[i] = 1.0f;
		qso_idct_float(e, B);
		for (y = 0; y < 8; y++) for (x = 0; x < 8; x++) {
			t[y * 8 + x] = x < 7 ? B[y * 8 + x] - B[y * 8 + x + 1] : 0.0f;
			t[96 + y * 8 + x] = y < 7 ? B[y * 8 + x] - B[(y + 1) * 8 + x] : 0.0f;
		}
		for (x = 0; x < 8; x++) {
			t[64 + x] = B[x] * bcoef;           /* top row    */
			t[72 + x] = B[56 + x] * bcoef;      /* bottom row */
			t[80 + x] = B[x * 8] * bcoef;       /* left col   */
			t[88 + x] = B[x * 8 + 7] * bcoef;   /* right col  */
		}
		if (flags & QSO_DIAGONALS) for (y = 0; y < 7; y++) {
			float *d = t + 160 + y * 16;
			for (x = 0; x < 7; x++) {
				d[x] = B[y * 8 + x] - B[(y + 1) * 8 + x + 1];
				d[8 + x] = B[y * 8 + x + 1] - B[(y + 1) * 8 + x];
			}
			d[7] = d[15] = 0.0f;
		}
	}
}

/* ---- quant table preparation, reference quantsmooth.h:2497-2511.
 *      q[i] = quantval with 0 replaced by 1.  Returns the OR of the raw values. */
int qso_quant_prepare(const uint16_t *raw, uint16_t *q) {
	int i, val = 0;
	for (i = 0; i < 64; i++) { val |= raw[i]; q[i] = raw[i] ? raw[i] : 1; }
	return val;
}

/* ---- original (quantized) coefficient value a0 = round_half_away(c / q) * q.
 *      Plain form, reference quantsmooth.h:338-341; SURVEY.md 8(a8) shows it equals the
 *      reciprocal form (324-337) exhaustively for q in [1,2047], c in [-0x4000,0x3fff]. */
static int orig_coef(int c, int q) {
	int h = q >> 1;
	return (c + (c < 0 ? -h : h)) / q * q;
}
int qso_orig_coef(int c, int q) { return orig_coef(c, q); }

static void clamp_bounds(int a0, int q, int *dl, int *dh) {   /* quantsmooth.h:1555-1556 */
	int d0 = (q - 1) >> 1, d1 = q >> 1;
	*dh = a0 + (a0 < 0 ? d1 : d0);
	*dl = a0 - (a0 > 0 ? d1 : d0);
}

/* ---- fdct_clamp, reference quantsmooth.h:343-347, 551-561 (scalar) */
void qso_fdct_clamp(float *buf, int16_t *coef, const uint16_t *q) {
	int x;
	qso_fdct_float(buf, buf);
	for (x = 0; x < 64; x++) {
		int dl, dh, add, a0 = orig_coef(coef[x], q[x]);
		clamp_bounds(a0, q[x], &dl, &dh);
		add = cvtt(roundf(buf[x]));
		if (add > dh) add = dh;
		if (add < dl) add = dl;
		coef[x] = (int16_t)add;
	}
}

/* ---- 3x3 luma/chroma regression shared by JOINT_YUV (quantsmooth.h:894-913) and
 *      upsample_row (2134-2155): weights centre 4, axial 2, diagonal 1. */
static float regress_scale(const uint8_t *A, const uint8_t *B, int stride, int32_t *psA, int32_t *psB) {
	int32_t sA = 0, sB = 0, sAA = 0, sAB = 0; float scale;
#define TAP(dx, dy) { int a = A[(dy) * stride + (dx)], b = B[(dy) * stride + (dx)]; \
	sA += a; sAA += a * a; sB += b; sAB += a * b; }
#define DBL sA += sA; sB += sB; sAA += sAA; sAB += sAB;
	TAP(0, 0) DBL
	TAP(0, -1) TAP(-1, 0) TAP(1, 0) TAP(0, 1) DBL
	TAP(-1, -1) TAP(1, -1) TAP(-1, 1) TAP(1, 1)
#undef TAP
#undef DBL
	sAA = sAA * 16 - sA * sA;
	sAB = sAB * 16 - sA * sB;
	scale = (float)sAA;
	if (sAA) scale = (float)sAB / scale;
	scale = scale < -16.0f ? -16.0f : scale;
	scale = scale > 16.0f ? 16.0f : scale;
	*psA = sA; *psB = sB;
	return scale;
}

/* ---- quantsmooth_block, reference quantsmooth.h:564-1849 (scalar branches:
 *      JOINT_YUV 894-921, main loop 1396-1409 + 1517-1565, rebalance 1566-1568 + 1823-1848).
 *      image  -> top-left pixel of this block in the component's sample plane
 *      image2 -> same position in the down-sampled luma plane, or NULL
 *      tables -> qso_tables() output (unused with LOW_QUALITY, quantsmooth.h:924-938, 1162-1178). */
/* measurement probe (tools/refresh_stats.py): per block, bit s-1 = "a coefficient of
 * anti-diagonal s changed in the last pass", i.e. the reference's need_refresh at the start of
 * the next diagonal.  Off unless qso_set_change_probe was called. */
static const int16_t *probe_base; static uint16_t *probe_out;
void qso_set_change_probe(const int16_t *coef_base, uint16_t *out) { probe_base = coef_base; probe_out = out; }

void qso_smooth_block(int16_t *coef, const uint16_t *q, const uint8_t *image,
		const uint8_t *image2, int stride, int flags, const float *tables, int luma) {
	uint8_t buf[64], border[32]; int k, x, y, need_refresh = 1;
	int tsize = qso_table_size(flags);
	unsigned probe_mask = 0;

	if (image2) {                                             /* 577-579, 894-921 */
		float fbuf[64];
		for (y = 0; y < 8; y++) for (x = 0; x < 8; x++) {
			int32_t sA, sB; float a;
			float scale = regress_scale(image2 + y * stride + x, image + y * stride + x, stride, &sA, &sB);
			a = ((float)(image2[y * stride + x] * 16 - sA) * scale + (float)sB) * (1.0f / 16);
			a = (a < 0 ? 0 : a) - 128;
			fbuf[y * 8 + x] = a > 128 ? 128 : a;
		}
		qso_fdct_clamp(fbuf, coef, q);
	}

	if (flags & QSO_LOW_QUALITY) {                            /* 924-938, 1162-1178 (scalar) */
		if (!image2) {
			float fbuf[64], range = 0, c0 = 2, c1 = c0 * sqrtf(0.5f); int sum = 0;
			for (x = 1; x < 64; x++) {
				int a = coef[x]; a = a < 0 ? -a : a;
				range = range + (float)(q[x] * a); sum += a;
			}
			if (sum) range = range * (4.0f / (float)sum);
			if (range > 128) range = 128;
			range = roundf(range);
			for (y = 0; y < 8; y++) for (x = 0; x < 8; x++) {
				int a = image[y * stride + x]; float a0 = 0, an = 0;
#define NB(c_, dx, dy) { float t0 = (float)(a - image[(y + (dy)) * stride + x + (dx)]), t = range - fabsf(t0), aw; \
	t = t < 0 ? 0 : t; t = t * t; aw = (c_) * t; a0 = a0 + t0 * t * aw; an = an + aw * aw; }
				NB(c1, -1, -1) NB(c0, 0, -1) NB(c1, 1, -1)
				NB(c0, -1, 0) NB(c0, 1, 0)
				NB(c1, -1, 1) NB(c0, 0, 1) NB(c1, 1, 1)
#undef NB
				if (an > 0.0f) a = cvtt((float)a - a0 / an);   /* int a -= float: truncates */
				fbuf[y * 8 + x] = (float)(a - 128);
			}
			qso_fdct_clamp(fbuf, coef, q);
		}
		goto rebalance;
	}

	for (x = 0; x < 8; x++) {                                 /* 1396-1401 */
		border[x] = image[x - stride];                        /* above        */
		border[8 + x] = image[x + stride * 8];                /* below        */
		border[16 + x] = image[x * stride - 1];               /* left         */
		border[24 + x] = image[x * stride + 8];               /* right        */
	}

	for (k = 63; k > 0; k--) {                                /* 1403 */
		int i = zz_to_natural[k], r;
		const float *tab = tables + i * tsize;
		float a2 = 0, a3 = 0, R = (float)(q[i] * 2);
		/* zigzag_refresh (313-322) is 1 exactly at the first-visited coefficient of each
		 * anti-diagonal, i.e. where the previous scan position lies on another diagonal */
		int first_of_diag = k == 63 || ((zz_to_natural[k + 1] >> 3) + (zz_to_natural[k + 1] & 7)) != ((i >> 3) + (i & 7));
		if (need_refresh && first_of_diag) { qso_idct_islow(coef, buf, 8); need_refresh = 0; }

#define TERM(d_, w_) { float a0 = (float)(d_), a1 = (w_), t = R - fabsf(a0); \
	t = t < 0 ? 0 : t; t = t * t; a0 = a0 * t; a1 = a1 * t; a2 = a2 + a0 * a1; a3 = a3 + a1 * a1; }
		if (i & 7) for (y = 0; y < 8; y++) for (x = 0; x < 7; x++)         /* 1527 */
			TERM(buf[y * 8 + x] - buf[y * 8 + x + 1], tab[y * 8 + x])
		for (x = 0; x < 8; x++) TERM(buf[x] - border[x], tab[64 + x])            /* 1529 */
		for (x = 0; x < 8; x++) TERM(buf[56 + x] - border[8 + x], tab[72 + x])
		for (y = 0; y < 8; y++) TERM(buf[y * 8] - border[16 + y], tab[80 + y])   /* 1530 */
		for (y = 0; y < 8; y++) TERM(buf[y * 8 + 7] - border[24 + y], tab[88 + y])
		if (i > 7) for (y = 0; y < 7; y++) for (x = 0; x < 8; x++)          /* 1531 */
			TERM(buf[y * 8 + x] - buf[y * 8 + 8 + x], tab[96 + y * 8 + x])
		if (flags & QSO_DIAGONALS) for (y = 0; y < 7; y++) for (x = 0; x < 7; x++) {  /* 1533-1540 */
			TERM(buf[y * 8 + x] - buf[y * 8 + 9 + x], tab[160 + y * 16 + x])
			TERM(buf[y * 8 + x + 1] - buf[y * 8 + 8 + x], tab[160 + y * 16 + 8 + x])
		}
#undef TERM
		r = cvtt(roundf(a2 / a3));                                            /* 1548-1549 */
		if (r) {                                                              /* 1551-1564 */
			int c = coef[i], dl, dh, add, a0 = orig_coef(c, q[i]);
			clamp_bounds(a0, q[i], &dl, &dh);
			add = (int)((unsigned)c - (unsigned)r);   /* wraps like the reference's int subtract */
			if (add > dh) add = dh;
			if (add < dl) add = dl;
			coef[i] = (int16_t)add;
			need_refresh |= add ^ c;
			if (add != c) probe_mask |= 1u << ((i >> 3) + (i & 7) - 1);
		}
	}
	if (probe_out) probe_out[(coef - probe_base) / 64] = (uint16_t)probe_mask;

rebalance:
	if (flags & QSO_NO_REBALANCE) return;                                     /* 1566-1568 */
	if (!luma && (flags & QSO_NO_REBALANCE_UV)) return;
	{                                                                         /* 1823-1848 */
		int orig[64]; int64_t m0 = 0, m1 = 0;
		for (k = 1; k < 64; k++) {
			int a0 = orig_coef(coef[k], q[k]);
			orig[k] = a0; m0 += coef[k] * a0; m1 += a0 * a0;
		}
		if (m1 > m0) {
			int mul = (int)(((m1 << 13) + (m0 >> 1)) / m0);
			for (k = 1; k < 64; k++) {
				int dl, dh, add;
				clamp_bounds(orig[k], q[k], &dl, &dh);
				add = (coef[k] * mul + 0x1000) >> 13;
				if (add > dh) add = dh;
				if (add < dl) add = dl;
				coef[k] = (int16_t)add;
			}
		}
	}
}

/* ---- one 8-row band of upsample_row, reference quantsmooth.h:1851-1865, 2134-2158
 *      (scale), 2364-2389 (emit).  Planes are addressed WITHOUT their border offset:
 *      C/Yd: chroma plane / down-sampled luma, pixel (0,0) at [0], 1-px border around;
 *      Yf: full-resolution luma likewise.  Writes rows [y0*hs, y1*hs) x [0, w1*ws) of mem. */
static void upsample_band(int w1, int y0, int y1, const uint8_t *C, const uint8_t *Yd, int stride,
		const uint8_t *Yf, int stride1, uint8_t *mem, int st, int ws, int hs) {
	int x, y, xx, yy;
	for (y = y0; y < y1; y++) for (x = 0; x < w1; x++) {
		int32_t sA, sB;
		float scale = regress_scale(Yd + y * stride + x, C + y * stride + x, stride, &sA, &sB);
		float offset = (float)C[y * stride + x] - (float)Yd[y * stride + x] * scale + 0.5f;
		for (yy = 0; yy < hs; yy++) for (xx = 0; xx < ws; xx++) {
			int a = cvtt((float)Yf[(y * hs + yy) * stride1 + x * ws + xx] * scale + offset);
			mem[(y * hs + yy) * st + x * ws + xx] = a < 0 ? 0 : a > 255 ? 255 : a;
		}
	}
}

/* ------------------------------------------------------------------------------------
 * Image driver: flat restatement of do_quantsmooth, reference quantsmooth.h:2404-2878.
 * ------------------------------------------------------------------------------------ */
typedef struct {
	int16_t *coef;              /* [hblk][wblk][64], quantized in, smoothed out (in place) */
	uint32_t wblk, hblk;
	int h_samp, v_samp;
	int has_qtbl;               /* 0: component has no quant table -> skipped (2494)       */
	uint16_t quant[64];         /* raw quantval; overwritten with 1 on return (2851-2859)  */
	int16_t *coef_up;           /* out: luma-sized buffer for UPSAMPLE_UV (may be NULL if unused) */
} qso_comp;

typedef struct {
	int ncomp, is_ycbcr;
	uint32_t image_width, image_height;
	qso_comp comp[4];
	int upsampled;              /* out: 1 when comp[1,2] results live in coef_up at luma dims */
} qso_image;

typedef int (*qso_progress_fn)(void *data, int cur, int max);

#define PLANE(p, st, x, y) ((p) + ((y) + 1) * (size_t)(st) + (x) + 1)

static uint8_t *plane_alloc(uint32_t wblk, uint32_t hblk, int *stride) {
	*stride = wblk * 8 + 8;                                             /* 2545 */
	return (uint8_t*)malloc(((size_t)hblk * 8 + 2) * *stride + 8);
}

static void plane_borders(uint8_t *p, int st, int w, int h) {           /* 2612-2620 */
	int y;
	for (y = 1; y < h + 1; y++) { p[y * (size_t)st] = p[y * (size_t)st + 1]; p[y * (size_t)st + w + 1] = p[y * (size_t)st + w]; }
	memcpy(p, p + st, st);
	memcpy(p + (size_t)(h + 1) * st, p + (size_t)h * st, st);
}

int qso_run(qso_image *im, int flags, int niter, int progprec, qso_progress_fn progress, void *userdata) {
	int ci, stop = 0, need_downsample = 0, stride = 0, stride1 = 0, stride2 = 0;
	uint8_t *image1 = NULL, *image2 = NULL;   /* full-res Y, down-sampled Y (2753-2815) */
	int prog_next = 0, prog_max = 0, prog_thr = 0;
	float *tables;
	im->upsampled = 0;

	if ((flags & (QSO_JOINT_YUV | QSO_UPSAMPLE_UV)) && im->is_ycbcr && im->ncomp >= 3 &&    /* 2447-2453 */
			im->comp[1].h_samp == 1 && im->comp[1].v_samp == 1 &&
			im->comp[2].h_samp == 1 && im->comp[2].v_samp == 1) need_downsample = 1;
	if (niter < 0) niter = 0;
	if (niter > 100) niter = 100;
	if (niter <= 0 && !((flags & QSO_UPSAMPLE_UV) && need_downsample)) return 0;   /* 2458 */

	tables = (float*)malloc(64 * sizeof(float) * qso_table_size(flags));
	qso_tables(flags, tables);

	if (progress) {                                                     /* 2474-2482 */
		for (ci = 0; ci < im->ncomp; ci++) prog_max += im->comp[ci].hblk * im->comp[ci].v_samp * niter;
		if (progprec == 0) progprec = 20;
		if (progprec < 0) progprec = prog_max;
		prog_thr = (unsigned)(prog_max + progprec - 1) / (unsigned)progprec;
	}

	for (ci = 0; ci < im->ncomp; ci++) {                                /* 2484 */
		qso_comp *c = &im->comp[ci];
		uint16_t q[64]; uint8_t *image = NULL;
		int W = c->wblk, H = c->hblk, iter, val, niter2 = niter, extra = 0;
		int prog_cur = prog_next, prog_inc = c->v_samp;
		int luma = !ci || !im->is_ycbcr;                                /* 2639 */
		int64_t by;
		prog_next += H * prog_inc * niter;
		if (!c->has_qtbl) continue;
		if (image1 || (!ci && need_downsample)) extra = 1;              /* 2495 */
		val = qso_quant_prepare(c->quant, q);
		if (val <= 1) niter2 = 0;                                       /* 2501 */
		if (val >= 0x800) stop = 1;                                     /* 2504 */
		if (niter2 + extra == 0) continue;                              /* 2542 */
		if (!stop) image = plane_alloc(W, H, &stride);
		if (!image) {                                                   /* 2551-2566: dequantize only */
			for (by = 0; by < (int64_t)H * W * 64; by++)
				c->coef[by] = (int16_t)(c->coef[by] * c->quant[by & 63]);
			continue;
		}
		for (iter = 0; iter < niter2 + extra; iter++) {                 /* 2580 */
			int bad = 0;
#pragma omp parallel for schedule(dynamic) reduction(|:bad)
			for (by = 0; by < H; by++) {                                /* 2589-2609 */
				int bx, k;
				for (bx = 0; bx < W; bx++) {
					int16_t *cf = c->coef + ((size_t)by * W + bx) * 64;
					if (!iter) for (k = 0; k < 64; k++) {
						int t = cf[k] * c->quant[k];
						cf[k] = (int16_t)t;
						if ((t + 0x800) >> 12) bad = 1;
					}
					qso_idct_islow(cf, PLANE(image, stride, bx * 8, by * 8), stride);
				}
			}
			if (bad) { stop = 1; break; }                               /* 2610 */
			plane_borders(image, stride, W * 8, H * 8);
			if (iter == niter2) break;                                  /* 2622 */
#pragma omp parallel for schedule(dynamic)
			for (by = 0; by < H; by++) {                                /* 2627-2640 */
				int bx;
				for (bx = 0; bx < W; bx++)
					qso_smooth_block(c->coef + ((size_t)by * W + bx) * 64, q,
							PLANE(image, stride, bx * 8, by * 8),
							image2 && (flags & QSO_JOINT_YUV) ? PLANE(image2, stride2, bx * 8, by * 8) : NULL,
							stride, flags, tables, luma);
			}
			if (progress) {                                             /* 2656-2664 */
				int cur = prog_cur += H * prog_inc;
				if (cur >= prog_thr) {
					cur = (int)((int64_t)progprec * cur / prog_max);
					prog_thr = (int)(((int64_t)(cur + 1) * prog_max + progprec - 1) / progprec);
					stop = progress(userdata, cur, progprec);
				}
				if (stop) break;
			}
		}
		for (by = 0; by < (int64_t)H * W * 64; by++) {                  /* 2670-2689 */
			int a = c->coef[by];
			c->coef[by] = (int16_t)(a > 1023 ? 1023 : a < -1023 ? -1023 : a);
		}

		if (!stop && image1) {                                          /* 2691-2752 */
			int ws = im->comp[0].h_samp, hs = im->comp[0].v_samp;
			int w1 = (im->image_width + ws - 1) / ws, h1 = (im->image_height + hs - 1) / hs;
			int W0 = im->comp[0].wblk, H0 = im->comp[0].hblk, ww = W0 * 8, hh = H0 * 8;
			int st = ((w1 + 8) & -8) * ws, h2 = ((h1 + 8) & -8) * hs, y;
			uint8_t *mem = (uint8_t*)calloc((size_t)h2, st);
			if (mem && c->coef_up) {
#pragma omp parallel for schedule(dynamic)
				for (y = 0; y < h1; y += 8)
					upsample_band(w1, y, y + 8 < h1 ? y + 8 : h1, PLANE(image, stride, 0, 0),
							PLANE(image2, stride2, 0, 0), stride, PLANE(image1, stride1, 0, 0), stride1,
							mem, st, ws, hs);
				/* right edge: replicate the last produced column (intent of 2390-2393; the
				 * reference only does this for the first band - see DESIGN.md "reference
				 * quirks"; shapes with w1*ws == ww, i.e. all BASELINE configs, are unaffected) */
				for (y = 0; y < h1 * hs; y++) { int x; for (x = w1 * ws; x < ww; x++) mem[(size_t)y * st + x] = mem[(size_t)y * st + w1 * ws - 1]; }
				for (y = h1 * hs; y < hh; y++) memcpy(mem + (size_t)y * st, mem + (size_t)(h1 * hs - 1) * st, st);  /* 2729-2730 */
#pragma omp parallel for schedule(dynamic)
				for (by = 0; by < H0; by++) {                           /* 2735-2750 */
					int bx, x, yy;
					for (bx = 0; bx < W0; bx++) {
						float fb[64]; int16_t *cf = c->coef_up + ((size_t)by * W0 + bx) * 64;
						for (yy = 0; yy < 8; yy++) for (x = 0; x < 8; x++)
							fb[yy * 8 + x] = (float)(mem[(size_t)(by * 8 + yy) * st + bx * 8 + x] - 128);
						qso_fdct_float(fb, fb);
						for (x = 0; x < 64; x++) cf[x] = (int16_t)cvtt(roundf(fb[x]));
					}
				}
			}
			free(mem);
		} else if (!stop && !ci && need_downsample) {                   /* 2753-2815 */
			int ws = c->h_samp, hs = c->v_samp;
			if (ws == 1 && hs == 1) { image2 = image; stride2 = stride; }
			else {
				int w = im->comp[1].wblk * 8, h = im->comp[1].hblk * 8, st = w + 8, x, y;
				int w1 = (W * 8 + ws - 1) / ws, h1 = (H * 8 + hs - 1) / hs;
				if (flags & QSO_UPSAMPLE_UV) { image1 = image; stride1 = stride; }
				image2 = (uint8_t*)malloc(((size_t)h + 2) * st + 8); stride2 = st;
				for (y = 0; y < h1; y++) {                              /* 2787-2802 (2774-2785 is its 2x2 case) */
					int h2 = H * 8 - y * hs; h2 = h2 < hs ? h2 : hs;
					for (x = 0; x < w1; x++) {
						const uint8_t *p = PLANE(image, stride, x * ws, y * hs);
						int xx, yy, sum = 0, w2 = W * 8 - x * ws, div;
						w2 = w2 < ws ? w2 : ws; div = w2 * h2;
						for (yy = 0; yy < h2; yy++) for (xx = 0; xx < w2; xx++) sum += p[yy * stride + xx];
						*PLANE(image2, st, x, y) = (uint8_t)((sum + div / 2) / div);
					}
				}
				for (y = 1; y < h1 + 1; y++) {                          /* 2805-2813 */
					uint8_t a = image2[(size_t)y * st + w1];
					image2[(size_t)y * st] = image2[(size_t)y * st + 1];
					for (x = w1 + 1; x < w + 2; x++) image2[(size_t)y * st + x] = a;
				}
				memcpy(image2, image2 + st, st);
				for (y = h1 + 1; y < h + 2; y++) memcpy(image2 + (size_t)y * st, image2 + (size_t)h1 * st, st);
			}
		}
		if (image != image1 && image != image2) free(image);            /* 2817 */
	}

	free(tables);
	if (image1 && !stop) im->upsampled = 1;                             /* 2835-2849 (dims rewritten by caller) */
	if (image2) free(image2);                                           /* 2831-2832 */
	if (image1) free(image1);
	for (ci = 0; ci < im->ncomp; ci++) {                                /* 2851-2859 */
		int k; if (im->comp[ci].has_qtbl) for (k = 0; k < 64; k++) im->comp[ci].quant[k] = 1;
	}
	return stop;
}

int qso_num_procs(void) {
#ifdef _OPENMP
	return omp_get_num_procs();
#else
	return 1;
#endif
}
void qso_set_threads(int n) {
#ifdef _OPENMP
	omp_set_num_threads(n > 0 ? n : omp_get_num_procs());
#else
	(void)n;
#endif
}
