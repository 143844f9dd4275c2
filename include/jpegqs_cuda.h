/*
 * jpegqs_cuda.h - C ABI of the B200 (sm_100a) back end of libjpegqs.
 *
 * This is the boundary between the libjpeg-facing host code (csrc/do_quantsmooth.c, which
 * keeps the reference's own entry points of libjpegqs.h) and the CUDA implementation.  It
 * occupies the slot of the reference's per-ISA workers do_quantsmooth_{base,sse2,avx2,avx512}
 * (reference libjpegqs.c:38-58, selected at libjpegqs.c:80-156): plain pointers and sizes,
 * no libjpeg types, no C++/torch types.  Every entry point cites the reference code it
 * replaces.  There is NO CPU fallback behind these calls: without a usable CUDA device they
 * fail with a negative return code.
 *
 * Layouts
 *   coefficients  int16 [hblk][wblk][64], natural (row-major) order inside a block - exactly
 *                 libjpeg's JBLOCKROW rows laid end to end (jpeglib.h JBLOCK / JCOEF).
 *   quant         the raw UINT16 quantval[64] of the component's JQUANT_TBL.
 */
#ifndef JPEGQS_CUDA_H
#define JPEGQS_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JPEGQS_CUDA_MAX_COMP 10        /* libjpeg MAX_COMPONENTS */

/* error codes (all negative); >= 0 return values are the reference's `stop` value */
#define JPEGQS_ERR_CUDA  (-1)          /* CUDA runtime failure, see jpegqs_cuda_last_error */
#define JPEGQS_ERR_ARG   (-2)          /* malformed arguments */
#define JPEGQS_ERR_UNSUPPORTED (-3)    /* a knob of a measurement build asked of the shipped library */
#define JPEGQS_ERR_TIMEOUT (-4)        /* sharded run: a peer rank did not answer (see last_error) */

typedef struct jpegqs_cuda_ctx jpegqs_cuda_ctx;

/* One colour component as do_quantsmooth sees it: fields of jpeg_component_info that the
 * reference reads at quantsmooth.h:2484-2494 plus its coefficient array. */
typedef struct {
	int16_t *coef;          /* in: quantized; out: de-quantized + smoothed (in place)     */
	uint32_t wblk, hblk;    /* width_in_blocks, height_in_blocks                          */
	int32_t h_samp, v_samp; /* h_samp_factor, v_samp_factor                               */
	int32_t has_qtbl;       /* 0 when compptr->quant_table == NULL (component skipped)    */
	uint16_t quant[64];     /* raw quantval; overwritten with 1 on return (2851-2859)     */
	int16_t *coef_up;       /* out, comps 1..2 only: luma-sized array filled when
	                           UPSAMPLE_UV replaces the chroma arrays (2691-2752); may be
	                           NULL when UPSAMPLE_UV cannot trigger                        */
	/* Host entry points only - libjpeg's own layout: hblk pointers to block rows of wblk*64
	 * coefficients each, rows not necessarily adjacent (access_virt_barray, quantsmooth.h:
	 * 2592-2594).  When rows != NULL it replaces coef (which may be NULL), rows_up likewise
	 * replaces coef_up: the library gathers the rows into its pinned staging memory band by band
	 * on worker threads, overlapped with the uploads, and scatters the results back the same
	 * way.  The row memory must stay valid and untouched by the caller during the call. */
	int16_t **rows;
	int16_t **rows_up;
} jpegqs_cuda_comp;

typedef struct {
	int32_t ncomp;
	int32_t is_ycbcr;                   /* jpeg_color_space == JCS_YCbCr                   */
	uint32_t image_width, image_height;
	jpegqs_cuda_comp comp[JPEGQS_CUDA_MAX_COMP];
	int32_t upsampled;                  /* out: 1 = comps 1,2 now live in coef_up at the
	                                       luma geometry with 1x1 sampling (2835-2849)     */
} jpegqs_cuda_image;

typedef int (*jpegqs_cuda_progress_fn)(void *userdata, int cur, int max);

/* ---- context -------------------------------------------------------------------------- */
/* device < 0: the current CUDA device.  Returns 0 or a negative error code. */
int jpegqs_cuda_create(int device, jpegqs_cuda_ctx **out);
void jpegqs_cuda_destroy(jpegqs_cuda_ctx *ctx);
const char *jpegqs_cuda_last_error(const jpegqs_cuda_ctx *ctx);   /* ctx may be NULL */
const char *jpegqs_cuda_device_name(const jpegqs_cuda_ctx *ctx);
/* device time (CUDA events) of the kernels of the last run_* call, milliseconds */
float jpegqs_cuda_last_device_ms(const jpegqs_cuda_ctx *ctx);
/* number of kernel launches issued by the last run_* call */
int jpegqs_cuda_last_launches(const jpegqs_cuda_ctx *ctx);

/* optional per-kernel timing of the following run_* calls (CUDA event pairs around every
 * IDCT-pass and smoothing-pass launch, on the stream they are launched on); the sums are
 * read back with jpegqs_cuda_kernel_stats after the call.  Measurement aid for bench.py. */
void jpegqs_cuda_set_profiling(jpegqs_cuda_ctx *ctx, int on);
void jpegqs_cuda_kernel_stats(const jpegqs_cuda_ctx *ctx, float *idct_ms, int *idct_launches,
		float *smooth_ms, int *smooth_launches);

/* knobs for tuning runs and tests; results are bit-identical for every setting.
 * key 1: maximum coefficients per accumulation chunk (1..4, default 4)
 * key 5: uniform-quant chunks share t and d*t (default 1)
 * key 6: slab-pipelined upload / download in the host entry points (default 1)
 * key 7: blocks per slab wave for key 6; 0 = SM count x resident warps x 32 (tests force small values)
 * key 8: the two edge coefficients of an anti-diagonal ride along with up to two of its full
 *        coefficients in one "mixed" chunk instead of forming their own
 * keys 0, 2, 4 (lock-step level, warps per sub-partition, packed FP32x2 path) only exist in the
 * measurement build (make -C csrc experiments); the shipped library accepts their default values
 * and answers JPEGQS_ERR_UNSUPPORTED otherwise.  key 3: retired, ignored. */
int jpegqs_cuda_set_tuning(jpegqs_cuda_ctx *ctx, int key, int value);

/* pinned host memory for coefficient arrays: the copy engines read / write it directly.  Plain
 * malloc'd memory (flat or as block-row tables, see jpegqs_cuda_comp.rows) works too and goes
 * through the context's pinned staging buffer, which is kept between calls (grow-only).
 * Environment: JPEGQS_IO_THREADS = threads used for that gather / scatter (default: up to 8). */
void *jpegqs_cuda_host_alloc(size_t bytes);
void jpegqs_cuda_host_free(void *p);

/* ---- whole-image entry points: the body of do_quantsmooth (quantsmooth.h:2404-2878) ----
 * flags/niter/progprec/progress/userdata = jpegqs_control_t fields (libjpegqs.h:41-45).
 * With progress == NULL independent components are processed in the same kernel launches;
 * with a callback components run one after another so the callback sequence (cur, max) is
 * the reference's (quantsmooth.h:2656-2664).
 * Return: the reference's `stop` (0 = done, non-zero = stopped early) or a negative error. */
int jpegqs_cuda_run_host(jpegqs_cuda_ctx *ctx, jpegqs_cuda_image *img, int flags, int niter,
		int progprec, jpegqs_cuda_progress_fn progress, void *userdata);
/* same, but comp[].coef / coef_up are DEVICE pointers; stream = cudaStream_t or NULL */
int jpegqs_cuda_run_device(jpegqs_cuda_ctx *ctx, jpegqs_cuda_image *img, int flags, int niter,
		int progprec, jpegqs_cuda_progress_fn progress, void *userdata, void *stream);
/* n independent images in shared launches (no progress callback); host or device pointers.
 * ret[i] receives each image's stop value.  Returns 0 or a negative error. */
int jpegqs_cuda_run_batch(jpegqs_cuda_ctx *ctx, int nimages, jpegqs_cuda_image *imgs, int flags,
		int niter, int on_device, int *ret, void *stream);

/* ---- one image sharded by MCU rows over several GPUs (SURVEY.md 8e) ----------------------
 * Every rank - a device of this process, or another process on the same box - smooths one slab
 * of contiguous MCU rows and exchanges ONE pixel row per plane with each neighbour after every
 * IDCT pass (quantsmooth.h:1396-1401: a pass reads only start-of-pass neighbour pixels).  The
 * exchange runs inside CUDA kernels over peer memory (NVLink P2P / CUDA IPC mailboxes, sequence
 * numbers instead of events): no host round trip, no NCCL call on the data path.  The
 * reference's `stop` logic is evaluated on the device from flags the ranks OR-combine, so all
 * ranks issue the same schedule whatever their data.  Results are bit-identical to the
 * unsharded run for any rank count.
 *
 *   link_create on every rank -> link_export + (all-gather of the handles by the caller) +
 *   link_connect_ipc, or link_connect_local for the devices of one process -> run_slab, as often
 *   as wanted, by all ranks alike -> link_destroy.                                            */
typedef struct jpegqs_cuda_link jpegqs_cuda_link;
typedef struct {
	int32_t rank, world;
	uint32_t row0[JPEGQS_CUDA_MAX_COMP];        /* first block row of the slab inside component c  */
	uint32_t hblk_total[JPEGQS_CUDA_MAX_COMP];  /* block rows of the whole component               */
} jpegqs_cuda_slab;
/* max_wblk: widest component (in blocks) any later run will exchange */
int jpegqs_cuda_link_create(jpegqs_cuda_ctx *ctx, int rank, int world, uint32_t max_wblk, jpegqs_cuda_link **out);
void jpegqs_cuda_link_destroy(jpegqs_cuda_link *link);
int jpegqs_cuda_link_handle_bytes(void);
int jpegqs_cuda_link_export(jpegqs_cuda_link *link, void *handle);
int jpegqs_cuda_link_connect_ipc(jpegqs_cuda_link *link, const void *handles_in_rank_order);
int jpegqs_cuda_link_connect_local(jpegqs_cuda_link **links_in_rank_order, int world);
/* slab: the image with comp[].hblk = block rows held by this rank and coef / rows / coef_up
 * covering exactly those rows (host memory, or device memory with on_device != 0);
 * image_width / image_height are the WHOLE image's.  No progress callback.  link may be NULL
 * for world == 1.  Returns the reference's stop value (identical on every rank) or an error. */
int jpegqs_cuda_run_slab(jpegqs_cuda_ctx *ctx, jpegqs_cuda_link *link, jpegqs_cuda_image *slab,
		const jpegqs_cuda_slab *geom, int flags, int niter, int on_device, void *stream);

/* The devices of ONE process behind one call (what do_quantsmooth uses when JPEGQS_GPUS is
 * set): contexts + links for ndev devices (devices == NULL: ordinals 0..ndev-1; ndev <= 0: all),
 * one host thread per device inside run_host_multi.  An image is spread over as many devices as
 * it has waves of the smoothing kernel (JPEGQS_MIN_BLOCKS_PER_GPU luma blocks per device,
 * default 148*16*32), so a small image stays on device 0 with the slab-pipelined run_host. */
typedef struct jpegqs_cuda_multi jpegqs_cuda_multi;
int jpegqs_cuda_multi_create(int ndev, const int *devices, jpegqs_cuda_multi **out);
void jpegqs_cuda_multi_destroy(jpegqs_cuda_multi *m);
int jpegqs_cuda_multi_devices(const jpegqs_cuda_multi *m);
jpegqs_cuda_ctx *jpegqs_cuda_multi_ctx(jpegqs_cuda_multi *m, int i);
const char *jpegqs_cuda_multi_last_error(const jpegqs_cuda_multi *m);
int jpegqs_cuda_multi_plan(const jpegqs_cuda_multi *m, const jpegqs_cuda_image *img);   /* devices it would use */
/* host buffers / block-row tables like jpegqs_cuda_run_host; no progress callback */
int jpegqs_cuda_run_host_multi(jpegqs_cuda_multi *m, jpegqs_cuda_image *img, int flags, int niter);

/* ---- geometry of the device's pixel planes -----------------------------------------------
 * stride = 8*wblk + 2*pad bytes per row; hblk*8 pixel rows plus one halo row above and below */
size_t jpegqs_cuda_plane_bytes(uint32_t wblk, uint32_t hblk);
int jpegqs_cuda_plane_stride(uint32_t wblk);
int jpegqs_cuda_plane_pad(void);   /* byte offset of pixel column 0 inside a plane row */

/* ---- decode to interleaved 8-bit RGB (SURVEY.md 8f row f2) -----------------------------
 * What libjpeg produces after the reference's jpegqs_start_decompress (quantsmooth.h:2880-2904):
 * islow IDCT, libjpeg's "fancy" chroma up-sampling (h2v1 / h2v2; other ratios: replication),
 * YCbCr -> RGB with libjpeg's fixed-point constants.  1 or 3 components.  Components whose
 * quant table is not all ones are de-quantized first, so the call also decodes an untouched
 * coefficient set.  rgb: image_width * image_height * 3 bytes (host, or device if on_device;
 * device coefficient arrays that still carry quant tables are de-quantized in place). */
int jpegqs_cuda_render_rgb(jpegqs_cuda_ctx *ctx, const jpegqs_cuda_image *img, int on_device,
		uint8_t *rgb, void *stream);

/* ---- introspection used by the parity tests ------------------------------------------- */
/* the 64 weight tables exactly as the device consumes them but WITHOUT the power-of-two
 * pre-scale, natural coefficient order, 160 (or 272 with JPEGQS_DIAGONALS) floats each;
 * replaces quantsmooth_init (quantsmooth.h:251-301).  Returns floats per coefficient. */
int jpegqs_cuda_tables(int flags, float *out);
/* host evaluation of the device's exact-division helper (GET_ORIG_COEF, 324-341) */
int jpegqs_cuda_orig_coef(int coef, int q);
/* the smoothing kernel's chunk schedule for one quant table (host-only; DESIGN.md 3.3): the 63
 * AC coefficients in the reference's anti-diagonal visiting order (quantsmooth.h:313-322,
 * 1403-1409), grouped into chunks.  out: 12 bytes per chunk = {type, n, first, 0, idx[8]} with
 * type 0 = plain, 1 = the diagonal's two edge coefficients, 2 = equal quant values (shared
 * threshold work), 3 = mixed (n full coefficients, then the row-0 and the column-0 one: n + 2
 * indices); idx = natural-order coefficient indices.  uniform: bit 0 = uniform chunks, bit 1 =
 * mixed chunks; quant == NULL gives the table-independent schedule.  Returns the chunk count (<= 64), or JPEGQS_ERR_ARG. */
int jpegqs_cuda_chunk_schedule(const uint16_t *quant, int max_coefs, int uniform, uint8_t *out);

#ifdef __cplusplus
}
#endif
#endif
