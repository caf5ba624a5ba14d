/*
 * p2p.h - C ABI of the B200-native panorama -> plane projection library (libp2p_b200.so).
 *
 * This is the drop-in boundary for ONE hot path of Maxiviper117/360-to-planer-images:
 * the per-view projection in app/panorama_to_plane-pitch.py.  The reference has no FFI seam
 * of its own (it is a single Python script calling NumPy and cv2.remap), so each entry point
 * below names the reference lines it replaces; INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - plain C types only; all functions return 0 (P2P_OK) or a negative p2p_status;
 *     p2p_last_error(ctx) returns a human readable message for the calling thread's last failure on ctx
 *     (kept per thread, like errno; valid until that thread's next failing call).
 *   - images are 8-bit, 3 channels, interleaved, channel order preserved (the reference keeps
 *     cv2's BGR end to end, ref :244; channels are independent in the arithmetic).
 *   - the caller owns every host buffer; the library owns device memory inside the context.
 *   - a context belongs to one CUDA device and is thread-safe (calls are serialised on an
 *     internal mutex and only enqueue work); work of different "slots" runs on different
 *     CUDA streams so upload / projection / readback of consecutive images overlap.
 *   - there is no CPU fallback: p2p_create fails if no CUDA device is usable.
 */
#ifndef P2P_B200_H
#define P2P_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define P2P_ABI_VERSION 1

typedef struct p2p_ctx p2p_ctx;

typedef enum p2p_status {
    P2P_OK = 0,
    P2P_ERR_INVALID = -1, /* bad argument (null pointer, non-positive size, bad slot ...) */
    P2P_ERR_CUDA = -2,    /* a CUDA runtime call failed; see p2p_last_error */
    P2P_ERR_NOMEM = -3,   /* device or pinned-host allocation failed */
    P2P_ERR_STATE = -4,   /* slot holds no panorama / size mismatch */
    P2P_ERR_LIMIT = -5,   /* size beyond the limits inherited from cv2.remap (< 32767) */
    P2P_ERR_UNSUPPORTED = -6 /* input file outside the subset the device decoder handles: use cv2.imread */
} p2p_status;

/* Per-pitch constants of the pitch map, formed on the host exactly as the reference does
 * (ref precompute_pitch_mapping :119 focal length, :142-149 R_pitch entries, cast to f32). */
typedef struct p2p_pitch_consts {
    float f; /* float32(0.5 * W / tan(FOV_rad / 2))           ref :119, :131 */
    float c; /* float32(cos(pitch_rad))                        ref :145-147   */
    float s; /* float32(sin(pitch_rad))                        ref :145-147   */
} p2p_pitch_consts;

/* option keys for p2p_set_option */
typedef enum p2p_option {
    P2P_OPT_SAMPLER = 0, /* 0 = global-load gather, 1 = texture gather4 point fetch (default) */
    P2P_OPT_WARP_W = 1,  /* output pixels per warp row: 32 (default) or 8 (8 x 4 warp tiles) */
    P2P_OPT_YAWS_PER_THREAD = 2, /* 1..4 views sharing one coordinate evaluation (default 4) */
    P2P_OPT_COUNT_LAUNCHES = 3,  /* read-only via p2p_get_option: kernels launched so far (the fold of a panorama into
                                    its quarter-turn planes, like the refresh of its texture array, is not counted) */
    P2P_OPT_IMAGES_PER_LAUNCH = 4, /* 2 or 4: consecutive resident panoramas of p2p_project_batch share one launch
                                     (and one coordinate evaluation) of the generic kernel's multi-image variants.
                                     1 (default): the row-segment kernel pairs same-stream resident panoramas of one
                                     size by itself (their quarter-turn groups share launches) */
    P2P_OPT_MIRROR = 5            /* with the texture sampler and W % 8 == 0 the pixel pair (W/2 + t, W/2 - t) shares
                                     one coordinate evaluation.  2 (default): row-segment kernel - a warp walks a
                                     row segment, every output byte leaves in a packed 32-bit store, any flat view
                                     list is one launch; 1: the round-1 pair kernel (byte stores for the mirrored
                                     half, one launch per pitch-list chunk); 0: every pixel evaluates its own */
    ,P2P_OPT_INTERP = 6            /* 0 (default): cv2.remap fixed-point bilinear, the reference's arithmetic
                                     (ref :192-199, :212-218); 1: exact bilinear - un-quantised fractions with the
                                     arithmetic of scipy.ndimage.map_coordinates(order=1) (double precision, round
                                     half up); integer-roll yaws only */
    ,P2P_OPT_TRIG = 7              /* 0 (default): f32 arccos / arctan2 exactly as NumPy evaluates them on AVX-512
                                     hosts (Intel SVML, ref :162-164) - coordinates and pixels then match the
                                     reference bit for bit there; 1: table-free minimax fits (acos <= 1.07 ulp,
                                     atan2 <= 1.76 ulp, measured on a B200) */
    ,P2P_OPT_GPU_HUFFMAN = 9       /* 1 (default): JPEG inputs are Huffman-decoded on the device (self-synchronising
                                     subsequences, restart intervals as independent scans), the FF 00 stuffing of files
                                     without restart markers is removed on the device too, and the whole stage is queued
                                     without waiting for it (a fixed number of rounds, then a device-side verdict gates the
                                     write pass; a file that needs more rounds continues with host-checked rounds); the
                                     library's host decoder takes over when that does not converge; 0: always the host
                                     decoder; 3: the device stage with destuffing on the calling thread and a host check
                                     after every few rounds; 2: like 3 with the plain synchronisation rounds (tables in
                                     global memory - the yardstick the shared-memory rounds are tested against) */
    ,P2P_OPT_GPU_HUFFMAN_COUNT = 10 /* read-only: JPEG inputs whose Huffman stage ran on the device so far */
    ,P2P_OPT_SEAM_WRAP = 12        /* exact-bilinear mode only (P2P_OPT_INTERP = 1).  0 (default): U is clipped to Wp - 1 like the
                                     reference does (ref :172) - no interpolation across the 0 / 360 degree seam; 1: U runs over
                                     [0, Wp) and a pixel between the last and the first panorama column blends the two (true wrap,
                                     scipy's mode='grid-wrap'; the north-star's "edge / wrap mode", SURVEY 8f-3) */
    ,P2P_OPT_HOST_WAIT = 13        /* how a host thread waits for its slot's stream.  0 (default): cudaStreamSynchronize (CUDA's
                                     default spins: lowest latency, one busy core per waiting thread - the reference's
                                     ThreadPoolExecutor workers, ref :252-265, block in cv2 instead); 1: the thread sleeps on a
                                     blocking-sync event, for more images in flight than cores (several ranks on one box) */
    ,P2P_OPT_PNG_FORMATS = 14      /* PNG files the device decoder takes (p2p_upload_pano_png, p2p_decode_png; ref :244).
                                     0 (default): 8-bit gray / RGB / gray + alpha / RGBA, not interlaced, no PLTE, no tRNS;
                                     1: also 1/2/4/16-bit gray, 16-bit RGB / gray + alpha / RGBA, palette images (1/2/4/8
                                     bit) and Adam7 interlacing, tRNS on gray / RGB / palette images - with the pixels
                                     cv2.imread's IMREAD_COLOR returns (high byte of 16-bit samples, palette alpha dropped) */
    ,P2P_OPT_PNG_HOST_BLOCKS = 15  /* read-only: dynamic-Huffman deflate blocks of PNG inputs so far that the device's block-start
                                     search did not return, so the host's chain walk measured them itself (stored and fixed
                                     blocks, which the search never looks for, are not counted).  0 for files whose every
                                     dynamic block was found */
    ,P2P_OPT_SEG_CHUNKS = 11       /* row-segment kernel: chunks of 32 pixel pairs per warp (default 4, 1..64) */
    ,P2P_OPT_PARTIAL_UPLOAD = 8    /* 1 (default): p2p_process_image copies only the panorama rows its views can
                                     touch (p2p_view_row_range) over PCIe; 0: always the whole panorama */
    ,P2P_OPT_POISON = 16           /* debug: -1 (default) = off; 0..255: every buffer the context allocates from now on (device
                                     scratch, panorama, gather arrays and folded planes, pinned and mapped host buffers) is
                                     filled with this byte before its first use, so that a result which depends on memory no
                                     call has written differs from the one of a run with another byte (see p2p_debug_poison) */

} p2p_option;

/* ---- life cycle ------------------------------------------------------------------------- */
int p2p_abi_version(void);
int p2p_device_count(void);
/* n_slots independent panorama slots (each with its own stream and device buffers). */
int p2p_create(int device, int n_slots, p2p_ctx **out);
void p2p_destroy(p2p_ctx *ctx);
const char *p2p_last_error(p2p_ctx *ctx);
const char *p2p_status_string(int status);
int p2p_set_option(p2p_ctx *ctx, int key, int value);
int p2p_get_option(p2p_ctx *ctx, int key, int *value);

/* ---- host helpers (no GPU work) --------------------------------------------------------- */
/* libm restatement of the reference's host scalars: np.radians (:64, :68), focal (:119),
 * cos / sin (:142-149).  The Python host forms them with NumPy instead (identical by
 * construction); this export is for non-Python callers. */
int p2p_pitch_constants(double fov_deg, double pitch_deg, int W, p2p_pitch_consts *out);
/* Quantised yaw column table: (ix, fx) = cv2's 1/32-px fixed point form of one row of the
 * reference yaw map (precompute_yaw_mapping :85-105; all rows are equal, V = v :102).
 * Returns in *shift the column roll if the table is a pure integer roll, else -1. */
int p2p_yaw_table(int Wp, double yaw_deg, int32_t *ix, int32_t *fx, int32_t *shift);
/* page-locked host memory for overlapped transfers */
int p2p_host_alloc(void **ptr, size_t bytes);
int p2p_host_free(void *ptr);
int p2p_host_register(void *ptr, size_t bytes);
int p2p_host_unregister(void *ptr);

/* ---- panorama upload (replaces holding the cv2.imread result, ref :244) ------------------ */
/* Copy a host BGR panorama (row_stride bytes between rows) into `slot` and pack it to the
 * device layout (RGBA-packed uint32, one duplicated wrap column and clamp row).  Asynchronous
 * on the slot's stream when `bgr` is page-locked. */
int p2p_upload_pano(p2p_ctx *ctx, int slot, const uint8_t *bgr, int Wp, int Hp, size_t row_stride);
/* Same, but `d_bgr` is a device pointer on ctx's device (no PCIe transfer). */
int p2p_upload_pano_device(p2p_ctx *ctx, int slot, const void *d_bgr, int Wp, int Hp, size_t row_stride);

/* Yaw pass for yaws that are not an integer column roll: materialise the rotated panorama
 * of `src_slot` into `dst_slot` with the Wp-entry table from p2p_yaw_table.  Bit-exact form of
 * the reference's first cv2.remap (ref :191-199). */
int p2p_rotate_pano(p2p_ctx *ctx, int src_slot, int dst_slot, const int32_t *ix, const int32_t *fx);

/* ---- the hot path (replaces process_yaw_and_pitchs, ref :181-221, for a whole batch of
 *      yaws: the ThreadPoolExecutor fan-out of ref :252-265 becomes one launch) ------------- */
/* Computes n_yaw * n_pitch views of the panorama in `slot`:
 *   out[(k * n_pitch + j)][v][u][ch], k = yaw index, j = pitch index, u8, W*H*3 bytes per view.
 * yaw_shift[k] in [0, Wp) is the integer column roll of yaw k (p2p_yaw_table); for other yaws
 * project from a slot produced by p2p_rotate_pano with shift 0.
 * out_on_device = 0: `out` is host memory, a device->host copy is enqueued after the kernel
 *                    (asynchronous if `out` is page-locked); call p2p_sync before reading.
 * out_on_device = 1: `out` is a device pointer, results stay in HBM. */
int p2p_project_views(p2p_ctx *ctx, int slot, int n_yaw, const int32_t *yaw_shift, int n_pitch,
                      const p2p_pitch_consts *pitch, int W, int H, uint8_t *out, int out_on_device);

/* p2p_project_views for yaws that are NOT integer column rolls, in one pass: yaw k is given by its Wp-entry column table
 * (ix[k][c], fx[k][c]) from p2p_yaw_table.  Both cv2.remap passes of the reference - the yaw pass over the whole panorama
 * (precompute_yaw_mapping, ref :79-108, :191-199) and the pitch pass (ref :212-218) - are evaluated per output pixel from the
 * 2 x 3 source texels under its footprint; the result is bit-identical to p2p_rotate_pano + p2p_project_views with shift 0,
 * without materialising a rotated panorama per yaw.  The slot must hold a whole panorama.  `out` as in p2p_project_views. */
int p2p_project_views_table(p2p_ctx *ctx, int slot, int n_yaw, const int32_t *const *ix, const int32_t *const *fx, int n_pitch,
                            const p2p_pitch_consts *pitch, int W, int H, uint8_t *out, int out_on_device);

/* The same views for a batch of panoramas that are already resident (one launch per image,
 * each on its slot's stream): slots[i] -> outs[i].  One host call per batch keeps the launch
 * queue full when a launch is only tens of microseconds (BASELINE configs[2]). */
int p2p_project_batch(p2p_ctx *ctx, int n_images, const int32_t *slots, int n_yaw, const int32_t *yaw_shift,
                      int n_pitch, const p2p_pitch_consts *pitch, int W, int H, uint8_t *const *outs,
                      int out_on_device);

/* A flat list of views in one launch, optionally only a band of output rows: view i = (yaw_shift[i], pitch[i]) is written
 * to out + i * W * H * 3 (rows row_begin .. row_end - 1 of it; the other rows of `out` are not touched).  This is the
 * unit the reference parallelises over (one (yaw, pitch) pair of the nested loops at ref :202-219 / :253-265) without the
 * yaw x pitch product structure of p2p_project_views: the six cube faces of BASELINE configs[4] - four yaws at pitch 90
 * plus the two pole pitches - are one call and one kernel launch.  Views whose pitch constants are bit-identical share one
 * coordinate evaluation (the reference's pitch_mapping_cache key has no yaw, ref :55-73); four of them whose rolls are
 * quarter turns apart (r0 + k Wp / 4, Wp % 4 == 0) are read automatically from the slot's yaw-folded copy, 3 texture
 * gathers per pixel for the four views instead of 4, from the second such render of a panorama on (the fold is built
 * then, once per panorama, and not counted in P2P_OPT_COUNT_LAUNCHES).  The row band is how one image
 * is split over several GPUs (SURVEY 8e): every device renders rows [H r / n, H (r + 1) / n) of all views into the same
 * host array.  out_on_device as in p2p_project_views (a host `out` receives only the band, one strided copy). */
int p2p_project_view_list(p2p_ctx *ctx, int slot, int n_views, const int32_t *yaw_shift, const p2p_pitch_consts *pitch,
                          int W, int H, int row_begin, int row_end, uint8_t *out, int out_on_device);

/* p2p_project_view_list for any yaw: view i is the integer roll yaw_shift[i] in [0, Wp), or, if yaw_shift[i] < 0, the
 * Wp-entry column table (ix[i], fx[i]) of p2p_yaw_table (ref :79-108, :191-199, :212-218) - both remap passes of the
 * reference per output pixel, the bytes of p2p_project_views_table.  ix / fx may be NULL when no shift is negative, and
 * their entries of integer-roll views are not read.  Views that pass the same table pointers share one device table; views
 * with bit-identical pitch constants share a coordinate evaluation (up to 4 per group).  The table views go out in a second
 * launch behind the integer rolls on the slot's stream (row-segment kernel; other geometries: one launch per view).  A
 * partial slot (p2p_process_image) serves the views whose rows it holds (the yaw pass reads the view's own rows only:
 * p2p_view_row_range), else P2P_ERR_STATE.  Table views need the fixed-point interpolation mode (P2P_OPT_INTERP = 0). */
int p2p_project_view_list_tables(p2p_ctx *ctx, int slot, int n_views, const int32_t *yaw_shift,
                                 const int32_t *const *ix, const int32_t *const *fx, const p2p_pitch_consts *pitch,
                                 int W, int H, int row_begin, int row_end, uint8_t *out, int out_on_device);

/* Replicate the (possibly partial) panorama held by src's slot into dst's slot; the two contexts may live on different
 * devices of one box (cudaMemcpyPeerAsync: NVLink when peer access is available, staged by the driver otherwise) - one
 * PCIe upload plus peer copies instead of one upload per GPU when a single image is split over GPUs (SURVEY 5, 8e).
 * Asynchronous on the destination slot's stream and ordered after the work enqueued on the source slot; keep the source
 * slot unchanged until the destination slot has been synchronised. */
int p2p_copy_pano(p2p_ctx *dst, int dst_slot, p2p_ctx *src, int src_slot);

/* A panorama assembled from pieces: when ONE image is split over n GPUs every device uploads 1 / n of the rows over its
 * own PCIe link (p2p_upload_pano_rows) and fetches the other pieces from its peers over NVLink (p2p_copy_pano_rows) - an
 * all-gather built from peer copies, so the PCIe time of the panorama shrinks with n instead of being paid by one GPU.
 * p2p_upload_pano_rows copies + packs host rows [row_begin, row_end) (row_end == Hp also writes the clamp row);
 * p2p_copy_pano_rows copies packed rows [row_begin, row_end) of the source slot (packed rows run 0 .. Hp, the clamp row
 * included: row_end <= Hp + 1; row_begin < 0: everything the source holds).  A piece that touches the rows a slot already
 * holds (same panorama size) extends them; otherwise the slot holds just the new piece.  Both are asynchronous on the
 * destination slot's stream; the copy is ordered after the work enqueued on the source slot. */
int p2p_upload_pano_rows(p2p_ctx *ctx, int slot, const uint8_t *bgr, int Wp, int Hp, size_t row_stride, int row_begin,
                         int row_end);
int p2p_copy_pano_rows(p2p_ctx *dst, int dst_slot, p2p_ctx *src, int src_slot, int row_begin, int row_end);

/* upload + project + readback of one image in one call (all asynchronous on the slot stream).
 * Because the views are known before the transfer, only the panorama rows they can touch are copied to the
 * device (P2P_OPT_PARTIAL_UPLOAD); the slot then holds a partial panorama: projecting other views from it
 * returns P2P_ERR_STATE, upload it again instead. */
int p2p_process_image(p2p_ctx *ctx, int slot, const uint8_t *bgr, int Wp, int Hp, size_t row_stride,
                      int n_yaw, const int32_t *yaw_shift, int n_pitch, const p2p_pitch_consts *pitch,
                      int W, int H, uint8_t *out_host);

/* First and last panorama row (inclusive) the 4-tap sampler reads for these pitches - every yaw, any image: the
 * pitch map has no yaw and no image in it (the key of the reference's pitch_mapping_cache, ref :55-73).  Evaluated
 * on the device with the projection kernel's own arithmetic (exact), memoised per geometry in the context. */
int p2p_view_row_range(p2p_ctx *ctx, int n_pitch, const p2p_pitch_consts *pitch, int W, int H, int Wp, int Hp,
                       int *first_row, int *last_row);

/* ---- JPEG files of the views (replaces cv2.imwrite(<name>.jpg, view), ref :277, for --output_format
 *      jpg | jpeg, ref :400-405) ------------------------------------------------------------------------ */
/* Baseline JPEG files of n_images images (BGR u8, H x W x 3, tightly packed; `bgr` is host memory when
 * on_device = 0, a device pointer on ctx's device when 1), encoded on the GPU.  With quality = 95 the files are
 * byte-identical to what cv2.imwrite / cv2.imencode('.jpg') produce with OpenCV's defaults (libjpeg-turbo:
 * 4:2:0, integer "islow" DCT, Annex K Huffman tables, JFIF header).  File i is written to
 * out_host + i * out_stride, its length to sizes[i].  Synchronous (returns when the files are in out_host).
 * P2P_ERR_LIMIT if a file does not fit out_stride bytes (W * H * 3 + 2048 always suffices). */
int p2p_encode_jpeg(p2p_ctx *ctx, int slot, const uint8_t *bgr, int on_device, int n_images, int W, int H,
                    int quality, uint8_t *out_host, size_t out_stride, size_t *sizes);
/* p2p_project_views followed by p2p_encode_jpeg without the pixels leaving the device: view (k, j) becomes
 * file k * n_pitch + j. */
int p2p_project_views_jpeg(p2p_ctx *ctx, int slot, int n_yaw, const int32_t *yaw_shift, int n_pitch,
                           const p2p_pitch_consts *pitch, int W, int H, int quality, uint8_t *out_host,
                           size_t out_stride, size_t *sizes);

/* upload (only the rows the views can touch, like p2p_process_image) + project + encode in one call: what the
 * reference does per image with --output_format jpg between cv2.imread (ref :244) and its cv2.imwrite calls (:277).
 * Synchronous for this slot; other slots / threads keep running (the context lock is not held while waiting). */
int p2p_process_image_jpeg(p2p_ctx *ctx, int slot, const uint8_t *bgr, int Wp, int Hp, size_t row_stride, int n_yaw,
                           const int32_t *yaw_shift, int n_pitch, const p2p_pitch_consts *pitch, int W, int H,
                           int quality, uint8_t *out_host, size_t out_stride, size_t *sizes);

/* ---- PNG files of the views (replaces cv2.imwrite(<name>.png, view), ref :277: the default --output_format) ---- */
/* PNG files of n_images images (BGR u8, tightly packed, host or device memory), encoded on the GPU and byte-identical
 * to cv2.imwrite / cv2.imencode('.png') at OpenCV's defaults (filter Sub, zlib level 1, strategy Z_RLE, 8192-byte IDAT
 * chunks), including libpng's small-image cases (window bits in the zlib header of images with at most 16384 bytes
 * of data, filter type 0 for images one pixel wide) and the blocks zlib stores uncompressed (white noise).  sizes[i] = 0
 * is kept as the "not handled on the device, use cv2.imwrite" signal; no input produces it any more.
 * Synchronous.  P2P_ERR_LIMIT if a file does not fit out_stride bytes (W * H * 4 + 4096 always suffices). */
int p2p_encode_png(p2p_ctx *ctx, int slot, const uint8_t *bgr, int on_device, int n_images, int W, int H,
                   uint8_t *out_host, size_t out_stride, size_t *sizes);
/* upload (rows the views touch; bgr = NULL: project from the panorama resident in the slot) + project + PNG-encode.
 * pixels_host (optional, n_yaw * n_pitch * H * W * 3 bytes) also receives the pixels, so the caller can write the views
 * the device encoder did not handle (sizes[i] = 0) with cv2.imwrite. */
int p2p_process_image_png(p2p_ctx *ctx, int slot, const uint8_t *bgr, int Wp, int Hp, size_t row_stride, int n_yaw,
                          const int32_t *yaw_shift, int n_pitch, const p2p_pitch_consts *pitch, int W, int H,
                          uint8_t *out_host, size_t out_stride, size_t *sizes, uint8_t *pixels_host);

/* The files of a flat view list of any yaws (p2p_project_view_list_tables): view i -> file i, encoded on the device like
 * p2p_process_image_jpeg / _png.  bgr == NULL: the panorama resident in the slot (e.g. decoded there by
 * p2p_upload_pano_jpeg / _png, which may also be a partial slot covering the views); else only the rows the views touch
 * are uploaded (P2P_OPT_PARTIAL_UPLOAD).  Fractional yaws then move no pixels over PCIe either.  Synchronous for this
 * slot; pixels_host (optional, n_views * H * W * 3 bytes) as in p2p_process_image_png. */
int p2p_process_view_list_jpeg(p2p_ctx *ctx, int slot, const uint8_t *bgr, int Wp, int Hp, size_t row_stride, int n_views,
                               const int32_t *yaw_shift, const int32_t *const *ix, const int32_t *const *fx,
                               const p2p_pitch_consts *pitch, int W, int H, int quality, uint8_t *out_host,
                               size_t out_stride, size_t *sizes);
int p2p_process_view_list_png(p2p_ctx *ctx, int slot, const uint8_t *bgr, int Wp, int Hp, size_t row_stride, int n_views,
                              const int32_t *yaw_shift, const int32_t *const *ix, const int32_t *const *fx,
                              const p2p_pitch_consts *pitch, int W, int H, uint8_t *out_host, size_t out_stride,
                              size_t *sizes, uint8_t *pixels_host);

/* ---- JPEG panoramas decoded on the device (replaces cv2.imread(path) of a .jpg / .jpeg input, ref :244) ---- */
/* Headers only: size of the image if the file is in the supported subset (8-bit YCbCr 4:4:4 / 4:2:2 / 4:2:0 or
 * grayscale, baseline or extended sequential Huffman with one scan, or progressive (SOF2: any standard scan progression that
 * reaches full precision), restart markers allowed, YCbCr by libjpeg's own rule (JFIF marker, or an Adobe marker with a non-zero transform flag
 * as Photoshop / Lightroom write it, or component ids other than 'R' 'G' 'B'), EXIF
 * orientation 1 or absent), else P2P_ERR_UNSUPPORTED - the caller then reads the file with cv2.imread as before. */
int p2p_jpeg_probe(const uint8_t *file, size_t len, int *W, int *H);
/* Host stage only (no GPU, debug / tests): layout[10] = {W, H, hmax, vmax, blocks per row and column of Y, Cb, Cr};
 * if coef != NULL the quantised coefficients (int16, natural order, component planes [by][bx][64], Y then Cb then Cr;
 * capacity in elements) exactly as jdhuff.c decodes them. */
int p2p_jpeg_coefficients(const uint8_t *file, size_t len, int16_t *coef, size_t capacity, int32_t *layout);
/* Host only (no GPU, debug / tests): the Huffman tables the device stage uploads for a baseline file, byte for byte (the
 * DevTables block of csrc/p2p_jpegdec.cuh: per component DevHuff, then SyncLut), into out[capacity] if out != NULL;
 * layout[16] = {sizeof DevTables, sizeof DevHuff, offsets in DevHuff of dc_look, dc_maxcode, dc_valoff, dc_vals, ac_fast,
 * ac_look, ac_maxcode, ac_valoff, ac_vals, entries of dc_vals, of ac_vals, offset of SyncLut, offset of SyncLut.w,
 * lookahead bits of ac_fast / SyncLut}.  P2P_ERR_UNSUPPORTED for files outside the subset and progressive files. */
int p2p_jpeg_device_tables(const uint8_t *file, size_t len, uint8_t *out, size_t capacity, int32_t *layout);
/* Decode the file into `slot` as its panorama (like cv2.imread + p2p_upload_pano, bit-identical pixels): Huffman
 * decoding (self-synchronising subsequences; P2P_OPT_GPU_HUFFMAN), inverse DCT, chroma upsampling and colour
 * conversion all run on the device (the FF 00 byte stuffing is removed there too when the file has no restart markers); the
 * pixels never exist in host memory.  The scans of a progressive file are decoded on host threads (jdphuff.c; up to four: DC, AC per component), everything
 * behind them on the device.  If the device Huffman stage does not converge the library's own host decoder (calling thread, outside the
 * context lock) takes over.  Returns after the decode has finished on the device: a damaged file (truncated scan,
 * restart markers out of sequence, codes or coefficient blocks no 8-bit encoder writes) gives P2P_ERR_UNSUPPORTED
 * and leaves the slot without a panorama - such files are decoded like libjpeg or not at all, never differently. */
int p2p_upload_pano_jpeg(p2p_ctx *ctx, int slot, const uint8_t *file, size_t len, int *Wp, int *Hp);
/* Same decoder, pixels returned to the host (BGR, row_stride bytes per row, at least capacity_rows rows): the array
 * cv2.imread / cv2.imdecode would return.  Synchronous; the slot's panorama is invalidated. */
int p2p_decode_jpeg(p2p_ctx *ctx, int slot, const uint8_t *file, size_t len, uint8_t *bgr_host, size_t row_stride,
                    size_t capacity_rows);

/* ---- PNG panoramas decoded on the device (replaces cv2.imread(path) of a .png input, ref :244; the reference's own
 *      default output format, ref :400-405, is the usual input of a second pass) ---------------------------------- */
/* Chunk structure only: size of the image if the file is in the supported subset (8-bit gray / RGB / gray + alpha / RGBA,
 * not interlaced, no APNG, no tRNS, every chunk CRC intact), else P2P_ERR_UNSUPPORTED - the caller then reads the file
 * with cv2.imread as before. */
int p2p_png_probe(const uint8_t *file, size_t len, int *W, int *H);
/* p2p_png_probe for a subset: formats as P2P_OPT_PNG_FORMATS (0: p2p_png_probe; 1: every PNG colour type, bit depth and
 * Adam7).  The same rule cv2.imread(path) of a .png input is replaced by (ref :244). */
int p2p_png_probe_ex(const uint8_t *file, size_t len, int formats, int *W, int *H);
/* Host model of the device decoder (no GPU, debug / tests): the same routines - block-start search, chain walk, inflate
 * with symbolic history, resolution, Adler-32 / CRC-32 checks, unfilter - run serially.  bgr: capacity_rows rows of
 * row_stride bytes, the array cv2.imread(path) returns.  stats (optional, 4 values): bit positions passing the first
 * header test, block-start candidates, deflate blocks of the stream, blocks the chain walk had to measure itself. */
int p2p_png_decode_host(const uint8_t *file, size_t len, uint8_t *bgr, size_t row_stride, size_t capacity_rows,
                        uint64_t *stats);
/* p2p_png_decode_host for a subset (formats as P2P_OPT_PNG_FORMATS; ref :244): also the unpacking of 1/2/4-bit samples,
 * the palette look-up, the high byte of 16-bit samples and the Adam7 passes, by the routines the device runs. */
int p2p_png_decode_host_ex(const uint8_t *file, size_t len, int formats, uint8_t *bgr, size_t row_stride, size_t capacity_rows,
                           uint64_t *stats);
/* Decode the file into `slot` as its panorama (like cv2.imread + p2p_upload_pano, identical pixels): the deflate stream is
 * inflated in parallel on the device (block starts found by testing every bit position for a dynamic-block header, every
 * block decoded independently with symbolic history, back-references resolved afterwards), the scanline filters are undone
 * there too (independent row runs, skewed wavefront inside a run); the pixels never exist in host memory.  Returns after
 * the decode has finished: a damaged file (CRC-32 / Adler-32 mismatch, invalid codes or distances, wrong amount of data)
 * or a stream the parallel decoder is not worth running on (fixed-Huffman-only writers, single huge blocks) gives
 * P2P_ERR_UNSUPPORTED and leaves the slot without a panorama. */
int p2p_upload_pano_png(p2p_ctx *ctx, int slot, const uint8_t *file, size_t len, int *Wp, int *Hp);
/* Same decoder, pixels returned to the host (BGR, row_stride bytes per row, at least capacity_rows rows): the array
 * cv2.imread / cv2.imdecode would return.  Synchronous; the slot's panorama is invalidated. */
int p2p_decode_png(p2p_ctx *ctx, int slot, const uint8_t *file, size_t len, uint8_t *bgr_host, size_t row_stride,
                   size_t capacity_rows);

/* wait for everything enqueued on `slot` (slot < 0: all slots) */
int p2p_sync(p2p_ctx *ctx, int slot);
/* run the slot's work on a caller supplied cudaStream_t (e.g. torch's current stream) */
int p2p_set_stream(p2p_ctx *ctx, int slot, void *cuda_stream);
/* the cudaStream_t a slot currently runs on (e.g. to put several slots on one stream) */
int p2p_get_stream(p2p_ctx *ctx, int slot, void **cuda_stream);

/* ---- device timing on the launching stream ----------------------------------------------- */
int p2p_event_create(p2p_ctx *ctx, void **event);
int p2p_event_destroy(p2p_ctx *ctx, void *event);
int p2p_event_record(p2p_ctx *ctx, void *event, int slot);
/* make everything enqueued on `slot` from now on wait for `event` (fork / join of several slot streams around a timed
 * region: record on one stream, wait on the others, and the reverse at the end) */
int p2p_event_wait(p2p_ctx *ctx, void *event, int slot);
int p2p_event_elapsed_ms(p2p_ctx *ctx, void *start, void *stop, float *ms); /* syncs on stop */
/* overwrite `bytes` of scratch device memory on the slot's stream (L2 flush between reps) */
int p2p_flush_l2(p2p_ctx *ctx, int slot, size_t bytes);

/* ---- stage-isolated debug exports (parity tests) ----------------------------------------- */
/* device self-test of the range-check-free sqrt / division sequences against the generic IEEE
 * intrinsics: number of pixels of a W x H view whose rotated ray differs in any bit, and (if
 * exhaustive_div) number of floats in {0} U [2^-64, 2^24) whose division by 2pi / pi differs (the
 * kernel's numerators never leave that set). Both must be 0. */
int p2p_selftest(p2p_ctx *ctx, const p2p_pitch_consts *pitch, int W, int H, int exhaustive_div,
                 unsigned long long *ray_mismatches, unsigned long long *div_mismatches);
/* coordinates only: the (U, V) f32 maps of ref precompute_pitch_mapping :114-175, to host */
int p2p_coords(p2p_ctx *ctx, const p2p_pitch_consts *pitch, int W, int H, int Wp, int Hp,
               float *U_host, float *V_host);
/* sampler only: injected host (U, V) maps, one integer yaw shift; ref :212-218 */
int p2p_sample_with_maps(p2p_ctx *ctx, int slot, int yaw_shift, const float *U_host,
                         const float *V_host, int W, int H, uint8_t *out_host);
/* read back the packed panorama of a slot as BGR (checks upload / rotate) */
int p2p_download_pano(p2p_ctx *ctx, int slot, uint8_t *bgr_host, size_t row_stride);
/* fill everything the slot does not hold with `byte` (0..255), at full capacity: staging, output and table buffers, the
 * scratch of every encoder and decoder (mapped flags and size arrays included), and the rows of the packed panorama, of
 * its gather array and of its folded planes outside the rows the slot holds (plus the pitch padding of the held rows).
 * What the slot holds and the context-wide caches are kept.  Waits for the slot's stream.  P2P_ERR_STATE while a JPEG
 * decode's Huffman verdict is still pending on the slot.  Reuse of the slot then reads the byte wherever a call reads
 * memory it has not written. */
int p2p_debug_poison(p2p_ctx *ctx, int slot, int byte);

#ifdef __cplusplus
}
#endif
#endif /* P2P_B200_H */
