/* b200timg.h -- C ABI of the B200-native timg hot path.
 *
 * Drop-in boundary for hzeller/timg's per-pixel hot path (paths below are relative to
 * the reference tree):
 *   scale      ImageScaler::Create/Scale                 src/image-scaler.h:33-39, .cc:75-97
 *   compose    Framebuffer::AlphaComposeBackground       src/framebuffer.h:103-106, .cc:108-150
 *   blocks     UnicodeBlockCanvas::Send (+FindBestGlyph, AppendDoubleRow)
 *                                                         src/unicode-block-canvas.cc:162-403
 *   sixel      the libsixel calls inside SixelCanvas::Send's encode lambda
 *                                                         src/sixel-canvas.cc:134-148
 *   geometry   ImageSource::CalcScaleToFitDisplay        src/image-source.cc:47-153
 *
 * Plain pointers and sizes only; no C++/torch types.  All pixel buffers are RGBA8,
 * row-major, tightly packed (src/framebuffer.h:26-61).  Colours passed as uint32_t are
 * the four rgba_t bytes in memory order: r | g<<8 | b<<16 | a<<24.
 *
 * Every entry point runs hand-written sm_100a CUDA kernels.  There is NO CPU fallback:
 * if no CUDA device is usable, b200timg_ctx_create fails with B200TIMG_ENODEV and nothing
 * else can be called.
 *
 * Return value: 0 (B200TIMG_OK) or a negative B200TIMG_E* code; b200timg_last_error()
 * gives a human-readable reason.  The reference's methods return void and cannot fail
 * (src/terminal-canvas.h:39, src/image-scaler.h:38); the adapters in INTEGRATION.md abort
 * on a negative code, which is the reference's behaviour on allocation failure too.
 *
 * Threading: a ctx is thread-compatible (one caller at a time per ctx), like the
 * reference's canvases (src/unicode-block-canvas.h:70-79 are plain members).
 * Current device: every entry point that takes a ctx makes the ctx's device the calling thread's current CUDA
 * device (cudaSetDevice) and leaves it so; hosts that juggle several devices in one thread re-select theirs.
 */
#ifndef B200TIMG_H
#define B200TIMG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200TIMG_OK        0
#define B200TIMG_EINVAL   (-1)  /* bad argument (null pointer, non-positive size, odd width in quarter mode) */
#define B200TIMG_ENOMEM   (-2)  /* device or pinned-host allocation failed */
#define B200TIMG_ECUDA    (-3)  /* a CUDA call or kernel failed; see b200timg_last_error */
#define B200TIMG_ENOSPC   (-4)  /* caller's output buffer too small; *size holds the needed size */
#define B200TIMG_ENODEV   (-5)  /* no usable CUDA device (this library has no CPU path) */

/* flags for the block encoders: UnicodeBlockCanvas ctor args, src/unicode-block-canvas.h:38-39 */
#define B200TIMG_QUARTER   1    /* use_quarter: 2x2 px per cell instead of 1x2 */
#define B200TIMG_UPPER     2    /* use_upper_half_block (TIMG_USE_UPPER_BLOCK) */
#define B200TIMG_COLOR8    4    /* use_256_color (--color8) */
/* batch flag (not a reference option): let the scaler use fused multiply-adds and skip the
 * byte*(1/255) .. *255 round trip where a kernel offers it.  Result within 1 LSB per channel of
 * ImageScaler::Scale's instead of bit-identical.  Meant for -p sixel, whose quantiser is compared
 * by a colour-difference tolerance anyway; never set it for the block modes' byte parity. */
#define B200TIMG_FAST_SCALE 8
/* batch flag: scale RGBA with the libswscale-style bilinear (triangle) filter of the reference's default
 * build (src/image-scaler.cc:45-72) instead of the STB build's Mitchell/box.  libswscale is not part of
 * the reference tree and its result is version/SIMD dependent: parity unpinned, distance measured in tests. */
#define B200TIMG_BILINEAR_SCALE 16

/* input colour formats: ImageScaler::ColorFmt, src/image-scaler.h:26-29 */
#define B200TIMG_FMT_RGBA  0
#define B200TIMG_FMT_RGB32 1    /* BGRA in memory */
/* decoder output of the video source (src/video-source.cc:59-89): planar / semi-planar YUV 4:2:0, converted
 * and scaled to RGBA in one pass (batch entry points and b200timg_yuv_scale only).  A frame is w*h luma bytes
 * followed by the chroma planes (I420: U then V, each (w/2)*(h/2); NV12: interleaved UV); w and h even.
 * Limited ("TV") range BT.601 unless B200TIMG_FMT_FULL_RANGE is or'ed in (the reference's YUVJ formats). */
#define B200TIMG_FMT_I420  2
#define B200TIMG_FMT_NV12  3
#define B200TIMG_FMT_FULL_RANGE 0x10

typedef struct b200timg_ctx b200timg_ctx;

/* device: CUDA ordinal.  stream: a cudaStream_t (as void*) to launch on, or NULL for a
 * stream owned by the ctx. */
int  b200timg_ctx_create(int device, void *stream, b200timg_ctx **out);
void b200timg_ctx_destroy(b200timg_ctx *ctx);
const char *b200timg_last_error(const b200timg_ctx *ctx);
int  b200timg_version(void);
/* Number of this library's kernels launched through ctx since creation. */
uint64_t b200timg_kernel_launches(const b200timg_ctx *ctx);

/* ---- geometry (host only) : ImageSource::CalcScaleToFitDisplay, src/image-source.cc:47-153.
 * Fields mirror DisplayOptions (src/display-options.h:33-55). Returns 1 if the image needs
 * scaling, 0 if not, negative on error. */
typedef struct {
    int width, height;          /* available pixels */
    int cell_x_px, cell_y_px;   /* 1x2 half, 2x2 quarter, font cell size for sixel */
    float width_stretch;
    int upscale, upscale_integer, fill_width, fill_height;
} b200timg_fit_opts;
int b200timg_calc_fit(const b200timg_fit_opts *opts, int img_w, int img_h,
                      int fit_in_rotated, int *target_w, int *target_h);

/* rgba_t::As256TermColor, src/framebuffer.h:37-52 (host helper, used by tests). */
int b200timg_as256(uint32_t rgba);

/* ======================= single frame, HOST buffers ==============================
 * These are the bodies of the reference's methods: they upload, run the kernels,
 * and download inside the call. */

/* ImageScaler::Scale with the STB scaler's semantics (src/image-scaler.cc:75-97):
 * Mitchell when shrinking, BOX when enlarging, point-sample copy at scale 1, edge clamp,
 * alpha-weighted, per axis.  in: iw*ih*4 bytes, out: ow*oh*4 bytes. */
int b200timg_scale_rgba(b200timg_ctx *ctx, const uint8_t *in, int iw, int ih, int fmt,
                        uint8_t *out, int ow, int oh);
/* mode 0: as above; 1: the <= 1 LSB arithmetic described at B200TIMG_FAST_SCALE; 2: the libswscale-style
 * bilinear filter described at B200TIMG_BILINEAR_SCALE. */
int b200timg_scale_rgba_mode(b200timg_ctx *ctx, const uint8_t *in, int iw, int ih, int fmt,
                             uint8_t *out, int ow, int oh, int fast);

/* The video source's sws_scale(decoder YUV -> RGBA at the target size), src/video-source.cc:59-89,352-354:
 * fmt = B200TIMG_FMT_I420 or _NV12 (| B200TIMG_FMT_FULL_RANGE); in: iw*ih*3/2 bytes; out: ow*oh*4 bytes. */
int b200timg_yuv_scale(b200timg_ctx *ctx, const uint8_t *in, int iw, int ih, int fmt,
                       uint8_t *out, int ow, int oh);

/* Framebuffer::AlphaComposeBackground (src/framebuffer.cc:108-150), in place on fb.
 * has_bg==0 models a null bgcolor_getter ("-b none"); the lazy getter itself stays on
 * the C++ side: the adapter resolves it only if this frame has a pixel with a<255
 * (b200timg_has_transparency). */
int b200timg_compose_bg(b200timg_ctx *ctx, uint8_t *fb, int w, int h, int has_bg,
                        uint32_t bg, uint32_t pattern, int pattern_w, int pattern_h,
                        int start_row);
/* b200timg_compose_bg on the copy b200timg_has_transparency(fb, w, h) just uploaded (one upload for "scan, fetch the
 * background colour lazily, compose"); falls back to b200timg_compose_bg if that copy is gone. */
int b200timg_compose_bg_resident(b200timg_ctx *ctx, uint8_t *fb, int w, int h, int has_bg,
                                 uint32_t bg, uint32_t pattern, int pattern_w, int pattern_h,
                                 int start_row);
/* *result = 1 if any pixel at or after start_row has alpha < 255 (the reference's
 * early-out scan, src/framebuffer.cc:113-117). */
int b200timg_has_transparency(b200timg_ctx *ctx, const uint8_t *fb, int w, int h,
                              int start_row, int *result);

/* Worst-case encoded size of one block frame: UnicodeBlockCanvas::RequestBuffers,
 * src/unicode-block-canvas.cc:405-424. */
size_t b200timg_blocks_bound(int w, int h);

/* UnicodeBlockCanvas::Send's image bytes (everything after the prefix):
 * row pairs -> glyph pick -> ANSI bytes, src/unicode-block-canvas.cc:361-399.
 * prev_fb: NULL for a full frame, else the previous frame (same w,h) for
 * emit_difference (:344-346; the backing store equals the previous frame).
 * x_indent_cells: the reference's x after "x /= 2" (:334).
 * *size == 0 means "nothing changed" (:390-395). */
int b200timg_blocks_encode(b200timg_ctx *ctx, const uint8_t *fb, int w, int h,
                           const uint8_t *prev_fb, int flags, int x_indent_cells,
                           char *out, size_t cap, size_t *size);

/* Worst-case encoded size of one sixel frame of w x h (h a multiple of 6).
 * Size limits of the sixel path (the reference has none; both are far beyond any terminal): w <= 99999 and
 * h <= 65536.  Frames up to 4095 px wide take the fast emit kernel, wider ones a column-tiled one. */
size_t b200timg_sixel_bound(int w, int h);

/* What libsixel does inside SixelCanvas::Send (src/sixel-canvas.cc:134-148):
 * sixel_dither_new(256) + sixel_dither_initialize(RGBA8888, LARGE_LUM,
 * REP_AVERAGE_COLORS, QUALITY_AUTO) + sixel_encode: 15-bit histogram -> median cut
 * (<=256) -> Floyd-Steinberg -> DCS q ... ST stream.  fb must already be padded to a
 * multiple of 6 rows (round_to_sixel, :91-94) and composed; alpha is ignored. */
int b200timg_sixel_encode(b200timg_ctx *ctx, const uint8_t *fb, int w, int h,
                          char *out, size_t cap, size_t *size);

/* ======================= batches, many frames per call ===========================
 * A batch is n_frames independent source frames of identical geometry, contiguous in
 * memory (frame f at src + f*src_w*src_h*4).  Each runs
 *     scale (src -> out_w x out_h) -> compose -> encode
 * entirely on the device; the scaled framebuffer never leaves it.  Encoded frames are
 * written back to back into `out`; offsets[f]..offsets[f+1] delimit frame f
 * (offsets has n_frames+1 entries).  This is the unit the renderer's grid
 * (src/renderer.cc:103-148) and the animation loops (src/video-source.cc:298-366)
 * produce one Send() at a time in the reference. */
typedef struct {
    int n_frames;
    int src_w, src_h, src_fmt;
    int out_w, out_h;           /* from b200timg_calc_fit */
    /* compose (DisplayOptions: bgcolor_getter result, bg_pattern_color, pattern_size) */
    int has_bg;
    uint32_t bg, pattern;
    int pattern_w, pattern_h;
    /* block modes */
    int flags;                  /* B200TIMG_QUARTER | _UPPER | _COLOR8 */
    int x_indent_cells;
    int animation;              /* 1: frame f>0 is delta-encoded against frame f-1
                                   (Send with dy == -height, :344-346); frame 0 is full.
                                   2: the same, but frame 0 is a HALO -- scaled and used as frame 1's
                                   predecessor, never emitted (offsets[0] == offsets[1]).  A rank that owns
                                   frames [lo, hi) of a sharded animation passes frames [lo-1, hi) this way
                                   and produces exactly the bytes an unsharded run produces for lo..hi-1. */
} b200timg_batch;

/* Device-resident variants: d_src, d_out, d_offsets are DEVICE pointers; nothing crosses
 * PCIe.  The call is asynchronous on the ctx stream (no size is read back).
 * OUTPUT CAPACITY CONTRACT: the call cannot fail with B200TIMG_ENOSPC because it never learns the sizes on the
 * host.  d_offsets is always complete and exact (d_offsets[n_frames] = the bytes the batch needs); a frame whose
 * end would lie beyond out_cap is NOT written (nothing is ever written out of bounds, earlier frames are intact).
 * The caller therefore either passes out_cap >= n_frames * b200timg_{blocks,sixel}_bound(out_w, padded out_h)
 * (cannot overflow) or compares d_offsets[n_frames] with out_cap when it reads the offsets, and repeats the call
 * with a larger buffer if it is greater -- exactly what the host variants do internally. */
int b200timg_blocks_batch_dev(b200timg_ctx *ctx, const b200timg_batch *b,
                              const uint8_t *d_src, char *d_out, size_t out_cap,
                              uint64_t *d_offsets);
int b200timg_sixel_batch_dev(b200timg_ctx *ctx, const b200timg_batch *b,
                             const uint8_t *d_src, char *d_out, size_t out_cap,
                             uint64_t *d_offsets);

/* Host variants (the plugin-level call): src/out/offsets are HOST pointers (pinned or
 * pageable); upload, kernels, and download of exactly the encoded bytes happen inside. */
int b200timg_blocks_batch(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *src,
                          char *out, size_t out_cap, uint64_t *offsets);
int b200timg_sixel_batch(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *src,
                         char *out, size_t out_cap, uint64_t *offsets);

/* Device-resident single stages, for tests and for callers that keep frames on the GPU
 * (e.g. an NVDEC front end).  All pointers are DEVICE pointers. */
int b200timg_scale_dev(b200timg_ctx *ctx, const uint8_t *d_in, int iw, int ih, int fmt,
                       uint8_t *d_out, int ow, int oh, int n_frames);
int b200timg_compose_dev(b200timg_ctx *ctx, uint8_t *d_fb, int w, int h, int n_frames,
                         int has_bg, uint32_t bg, uint32_t pattern, int pattern_w,
                         int pattern_h, int start_row);

/* The sixel stage alone on n device-resident frames that are already scaled, padded to a
 * multiple of 6 rows and composed (e.g. BASELINE config 5: 1280x720 frames shown unscaled). */
int b200timg_sixel_dev(b200timg_ctx *ctx, const uint8_t *d_fb, int w, int h, int n_frames,
                       char *d_out, size_t out_cap, uint64_t *d_offsets);

/* Per-kernel timing with CUDA events recorded on the ctx stream around every launch.
 * profile(ctx,1) clears and starts, profile(ctx,0) stops and clears.  The report is text, one
 * line per kernel: "<name> <launches> <total_ms>".  Timing adds two event records per launch,
 * so throughput numbers are taken with profiling off. */
int b200timg_profile(b200timg_ctx *ctx, int enable);
int b200timg_profile_report(b200timg_ctx *ctx, char *buf, size_t cap);

/* Introspection for tests: after b200timg_sixel_encode, the palette (256 words r|g<<8|b<<16),
 * counts[0] = palette entries in use, counts[1] = occupied 15-bit histogram cells, and the
 * palette-index plane (w*h bytes) of that frame.  Any pointer may be NULL. */
int b200timg_sixel_debug(b200timg_ctx *ctx, uint32_t *palette, uint32_t *counts, uint8_t *index,
                         size_t index_bytes);

/* Host-only introspection of the resampling plan behind b200timg_scale_* (no GPU needed):
 * the per-axis contributor tables and the pass order that reproduce the reference scaler's
 * arithmetic (third_party/stb/stb_image_resize2.h:3267-3635, 6859-6905).  axis 0 = horizontal,
 * 1 = vertical.  first/count/lead have out_w (or out_h) entries, coeff has entries*widest.
 * flags: bit0 vertical pass first, bit1 plain copy (both axes at scale 1), bit2 horizontal taps
 * use a single accumulator.  Any output pointer may be NULL. */
int b200timg_resample_plan(int in_w, int in_h, int out_w, int out_h, int axis, int *widest,
                           int *flags, int32_t *first, int32_t *count, int32_t *lead,
                           float *coeff, size_t coeff_cap);

/* ======================= geometry passes around the path (SURVEY 8f rank 3, row a15) ===============
 * ApplyExifOp (src/jpeg-source.cc:84-119): mirror each row, then rotate by 0, 180, 90 or -90 degrees exactly as
 * the reference's loops do (90 / -90: out is h x w).  in and out: w*h*4 bytes. */
int b200timg_exif_op(b200timg_ctx *ctx, const uint8_t *fb, int w, int h, int mirror, int angle, uint8_t *out);
int b200timg_exif_op_dev(b200timg_ctx *ctx, const uint8_t *d_in, uint8_t *d_out, int w, int h, int mirror, int angle,
                         int n_frames);
/* --auto-crop = Magick::Image::trim() (src/graphics-magick-source.cc:238-240; GraphicsMagick is not in the tree:
 * its documented rule with fuzz 0 is restated, parity unpinned): rect = {x, y, w, h} of the bounding box of the
 * pixels differing from the corner colours (left and top edges against the top-left pixel, right edge against the
 * top-right, bottom edge against the bottom-left).  A single-colour image keeps its full size. */
int b200timg_trim_bbox(b200timg_ctx *ctx, const uint8_t *fb, int w, int h, int rect_xywh[4]);
/* n_pos windows of dw x dh pixels cut from one w x h image, window k at
 *     ((x0 + dx*(first_pos + k)) mod w, (y0 + dy*(first_pos + k)) mod h), wrapping around
 * -- the scroll animation of src/graphics-magick-source.cc:383-389 (one launch for many positions) and, with
 * n_pos = 1 and dx = dy = 0, a plain crop (--crop-border, :232-237).  out: n_pos * dw*dh*4 bytes. */
int b200timg_windows(b200timg_ctx *ctx, const uint8_t *img, int w, int h, int dw, int dh, long long x0, long long y0,
                     int dx, int dy, long long first_pos, int n_pos, uint8_t *out);
int b200timg_windows_dev(b200timg_ctx *ctx, const uint8_t *d_img, int w, int h, int dw, int dh, long long x0,
                         long long y0, int dx, int dy, long long first_pos, int n_pos, uint8_t *d_out);

/* ======================= Kitty / iTerm2 canvases: PNG + base64 (SURVEY 8f rank 2) ===================
 * png::Encode (src/timg-png.cc:90-152): signature, IHDR, one IDAT holding the zlib stream of the scanlines (each
 * row filtered with "Sub"), IEND.  rgb24 != 0: colour type 2 (png::ColorEncoding::kRGB_24), else RGBA.  The
 * reference deflates with libdeflate (third party, not in its tree) at DisplayOptions::compress_pixel_level
 * (timg's --compress, 1 by default).  The stream here decodes to the same pixels but is not the same bytes.
 * EncodeBase64 (src/timg-base64.h:28-53) of the file goes to b64 when given.  The protocol framing
 * (src/kitty-canvas.cc:196-226, src/iterm2-canvas.cc:66-72) stays in the host adapter.
 *
 * Level 0 (and the calls without a level): stored deflate blocks, exactly b200timg_png_size() bytes.
 * Levels 1..9: the device deflate encoder -- greedy LZ77 over 16 KiB segments whose matches reach 32 KiB back,
 * dynamic / fixed / stored Huffman blocks by exact cost.  All of 1..9 currently run this one level-1-style
 * encoder: a higher level is accepted and not yet stronger.  A frame that would not come out smaller than its
 * stored form is sent stored (the level-0 bytes), so the output never exceeds b200timg_png_size(). */
size_t b200timg_png_size(int w, int h, int rgb24);
size_t b200timg_base64_size(size_t n_bytes);
int b200timg_png_encode(b200timg_ctx *ctx, const uint8_t *fb, int w, int h, int rgb24, uint8_t *out, size_t cap,
                        char *b64, size_t b64_cap);
/* n device-resident frames -> n files at d_png + f*png_size (and their base64 at d_b64 + f*base64_size, or NULL) */
int b200timg_png_batch_dev(b200timg_ctx *ctx, const uint8_t *d_frames, int w, int h, int n_frames, int rgb24,
                           uint8_t *d_png, char *d_b64);
/* Upper bound of a PNG at this level (closed formula, host only); at level 0 it equals b200timg_png_size. */
size_t b200timg_png_bound(int w, int h, int rgb24, int level);
/* One frame, host buffers.  level 0..9 (timg's --compress range; anything else: B200TIMG_EINVAL).
 * *png_size = bytes written.  B200TIMG_ENOSPC (nothing written, *png_size = the need) when cap or b64_cap is too
 * small; cap = b200timg_png_bound() and b64_cap = b200timg_base64_size(cap) always suffice.
 * b64 (optional) receives base64(png) = b200timg_base64_size(*png_size) characters. */
int b200timg_png_encode_level(b200timg_ctx *ctx, const uint8_t *fb, int w, int h, int rgb24, int level,
                              uint8_t *out, size_t cap, size_t *png_size, char *b64, size_t b64_cap);
/* n device-resident frames (n <= 65535) -> files back to back at d_png, frame f at
 * d_png_offsets[f]..d_png_offsets[f+1] (n+1 entries); base64 likewise at d_b64 / d_b64_offsets (d_b64 may be NULL,
 * then d_b64_offsets may be NULL too).  Asynchronous on the ctx stream.  Same OUTPUT CAPACITY CONTRACT as the
 * blocks / sixel *_dev calls: the offsets are always complete and exact; a frame whose file end lies beyond
 * png_cap, or whose text end lies beyond b64_cap, is not written (neither its file nor its text); nothing is ever
 * written out of bounds.  n * b200timg_png_bound() bytes (and their base64 sizes) cannot overflow. */
int b200timg_png_batch_level_dev(b200timg_ctx *ctx, const uint8_t *d_frames, int w, int h, int n_frames,
                                 int rgb24, int level, uint8_t *d_png, size_t png_cap, uint64_t *d_png_offsets,
                                 char *d_b64, size_t b64_cap, uint64_t *d_b64_offsets);

/* ======================= K7: gather of the encoded frames over NCCL ==============================
 * One process per GPU (SURVEY 8e).  The reference is a single process and has no counterpart; frames are
 * independent units, every rank encodes its own batch (b200timg_*_batch_dev) and this call moves the
 * encoded bytes to `root`.  Fixed-slot protocol without any host synchronisation: every rank passes the same
 * slot_bytes (>= the size of any rank's batch, <= the capacity of d_payload); on root, rank r's bytes land at
 * d_dst + r*slot_bytes and frame i of rank r is
 *     [d_dst_offsets[r*(n_frames+1) + i], d_dst_offsets[r*(n_frames+1) + i + 1])   (absolute, inside d_dst).
 * d_dst: nranks*slot_bytes bytes, d_dst_offsets: nranks*(n_frames+1) entries, both only read on root.
 * *d_status (optional, root): bit r set if rank r's batch did not fit its slot (its frames are then truncated
 * at the slot end, nothing is read or written out of bounds).  The transfer runs on the context's gather
 * stream behind the compute stream, so the next batch's kernels overlap it.  b200timg_gather returns a ticket
 * (>= 0) or a negative error; b200timg_gather_wait(ctx, ticket, block_host) orders the compute stream (or the
 * host) after that gather -- call it before consuming d_dst or overwriting d_payload.  The last four gathers
 * can be waited for individually (double-buffered callers wait for the one that used the buffer they reuse). */
#define B200TIMG_NCCL_ID_BYTES 128
int  b200timg_gather_unique_id(char id[B200TIMG_NCCL_ID_BYTES]);            /* ncclGetUniqueId; share it with all ranks */
int  b200timg_gather_init(b200timg_ctx *ctx, const char id[B200TIMG_NCCL_ID_BYTES], int rank, int nranks);   /* ncclCommInitRank */
int  b200timg_gather_attach(b200timg_ctx *ctx, void *nccl_comm, int rank, int nranks);  /* use the caller's ncclComm_t */
void b200timg_gather_shutdown(b200timg_ctx *ctx);
int  b200timg_gather(b200timg_ctx *ctx, const char *d_payload, const uint64_t *d_offsets, int n_frames,
                     size_t slot_bytes, char *d_dst, uint64_t *d_dst_offsets, uint32_t *d_status, int root);
int  b200timg_gather_wait(b200timg_ctx *ctx, int ticket, int block_host);

#ifdef __cplusplus
}
#endif
#endif /* B200TIMG_H */
