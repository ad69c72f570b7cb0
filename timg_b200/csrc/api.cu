// The extern "C" surface declared in include/b200timg.h: context management, host-buffer
// entry points (upload -> kernels -> download) and the batched pipelines.
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "common.cuh"

using namespace b200timg;

namespace {

// Every entry point starts here: a context belongs to one device, whatever the caller's current one is.
int check_ctx(b200timg_ctx *ctx) {
    if (!ctx) return B200TIMG_EINVAL;
    B2_CUDA(ctx, cudaSetDevice(ctx->device));
    return B200TIMG_OK;
}

// Upload helper: pageable or pinned host memory -> device, async on the ctx stream.
int upload(b200timg_ctx *ctx, void *dst, const void *src, size_t bytes) {
    B2_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return B200TIMG_OK;
}
int download(b200timg_ctx *ctx, void *dst, const void *src, size_t bytes) {
    B2_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return B200TIMG_OK;
}
int sync(b200timg_ctx *ctx) {
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200TIMG_OK;
}

inline int round_to_sixel(int px) { px += 5; return px - px % 6; }   // src/sixel-canvas.cc:91-94

}  // namespace

extern "C" {

int b200timg_version(void) { return 100; }

int b200timg_ctx_create(int device, void *stream, b200timg_ctx **out) {
    if (!out) return B200TIMG_EINVAL;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
        cudaGetLastError();
        return B200TIMG_ENODEV;   // no CPU fallback by design
    }
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return B200TIMG_ENODEV; }
    b200timg_ctx *ctx = new b200timg_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    if (stream) { ctx->stream = (cudaStream_t)stream; ctx->own_stream = false; }
    else {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete ctx; return B200TIMG_ECUDA;
        }
        ctx->own_stream = true;
    }
    *out = ctx;
    return B200TIMG_OK;
}

void b200timg_ctx_destroy(b200timg_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto &r : ctx->prof) { cudaEventDestroy(r.begin); cudaEventDestroy(r.end); }
    ctx->prof.clear();
    b200timg_gather_shutdown(ctx);
    ctx->gather_status.release();
    ctx->in_stage.release(); ctx->fb_scaled.release(); ctx->prev_stage.release();
    ctx->out_stage.release(); ctx->offsets.release(); ctx->cells.release(); ctx->rows.release();
    ctx->tables.release(); ctx->sixel_work.release(); ctx->misc.release(); ctx->deflate_work.release(); ctx->scale_list.release(); ctx->scale_tmp.release(); ctx->tri_tables.release();
    ctx->pinned.release(); ctx->pinned_io.release();
    for (int i = 0; i < 2; ++i) { ctx->pipe_in[i].release(); ctx->pipe_out[i].release(); }
    if (ctx->parts_ready) {
        for (int i = 0; i < 4; ++i) { cudaStreamSynchronize(ctx->part_stream[i]); cudaStreamDestroy(ctx->part_stream[i]); cudaEventDestroy(ctx->ev_part[i]); }
        cudaEventDestroy(ctx->ev_fork);
    }
    if (ctx->pipe_ready) {
        for (int i = 0; i < 2; ++i) { cudaEventDestroy(ctx->ev_up[i]); cudaEventDestroy(ctx->ev_write[i]); cudaEventDestroy(ctx->ev_d2h[i]); cudaEventDestroy(ctx->ev_scaled[i]); }
        cudaEventDestroy(ctx->ev_prep);
        cudaStreamDestroy(ctx->copy_stream); cudaStreamDestroy(ctx->d2h_stream);
    }
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    if (ctx->plan) free_plan(ctx->plan);
    delete ctx;
}

const char *b200timg_last_error(const b200timg_ctx *ctx) { return ctx ? ctx->err : "null ctx"; }
uint64_t b200timg_kernel_launches(const b200timg_ctx *ctx) { return ctx ? ctx->launches : 0; }

// ---- per-kernel timing --------------------------------------------------------------------
int b200timg_profile(b200timg_ctx *ctx, int enable) {
    if (const int rc = check_ctx(ctx)) return rc;
    cudaStreamSynchronize(ctx->stream);
    for (auto &r : ctx->prof) { cudaEventDestroy(r.begin); cudaEventDestroy(r.end); }
    ctx->prof.clear();
    ctx->profiling = enable != 0;
    return B200TIMG_OK;
}

int b200timg_profile_report(b200timg_ctx *ctx, char *buf, size_t cap) {
    if (!ctx || !buf || cap < 2) return B200TIMG_EINVAL;
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    struct Agg { const char *name; int n; double ms; };
    std::vector<Agg> agg;
    for (auto &r : ctx->prof) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.begin, r.end) != cudaSuccess) { cudaGetLastError(); continue; }
        bool found = false;
        for (auto &a : agg) if (strcmp(a.name, r.name) == 0) { a.n++; a.ms += ms; found = true; break; }
        if (!found) agg.push_back({r.name, 1, (double)ms});
    }
    size_t pos = 0;
    for (auto &a : agg) {
        const int n = snprintf(buf + pos, cap - pos, "%s %d %.6f\n", a.name, a.n, a.ms);
        if (n < 0 || (size_t)n >= cap - pos) return ctx->fail(B200TIMG_ENOSPC, "profile report truncated");
        pos += (size_t)n;
    }
    buf[pos] = 0;
    return B200TIMG_OK;
}

// Encode n device-resident, already scaled + padded + composed frames (w x h, h % 6 == 0).
int b200timg_sixel_dev(b200timg_ctx *ctx, const uint8_t *d_fb, int w, int h, int n_frames, char *d_out,
                       size_t out_cap, uint64_t *d_offsets) {
    B2_TRY(check_ctx(ctx));
    if (!d_fb || !d_out || !d_offsets || w <= 0 || h <= 0 || n_frames <= 0) return ctx->fail(B200TIMG_EINVAL, "sixel_dev: bad args");
    return launch_sixel(ctx, d_fb, w, h, n_frames, d_out, out_cap, d_offsets, 3);
}

// ---- geometry: ImageSource::CalcScaleToFitDisplay, src/image-source.cc:47-153 ------------
int b200timg_calc_fit(const b200timg_fit_opts *o, int img_w, int img_h, int rotated,
                      int *target_w, int *target_h) {
    if (!o || !target_w || !target_h || img_w <= 0 || img_h <= 0) return B200TIMG_EINVAL;
    int width = o->width, height = o->height;
    bool fill_w = o->fill_width != 0, fill_h = o->fill_height != 0;
    float stretch = o->width_stretch;
    if (rotated) {                                   // :52-56
        std::swap(width, height);
        std::swap(fill_w, fill_h);
        stretch = 1.0f / o->width_stretch;
    }
    const float kMaxAccept = 5.0f;                   // :59-63
    if (stretch > kMaxAccept) stretch = kMaxAccept;
    if (stretch < 1 / kMaxAccept) stretch = 1 / kMaxAccept;
    if (stretch > 1.0f) width = (int)((float)width / stretch);      // :65-70
    else height = (int)((float)height * stretch);
    const float wfrac = (float)width / (float)img_w;
    const float hfrac = (float)height / (float)img_h;
    if (!o->upscale && (fill_h || wfrac > 1.0f) && (fill_w || hfrac > 1.0f)) {   // :75-86
        *target_w = img_w; *target_h = img_h;
        if (o->cell_x_px == 2) { *target_w *= 2; return 1; }
        return 0;
    }
    int tw = width, th = height;
    if (fill_w && fill_h) {
        const float f = wfrac > hfrac ? wfrac : hfrac;
        tw = (int)roundf(f * (float)img_w); th = (int)roundf(f * (float)img_h);
    } else if (fill_h) {
        tw = (int)roundf(hfrac * (float)img_w);
    } else if (fill_w) {
        th = (int)roundf(wfrac * (float)img_h);
    } else {
        const float f = wfrac < hfrac ? wfrac : hfrac;
        tw = (int)roundf(f * (float)img_w); th = (int)roundf(f * (float)img_h);
    }
    if (stretch > 1.0f) tw = (int)((float)tw * stretch);            // :120-125
    else th = (int)((float)th / stretch);
    if (o->cell_x_px > 0 && o->cell_x_px <= 2 && o->cell_y_px > 0 && o->cell_y_px <= 2) {
        tw = tw / o->cell_x_px * o->cell_x_px;                      // :129-133
        th = th / o->cell_y_px * o->cell_y_px;
    }
    if (tw <= 0) tw = 1;
    if (th <= 0) th = 1;
    if (o->upscale_integer && tw > img_w && th > img_h) {           // :139-150
        const float aspect = o->cell_x_px == 2 ? 2.0f : 1.0f;
        const float wf = 1.0f * (float)tw / aspect / (float)img_w;
        const float hf = 1.0f * (float)th / (float)img_h;
        const float smaller = wf < hf ? wf : hf;
        if (smaller > 1.0f) {
            const double fl = std::floor((double)smaller);
            tw = (int)((double)aspect * fl * (double)img_w);
            th = (int)(fl * (double)img_h);
        }
    }
    *target_w = tw; *target_h = th;
    return (tw != img_w || th != img_h) ? 1 : 0;
}

int b200timg_as256(uint32_t p) {   // src/framebuffer.h:37-52
    const uint32_t r = p & 0xff, g = (p >> 8) & 0xff, b = (p >> 16) & 0xff;
    if (r == g && g == b) return (int)((232 + (r * 23 / 255)) & 0xff);
    auto cube = [](uint32_t v) -> uint32_t {
        return v < 47 ? 0 : v < 115 ? 1 : v < 155 ? 2 : v < 195 ? 3 : v < 235 ? 4 : 5;
    };
    return (int)(16 + 36 * cube(r) + 6 * cube(g) + cube(b));
}

// ---- compose ---------------------------------------------------------------------------
int b200timg_compose_dev(b200timg_ctx *ctx, uint8_t *d_fb, int w, int h, int n_frames, int has_bg,
                         uint32_t bg, uint32_t pattern, int pw, int ph, int start_row) {
    B2_TRY(check_ctx(ctx));
    if (!d_fb || w <= 0 || h <= 0 || n_frames <= 0) return ctx->fail(B200TIMG_EINVAL, "compose: bad args");
    return launch_compose(ctx, d_fb, w, h, n_frames, has_bg, bg, pattern, pw, ph, start_row);
}

int b200timg_compose_bg(b200timg_ctx *ctx, uint8_t *fb, int w, int h, int has_bg, uint32_t bg,
                        uint32_t pattern, int pw, int ph, int start_row) {
    B2_TRY(check_ctx(ctx));
    if (!fb || w <= 0 || h <= 0) return ctx->fail(B200TIMG_EINVAL, "compose: bad args");
    const size_t bytes = (size_t)w * h * 4;
    ctx->resident_fb = nullptr;
    B2_CUDA(ctx, ctx->fb_scaled.reserve(bytes));
    B2_TRY(upload(ctx, ctx->fb_scaled.p, fb, bytes));
    B2_TRY(launch_compose(ctx, ctx->fb_scaled.as<uint8_t>(), w, h, 1, has_bg, bg, pattern, pw, ph, start_row));
    B2_TRY(download(ctx, fb, ctx->fb_scaled.p, bytes));
    return sync(ctx);
}

// Compose the frame b200timg_has_transparency uploaded last (same fb, w, h) and download the result: the adapter's
// "scan, ask for the background colour only if needed, compose" costs one upload instead of two.
int b200timg_compose_bg_resident(b200timg_ctx *ctx, uint8_t *fb, int w, int h, int has_bg, uint32_t bg,
                                 uint32_t pattern, int pw, int ph, int start_row) {
    B2_TRY(check_ctx(ctx));
    if (!fb || w <= 0 || h <= 0) return ctx->fail(B200TIMG_EINVAL, "compose: bad args");
    if (ctx->resident_fb != fb || ctx->resident_w != w || ctx->resident_h != h)
        return b200timg_compose_bg(ctx, fb, w, h, has_bg, bg, pattern, pw, ph, start_row);     // nothing resident: plain path
    const size_t bytes = (size_t)w * h * 4;
    B2_TRY(launch_compose(ctx, ctx->fb_scaled.as<uint8_t>(), w, h, 1, has_bg, bg, pattern, pw, ph, start_row));
    B2_TRY(download(ctx, fb, ctx->fb_scaled.p, bytes));
    ctx->resident_fb = nullptr;
    return sync(ctx);
}

int b200timg_has_transparency(b200timg_ctx *ctx, const uint8_t *fb, int w, int h, int start_row,
                              int *result) {
    B2_TRY(check_ctx(ctx));
    if (!fb || !result || w <= 0 || h <= 0) return ctx->fail(B200TIMG_EINVAL, "has_transparency: bad args");
    const size_t bytes = (size_t)w * h * 4;
    B2_CUDA(ctx, ctx->fb_scaled.reserve(bytes));
    B2_CUDA(ctx, ctx->misc.reserve(64));
    B2_CUDA(ctx, ctx->pinned.reserve(64));
    B2_TRY(upload(ctx, ctx->fb_scaled.p, fb, bytes));
    B2_TRY(launch_has_transparency(ctx, ctx->fb_scaled.as<uint8_t>(), w, h, start_row < 0 ? 0 : start_row,
                                   ctx->misc.as<int>()));
    B2_TRY(download(ctx, ctx->pinned.p, ctx->misc.p, sizeof(int)));
    B2_TRY(sync(ctx));
    *result = *ctx->pinned.as<int>() ? 1 : 0;
    ctx->resident_fb = fb; ctx->resident_w = w; ctx->resident_h = h;      // still in ctx->fb_scaled for b200timg_compose_bg_resident
    return B200TIMG_OK;
}

// ---- blocks ----------------------------------------------------------------------------
size_t b200timg_blocks_bound(int w, int h) {   // src/unicode-block-canvas.cc:405-424
    const size_t max_cell = 2 + 5 + 11 + 1 + 5 + 11 + 1 + 3;
    const size_t rows = (size_t)(h + 1) / 2;
    return 9 + rows * (9 + (size_t)w * max_cell + 5);
}

int b200timg_blocks_encode(b200timg_ctx *ctx, const uint8_t *fb, int w, int h, const uint8_t *prev_fb,
                           int flags, int x_indent_cells, char *out, size_t cap, size_t *size) {
    B2_TRY(check_ctx(ctx));
    if (!fb || !size || w <= 0 || h <= 0 || (!out && cap)) return ctx->fail(B200TIMG_EINVAL, "blocks: bad args");
    const size_t bytes = (size_t)w * h * 4;
    const size_t bound = b200timg_blocks_bound(w, h) + 32;
    ctx->resident_fb = nullptr;
    B2_CUDA(ctx, ctx->fb_scaled.reserve(bytes));
    B2_CUDA(ctx, ctx->out_stage.reserve(bound));
    B2_CUDA(ctx, ctx->offsets.reserve(2 * sizeof(uint64_t)));
    B2_CUDA(ctx, ctx->pinned.reserve(64));
    B2_TRY(upload(ctx, ctx->fb_scaled.p, fb, bytes));
    if (prev_fb) {
        B2_CUDA(ctx, ctx->prev_stage.reserve(bytes));
        B2_TRY(upload(ctx, ctx->prev_stage.p, prev_fb, bytes));
    }
    B2_TRY(launch_blocks(ctx, ctx->fb_scaled.as<uint8_t>(), prev_fb ? ctx->prev_stage.as<uint8_t>() : nullptr,
                         prev_fb ? 1 : 0, w, h, 1, flags, x_indent_cells, ctx->out_stage.as<char>(), bound,
                         ctx->offsets.as<uint64_t>()));
    B2_TRY(download(ctx, ctx->pinned.p, ctx->offsets.p, 2 * sizeof(uint64_t)));
    B2_TRY(sync(ctx));
    const size_t n = (size_t)ctx->pinned.as<uint64_t>()[1];
    *size = n;
    if (n > cap) return ctx->fail(B200TIMG_ENOSPC, "blocks: need %zu bytes, have %zu", n, cap);
    if (n) { B2_TRY(download(ctx, out, ctx->out_stage.p, n)); B2_TRY(sync(ctx)); }
    return B200TIMG_OK;
}

// ---- scale -----------------------------------------------------------------------------
int b200timg_scale_dev(b200timg_ctx *ctx, const uint8_t *d_in, int iw, int ih, int fmt, uint8_t *d_out,
                       int ow, int oh, int n_frames) {
    B2_TRY(check_ctx(ctx));
    if (!d_in || !d_out || iw <= 0 || ih <= 0 || ow <= 0 || oh <= 0 || n_frames <= 0)
        return ctx->fail(B200TIMG_EINVAL, "scale: bad args");
    return launch_scale(ctx, d_in, iw, ih, fmt, d_out, ow, oh, oh, n_frames);
}

int b200timg_scale_rgba(b200timg_ctx *ctx, const uint8_t *in, int iw, int ih, int fmt, uint8_t *out,
                        int ow, int oh) {
    return b200timg_scale_rgba_mode(ctx, in, iw, ih, fmt, out, ow, oh, 0);
}

int b200timg_scale_rgba_mode(b200timg_ctx *ctx, const uint8_t *in, int iw, int ih, int fmt, uint8_t *out,
                             int ow, int oh, int fast) {
    B2_TRY(check_ctx(ctx));
    if (!in || !out || iw <= 0 || ih <= 0 || ow <= 0 || oh <= 0) return ctx->fail(B200TIMG_EINVAL, "scale: bad args");
    const size_t ib = (size_t)iw * ih * 4, ob = (size_t)ow * oh * 4;
    B2_CUDA(ctx, ctx->in_stage.reserve(ib));
    ctx->resident_fb = nullptr;
    B2_CUDA(ctx, ctx->fb_scaled.reserve(ob));
    B2_TRY(upload(ctx, ctx->in_stage.p, in, ib));
    if (fast == 2) B2_TRY(launch_scale_bilinear(ctx, ctx->in_stage.as<uint8_t>(), iw, ih, fmt, ctx->fb_scaled.as<uint8_t>(), ow, oh, oh, 1, nullptr));
    else B2_TRY(launch_scale(ctx, ctx->in_stage.as<uint8_t>(), iw, ih, fmt, ctx->fb_scaled.as<uint8_t>(), ow, oh, oh, 1, nullptr, fast));
    B2_TRY(download(ctx, out, ctx->fb_scaled.p, ob));
    return sync(ctx);
}

int b200timg_yuv_scale(b200timg_ctx *ctx, const uint8_t *in, int iw, int ih, int fmt, uint8_t *out, int ow, int oh) {
    B2_TRY(check_ctx(ctx));
    const int f = fmt & 0xf;
    if (!in || !out || iw <= 0 || ih <= 0 || ow <= 0 || oh <= 0 || (f != B200TIMG_FMT_I420 && f != B200TIMG_FMT_NV12))
        return ctx->fail(B200TIMG_EINVAL, "yuv_scale: bad args");
    const size_t ib = (size_t)iw * ih + 2 * (size_t)(iw / 2) * (ih / 2), ob = (size_t)ow * oh * 4;
    B2_CUDA(ctx, ctx->in_stage.reserve(ib));
    ctx->resident_fb = nullptr;
    B2_CUDA(ctx, ctx->fb_scaled.reserve(ob));
    B2_TRY(upload(ctx, ctx->in_stage.p, in, ib));
    B2_TRY(launch_yuv_scale(ctx, ctx->in_stage.as<uint8_t>(), iw, ih, fmt, ctx->fb_scaled.as<uint8_t>(), ow, oh, oh, 1));
    B2_TRY(download(ctx, out, ctx->fb_scaled.p, ob));
    return sync(ctx);
}

// ---- sixel -----------------------------------------------------------------------------
size_t b200timg_sixel_bound(int w, int h) {
    // our stream: header + <=256 palette definitions; per 6-row band every column has <= 6
    // (colour, bits) entries of <= 8 bytes ("!nnnnn?" gap + char), plus "#ccc" and "$" per colour and
    // column tile (tiles of <= 4096 columns), plus "-"
    const size_t bands = (size_t)(h + 5) / 6, tiles = (size_t)(w + 4095) / 4096;
    return 32 + 256 * 18 + bands * ((size_t)w * 48 + tiles * 256 * 5 + 1) + 2;
}

int b200timg_sixel_encode(b200timg_ctx *ctx, const uint8_t *fb, int w, int h, char *out, size_t cap,
                          size_t *size) {
    B2_TRY(check_ctx(ctx));
    if (!fb || !size || w <= 0 || h <= 0 || (h % 6) != 0 || (!out && cap))
        return ctx->fail(B200TIMG_EINVAL, "sixel: bad args (height must be a multiple of 6)");
    // one pass: the frame is encoded into a device staging buffer of worst-case size, and exactly the
    // encoded bytes come back (or ENOSPC with the size needed, nothing copied)
    const size_t bytes = (size_t)w * h * 4, bound = b200timg_sixel_bound(w, h);
    ctx->resident_fb = nullptr;
    B2_CUDA(ctx, ctx->fb_scaled.reserve(bytes));
    B2_CUDA(ctx, ctx->out_stage.reserve(bound));
    B2_CUDA(ctx, ctx->offsets.reserve(2 * sizeof(uint64_t)));
    B2_CUDA(ctx, ctx->pinned.reserve(64));
    B2_TRY(upload(ctx, ctx->fb_scaled.p, fb, bytes));
    B2_TRY(launch_sixel(ctx, ctx->fb_scaled.as<uint8_t>(), w, h, 1, ctx->out_stage.as<char>(), bound,
                        ctx->offsets.as<uint64_t>(), 3));
    B2_TRY(download(ctx, ctx->pinned.p, ctx->offsets.p, 2 * sizeof(uint64_t)));
    B2_TRY(sync(ctx));
    const size_t n = (size_t)ctx->pinned.as<uint64_t>()[1];
    *size = n;
    if (n > bound) return ctx->fail(B200TIMG_ECUDA, "sixel: encoded size %zu exceeds the bound %zu", n, bound);
    if (n > cap) return ctx->fail(B200TIMG_ENOSPC, "sixel: need %zu bytes, have %zu", n, cap);
    B2_TRY(download(ctx, out, ctx->out_stage.p, n));
    return sync(ctx);
}

int b200timg_sixel_debug(b200timg_ctx *ctx, uint32_t *palette, uint32_t *counts, uint8_t *index, size_t index_bytes) {
    B2_TRY(check_ctx(ctx));
    return sixel_debug_fetch(ctx, palette, counts, index, index_bytes);
}

// ---- batches -----------------------------------------------------------------------------
static int validate_batch(b200timg_ctx *ctx, const b200timg_batch *b) {
    if (!b || b->n_frames <= 0 || b->src_w <= 0 || b->src_h <= 0 || b->out_w <= 0 || b->out_h <= 0)
        return ctx->fail(B200TIMG_EINVAL, "batch: bad geometry");
    return B200TIMG_OK;
}

static size_t src_frame_bytes(const b200timg_batch *b) {
    const int f = b->src_fmt & 0xf;
    if (f == B200TIMG_FMT_I420 || f == B200TIMG_FMT_NV12) return (size_t)b->src_w * b->src_h + 2 * (size_t)(b->src_w / 2) * (b->src_h / 2);
    return (size_t)b->src_w * b->src_h * 4;
}

// scale stage of a batch: the STB-semantics scaler (exact or B200TIMG_FAST_SCALE), the libswscale-style bilinear
// one (B200TIMG_BILINEAR_SCALE), or colour conversion + bilinear scaling of decoder YUV in one pass
static int batch_scale(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *d_src, uint8_t *d_fb, int frame_rows,
                       const ComposeSpec *cs) {
    const int f = b->src_fmt & 0xf;
    if (f == B200TIMG_FMT_I420 || f == B200TIMG_FMT_NV12)
        return launch_yuv_scale(ctx, d_src, b->src_w, b->src_h, b->src_fmt, d_fb, b->out_w, b->out_h, frame_rows, b->n_frames);
    if (f != B200TIMG_FMT_RGBA && f != B200TIMG_FMT_RGB32) return ctx->fail(B200TIMG_EINVAL, "batch: unknown source format %d", b->src_fmt);
    if (b->flags & B200TIMG_BILINEAR_SCALE)
        return launch_scale_bilinear(ctx, d_src, b->src_w, b->src_h, f, d_fb, b->out_w, b->out_h, frame_rows, b->n_frames, cs);
    return launch_scale(ctx, d_src, b->src_w, b->src_h, f, d_fb, b->out_w, b->out_h, frame_rows, b->n_frames, cs,
                        (b->flags & B200TIMG_FAST_SCALE) != 0);
}

int b200timg_blocks_batch_dev(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *d_src,
                              char *d_out, size_t out_cap, uint64_t *d_offsets) {
    B2_TRY(check_ctx(ctx));
    B2_TRY(validate_batch(ctx, b));
    if (!d_src || !d_out || !d_offsets) return ctx->fail(B200TIMG_EINVAL, "batch: null pointer");
    const size_t fb_bytes = (size_t)b->out_w * b->out_h * 4 * b->n_frames;
    ctx->resident_fb = nullptr;
    B2_CUDA(ctx, ctx->fb_scaled.reserve(fb_bytes));
    uint8_t *d_fb = ctx->fb_scaled.as<uint8_t>();
    const ComposeSpec cs = make_compose_spec(b->has_bg, b->bg, b->pattern, b->pattern_w, b->pattern_h);
    B2_TRY(batch_scale(ctx, b, d_src, d_fb, b->out_h, &cs));
    if (ctx->ev_after_scale) B2_CUDA(ctx, cudaEventRecord(ctx->ev_after_scale, ctx->stream));
    return launch_blocks(ctx, d_fb, nullptr, b->animation == 2 ? 3 : b->animation ? 2 : 0, b->out_w, b->out_h, b->n_frames, b->flags,
                         b->x_indent_cells, d_out, out_cap, d_offsets);
}

// One slice of a sixel batch: scale (+ fused compose), pad strip, then the per-frame front kernels.
static int sixel_slice_front(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *d_src, int f0, int n, bool reserve) {
    const int hp = round_to_sixel(b->out_h);
    const size_t frame_bytes = (size_t)b->out_w * hp * 4;
    uint8_t *d_fb_all = ctx->fb_scaled.as<uint8_t>(), *d_fb = d_fb_all + (size_t)f0 * frame_bytes;
    // scale with AlphaComposeBackground fused into the epilogue (what the sources do, e.g.
    // src/stb-image-source.cc:56-60); then only the pad strip is cleared and composed, exactly the
    // canvas' own start_row = height call (src/sixel-canvas.cc:115-118).
    const ComposeSpec cs = make_compose_spec(b->has_bg, b->bg, b->pattern, b->pattern_w, b->pattern_h);
    b200timg_batch sub = *b;
    sub.n_frames = n;
    B2_TRY(batch_scale(ctx, &sub, d_src + (size_t)f0 * src_frame_bytes(b), d_fb, hp, &cs));
    if (ctx->ev_after_scale) B2_CUDA(ctx, cudaEventRecord(ctx->ev_after_scale, ctx->stream));
    if (hp != b->out_h) {
        B2_CUDA(ctx, cudaMemset2DAsync(d_fb + (size_t)b->out_h * b->out_w * 4, frame_bytes, 0,
                                       (size_t)(hp - b->out_h) * b->out_w * 4, n, ctx->stream));
        B2_TRY(launch_compose(ctx, d_fb, b->out_w, hp, n, b->has_bg, b->bg, b->pattern, b->pattern_w, b->pattern_h, b->out_h));
    }
    return launch_sixel_front(ctx, d_fb_all, b->out_w, hp, b->n_frames, f0, n, reserve);
}

static int parts_init(b200timg_ctx *ctx) {
    if (ctx->parts_ready) return B200TIMG_OK;
    for (int i = 0; i < 4; ++i) {
        B2_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->part_stream[i], cudaStreamNonBlocking));
        B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_part[i], cudaEventDisableTiming));
    }
    B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    ctx->parts_ready = true;
    return B200TIMG_OK;
}

static int sixel_batch_phases(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *d_src,
                              char *d_out, size_t out_cap, uint64_t *d_offsets, int phases) {
    const int hp = round_to_sixel(b->out_h);
    if (phases == 2)     // scaled frames are still in ctx->fb_scaled from the prepare phase
        return launch_sixel_back(ctx, b->out_w, hp, b->n_frames, d_out, out_cap, d_offsets, 2);
    // SixelCanvas::Send (src/sixel-canvas.cc:109-120): pad to a multiple of 6 rows with
    // transparent pixels, compose the background into the pad strip only, keep the rest.
    const size_t frame_bytes = (size_t)b->out_w * hp * 4;
    ctx->resident_fb = nullptr;
    B2_CUDA(ctx, ctx->fb_scaled.reserve(frame_bytes * b->n_frames));
    // Large device-resident batches run as slices on separate streams: the palette and dither kernels of a slice are
    // latency-bound (one CTA per frame), so the scaler and the emitter of the other slices fill the machine meanwhile.
    // Timing runs (b200timg_profile) keep the plain in-order chain so that per-kernel durations stay meaningful.
    int parts = 1;
    // measured (run r2k): 1250 unscaled 720p frames 29.9 -> 28.3 ms with 4 slices; 148 4K frames 14.28 vs 14.25 ms with 2 -- not
    // worth a second launch sequence, so batches below 512 frames stay one in-order chain
    if (phases == 3 && !ctx->profiling && !ctx->ev_after_scale && b->n_frames >= 512) parts = 4;
    if (const char *e = getenv("B200TIMG_PARTS")) parts = std::max(1, std::min(4, std::min(atoi(e), b->n_frames)));
    if (parts == 1) {
        B2_TRY(sixel_slice_front(ctx, b, d_src, 0, b->n_frames, true));
        return launch_sixel_back(ctx, b->out_w, hp, b->n_frames, d_out, out_cap, d_offsets, phases);
    }
    B2_TRY(parts_init(ctx));
    cudaStream_t main_stream = ctx->stream;
    const int per = (b->n_frames + parts - 1) / parts;
    // everything a slice would allocate is sized for the whole batch first: nothing may be re-allocated while slices run
    ctx->part_slots = parts; ctx->part_max_frames = per;
    B2_CUDA(ctx, cudaEventRecord(ctx->ev_fork, main_stream));
    int rc = B200TIMG_OK;
    for (int k = 0; k < parts && rc == B200TIMG_OK; ++k) {
        const int f0 = k * per, n = std::min(per, b->n_frames - f0);
        if (n <= 0) break;
        ctx->stream = ctx->part_stream[k];
        ctx->part_slot = k;
        if (cudaStreamWaitEvent(ctx->stream, ctx->ev_fork, 0) != cudaSuccess) rc = ctx->fail(B200TIMG_ECUDA, "batch: stream wait failed");
        if (rc == B200TIMG_OK) rc = sixel_slice_front(ctx, b, d_src, f0, n, k == 0);
        if (rc == B200TIMG_OK && cudaEventRecord(ctx->ev_part[k], ctx->stream) != cudaSuccess) rc = ctx->fail(B200TIMG_ECUDA, "batch: event record failed");
        if (rc == B200TIMG_OK && cudaStreamWaitEvent(main_stream, ctx->ev_part[k], 0) != cudaSuccess) rc = ctx->fail(B200TIMG_ECUDA, "batch: stream wait failed");
    }
    ctx->stream = main_stream;
    ctx->part_slot = 0; ctx->part_slots = 1; ctx->part_max_frames = 0;
    if (rc != B200TIMG_OK) {                       // leave no slice running behind the caller's back
        for (int k = 0; k < parts; ++k) cudaStreamSynchronize(ctx->part_stream[k]);
        return rc;
    }
    return launch_sixel_back(ctx, b->out_w, hp, b->n_frames, d_out, out_cap, d_offsets, phases);
}

int b200timg_sixel_batch_dev(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *d_src,
                             char *d_out, size_t out_cap, uint64_t *d_offsets) {
    B2_TRY(check_ctx(ctx));
    B2_TRY(validate_batch(ctx, b));
    if (!d_src || !d_out || !d_offsets) return ctx->fail(B200TIMG_EINVAL, "batch: null pointer");
    return sixel_batch_phases(ctx, b, d_src, d_out, out_cap, d_offsets, 3);
}

static int pipe_init(b200timg_ctx *ctx) {
    if (ctx->pipe_ready) return B200TIMG_OK;
    B2_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    B2_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_up[i], cudaEventDisableTiming));
        B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_write[i], cudaEventDisableTiming));
        B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_d2h[i], cudaEventDisableTiming));
        B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_scaled[i], cudaEventDisableTiming));
    }
    B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_prep, cudaEventDisableTiming));
    ctx->pipe_ready = true;
    return B200TIMG_OK;
}

// Host-buffer batch: the batch is cut into chunks; while chunk k runs its kernels, chunk k+1 is
// uploading and chunk k-1's encoded bytes are downloading (three streams, double-buffered staging).
// Per chunk the encoded size is known before anything is written (sixel) or bounded (blocks), so
// the caller's buffer is never overrun and *exactly* the encoded bytes cross PCIe on the way back.
static int batch_host_impl(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *src, char *out,
                           size_t out_cap, uint64_t *offsets, bool sixel);
static int batch_host(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *src, char *out,
                      size_t out_cap, uint64_t *offsets, bool sixel) {
    const int rc = batch_host_impl(ctx, b, src, out, out_cap, offsets, sixel);
    if (rc != B200TIMG_OK && ctx && ctx->pipe_ready) {      // nothing may still be reading or writing the caller's buffers
        cudaStreamSynchronize(ctx->copy_stream); cudaStreamSynchronize(ctx->stream); cudaStreamSynchronize(ctx->d2h_stream);
        cudaGetLastError();
    }
    return rc;
}
static int batch_host_impl(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *src, char *out,
                           size_t out_cap, uint64_t *offsets, bool sixel) {
    B2_TRY(check_ctx(ctx));
    B2_TRY(validate_batch(ctx, b));
    if (!src || !out || !offsets) return ctx->fail(B200TIMG_EINVAL, "batch: null pointer");
    B2_TRY(pipe_init(ctx));
    const size_t frame_bytes = src_frame_bytes(b);
    int chunk = (int)std::max<size_t>(1, ((size_t)672 << 20) / frame_bytes);
    if (const char *e = getenv("B200TIMG_CHUNK_FRAMES")) chunk = std::max(1, atoi(e));      // test knob
    // delta-encoded animations chain frame to frame: every chunk after the first re-uploads its predecessor's last
    // frame as a halo (animation = 2: scaled, used as the reference of the chunk's first frame, not emitted)
    const bool anim = !sixel && b->animation != 0;
    chunk = std::min(chunk, b->n_frames);
    const int n_chunks = (b->n_frames + chunk - 1) / chunk;
    const size_t blocks_bound = sixel ? b200timg_sixel_bound(b->out_w, round_to_sixel(b->out_h)) * (size_t)chunk
                                      : b200timg_blocks_bound(b->out_w, b->out_h) * (size_t)chunk + 64;
    for (int i = 0; i < 2 && i < n_chunks; ++i) B2_CUDA(ctx, ctx->pipe_in[i].reserve(frame_bytes * (chunk + 1)));
    B2_CUDA(ctx, ctx->offsets.reserve((size_t)(chunk + 2) * sizeof(uint64_t)));
    B2_CUDA(ctx, ctx->pinned.reserve((size_t)(chunk + 2) * sizeof(uint64_t)));
    uint64_t *h_offs = ctx->pinned.as<uint64_t>();

    auto upload_chunk = [&](int k) -> int {
        const int i = k & 1, halo = (anim && k > 0) ? 1 : 0;
        const int f0 = k * chunk - halo, nf = std::min(chunk, b->n_frames - k * chunk) + halo;
        B2_CUDA(ctx, cudaMemcpyAsync(ctx->pipe_in[i].p, src + (size_t)f0 * frame_bytes, frame_bytes * nf,
                                     cudaMemcpyHostToDevice, ctx->copy_stream));
        B2_CUDA(ctx, cudaEventRecord(ctx->ev_up[i], ctx->copy_stream));
        return B200TIMG_OK;
    };
    B2_TRY(upload_chunk(0));
    if (n_chunks > 1) B2_TRY(upload_chunk(1));
    size_t base_bytes = 0;
    offsets[0] = 0;
    for (int k = 0; k < n_chunks; ++k) {
        const int i = k & 1, f0 = k * chunk, nf = std::min(chunk, b->n_frames - f0);
        const int halo = (anim && k > 0) ? 1 : 0;             // the sub-batch then starts one frame early
        b200timg_batch sub = *b;
        sub.n_frames = nf + halo;
        if (halo) sub.animation = 2;
        const uint8_t *d_in = ctx->pipe_in[i].as<uint8_t>();
        B2_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_up[i], 0));
        if (k >= 2) B2_CUDA(ctx, cudaEventSynchronize(ctx->ev_d2h[i]));            // pipe_out[i] is free again
        B2_CUDA(ctx, ctx->pipe_out[i].reserve(blocks_bound));
        ctx->ev_after_scale = ctx->ev_scaled[i];                                   // recorded once pipe_in[i] has been consumed
        const int rc_k = sixel ? sixel_batch_phases(ctx, &sub, d_in, ctx->pipe_out[i].as<char>(), blocks_bound, ctx->offsets.as<uint64_t>(), 3)
                               : b200timg_blocks_batch_dev(ctx, &sub, d_in, ctx->pipe_out[i].as<char>(), blocks_bound,
                                                           ctx->offsets.as<uint64_t>());
        ctx->ev_after_scale = nullptr;
        B2_TRY(rc_k);
        if (k + 2 < n_chunks) {                                                    // refill pipe_in[i] as soon as this chunk's scaler is done
            B2_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_scaled[i], 0));
            B2_TRY(upload_chunk(k + 2));
        }
        B2_CUDA(ctx, cudaMemcpyAsync(h_offs, ctx->offsets.p, (size_t)(nf + halo + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        B2_CUDA(ctx, cudaEventRecord(ctx->ev_prep, ctx->stream));
        B2_CUDA(ctx, cudaEventSynchronize(ctx->ev_prep));                          // sizes of this chunk are on the host
        const size_t total = (size_t)h_offs[nf + halo];                            // a halo frame contributes no bytes
        for (int j = 1; j <= nf; ++j) offsets[f0 + j] = base_bytes + h_offs[j + halo];
        if (base_bytes + total > out_cap) {
            return ctx->fail(B200TIMG_ENOSPC, "batch: need more than %zu bytes (have %zu)", base_bytes + total, out_cap);
        }
        if (total > blocks_bound) return ctx->fail(B200TIMG_ECUDA, "batch: encoded size %zu exceeds the staging bound %zu", total, blocks_bound);
        B2_CUDA(ctx, cudaEventRecord(ctx->ev_write[i], ctx->stream));
        B2_CUDA(ctx, cudaStreamWaitEvent(ctx->d2h_stream, ctx->ev_write[i], 0));
        if (total) B2_CUDA(ctx, cudaMemcpyAsync(out + base_bytes, ctx->pipe_out[i].p, total, cudaMemcpyDeviceToHost, ctx->d2h_stream));
        B2_CUDA(ctx, cudaEventRecord(ctx->ev_d2h[i], ctx->d2h_stream));
        base_bytes += total;
    }
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->d2h_stream));
    return sync(ctx);
}

int b200timg_blocks_batch(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *src, char *out,
                          size_t out_cap, uint64_t *offsets) {
    return batch_host(ctx, b, src, out, out_cap, offsets, false);
}
int b200timg_sixel_batch(b200timg_ctx *ctx, const b200timg_batch *b, const uint8_t *src, char *out,
                         size_t out_cap, uint64_t *offsets) {
    return batch_host(ctx, b, src, out, out_cap, offsets, true);
}

}  // extern "C"
