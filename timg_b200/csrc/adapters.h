// C++ adapters that put libb200timg behind the reference's own plugin surface.  This header is
// meant to be compiled INSIDE the timg source tree (it includes timg's headers, which are not part
// of this repository); INTEGRATION.md shows the three call sites that change.  It is
// syntax-checked against /root/reference/src by tests/test_adapters_compile.py when that tree is
// present.
//
//   B200ImageScaler  : timg::ImageScaler      (src/image-scaler.h:24-40)
//   B200AlphaCompose : free function with Framebuffer::AlphaComposeBackground's signature
//                                              (src/framebuffer.h:103-106)
//   B200BlockCanvas  : timg::TerminalCanvas    (src/terminal-canvas.h:28-60), replaces
//                                              UnicodeBlockCanvas (src/unicode-block-canvas.h:33-80)
//   B200SixelCanvas  : timg::TerminalCanvas,   replaces SixelCanvas (src/sixel-canvas.h:29-47)
//   B200ITerm2Canvas / B200KittyCanvas : timg::TerminalCanvas, replace ITerm2GraphicsCanvas / KittyGraphicsCanvas
//                                              (src/iterm2-canvas.h, src/kitty-canvas.h; no tmux passthrough)
//
// Ownership follows the reference (SURVEY 8b): the OutBuffer handed to the write sequencer holds
// a `new char[]` that the writer thread frees; the input Framebuffer is only borrowed during Send.
#ifndef B200TIMG_ADAPTERS_H
#define B200TIMG_ADAPTERS_H

#include <cassert>
#include <cstdio>
#include <ctime>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <utility>

#include "b200timg.h"
#include "buffered-write-sequencer.h"
#include "display-options.h"
#include "framebuffer.h"
#include "image-scaler.h"
#include "terminal-canvas.h"
#include "term-query.h"

namespace timg {

// One context per process and device; timg's loaders run on a thread pool, so calls are serialised.
class B200Context {
public:
    static b200timg_ctx *Get() {
        static B200Context instance;
        return instance.ctx_;
    }
    static std::mutex &Lock() { static std::mutex m; return m; }
    // The reference's methods return void; a failing CUDA call is as fatal as a failing new[].
    static void Check(int rc, const char *what) {
        if (rc == B200TIMG_OK) return;
        fprintf(stderr, "b200timg: %s failed (%d): %s\n", what, rc, b200timg_last_error(Get()));
        abort();
    }

private:
    B200Context() {
        const char *dev = getenv("TIMG_B200_DEVICE");
        const int rc = b200timg_ctx_create(dev ? atoi(dev) : 0, nullptr, &ctx_);
        if (rc != B200TIMG_OK) {   // no CPU fallback by design
            fprintf(stderr, "b200timg: no usable B200 (error %d)\n", rc);
            abort();
        }
    }
    ~B200Context() { b200timg_ctx_destroy(ctx_); }
    b200timg_ctx *ctx_ = nullptr;
};

inline uint32_t B200PackColor(rgba_t c) {
    uint32_t v;
    memcpy(&v, &c, 4);
    return v;
}

// ---- ImageScaler ---------------------------------------------------------------------------
class B200ImageScaler final : public ImageScaler {
public:
    explicit B200ImageScaler(ColorFmt fmt) : fmt_(fmt) {}
    void Scale(Framebuffer &in, Framebuffer *out) final {
        std::lock_guard<std::mutex> l(B200Context::Lock());
        B200Context::Check(
            b200timg_scale_rgba(B200Context::Get(), (const uint8_t *)in.begin(), in.width(), in.height(),
                                fmt_ == ColorFmt::kRGBA ? B200TIMG_FMT_RGBA : B200TIMG_FMT_RGB32,
                                (uint8_t *)out->begin(), out->width(), out->height()),
            "scale");
    }

private:
    const ColorFmt fmt_;
};
// Body for ImageScaler::Create (src/image-scaler.cc:101-115).
inline std::unique_ptr<ImageScaler> B200CreateImageScaler(int, int, ImageScaler::ColorFmt fmt, int, int) {
    return std::unique_ptr<ImageScaler>(new B200ImageScaler(fmt));
}

// ---- Framebuffer::AlphaComposeBackground ----------------------------------------------------
// Same lazy background query as the reference (src/framebuffer.cc:113-121): the getter is only
// called when the frame really has a pixel with alpha < 255 at or after start_row.
inline void B200AlphaComposeBackground(Framebuffer *fb, const Framebuffer::bgcolor_query &get_bg,
                                       rgba_t pattern, int pwidth, int pheight, int start_row = 0) {
    if (!get_bg || start_row >= fb->height()) return;
    std::lock_guard<std::mutex> l(B200Context::Lock());
    int transparent = 0;
    B200Context::Check(b200timg_has_transparency(B200Context::Get(), (const uint8_t *)fb->begin(), fb->width(),
                                                 fb->height(), start_row, &transparent),
                       "has_transparency");
    if (!transparent) return;
    const rgba_t bg = get_bg();
    // the frame is still on the device from the transparency test: compose that copy, one upload in total
    B200Context::Check(b200timg_compose_bg_resident(B200Context::Get(), (uint8_t *)fb->begin(), fb->width(), fb->height(), 1,
                                                    B200PackColor(bg), B200PackColor(pattern), pwidth, pheight, start_row),
                       "compose");
}

// ---- UnicodeBlockCanvas ---------------------------------------------------------------------
class B200BlockCanvas final : public TerminalCanvas {
public:
    B200BlockCanvas(BufferedWriteSequencer *ws, bool use_quarter, bool use_upper_half_block, bool use_256_color)
        : TerminalCanvas(ws),
          quarter_(use_quarter),
          flags_((use_quarter ? B200TIMG_QUARTER : 0) | (use_upper_half_block ? B200TIMG_UPPER : 0) |
                 (use_256_color ? B200TIMG_COLOR8 : 0)) {}

    int cell_height_for_pixels(int pixels) const final { return (pixels - 1) / 2; }   // .h:42-45

    void Send(int x, int dy, const Framebuffer &fb, SeqType seq_type, Duration end_of_frame) override {
        const int w = fb.width(), h = fb.height();
        if (dy < 0) MoveCursorDY(cell_height_for_pixels(dy));                           // .cc:329
        if (quarter_) x /= 2;                                                           // .cc:334
        const bool emit_difference = (x == last_x_indent_) && (last_height_ > 0) && abs(dy) == last_height_ &&
                                     prev_ && prev_->width() == w && prev_->height() == h;   // .cc:344-346
        const size_t bound = b200timg_blocks_bound(w, h) + 64;
        // prefix goes first (.cc:332); it is only known now, and is dropped again if nothing changed
        char *buffer = new char[bound + 4096];
        char *pos = AppendPrefixToBuffer(buffer);
        size_t n = 0;
        {
            std::lock_guard<std::mutex> l(B200Context::Lock());
            B200Context::Check(b200timg_blocks_encode(B200Context::Get(), (const uint8_t *)fb.begin(), w, h,
                                                      emit_difference ? (const uint8_t *)prev_->begin() : nullptr,
                                                      flags_, x, pos, bound, &n),
                               "blocks_encode");
        }
        prev_.reset(new Framebuffer(fb));          // the backing store of .cc:139-152, kept as the frame itself
        last_height_ = h;
        last_x_indent_ = x;
        OutBuffer out(buffer, n ? (size_t)(pos - buffer) + n : 0);                      // .cc:390-395
        write_sequencer_->WriteBuffer(std::move(out), seq_type, end_of_frame);
    }

private:
    const bool quarter_;
    const int flags_;
    std::unique_ptr<Framebuffer> prev_;
    int last_height_ = 0, last_x_indent_ = 0;
};

// ---- SixelCanvas ----------------------------------------------------------------------------
class B200SixelCanvas final : public TerminalCanvas {
public:
    B200SixelCanvas(BufferedWriteSequencer *ws, const SixelOptions &sixel_options, const DisplayOptions &opts)
        : TerminalCanvas(ws), options_(opts), full_cell_jump_(sixel_options.full_cell_jump) {
        if (!sixel_options.known_broken_cursor_placement) {                             // .cc:66-79
            before_ = "\033[80h\033[?7730h\033[?8452l"; after_ = "\r";
        } else {
            before_ = "\033[80l\033[?7730l\033[?8452h"; after_ = "\n";
        }
    }

    int cell_height_for_pixels(int pixels) const final {                                // .cc:157-172
        pixels = -pixels;
        if (full_cell_jump_) return -((RoundToSixel(pixels) - 6) / options_.cell_y_px + 1);
        return -((RoundToSixel(pixels) + options_.cell_y_px - 1) / options_.cell_y_px);
    }

    void Send(int x, int dy, const Framebuffer &fb_orig, SeqType seq_type, Duration end_of_frame) override {
        if (dy < 0) MoveCursorDY(cell_height_for_pixels(dy));                           // .cc:102-105
        MoveCursorDX(x / options_.cell_x_px);
        const int w = fb_orig.width(), hp = RoundToSixel(fb_orig.height());
        Framebuffer fb(w, hp);                                                          // .cc:111-120
        // the pad strip (<= 5 rows) is composed by the reference's own member function, exactly as the reference does
        fb.AlphaComposeBackground(options_.bgcolor_getter, options_.bg_pattern_color,
                                  options_.pattern_size * options_.cell_x_px,
                                  options_.pattern_size * options_.cell_y_px / 2, fb_orig.height());
        std::copy(fb_orig.begin(), fb_orig.end(), fb.begin());
        // One encode pass.  Start with the reference's own guess (.cc:123); the library reports the exact size
        // needed (and writes nothing) should a frame ever exceed it.
        size_t cap = 1024 + (size_t)w * hp * 5, n = 0;
        const size_t extra = 1024;
        char *buffer = new char[cap + extra];
        char *pos = AppendPrefixToBuffer(buffer);
        const size_t prefix_len = (size_t)(pos - buffer);
        pos = (char *)memcpy(pos, before_, strlen(before_)) + strlen(before_);          // .cc:133
        std::lock_guard<std::mutex> l(B200Context::Lock());
        int rc = b200timg_sixel_encode(B200Context::Get(), (const uint8_t *)fb.begin(), w, hp, pos, cap - prefix_len, &n);
        if (rc == B200TIMG_ENOSPC) {
            char *bigger = new char[n + prefix_len + extra];
            memcpy(bigger, buffer, (size_t)(pos - buffer));
            pos = bigger + (pos - buffer);
            delete[] buffer;
            buffer = bigger;
            rc = b200timg_sixel_encode(B200Context::Get(), (const uint8_t *)fb.begin(), w, hp, pos, n, &n);
        }
        B200Context::Check(rc, "sixel_encode");
        pos += n;
        pos = (char *)memcpy(pos, after_, strlen(after_)) + strlen(after_);             // .cc:150
        write_sequencer_->WriteBuffer(OutBuffer(buffer, (size_t)(pos - buffer)), seq_type, end_of_frame);
    }

private:
    static int RoundToSixel(int px) { px += 5; return px - px % 6; }                    // .cc:91-94
    const DisplayOptions &options_;
    const bool full_cell_jump_;
    const char *before_, *after_;
};

// ---- ITerm2GraphicsCanvas / KittyGraphicsCanvas -------------------------------------------------
// The PNG file and its base64 text come from the device (b200timg_png_encode_level at
// DisplayOptions::compress_pixel_level, timg's --compress: 0 stored blocks, 1..9 deflate-compressed, 1 by default);
// the protocol framing is the reference's, byte for byte (src/iterm2-canvas.cc:66-72, src/kitty-canvas.cc:196-226
// without the tmux passthrough variant, which only wraps the same chunks).  Buffers are sized with
// b200timg_png_bound and the framing uses the size the encode returns.  The compressed bytes are not libdeflate's
// but decode to the same pixels.
class B200ITerm2Canvas final : public TerminalCanvas {
public:
    B200ITerm2Canvas(BufferedWriteSequencer *ws, const DisplayOptions &opts) : TerminalCanvas(ws), options_(opts) {}
    int cell_height_for_pixels(int pixels) const final {                                // src/iterm2-canvas.cc:91-95
        assert(pixels <= 0);
        return -((-pixels + options_.cell_y_px - 1) / options_.cell_y_px);
    }
    void Send(int x, int dy, const Framebuffer &fb, SeqType seq_type, Duration end_of_frame) override {
        if (dy < 0) MoveCursorDY(cell_height_for_pixels(dy));
        MoveCursorDX(x / options_.cell_x_px);
        const int w = fb.width(), h = fb.height(), rgb24 = options_.local_alpha_handling ? 1 : 0;
        const size_t png_cap = b200timg_png_bound(w, h, rgb24, options_.compress_pixel_level), b64_cap = b200timg_base64_size(png_cap);
        std::unique_ptr<uint8_t[]> png(new uint8_t[png_cap]);
        std::unique_ptr<char[]> b64(new char[b64_cap]);
        size_t png_size = 0;
        {
            std::lock_guard<std::mutex> l(B200Context::Lock());
            B200Context::Check(b200timg_png_encode_level(B200Context::Get(), (const uint8_t *)fb.begin(), w, h, rgb24,
                                                         options_.compress_pixel_level, png.get(), png_cap, &png_size,
                                                         b64.get(), b64_cap), "png_encode");
        }
        const size_t b64_size = b200timg_base64_size(png_size);
        char *buffer = new char[b64_size + 4096];
        char *pos = AppendPrefixToBuffer(buffer);
        pos += sprintf(pos, "\033]1337;File=size=%d;width=%dpx;height=%dpx;inline=1:", (int)png_size, w, h);   // .cc:66-68
        memcpy(pos, b64.get(), b64_size);
        pos += b64_size;
        *pos++ = '\007';
        *pos++ = '\n';                                                                   // .cc:71-72
        write_sequencer_->WriteBuffer(OutBuffer(buffer, (size_t)(pos - buffer)), seq_type, end_of_frame);
    }

private:
    const DisplayOptions &options_;
};

class B200KittyCanvas final : public TerminalCanvas {
public:
    B200KittyCanvas(BufferedWriteSequencer *ws, const DisplayOptions &opts) : TerminalCanvas(ws), options_(opts) {}
    int cell_height_for_pixels(int pixels) const final {                                // src/kitty-canvas.cc:248-252
        assert(pixels <= 0);
        return -((-pixels + options_.cell_y_px - 1) / options_.cell_y_px);
    }
    void Send(int x, int dy, const Framebuffer &fb, SeqType seq_type, Duration end_of_frame) override {
        if (dy < 0) MoveCursorDY(cell_height_for_pixels(dy));
        MoveCursorDX(x / options_.cell_x_px);
        uint32_t id = 0;                                                                 // .cc:142-172
        switch (seq_type) {
        case SeqType::FrameImmediate: id = CreateId(); break;
        case SeqType::StartOfAnimation: id = CreateId(); CreateId(); animation_id_ = id; flip_buffer_ = 0; break;
        case SeqType::AnimationFrame: ++flip_buffer_; id = animation_id_ + (flip_buffer_ % 2); break;
        case SeqType::ControlWrite: break;
        }
        const int w = fb.width(), h = fb.height(), rgb24 = options_.local_alpha_handling ? 1 : 0;
        const size_t png_cap = b200timg_png_bound(w, h, rgb24, options_.compress_pixel_level), b64_cap = b200timg_base64_size(png_cap);
        std::unique_ptr<uint8_t[]> png(new uint8_t[png_cap]);
        std::unique_ptr<char[]> b64(new char[b64_cap]);
        size_t encoded = 0;
        {
            std::lock_guard<std::mutex> l(B200Context::Lock());
            B200Context::Check(b200timg_png_encode_level(B200Context::Get(), (const uint8_t *)fb.begin(), w, h, rgb24,
                                                         options_.compress_pixel_level, png.get(), png_cap, &encoded,
                                                         b64.get(), b64_cap), "png_encode");
        }
        int png_size = (int)encoded;
        const size_t b64_size = b200timg_base64_size(encoded);
        constexpr int kChunk = 4096, kByteChunk = kChunk / 4 * 3;                        // .cc:43-44
        char *buffer = new char[b64_size + (b64_size / kChunk + 2) * 32 + 4096];
        char *pos = AppendPrefixToBuffer(buffer);
        pos += sprintf(pos, "\033_Ga=T,i=%u,q=2,f=100,m=%d;", id, png_size > kByteChunk);   // .cc:197-203
        const char *src = b64.get();
        while (png_size) {                                                               // .cc:206-219: chunks of <= 4096 base64 characters
            const int chunk_bytes = std::min(png_size, kByteChunk);
            const size_t chars = (size_t)(chunk_bytes + 2) / 3 * 4;                      // every chunk but the last is a multiple of 3 bytes
            memcpy(pos, src, chars); pos += chars; src += chars;
            png_size -= chunk_bytes;
            if (png_size) pos += sprintf(pos, "\033\\\033_Gq=2,m=%d;", png_size > kByteChunk);
        }
        *pos++ = '\033'; *pos++ = '\\';                                                  // .cc:220
        *pos++ = '\n';                                                                   // .cc:227
        write_sequencer_->WriteBuffer(OutBuffer(buffer, (size_t)(pos - buffer)), seq_type, end_of_frame);
    }

private:
    static uint32_t CreateId() {                                                         // .cc:48-53
        static const uint32_t kStart = (uint32_t)time(nullptr) << 7;
        static uint32_t counter = 0;
        counter++;
        return kStart + counter;
    }
    const DisplayOptions &options_;
    uint32_t animation_id_ = 0;
    uint8_t flip_buffer_ = 0;
};

}  // namespace timg
#endif  // B200TIMG_ADAPTERS_H
