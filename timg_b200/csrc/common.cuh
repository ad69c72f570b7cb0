// Shared internals of libb200timg: context, scratch arena, error plumbing and the
// strict-IEEE float helpers every bit-exact kernel uses.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/b200timg.h"

namespace b200timg {

// A grow-only device buffer (never shrinks; freed with the ctx).
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + (bytes >> 3) + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

struct HostBuf {   // pinned staging
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + (bytes >> 3) + 256;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

}  // namespace b200timg

namespace b200timg { struct ResamplePlan; void free_plan(ResamplePlan *); }

struct b200timg_ctx {
    int device = 0;
    b200timg::ResamplePlan *plan = nullptr;   // cached resampling tables (host copy) ...
    int plan_key[4] = {0, 0, 0, 0};           // ... for this iw, ih, ow, oh (device copy in `tables`)
    long long fixed_geom_key = -1;            // which tile-origin arrays are uploaded behind ctx->misc + 4096
    size_t sixel_idx_off = 0;                 // where the last sixel encode put its index planes
    const void *resident_fb = nullptr;        // host frame whose copy b200timg_has_transparency left in fb_scaled ...
    int resident_w = 0, resident_h = 0;       // ... (cleared by anything else that writes fb_scaled)
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 148;
    uint64_t launches = 0;
    char err[512] = {0};
    // optional per-kernel timing (b200timg_profile): CUDA events on the launching stream
    bool profiling = false;
    const char *pending_kernel = "?";
    struct ProfRec { const char *name; cudaEvent_t begin, end; };
    std::vector<ProfRec> prof;

    // scratch, grown on demand
    b200timg::DevBuf in_stage;     // uploaded source frames (host entry points)
    b200timg::DevBuf fb_scaled;    // scaled (+padded) RGBA framebuffers of a batch
    b200timg::DevBuf prev_stage;   // previous frame for single-frame delta encode
    b200timg::DevBuf out_stage;    // encoded bytes (host entry points)
    b200timg::DevBuf offsets;      // uint64 [n+1]
    b200timg::DevBuf cells;        // per-cell records of the block encoder
    b200timg::DevBuf rows;         // per-rowpair records
    b200timg::DevBuf tables;       // resampler coefficient tables
    b200timg::DevBuf sixel_work;   // palettes, LUTs, index planes, band tables
    b200timg::DevBuf misc;         // small flags / sizes
    b200timg::DevBuf deflate_work; // compressed PNG: per-segment output slots, sizes and offsets (deflate.cu)
    b200timg::DevBuf tri_tables;   // bilinear / YUV scaler tap tables ...
    int tri_key[5] = {0, 0, 0, 0, 0};          // ... for this (kind, iw, ih, ow, oh), device pointers cached in tri_params
    std::vector<char> tri_params;
    int yuv_geom[4] = {0, 0, 0, 0};            // window extents of the tiled YUV kernel for the cached geometry
    bool yuv_geom_valid = false;
    b200timg::DevBuf scale_tmp;    // float4 intermediate + flags of the two-pass scaler (long filters)
    b200timg::DevBuf scale_list;   // work list of tiles the opaque-only scaler hands to the general one
    b200timg::HostBuf pinned;      // staging for sizes / offsets
    b200timg::HostBuf pinned_io;   // staging for pageable payloads
    // host-batch pipeline: upload of chunk k+1 / download of chunk k-1 overlap the kernels of chunk k
    cudaStream_t copy_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev_up[2] = {nullptr, nullptr}, ev_write[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr}, ev_scaled[2] = {nullptr, nullptr}, ev_prep = nullptr;
    cudaEvent_t ev_after_scale = nullptr;      // set by the host pipeline: recorded right after the scaler of a batch call
    b200timg::DevBuf pipe_in[2], pipe_out[2];
    bool pipe_ready = false;
    // slices of a large device-resident batch on their own streams (api.cu: sixel_batch_phases)
    cudaStream_t part_stream[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_part[4] = {nullptr, nullptr, nullptr, nullptr}, ev_fork = nullptr;
    bool parts_ready = false;
    int part_slot = 0, part_slots = 1, part_max_frames = 0;   // which slice is being launched / how many / frames per slice
    bool sixel_attrs_set = false;            // cudaFuncSetAttribute done for this context's device
    // K7 gather (gather.cu): NCCL communicator (owned or attached), its stream and ordering events
    void *nccl_comm = nullptr;
    bool nccl_owned = false;
    int nccl_rank = 0, nccl_nranks = 1;
    cudaStream_t gather_stream = nullptr;
    cudaEvent_t ev_gather_ready = nullptr, ev_gather_done[4] = {nullptr, nullptr, nullptr, nullptr};
    uint64_t gather_seq = 0;
    b200timg::DevBuf gather_status;

    int fail(int code, const char *fmt, ...) {
        va_list ap; va_start(ap, fmt);
        vsnprintf(err, sizeof err, fmt, ap);
        va_end(ap);
        return code;
    }
};

#define B2_CUDA(ctx, call)                                                         \
    do {                                                                           \
        cudaError_t e__ = (call);                                                  \
        if (e__ != cudaSuccess)                                                    \
            return (ctx)->fail(e__ == cudaErrorMemoryAllocation ? B200TIMG_ENOMEM  \
                                                                : B200TIMG_ECUDA,  \
                               "%s:%d %s -> %s", __FILE__, __LINE__, #call,        \
                               cudaGetErrorString(e__));                           \
    } while (0)

#define B2_KERNEL(ctx, kname)                                                      \
    do {                                                                           \
        (ctx)->pending_kernel = (kname);                                           \
        if ((ctx)->profiling) {                                                    \
            b200timg_ctx::ProfRec r__;                                             \
            r__.name = (kname);                                                    \
            cudaEventCreate(&r__.begin); cudaEventCreate(&r__.end);                \
            cudaEventRecord(r__.begin, (ctx)->stream);                             \
            (ctx)->prof.push_back(r__);                                            \
        }                                                                          \
    } while (0)

#define B2_LAUNCH_CHECK(ctx)                                                       \
    do {                                                                           \
        (ctx)->launches++;                                                         \
        if ((ctx)->profiling && !(ctx)->prof.empty())                              \
            cudaEventRecord((ctx)->prof.back().end, (ctx)->stream);                \
        cudaError_t e__ = cudaGetLastError();                                      \
        if (e__ != cudaSuccess)                                                    \
            return (ctx)->fail(B200TIMG_ECUDA, "%s:%d kernel %s launch -> %s",     \
                               __FILE__, __LINE__, (ctx)->pending_kernel,          \
                               cudaGetErrorString(e__));                           \
    } while (0)

#define B2_TRY(expr)                          \
    do {                                      \
        int rc__ = (expr);                    \
        if (rc__ != B200TIMG_OK) return rc__; \
    } while (0)

namespace b200timg {

// ---- strict IEEE-754 single precision, never contracted into FMA ------------------
// The reference is compiled for baseline x86-64 (SSE2, no FMA): every * and + rounds
// separately.  These intrinsics map to single SASS FMUL/FADD/MUFU+fixup and are never
// fused by ptxas, independent of -fmad.
__device__ __forceinline__ float fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fdiv(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float fsqrt(float a) { return __fsqrt_rn(a); }

// LinearColor::gamma (src/framebuffer.h:169-172): sqrt, saturate at 255, truncate.
__device__ __forceinline__ uint32_t ungamma(float v) {
    const float s = fsqrt(v);
    return (s > 255.0f) ? 255u : __float2uint_rz(s);
}

struct __align__(4) px4 { uint8_t r, g, b, a; };

__device__ __forceinline__ uint32_t pack_rgba(uint32_t r, uint32_t g, uint32_t b, uint32_t a) {
    return r | (g << 8) | (b << 16) | (a << 24);
}

// LinearColor::AlphaBlend + repack (src/framebuffer.h:142-161,169-172) of one RGBA8 pixel onto a
// linearised background colour; opaque pixels pass through.
__device__ __forceinline__ uint32_t blend_px(uint32_t p, float bgr, float bgg, float bgb) {
    const uint32_t a8 = p >> 24;
    if (a8 == 0xffu) return p;
    const uint32_t r8 = p & 0xff, g8 = (p >> 8) & 0xff, b8 = (p >> 16) & 0xff;
    const float a = (float)a8, ia = (float)(0xff - a8);
    const float r = fdiv(fadd(fmul((float)(r8 * r8), a), fmul(bgr, ia)), 255.0f);
    const float g = fdiv(fadd(fmul((float)(g8 * g8), a), fmul(bgg, ia)), 255.0f);
    const float b = fdiv(fadd(fmul((float)(b8 * b8), a), fmul(bgb, ia)), 255.0f);
    return pack_rgba(ungamma(r), ungamma(g), ungamma(b), 0xffu);
}

// What AlphaComposeBackground would do to a pixel at (x, y): resolved once on the host.
struct ComposeSpec {
    int active;                  // 0: leave pixels alone (no getter, transparent bg)
    int use_pattern, pw, ph;
    float bg[2][3];              // linearised background and pattern colours
};
inline ComposeSpec make_compose_spec(int has_bg, uint32_t bg, uint32_t pattern, int pw, int ph) {
    ComposeSpec c;
    c.active = (has_bg && (bg >> 24) != 0) ? 1 : 0;                       // src/framebuffer.cc:111,121
    c.use_pattern = !((pattern >> 24) == 0 || pattern == bg || pw <= 0 || ph <= 0);   // :124-125
    c.pw = pw > 0 ? pw : 1; c.ph = ph > 0 ? ph : 1;
    const uint32_t cols[2] = {bg, pattern};
    for (int k = 0; k < 2; ++k)
        for (int ch = 0; ch < 3; ++ch) { const uint32_t v = (cols[k] >> (8 * ch)) & 0xff; c.bg[k][ch] = (float)(v * v); }
    return c;
}
__device__ __forceinline__ uint32_t compose_at(const ComposeSpec &c, uint32_t p, int x, int y) {
    if (!c.active || (p >> 24) == 0xffu) return p;
    const int sel = c.use_pattern ? (((x / c.pw) + (y / c.ph)) & 1) : 0;
    return blend_px(p, c.bg[sel][0], c.bg[sel][1], c.bg[sel][2]);
}

// per-stage launchers (defined in the .cu files); all device pointers
int launch_compose(b200timg_ctx *ctx, uint8_t *d_fb, int w, int h, int n_frames, int has_bg,
                   uint32_t bg, uint32_t pattern, int pw, int ph, int start_row);
int launch_has_transparency(b200timg_ctx *ctx, const uint8_t *d_fb, int w, int h,
                            int start_row, int *d_flag);
// Block encode of n frames of w x h at d_fb (frame stride w*h*4).  prev_mode: 0 none,
// 1 = explicit d_prev (single frame), 2 = animation (frame f vs f-1, frame 0 full).
int launch_blocks(b200timg_ctx *ctx, const uint8_t *d_fb, const uint8_t *d_prev, int prev_mode,
                  int w, int h, int n_frames, int flags, int x_indent, char *d_out,
                  size_t out_cap, uint64_t *d_offsets);
// cs != nullptr fuses AlphaComposeBackground (start_row 0) into the scaler's epilogue.
// fast != 0: the <= 1 LSB arithmetic (FMA, no 1/255 round trip) where a kernel offers it; 0: bit-exact.
int launch_scale(b200timg_ctx *ctx, const uint8_t *d_in, int iw, int ih, int fmt, uint8_t *d_out,
                 int ow, int oh, int out_frame_rows, int n_frames, const ComposeSpec *cs = nullptr, int fast = 0);
// libswscale-style bilinear (triangle) scalers, bilinear.cu: RGBA -> RGBA and YUV 4:2:0 -> RGBA
int launch_scale_bilinear(b200timg_ctx *ctx, const uint8_t *d_in, int iw, int ih, int fmt, uint8_t *d_out, int ow, int oh,
                          int out_frame_rows, int n_frames, const ComposeSpec *cs);
int launch_yuv_scale(b200timg_ctx *ctx, const uint8_t *d_in, int iw, int ih, int fmt, uint8_t *d_out, int ow, int oh,
                     int out_frame_rows, int n_frames);
int launch_sixel(b200timg_ctx *ctx, const uint8_t *d_fb, int w, int h, int n_frames, char *d_out,
                 size_t out_cap, uint64_t *d_offsets, int phases);
int launch_sixel_front(b200timg_ctx *ctx, const uint8_t *d_fb, int w, int h, int n_total, int f0, int n, bool reserve);
int launch_sixel_back(b200timg_ctx *ctx, int w, int h, int n_frames, char *d_out, size_t out_cap, uint64_t *d_offsets, int phases);
int sixel_debug_fetch(b200timg_ctx *ctx, uint32_t *h_palette, uint32_t *h_counts, uint8_t *h_index, size_t index_bytes);

}  // namespace b200timg
