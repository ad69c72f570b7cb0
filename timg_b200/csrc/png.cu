// Kitty / iTerm2 canvases' per-frame encode (SURVEY 8f rank 2): PNG container + base64.
//   png::Encode            src/timg-png.cc:90-152   signature, IHDR, one IDAT (zlib stream of the scanlines, every
//                                                   row filtered with the "Sub" filter, type 1), IEND, CRC per chunk
//   EncodeBase64           src/timg-base64.h:28-53
//   callers                src/kitty-canvas.cc:178-232, src/iterm2-canvas.cc:55-75 (protocol framing stays on the host)
// The reference compresses the filtered scanlines with libdeflate, a third-party library that is not part of its
// tree: the compressed bytes are not pinnable, the PIXELS the stream decodes to are.  Here the zlib stream uses
// stored (uncompressed) deflate blocks -- a valid stream any PNG decoder accepts, whose size is a closed formula,
// so every frame of a batch lands at a fixed offset and all stages are embarrassingly parallel:
//   png_fill_kernel   filter + block headers + chunk headers, one thread per output byte group
//   png_check_kernel  CRC-32 (IDAT) and Adler-32 (zlib) of 4 KB segments, one thread per segment
//   png_seal_kernel   combine the segment checksums (GF(2) polynomial arithmetic for CRC, modular for Adler) and
//                     write the trailers
//   base64_kernel     3 bytes -> 4 characters
// Parity test: the stream parses with Python's zlib/struct and decodes to the source pixels; chunk CRCs verify.
// This is timg's --compress=0.  Levels 1..9 (deflate.cu) reuse the checksum kernels with per-frame offsets and lengths.
#include "png.cuh"

namespace b200timg {

__global__ void __launch_bounds__(256)
png_fill_kernel(const uint8_t *__restrict__ frames, uint8_t *__restrict__ out, PngGeom g, int n_frames) {
    const long long per = g.png_len, total = per * n_frames;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const long long f = t / per, o = t - f * per;
        const uint8_t *fb = frames + f * (long long)g.w * g.h * 4;
        uint8_t v = 0;
        if (o < g.idat_data_off) v = png_head_byte(g, o, g.zlib_len);
        else if (o < g.idat_data_off + g.zlib_len) {
            const long long z = o - g.idat_data_off;
            if (z < 2) v = z == 0 ? 0x78 : 0x01;                       // zlib header: deflate, 32K window, no preset dictionary, level 0
            else if (z >= g.zlib_len - 4) v = 0;                       // Adler-32, filled by png_seal_kernel
            else v = stored_data_byte(fb, g, z - 2);
        } else if (o < g.idat_data_off + g.zlib_len + 4) v = 0;        // IDAT CRC, filled later
        else v = png_iend_byte(o - (g.idat_data_off + g.zlib_len + 4));
        out[t] = v;
    }
}

// one thread per PNG_SEG-byte segment of the region [type "IDAT" .. end of zlib stream] (CRC) and of the raw scanline
// stream (Adler); both are derived from the bytes png_fill_kernel wrote / would write.  png_off / zlens: per-frame file
// offsets and zlib lengths of a compressed batch (nullptr: the fixed stored-block layout); nseg_crc then covers the
// longest possible stream and the segments past a frame's own end are empty.
__global__ void __launch_bounds__(128)
png_check_kernel(const uint8_t *__restrict__ frames, const uint8_t *__restrict__ png, PngGeom g, int n_frames, int nseg_crc, int nseg_raw,
                 SegSum *__restrict__ seg, const uint64_t *__restrict__ png_off, const uint64_t *__restrict__ zlens) {
    const long long per = (long long)nseg_crc + nseg_raw, total = per * n_frames;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const long long f = t / per, s = t - f * per;
        const long long zlen = zlens ? (long long)zlens[f] : g.zlib_len;
        if (zlen == 0) continue;                                       // frame not written (beyond the capacity)
        SegSum r = {0, 0, 0};
        if (s < nseg_crc) {
            const long long lo = s * PNG_SEG, hi = min(lo + PNG_SEG, 4 + zlen);
            const uint8_t *p = png + (png_off ? (long long)png_off[f] : f * g.png_len) + (g.idat_data_off - 4);   // starts at the chunk type
            uint32_t c = 0xffffffffu;
            for (long long i = lo; i < hi; ++i) c = crc_byte(c, p[i]);
            r.crc = c ^ 0xffffffffu;
        } else {
            const long long lo = (s - nseg_crc) * PNG_SEG, hi = min(lo + PNG_SEG, g.raw_len);
            const uint8_t *fb = frames + f * (long long)g.w * g.h * 4;
            uint32_t a = 0, b = 0;
            for (long long i = lo; i < hi; ++i) { a += raw_byte(fb, g, i); b += a; }   // <= 4096 * 255 and its triangle sum: no overflow
            r.a = a % 65521u; r.b = b % 65521u;
        }
        seg[t] = r;
    }
}

__global__ void __launch_bounds__(32)
png_seal_kernel(uint8_t *__restrict__ png, PngGeom g, int nseg_crc, int nseg_raw, const SegSum *__restrict__ seg, uint32_t xn_full,
                const uint64_t *__restrict__ png_off, const uint64_t *__restrict__ zlens) {
    const int f = blockIdx.x;
    if (threadIdx.x != 0) return;
    const long long zlen = zlens ? (long long)zlens[f] : g.zlib_len;
    if (zlen == 0) return;
    uint8_t *p = png + (png_off ? (long long)png_off[f] : (long long)f * g.png_len);
    const SegSum *s = seg + (long long)f * (nseg_crc + nseg_raw);
    // Adler-32 of the raw stream: A = 1 + sum a_i, B = sum over segments (b_i + len_i * A_before_i)
    unsigned long long A = 1, B = 0;
    for (int i = 0; i < nseg_raw; ++i) {
        const long long len = min((long long)PNG_SEG, g.raw_len - (long long)i * PNG_SEG);
        B = (B + s[nseg_crc + i].b + (unsigned long long)(len % 65521) * A) % 65521ull;
        A = (A + s[nseg_crc + i].a) % 65521ull;
    }
    const uint32_t adler = (uint32_t)((B << 16) | A);
    uint8_t *ad = p + g.idat_data_off + zlen - 4;
    put_be32(ad, adler);
    // CRC-32 of "IDAT" + zlib stream: segment CRCs were computed with the Adler field still zero.  CRC is linear over
    // GF(2): crc(m ^ d) = crc(m) ^ crc0(d) for equal lengths (crc0 = without init / final xor), and the 4 Adler bytes
    // are the last 4 bytes of the region, so their contribution is the plain register update over those bytes.
    uint32_t crc = 0;
    const long long region = 4 + zlen;
    for (int i = 0; i < nseg_crc && (long long)i * PNG_SEG < region; ++i) {
        const long long len = min((long long)PNG_SEG, region - (long long)i * PNG_SEG);
        const uint32_t xn = len == PNG_SEG ? xn_full : x8nmodp((unsigned long long)len);
        crc = i == 0 ? s[i].crc : (multmodp(xn, crc) ^ s[i].crc);     // crc32_combine(crc, s[i].crc, len)
    }
    uint32_t d = 0;                                                    // zero-init, no final xor: pure linear part
    for (int k = 0; k < 4; ++k) d = crc_byte(d, ad[k]);
    crc ^= d;
    put_be32(p + g.idat_data_off + zlen, crc);
    // IHDR CRC (17 bytes: type + data)
    uint32_t c = 0xffffffffu;
    for (int k = 12; k < 29; ++k) c = crc_byte(c, p[k]);
    put_be32(p + 29, c ^ 0xffffffffu);
}

// ---- base64 (src/timg-base64.h:28-53): n bytes -> 4*ceil(n/3) characters, per frame ---------------------
// group gi of an n-byte input p -> 4 characters at o
__device__ __forceinline__ void base64_group(const uint8_t *__restrict__ p, long long n, long long gi, char *__restrict__ o) {
    p += gi * 3; o += gi * 4;
    const long long left = n - gi * 3;
    const uint32_t b0 = p[0], b1 = left > 1 ? p[1] : 0, b2 = left > 2 ? p[2] : 0;
    const char *tab = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/";
    o[0] = tab[b0 >> 2];
    o[1] = tab[((b0 & 3) << 4) | (b1 >> 4)];
    o[2] = left > 1 ? tab[((b1 & 15) << 2) | (b2 >> 6)] : '=';
    o[3] = left > 2 ? tab[b2 & 63] : '=';
}

__global__ void __launch_bounds__(256)
base64_kernel(const uint8_t *__restrict__ in, long long in_stride, long long n, char *__restrict__ out, long long out_stride, int n_frames) {
    const long long groups = (n + 2) / 3, total = groups * n_frames;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const long long f = t / groups, gi = t - f * groups;
        base64_group(in + f * in_stride, n, gi, out + f * out_stride);
    }
}

// frames of different lengths: frame blockIdx.y spans in[png_off[f], png_off[f+1]) -> out + b64_off[f]
__global__ void __launch_bounds__(256)
base64_var_kernel(const uint8_t *__restrict__ in, const uint64_t *__restrict__ png_off, const uint64_t *__restrict__ zlens,
                  char *__restrict__ out, const uint64_t *__restrict__ b64_off) {
    const int f = blockIdx.y;
    if (zlens[f] == 0) return;
    const long long n = (long long)(png_off[f + 1] - png_off[f]), groups = (n + 2) / 3;
    for (long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x; gi < groups; gi += (long long)gridDim.x * blockDim.x)
        base64_group(in + png_off[f], n, gi, out + b64_off[f]);
}

static unsigned png_grid(b200timg_ctx *ctx, long long items, int threads) {
    long long b = (items + threads - 1) / threads;
    const long long cap = (long long)ctx->sm_count * 32;
    if (b > cap) b = cap;
    return (unsigned)(b < 1 ? 1 : b);
}

int launch_png_checksums(b200timg_ctx *ctx, const uint8_t *d_frames, const PngGeom &g, int n_frames, uint8_t *d_png,
                         const uint64_t *d_png_off, const uint64_t *d_zlens) {
    const int nseg_crc = (int)((4 + g.zlib_len + PNG_SEG - 1) / PNG_SEG), nseg_raw = (int)((g.raw_len + PNG_SEG - 1) / PNG_SEG);
    B2_CUDA(ctx, ctx->cells.reserve(sizeof(SegSum) * (size_t)(nseg_crc + nseg_raw) * n_frames));
    SegSum *seg = ctx->cells.as<SegSum>();
    B2_KERNEL(ctx, "png_check_kernel");
    png_check_kernel<<<png_grid(ctx, (long long)(nseg_crc + nseg_raw) * n_frames, 128), 128, 0, ctx->stream>>>(d_frames, d_png, g, n_frames, nseg_crc, nseg_raw, seg,
                                                                                                            d_png_off, d_zlens);
    B2_LAUNCH_CHECK(ctx);
    B2_KERNEL(ctx, "png_seal_kernel");
    png_seal_kernel<<<n_frames, 32, 0, ctx->stream>>>(d_png, g, nseg_crc, nseg_raw, seg, x8nmodp(PNG_SEG), d_png_off, d_zlens);
    B2_LAUNCH_CHECK(ctx);
    return B200TIMG_OK;
}

int launch_base64_var(b200timg_ctx *ctx, const uint8_t *d_png, const uint64_t *d_png_off, const uint64_t *d_zlens,
                      int n_frames, char *d_b64, const uint64_t *d_b64_off) {
    B2_KERNEL(ctx, "base64_var_kernel");
    base64_var_kernel<<<dim3(n_frames < ctx->sm_count * 8 ? ctx->sm_count * 8 / n_frames : 1, n_frames), 256, 0, ctx->stream>>>(d_png, d_png_off, d_zlens, d_b64, d_b64_off);
    B2_LAUNCH_CHECK(ctx);
    return B200TIMG_OK;
}

// n frames (RGBA8, device) -> n PNG files at d_png + f * png_len; optionally their base64 text at d_b64 + f * b64_len
int launch_png(b200timg_ctx *ctx, const uint8_t *d_frames, int w, int h, int n_frames, int rgb24, uint8_t *d_png, char *d_b64) {
    const PngGeom g = png_geom(w, h, rgb24);
    if (g.zlib_len > 0x7fffffffll) return ctx->fail(B200TIMG_EINVAL, "png: frame too large for one IDAT chunk");
    B2_KERNEL(ctx, "png_fill_kernel");
    png_fill_kernel<<<png_grid(ctx, g.png_len * n_frames, 256), 256, 0, ctx->stream>>>(d_frames, d_png, g, n_frames);
    B2_LAUNCH_CHECK(ctx);
    B2_TRY(launch_png_checksums(ctx, d_frames, g, n_frames, d_png, nullptr, nullptr));
    if (d_b64) {
        const long long b64_len = (g.png_len + 2) / 3 * 4;
        B2_KERNEL(ctx, "base64_kernel");
        base64_kernel<<<png_grid(ctx, (g.png_len + 2) / 3 * n_frames, 256), 256, 0, ctx->stream>>>(d_png, g.png_len, g.png_len, d_b64, b64_len, n_frames);
        B2_LAUNCH_CHECK(ctx);
    }
    return B200TIMG_OK;
}

}  // namespace b200timg

using namespace b200timg;

extern "C" {

size_t b200timg_png_size(int w, int h, int rgb24) { return (size_t)png_geom(w, h, rgb24).png_len; }
size_t b200timg_base64_size(size_t n) { return (n + 2) / 3 * 4; }

int b200timg_png_batch_dev(b200timg_ctx *ctx, const uint8_t *d_frames, int w, int h, int n_frames, int rgb24, uint8_t *d_png, char *d_b64) {
    if (!ctx) return B200TIMG_EINVAL;
    B2_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!d_frames || !d_png || w <= 0 || h <= 0 || n_frames <= 0) return ctx->fail(B200TIMG_EINVAL, "png: bad args");
    return launch_png(ctx, d_frames, w, h, n_frames, rgb24, d_png, d_b64);
}

// one frame, host buffers: out gets the PNG (b200timg_png_size bytes), b64 (optional) its base64 text
int b200timg_png_encode(b200timg_ctx *ctx, const uint8_t *fb, int w, int h, int rgb24, uint8_t *out, size_t cap, char *b64, size_t b64_cap) {
    if (!ctx) return B200TIMG_EINVAL;
    B2_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!fb || !out || w <= 0 || h <= 0) return ctx->fail(B200TIMG_EINVAL, "png: bad args");
    const size_t n = b200timg_png_size(w, h, rgb24), nb = b200timg_base64_size(n);
    if (cap < n || (b64 && b64_cap < nb)) return ctx->fail(B200TIMG_ENOSPC, "png: need %zu (+%zu base64) bytes", n, nb);
    const size_t bytes = (size_t)w * h * 4;
    ctx->resident_fb = nullptr;
    B2_CUDA(ctx, ctx->in_stage.reserve(bytes));
    B2_CUDA(ctx, ctx->out_stage.reserve((n + 15) / 16 * 16 + nb + 16));
    B2_CUDA(ctx, cudaMemcpyAsync(ctx->in_stage.p, fb, bytes, cudaMemcpyHostToDevice, ctx->stream));
    uint8_t *d_png = ctx->out_stage.as<uint8_t>();
    char *d_b64 = b64 ? ctx->out_stage.as<char>() + (n + 15) / 16 * 16 : nullptr;
    B2_TRY(launch_png(ctx, ctx->in_stage.as<uint8_t>(), w, h, 1, rgb24, d_png, d_b64));
    B2_CUDA(ctx, cudaMemcpyAsync(out, d_png, n, cudaMemcpyDeviceToHost, ctx->stream));
    if (b64) B2_CUDA(ctx, cudaMemcpyAsync(b64, d_b64, nb, cudaMemcpyDeviceToHost, ctx->stream));
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200TIMG_OK;
}

}  // extern "C"
