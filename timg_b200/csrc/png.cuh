// Shared by png.cu (stored-block PNG) and deflate.cu (compressed PNG): the container geometry of a frame, the
// Sub-filtered scanline stream, the stored-block zlib bytes and the checksum arithmetic.
#pragma once
#include "common.cuh"

namespace b200timg {

struct PngGeom {
    int w, h, bpp;                 // bpp 4 (RGBA, colour type 6) or 3 (RGB, colour type 2)
    long long row_bytes;           // 1 + w*bpp
    long long raw_len;             // h * row_bytes : the filtered scanline stream
    long long nblocks;             // stored deflate blocks of <= 65535 bytes
    long long zlib_len;            // 2 + 5*nblocks + raw_len + 4
    long long png_len;             // 8 + 25 + 12 + zlib_len + 12
    long long idat_data_off;       // offset of the first zlib byte inside the PNG
};

static inline PngGeom png_geom(int w, int h, int rgb24) {
    PngGeom g;
    g.w = w; g.h = h; g.bpp = rgb24 ? 3 : 4;
    g.row_bytes = 1 + (long long)w * g.bpp;
    g.raw_len = g.row_bytes * h;
    g.nblocks = (g.raw_len + 65534) / 65535;
    if (g.nblocks == 0) g.nblocks = 1;
    g.zlib_len = 2 + 5 * g.nblocks + g.raw_len + 4;
    g.idat_data_off = 8 + 25 + 8;
    g.png_len = g.idat_data_off + g.zlib_len + 4 + 12;
    return g;
}

// byte o < g.idat_data_off of a PNG whose zlib stream is zlen bytes: signature, IHDR (its CRC left zero), IDAT length
// and type
__device__ __forceinline__ uint8_t png_head_byte(const PngGeom &g, long long o, long long zlen) {
    if (o < 8) { const uint8_t sig[8] = {0x89, 0x50, 0x4E, 0x47, '\r', '\n', 0x1A, '\n'}; return sig[o]; }
    if (o < 33) {                                                       // IHDR chunk, CRC filled by png_seal_kernel (bytes 29..32)
        const long long k = o - 8;
        const uint8_t hdr[21] = {0, 0, 0, 13, 'I', 'H', 'D', 'R', (uint8_t)(g.w >> 24), (uint8_t)(g.w >> 16), (uint8_t)(g.w >> 8), (uint8_t)g.w,
                                 (uint8_t)(g.h >> 24), (uint8_t)(g.h >> 16), (uint8_t)(g.h >> 8), (uint8_t)g.h, 8, (uint8_t)(g.bpp == 4 ? 6 : 2), 0, 0, 0};
        return k < 21 ? hdr[k] : 0;
    }
    const long long k = o - 33;                                         // IDAT length + type
    const uint8_t hd[8] = {(uint8_t)(zlen >> 24), (uint8_t)(zlen >> 16), (uint8_t)(zlen >> 8), (uint8_t)zlen, 'I', 'D', 'A', 'T'};
    return hd[k];
}
// byte k < 12 of the IEND chunk
__device__ __forceinline__ uint8_t png_iend_byte(long long k) {
    const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xAE, 0x42, 0x60, 0x82};
    return iend[k];
}

// byte c of row y of the filtered scanline stream of one frame (c < row_bytes < 2^31: 32-bit arithmetic)
__device__ __forceinline__ uint8_t raw_byte_yc(const uint8_t *__restrict__ fb, const PngGeom &g, long long y, uint32_t c) {
    if (c == 0) return 1;                                               // filter type: Sub
    const uint32_t x = (c - 1) / (uint32_t)g.bpp, ch = (c - 1) - x * (uint32_t)g.bpp;
    const uint8_t *px = fb + ((long long)y * g.w + x) * 4;
    const uint8_t cur = px[ch];
    return x == 0 ? cur : (uint8_t)(cur - px[(int)ch - 4]);                  // src/timg-png.cc:119-126
}

// byte i of the filtered scanline stream of one frame
__device__ __forceinline__ uint8_t raw_byte(const uint8_t *__restrict__ fb, const PngGeom &g, long long i) {
    const long long y = i / g.row_bytes;
    return raw_byte_yc(fb, g, y, (uint32_t)(i - y * g.row_bytes));
}

// byte d of the stored-block deflate data (the zlib stream without its 2-byte header and Adler-32 trailer)
__device__ __forceinline__ uint8_t stored_data_byte(const uint8_t *__restrict__ fb, const PngGeom &g, long long d) {
    const long long blk = d / 65540, in = d - blk * 65540;              // 5-byte header + up to 65535 bytes
    const long long start = blk * 65535;
    const long long len = min((long long)65535, g.raw_len - start);
    if (in == 0) return blk == g.nblocks - 1 ? 1 : 0;                   // BFINAL, BTYPE = 00 (stored)
    if (in == 1) return (uint8_t)len;
    if (in == 2) return (uint8_t)(len >> 8);
    if (in == 3) return (uint8_t)~len;
    if (in == 4) return (uint8_t)(~len >> 8);
    return raw_byte(fb, g, start + in - 5);
}

__device__ __forceinline__ void put_be32(uint8_t *p, uint32_t v) { p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v; }

// ---- checksums ---------------------------------------------------------------------------------------
constexpr uint32_t CRC_POLY = 0xedb88320u;
__device__ __forceinline__ uint32_t crc_byte(uint32_t c, uint8_t b) {
    c ^= b;
#pragma unroll
    for (int k = 0; k < 8; ++k) c = (c >> 1) ^ (CRC_POLY & (0u - (c & 1u)));
    return c;
}
// a(x) * b(x) mod p(x), reflected representation (the arithmetic of zlib's crc32_combine)
__host__ __device__ inline uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) { p ^= b; if ((a & (m - 1)) == 0) break; }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}
// x^(8*n) mod p(x)
__host__ __device__ inline uint32_t x8nmodp(unsigned long long n) {
    uint32_t sq = multmodp(multmodp(multmodp(1u << 30, 1u << 30), multmodp(1u << 30, 1u << 30)),
                           multmodp(multmodp(1u << 30, 1u << 30), multmodp(1u << 30, 1u << 30)));     // x^8 = (x^1)^8
    uint32_t p = 1u << 31;                                               // x^0
    while (n) { if (n & 1) p = multmodp(sq, p); sq = multmodp(sq, sq); n >>= 1; }
    return p;
}

constexpr int PNG_SEG = 4096;
struct SegSum { uint32_t crc, a, b; };     // finalized CRC-32 of the segment; Adler-32 partial sums of its raw bytes (a without the initial 1)

// The checksum and base64 stages of png.cu.  Frame f's file starts at png + (png_off ? png_off[f] : f * g.png_len)
// and its zlib stream is (zlens ? zlens[f] : g.zlib_len) bytes long; zlens[f] == 0 marks a frame that is not written.
int launch_png_checksums(b200timg_ctx *ctx, const uint8_t *d_frames, const PngGeom &g, int n_frames, uint8_t *d_png,
                         const uint64_t *d_png_off, const uint64_t *d_zlens);
int launch_base64_var(b200timg_ctx *ctx, const uint8_t *d_png, const uint64_t *d_png_off, const uint64_t *d_zlens,
                      int n_frames, char *d_b64, const uint64_t *d_b64_off);
int launch_png(b200timg_ctx *ctx, const uint8_t *d_frames, int w, int h, int n_frames, int rgb24, uint8_t *d_png, char *d_b64);

}  // namespace b200timg
