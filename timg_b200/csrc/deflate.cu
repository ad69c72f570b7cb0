// Compressed PNG for the kitty / iTerm2 canvases: what png::Encode (src/timg-png.cc:90-152) does with libdeflate at
// DisplayOptions::compress_pixel_level (1 by default, --compress=0..9).  Level 0 is png.cu's stored-block stream;
// levels 1..9 run the one encoder here (a greedy level-1 parse; higher levels are accepted and not yet stronger).
//
// The Sub-filtered scanline stream of each frame is cut into DF_SEG-byte segments, each encoded by one block on its
// own.  A segment's matches may reach back DF_HIST bytes into the same frame (the history is input, known up front),
// so the segments stay independent and lose little against one sequential compressor.
//   deflate_segment_kernel  window -> hash (one bucket per hash, nearest earlier position) -> greedy parse by one
//                           warp -> histograms -> length-limited Huffman codes -> exact bit cost of dynamic, fixed
//                           and stored -> the smallest, bit-packed by the whole block; a segment that is not its
//                           frame's last ends byte-aligned (empty stored block, "sync flush"), the last sets BFINAL
//   deflate_scan_kernel     per-frame prefix sums of the segment sizes -> file offsets, zlib lengths, base64 offsets;
//                           a frame whose stream would not be shorter than the stored one is sent stored (level 0 bytes)
//   deflate_place_kernel    container bytes + segment outputs copied to their final offsets
// then png.cu's checksum kernels (CRC-32 of the variable-length IDAT, Adler-32 of the filtered stream) and base64.
// Every frame's output depends on its pixels only (no atomic-order effects): a batch slice equals the one-frame call.
#include "png.cuh"

namespace b200timg {

constexpr int DF_SEG = 16384;                  // filtered bytes per segment
constexpr int DF_HIST = 32768;                 // how far back a match may reach (the deflate window)
constexpr int DF_WIN = DF_SEG + DF_HIST;
constexpr int DF_HASH_BITS = 14;
constexpr int DF_THREADS = 512;
constexpr int DF_MIN = 4, DF_MAX = 258;        // match lengths
constexpr int DF_SLOT = 16400;                 // >= worst segment output: stored block (5 + DF_SEG) + sync flush (5)
constexpr size_t DF_SMEM = DF_WIN + 4 * DF_SEG + 4 * (1 << DF_HASH_BITS);

// length 3..258 -> symbol 257..285 and its extra bits; distance 1..32768 -> symbol 0..29 and its extra bits
__device__ __forceinline__ void len_code(int len, int &sym, int &nextra, int &extra) {
    if (len == 258) { sym = 285; nextra = 0; extra = 0; return; }
    const int l = len - 3;
    if (l < 8) { sym = 257 + l; nextra = 0; extra = 0; return; }
    const int nb = 31 - __clz(l);
    sym = 257 + 4 * (nb - 1) + ((l >> (nb - 2)) & 3); nextra = nb - 2; extra = l & ((1 << (nb - 2)) - 1);
}
__device__ __forceinline__ void dist_code(int dist, int &sym, int &nextra, int &extra) {
    const int d = dist - 1;
    if (d < 4) { sym = d; nextra = 0; extra = 0; return; }
    const int nb = 31 - __clz(d);
    sym = 2 * nb + ((d >> (nb - 1)) & 1); nextra = nb - 1; extra = d & ((1 << (nb - 1)) - 1);
}
__device__ __forceinline__ int len_extra_bits(int sym) { return sym >= 265 && sym < 285 ? (sym - 261) / 4 : 0; }
__device__ __forceinline__ int dist_extra_bits(int sym) { return sym < 4 ? 0 : sym / 2 - 1; }
__device__ __forceinline__ int fixed_lit_len(int sym) { return sym < 144 ? 8 : sym < 256 ? 9 : sym < 280 ? 7 : 8; }

struct DfShared {
    uint32_t lfreq[288], dfreq[32], clfreq[19];
    uint8_t llen[288], dlen[32], cllen[19];
    uint16_t lcode[288], dcode[32], clcode[19];
    uint16_t rle[320];                          // code-length sequence: symbol | extra << 5
    int sorted[288], A[288];                    // Huffman construction scratch
    unsigned long long cost_dyn, cost_fix;
    uint32_t warp_sum[DF_THREADS / 32 + 1];
    int ntok, nrle, hlit, hdist, hclen, mode;   // mode 0 stored, 1 fixed, 2 dynamic
};

// Length-limited Huffman code lengths of n <= DF_THREADS symbols (whole block): rank sort by (frequency, symbol),
// minimum-redundancy lengths in place (Moffat & Katajainen), then the Kraft-sum repair that caps them at maxbits.
// Fewer than two used symbols get two codes of length 1, as a decoder expects a complete code.
__device__ void huff_lengths(const uint32_t *freq, int n, int maxbits, uint8_t *len, DfShared &S) {
    const int tid = threadIdx.x;
    const bool mine = tid < n && freq[tid] > 0;
    if (tid < n) len[tid] = 0;
    const int nused = __syncthreads_count(mine);
    if (mine) {
        const uint32_t key = freq[tid] << 9 | (uint32_t)tid;
        int r = 0;
        for (int u = 0; u < n; ++u) r += freq[u] > 0 && (freq[u] << 9 | (uint32_t)u) < key;
        S.sorted[r] = tid; S.A[r] = (int)freq[tid];
    }
    __syncthreads();
    if (tid == 0) {
        int *A = S.A;
        if (nused < 2) {
            const int a = nused ? S.sorted[0] : 0;
            len[a] = 1; len[a == 0 ? 1 : 0] = 1;
        } else {
            A[0] += A[1];
            int root = 0, leaf = 2, next;
            for (next = 1; next < nused - 1; ++next) {
                if (leaf >= nused || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = next; } else A[next] = A[leaf++];
                if (leaf >= nused || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = next; } else A[next] += A[leaf++];
            }
            A[nused - 2] = 0;
            for (next = nused - 3; next >= 0; --next) A[next] = A[A[next]] + 1;
            int avbl = 1, used = 0, dpth = 0;
            root = nused - 2; next = nused - 1;
            while (avbl > 0) {
                while (root >= 0 && A[root] == dpth) { ++used; --root; }
                while (avbl > used) { A[next--] = dpth; --avbl; }
                avbl = 2 * used; ++dpth; used = 0;
            }
            int num[33];
            for (int i = 0; i <= 32; ++i) num[i] = 0;
            for (int i = 0; i < nused; ++i) ++num[A[i] < 32 ? A[i] : 32];
            for (int i = maxbits + 1; i <= 32; ++i) num[maxbits] += num[i];
            uint32_t total = 0;
            for (int i = 1; i <= maxbits; ++i) total += (uint32_t)num[i] << (maxbits - i);
            while (total != 1u << maxbits) {
                --num[maxbits];
                for (int i = maxbits - 1; i > 0; --i)
                    if (num[i]) { --num[i]; num[i + 1] += 2; break; }
                --total;
            }
            int j = nused;
            for (int i = 1; i <= maxbits; ++i)
                for (int k = num[i]; k > 0; --k) len[S.sorted[--j]] = (uint8_t)i;
        }
    }
    __syncthreads();
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for the LSB-first writer; one thread
__device__ void huff_codes(const uint8_t *len, int n, uint16_t *code) {
    int cnt[16], next[16];
    for (int b = 0; b < 16; ++b) cnt[b] = 0;
    for (int s = 0; s < n; ++s) ++cnt[len[s]];
    cnt[0] = 0;
    int c = 0;
    for (int b = 1; b < 16; ++b) { c = (c + cnt[b - 1]) << 1; next[b] = c; }
    for (int s = 0; s < n; ++s) {
        const int l = len[s];
        code[s] = l ? (uint16_t)(__brev((uint32_t)next[l]++) >> (32 - l)) : 0;
    }
}

// one writer: append the n low bits of v at bit position pos of a zeroed word buffer
__device__ __forceinline__ void put_bits(uint32_t *w, uint32_t &pos, uint32_t v, int n) {
    if (!n) return;
    const uint32_t i = pos >> 5, sh = pos & 31;
    w[i] |= v << sh;
    if (sh + n > 32) w[i + 1] |= v >> (32 - sh);
    pos += n;
}
// many writers: OR up to 48 bits at pos (disjoint ranges, so the order of the atomics does not matter)
__device__ __forceinline__ void or_bits(uint32_t *w, uint32_t pos, unsigned long long v) {
    const uint32_t i = pos >> 5, sh = pos & 31;
    const unsigned long long lo = v << sh;
    const uint32_t hi = sh ? (uint32_t)(v >> (64 - sh)) : 0u;
    if ((uint32_t)lo) atomicOr(&w[i], (uint32_t)lo);
    if ((uint32_t)(lo >> 32)) atomicOr(&w[i + 1], (uint32_t)(lo >> 32));
    if (hi) atomicOr(&w[i + 2], hi);
}

// exclusive prefix sum over the block; *total gets the sum (same value in every thread)
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t x, uint32_t *warp_sum, uint32_t *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint32_t incl = x;
    for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += o; }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const uint32_t v = lane < nw ? warp_sum[lane] : 0u;
        uint32_t s = v;
        for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(0xffffffffu, s, d); if (lane >= d) s += o; }
        if (lane < nw) warp_sum[lane] = s - v;
        if (lane == 31) warp_sum[nw] = s;
    }
    __syncthreads();
    const uint32_t r = warp_sum[warp] + incl - x;
    *total = warp_sum[nw];
    __syncthreads();
    return r;
}

extern __shared__ __align__(16) uint8_t df_smem[];

__global__ void __launch_bounds__(DF_THREADS, 1)
deflate_segment_kernel(const uint8_t *__restrict__ frames, PngGeom g, int nseg, uint8_t *__restrict__ slots,
                       uint32_t *__restrict__ seg_bytes) {
    __shared__ DfShared S;
    uint8_t *win = df_smem;                                              // history + segment bytes
    uint32_t *tok = reinterpret_cast<uint32_t *>(df_smem + DF_WIN);      // match candidates, then the token list
    uint32_t *head = tok + DF_SEG;                                       // hash heads (position + 1), then the output bits
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long blk = blockIdx.x, f = blk / nseg, s = blk - f * nseg;
    const uint8_t *fb = frames + f * (long long)g.w * g.h * 4;
    const long long seg_lo = s * DF_SEG, seg_hi = min(seg_lo + DF_SEG, g.raw_len), hist_lo = max(0ll, seg_lo - DF_HIST);
    const int wlen = (int)(seg_hi - hist_lo), ss = (int)(seg_lo - hist_lo), slen = wlen - ss;
    const bool last = s == nseg - 1;

    // 1. the window of the filtered stream
    {
        const long long y0 = hist_lo / g.row_bytes;
        const uint32_t rb = (uint32_t)g.row_bytes, c0 = (uint32_t)(hist_lo - y0 * g.row_bytes);
        for (int i = tid; i < wlen; i += DF_THREADS) {
            const uint32_t t = c0 + (uint32_t)i, dy = t / rb;
            win[i] = raw_byte_yc(fb, g, y0 + dy, t - dy * rb);
        }
    }
    for (int i = tid; i < (1 << DF_HASH_BITS); i += DF_THREADS) head[i] = 0;
    for (int i = tid; i < 288; i += DF_THREADS) S.lfreq[i] = 0;
    if (tid < 32) S.dfreq[tid] = 0;
    if (tid < 19) S.clfreq[tid] = 0;
    if (tid == 0) { S.cost_dyn = 0; S.cost_fix = 0; }
    __syncthreads();

    // 2. every position's candidate: the nearest earlier position with the same hash of 4 bytes.  Chunks of
    //    DF_THREADS positions; inside a warp __match_any_sync finds the nearest earlier lane, otherwise the bucket head
    //    as it stood before the chunk.  The last position of each hash in the chunk becomes the head (atomicMax).
    for (int base = 0; base < wlen; base += DF_THREADS) {
        const int i = base + tid;
        const bool valid = i + DF_MIN <= wlen;
        uint32_t h = (1u << DF_HASH_BITS) + lane;                        // distinct dummy keys for invalid lanes
        if (valid) {
            const uint32_t v = win[i] | (uint32_t)win[i + 1] << 8 | (uint32_t)win[i + 2] << 16 | (uint32_t)win[i + 3] << 24;
            h = (v * 0x1E35A7BDu) >> (32 - DF_HASH_BITS);
        }
        const unsigned mask = __match_any_sync(0xffffffffu, h);
        const unsigned lower = mask & ((1u << lane) - 1u);
        uint32_t cand = 0;
        if (valid) cand = lower ? (uint32_t)(i - lane + (31 - __clz((int)lower))) + 1u : head[h];
        if (i >= ss && i < wlen) tok[i - ss] = cand;
        __syncthreads();
        if (valid && (mask >> lane) == 1u) atomicMax(&head[h], (uint32_t)i + 1u);
        __syncthreads();
    }

    // 3. greedy parse by warp 0, 32 positions at a time: a ballot of the positions whose candidate matches 4 bytes,
    //    literal runs written in parallel, each match extended 32 bytes per step.  Tokens are compacted into tok[]
    //    in place (a token never lands beyond the position it starts at).  The other warps clear the output buffer.
    if (warp == 0) {
        int nxt = ss, ntok = 0;
        while (nxt < wlen) {
            const int base = ss + ((nxt - ss) & ~31);
            const int i = base + lane;
            int cand = -1;
            bool ok = false;
            if (i >= nxt && i + DF_MIN <= wlen) {
                const uint32_t c = tok[i - ss];
                if (c && i - (int)(c - 1) <= DF_HIST) {
                    cand = (int)c - 1;
                    ok = win[i] == win[cand] && win[i + 1] == win[cand + 1] && win[i + 2] == win[cand + 2] && win[i + 3] == win[cand + 3];
                }
            }
            const unsigned M = __ballot_sync(0xffffffffu, ok);
            const int end = min(base + 32, wlen);
            while (nxt < end) {
                const unsigned m = M & (0xffffffffu << (nxt - base));
                const int stop = m ? base + __ffs((int)m) - 1 : end;
                if (lane < stop - nxt) tok[ntok + lane] = win[nxt + lane];
                ntok += stop - nxt;
                nxt = stop;
                if (!m) break;
                const int p = stop, c = __shfl_sync(0xffffffffu, cand, p - base);
                const int maxlen = min(DF_MAX, wlen - p);
                int len = DF_MIN;
                while (len < maxlen) {
                    const int k = len + lane;
                    const bool diff = k >= maxlen || win[p + k] != win[c + k];
                    const unsigned d = __ballot_sync(0xffffffffu, diff);
                    if (d) { len += __ffs((int)d) - 1; break; }
                    len += 32;
                }
                if (lane == 0) tok[ntok] = 0x80000000u | (uint32_t)len << 16 | (uint32_t)(p - c - 1);
                ++ntok;
                nxt = p + len;
            }
            __syncwarp();
        }
        if (lane == 0) S.ntok = ntok;
    } else {
        for (int i = tid - 32; i < DF_SLOT / 4 + 4; i += DF_THREADS - 32) head[i] = 0;
    }
    __syncthreads();
    const int ntok = S.ntok;

    // 4. histograms
    for (int t = tid; t < ntok; t += DF_THREADS) {
        const uint32_t v = tok[t];
        if (!(v >> 31)) atomicAdd(&S.lfreq[v], 1u);
        else {
            int sym, ne, ex;
            len_code((int)(v >> 16 & 0x1ff), sym, ne, ex);
            atomicAdd(&S.lfreq[sym], 1u);
            dist_code((int)(v & 0xffff) + 1, sym, ne, ex);
            atomicAdd(&S.dfreq[sym], 1u);
        }
    }
    if (tid == 0) S.lfreq[256] = 1;                                      // end of block
    __syncthreads();

    // 5. dynamic codes, their header and the exact cost of each block type
    huff_lengths(S.lfreq, 288, 15, S.llen, S);                        // 286, 287: never used, length 0
    huff_lengths(S.dfreq, 30, 15, S.dlen, S);
    if (tid == 0) {
        int hlit = 286, hdist = 30;
        while (hlit > 257 && !S.llen[hlit - 1]) --hlit;
        while (hdist > 1 && !S.dlen[hdist - 1]) --hdist;
        S.hlit = hlit; S.hdist = hdist;
        const int n = hlit + hdist;
        int nr = 0, i = 0;
        while (i < n) {
            const int v = i < hlit ? S.llen[i] : S.dlen[i - hlit];
            int run = 1;
            while (i + run < n && (i + run < hlit ? S.llen[i + run] : S.dlen[i + run - hlit]) == v) ++run;
            int r = run;
            if (v == 0) {
                while (r >= 11) { const int k = min(r, 138); S.rle[nr++] = (uint16_t)(18 | (k - 11) << 5); r -= k; }
                if (r >= 3) { S.rle[nr++] = (uint16_t)(17 | (r - 3) << 5); r = 0; }
                while (r-- > 0) S.rle[nr++] = 0;
            } else {
                S.rle[nr++] = (uint16_t)v; --r;
                while (r >= 3) { const int k = min(r, 6); S.rle[nr++] = (uint16_t)(16 | (k - 3) << 5); r -= k; }
                while (r-- > 0) S.rle[nr++] = (uint16_t)v;
            }
            i += run;
        }
        S.nrle = nr;
        for (int k = 0; k < nr; ++k) ++S.clfreq[S.rle[k] & 31];
    }
    __syncthreads();
    huff_lengths(S.clfreq, 19, 7, S.cllen, S);
    if (tid < 286 && S.lfreq[tid]) {
        const unsigned long long fr = S.lfreq[tid], ex = (unsigned long long)len_extra_bits(tid);
        atomicAdd(&S.cost_dyn, fr * (S.llen[tid] + ex));
        atomicAdd(&S.cost_fix, fr * (fixed_lit_len(tid) + ex));
    } else if (tid >= 288 && tid < 318 && S.dfreq[tid - 288]) {
        const int d = tid - 288;
        const unsigned long long fr = S.dfreq[d], ex = (unsigned long long)dist_extra_bits(d);
        atomicAdd(&S.cost_dyn, fr * (S.dlen[d] + ex));
        atomicAdd(&S.cost_fix, fr * (5 + ex));
    }
    __syncthreads();
    if (tid == 0) {
        const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        int hclen = 19;
        while (hclen > 4 && !S.cllen[order[hclen - 1]]) --hclen;
        S.hclen = hclen;
        unsigned long long hdr = 3 + 5 + 5 + 4 + 3ull * hclen;
        for (int k = 0; k < S.nrle; ++k) {
            const int sym = S.rle[k] & 31;
            hdr += S.cllen[sym] + (sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0);
        }
        const unsigned long long dyn = hdr + S.cost_dyn, fix = 3 + S.cost_fix, stored = 40 + 8ull * slen;
        S.mode = stored <= dyn && stored <= fix ? 0 : fix <= dyn ? 1 : 2;
        if (S.mode == 1) {                                               // RFC 1951 3.2.6
            for (int k = 0; k < 288; ++k) S.llen[k] = (uint8_t)fixed_lit_len(k);
            for (int k = 0; k < 30; ++k) S.dlen[k] = 5;
        }
    }
    __syncthreads();
    const int mode = S.mode;
    uint8_t *out = slots + blk * (long long)DF_SLOT;
    if (mode == 0) {                                                     // stored: header, LEN, NLEN, the bytes
        if (tid == 0) {
            out[0] = last ? 1 : 0;
            out[1] = (uint8_t)slen; out[2] = (uint8_t)(slen >> 8);
            out[3] = (uint8_t)~slen; out[4] = (uint8_t)(~slen >> 8);
            seg_bytes[blk] = 5u + (uint32_t)slen;
        }
        for (int i = tid; i < slen; i += DF_THREADS) out[5 + i] = win[ss + i];
        return;
    }
    if (tid == 0) huff_codes(S.llen, 288, S.lcode);
    else if (tid == 32) huff_codes(S.dlen, 30, S.dcode);
    else if (tid == 64 && mode == 2) huff_codes(S.cllen, 19, S.clcode);
    __syncthreads();

    // 6. bit packing: the block header by one thread, then the tokens by the whole block (prefix sum of their bit lengths)
    uint32_t *bits = head;
    uint32_t pos = 0;
    if (tid == 0) {
        put_bits(bits, pos, (last ? 1u : 0u) | (uint32_t)mode << 1, 3);
        if (mode == 2) {
            const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
            put_bits(bits, pos, S.hlit - 257, 5);
            put_bits(bits, pos, S.hdist - 1, 5);
            put_bits(bits, pos, S.hclen - 4, 4);
            for (int k = 0; k < S.hclen; ++k) put_bits(bits, pos, S.cllen[order[k]], 3);
            for (int k = 0; k < S.nrle; ++k) {
                const int sym = S.rle[k] & 31, ex = S.rle[k] >> 5;
                put_bits(bits, pos, S.clcode[sym], S.cllen[sym]);
                if (sym >= 16) put_bits(bits, pos, ex, sym == 16 ? 2 : sym == 17 ? 3 : 7);
            }
        }
        S.warp_sum[0] = pos;
    }
    __syncthreads();
    pos = S.warp_sum[0];
    __syncthreads();
    for (int base = 0; base < ntok; base += DF_THREADS) {
        const int t = base + tid;
        unsigned long long v = 0;
        int n = 0;
        if (t < ntok) {
            const uint32_t x = tok[t];
            if (!(x >> 31)) { v = S.lcode[x]; n = S.llen[x]; }
            else {
                int sym, ne, ex;
                len_code((int)(x >> 16 & 0x1ff), sym, ne, ex);
                v = S.lcode[sym]; n = S.llen[sym];
                v |= (unsigned long long)ex << n; n += ne;
                dist_code((int)(x & 0xffff) + 1, sym, ne, ex);
                v |= (unsigned long long)S.dcode[sym] << n; n += S.dlen[sym];
                v |= (unsigned long long)ex << n; n += ne;
            }
        }
        uint32_t total;
        const uint32_t off = block_excl_scan((uint32_t)n, S.warp_sum, &total);
        if (n) or_bits(bits, pos + off, v);
        pos += total;
    }
    __syncthreads();
    if (tid == 0) {
        put_bits(bits, pos, S.lcode[256], S.llen[256]);                 // end of block
        if (!last) {                                                     // sync flush: empty stored block, byte-aligned
            pos += 3;
            pos = (pos + 7) & ~7u;
            put_bits(bits, pos, 0xffff0000u, 32);
        }
        S.warp_sum[0] = (pos + 7) >> 3;
    }
    __syncthreads();
    const uint32_t nbytes = S.warp_sum[0];
    uint32_t *o32 = reinterpret_cast<uint32_t *>(out);
    for (uint32_t i = tid; i < (nbytes + 3) / 4; i += DF_THREADS) o32[i] = bits[i];
    if (tid == 0) seg_bytes[blk] = nbytes;
}

// One block: per frame, the exclusive prefix sum of its segment sizes; then, serially over frames, the zlib length
// (or the stored one when compression does not pay), file and base64 offsets, and whether the frame fits.
__global__ void __launch_bounds__(1024)
deflate_scan_kernel(const uint32_t *__restrict__ seg_bytes, uint32_t *__restrict__ seg_off, int nseg, int n_frames, PngGeom g,
                    unsigned long long png_cap, unsigned long long b64_cap, int want_b64, uint64_t *__restrict__ png_off,
                    uint64_t *__restrict__ b64_off, uint64_t *__restrict__ zlens, uint32_t *__restrict__ stored) {
    __shared__ uint32_t ws[33];
    for (int f = 0; f < n_frames; ++f) {
        uint32_t carry = 0;
        for (int base = 0; base < nseg; base += blockDim.x) {
            const int s = base + threadIdx.x;
            const uint32_t x = s < nseg ? seg_bytes[(long long)f * nseg + s] : 0u;
            uint32_t total;
            const uint32_t e = block_excl_scan(x, ws, &total);
            if (s < nseg) seg_off[(long long)f * nseg + s] = carry + e;
            carry += total;
        }
        if (threadIdx.x == 0) zlens[f] = 2ull + carry + 4ull;
    }
    if (threadIdx.x != 0) return;
    unsigned long long off = 0, boff = 0;
    for (int f = 0; f < n_frames; ++f) {
        unsigned long long z = zlens[f];
        const bool st = z >= (unsigned long long)g.zlib_len;
        if (st) z = (unsigned long long)g.zlib_len;
        const unsigned long long len = (unsigned long long)g.idat_data_off + z + 16;
        png_off[f] = off;
        if (b64_off) b64_off[f] = boff;
        off += len; boff += (len + 2) / 3 * 4;
        const bool fits = off <= png_cap && (!want_b64 || boff <= b64_cap);
        zlens[f] = fits ? z : 0;
        stored[f] = st;
    }
    png_off[n_frames] = off;
    if (b64_off) b64_off[n_frames] = boff;
}

// block (frame, segment): the segment's bytes to their place in the file; segment 0 also writes the container head,
// the last segment the (zeroed) trailers and IEND.  A frame sent stored gets png.cu's stored-block bytes instead.
__global__ void __launch_bounds__(256)
deflate_place_kernel(const uint8_t *__restrict__ frames, PngGeom g, int nseg, int level, const uint8_t *__restrict__ slots,
                     const uint32_t *__restrict__ seg_bytes, const uint32_t *__restrict__ seg_off, const uint64_t *__restrict__ png_off,
                     const uint64_t *__restrict__ zlens, const uint32_t *__restrict__ stored, uint8_t *__restrict__ png) {
    const long long blk = blockIdx.x, f = blk / nseg, s = blk - f * nseg;
    const long long zl = (long long)zlens[f];
    if (!zl) return;
    uint8_t *p = png + png_off[f];
    const bool st = stored[f] != 0;
    const int tid = threadIdx.x;
    if (s == 0 && tid < g.idat_data_off + 2) {
        uint8_t v;
        if (tid < g.idat_data_off) v = png_head_byte(g, tid, zl);
        else if (tid == g.idat_data_off) v = 0x78;                      // deflate, 32K window
        else {                                                           // FLEVEL as zlib maps the level, FDICT 0, check bits
            const uint32_t flevel = st ? 0 : level < 2 ? 0 : level < 6 ? 1 : level == 6 ? 2 : 3;
            v = st ? 0x01 : (uint8_t)((flevel << 6) + 31 - ((0x78u * 256 + (flevel << 6)) % 31));
        }
        p[tid] = v;
    }
    if (s == nseg - 1 && tid < 20) {                                     // Adler-32 and CRC (filled by png_seal_kernel), IEND
        const long long o = g.idat_data_off + zl - 4 + tid;
        p[o] = tid < 8 ? 0 : png_iend_byte(tid - 8);
    }
    uint8_t *data = p + g.idat_data_off + 2;
    if (st) {
        const long long dlen = zl - 6, per = (dlen + nseg - 1) / nseg, lo = s * per, hi = min(lo + per, dlen);
        const uint8_t *fb = frames + f * (long long)g.w * g.h * 4;
        for (long long d = lo + tid; d < hi; d += blockDim.x) data[d] = stored_data_byte(fb, g, d);
    } else {
        const uint8_t *src = slots + blk * (long long)DF_SLOT;
        uint8_t *dst = data + seg_off[blk];
        const uint32_t n = seg_bytes[blk];
        for (uint32_t i = tid; i < n; i += blockDim.x) dst[i] = src[i];
    }
}

// file (and base64) offsets of the stored layout: frame f at f * png_len
__global__ void __launch_bounds__(256)
png_offsets_kernel(int n_frames, unsigned long long png_len, uint64_t *__restrict__ png_off, uint64_t *__restrict__ b64_off) {
    for (int f = blockIdx.x * blockDim.x + threadIdx.x; f <= n_frames; f += gridDim.x * blockDim.x) {
        png_off[f] = png_len * f;
        if (b64_off) b64_off[f] = (png_len + 2) / 3 * 4 * f;
    }
}

static size_t deflate_work_bytes(long long nseg, int n_frames) {
    const long long total = nseg * n_frames;
    return (size_t)total * DF_SLOT + (size_t)total * 8 + (size_t)n_frames * 12 + 64;
}

// n frames (RGBA8, device) -> PNG files back to back at d_png, offsets in d_png_off[n+1] (and base64 likewise)
int launch_png_level(b200timg_ctx *ctx, const uint8_t *d_frames, int w, int h, int n_frames, int rgb24, int level,
                     uint8_t *d_png, size_t png_cap, uint64_t *d_png_off, char *d_b64, size_t b64_cap, uint64_t *d_b64_off) {
    const PngGeom g = png_geom(w, h, rgb24);
    if (g.zlib_len > 0x7fffffffll) return ctx->fail(B200TIMG_EINVAL, "png: frame too large for one IDAT chunk");
    if (level == 0) {                                                    // png.cu's stored blocks, at their fixed stride
        const unsigned long long b64_len = (g.png_len + 2) / 3 * 4;
        long long fit = (long long)(png_cap / (unsigned long long)g.png_len);
        if (d_b64) fit = min(fit, (long long)(b64_cap / b64_len));
        B2_KERNEL(ctx, "png_offsets_kernel");
        png_offsets_kernel<<<1, 256, 0, ctx->stream>>>(n_frames, (unsigned long long)g.png_len, d_png_off, d_b64_off);
        B2_LAUNCH_CHECK(ctx);
        const int n = (int)min((long long)n_frames, fit);
        return n > 0 ? launch_png(ctx, d_frames, w, h, n, rgb24, d_png, d_b64) : B200TIMG_OK;
    }
    const long long nseg = (g.raw_len + DF_SEG - 1) / DF_SEG;
    if (nseg * n_frames > 0x7fffffffll) return ctx->fail(B200TIMG_EINVAL, "png: batch too large");
    const long long total = nseg * n_frames;
    B2_CUDA(ctx, ctx->deflate_work.reserve(deflate_work_bytes(nseg, n_frames)));
    uint8_t *slots = ctx->deflate_work.as<uint8_t>();
    uint32_t *seg_bytes = reinterpret_cast<uint32_t *>(slots + (size_t)total * DF_SLOT);
    uint32_t *seg_off = seg_bytes + total;
    uint64_t *zlens = reinterpret_cast<uint64_t *>(seg_off + total);     // 2 * total words past a 16-byte boundary: 8-aligned
    uint32_t *stored = reinterpret_cast<uint32_t *>(zlens + n_frames);
    B2_CUDA(ctx, cudaFuncSetAttribute(deflate_segment_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DF_SMEM));
    B2_KERNEL(ctx, "deflate_segment_kernel");
    deflate_segment_kernel<<<(unsigned)total, DF_THREADS, DF_SMEM, ctx->stream>>>(d_frames, g, (int)nseg, slots, seg_bytes);
    B2_LAUNCH_CHECK(ctx);
    B2_KERNEL(ctx, "deflate_scan_kernel");
    deflate_scan_kernel<<<1, 1024, 0, ctx->stream>>>(seg_bytes, seg_off, (int)nseg, n_frames, g, (unsigned long long)png_cap,
                                                     (unsigned long long)b64_cap, d_b64 ? 1 : 0, d_png_off, d_b64_off, zlens, stored);
    B2_LAUNCH_CHECK(ctx);
    B2_KERNEL(ctx, "deflate_place_kernel");
    deflate_place_kernel<<<(unsigned)total, 256, 0, ctx->stream>>>(d_frames, g, (int)nseg, level, slots, seg_bytes, seg_off, d_png_off,
                                                                    zlens, stored, d_png);
    B2_LAUNCH_CHECK(ctx);
    B2_TRY(launch_png_checksums(ctx, d_frames, g, n_frames, d_png, d_png_off, zlens));
    if (d_b64) B2_TRY(launch_base64_var(ctx, d_png, d_png_off, zlens, n_frames, d_b64, d_b64_off));
    return B200TIMG_OK;
}

}  // namespace b200timg

using namespace b200timg;

extern "C" {

size_t b200timg_png_bound(int w, int h, int rgb24, int level) {
    // a frame whose compressed stream would not be shorter than the stored one is sent stored: the stored size is
    // the bound at every level
    (void)level;
    return b200timg_png_size(w, h, rgb24);
}

int b200timg_png_batch_level_dev(b200timg_ctx *ctx, const uint8_t *d_frames, int w, int h, int n_frames, int rgb24, int level,
                                 uint8_t *d_png, size_t png_cap, uint64_t *d_png_offsets, char *d_b64, size_t b64_cap,
                                 uint64_t *d_b64_offsets) {
    if (!ctx) return B200TIMG_EINVAL;
    B2_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!d_frames || !d_png || !d_png_offsets || (d_b64 && !d_b64_offsets) || w <= 0 || h <= 0 || n_frames <= 0 || n_frames > 65535)
        return ctx->fail(B200TIMG_EINVAL, "png: bad args");
    if (level < 0 || level > 9) return ctx->fail(B200TIMG_EINVAL, "png: level %d is outside 0..9", level);
    return launch_png_level(ctx, d_frames, w, h, n_frames, rgb24, level, d_png, png_cap, d_png_offsets, d_b64, b64_cap, d_b64_offsets);
}

int b200timg_png_encode_level(b200timg_ctx *ctx, const uint8_t *fb, int w, int h, int rgb24, int level, uint8_t *out, size_t cap,
                              size_t *png_size, char *b64, size_t b64_cap) {
    if (!ctx) return B200TIMG_EINVAL;
    B2_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!fb || !out || w <= 0 || h <= 0) return ctx->fail(B200TIMG_EINVAL, "png: bad args");
    if (level < 0 || level > 9) return ctx->fail(B200TIMG_EINVAL, "png: level %d is outside 0..9", level);
    if (level == 0) {
        const size_t n = b200timg_png_size(w, h, rgb24);
        if (png_size) *png_size = n;
        if (cap < n || (b64 && b64_cap < b200timg_base64_size(n))) return ctx->fail(B200TIMG_ENOSPC, "png: need %zu bytes", n);
        return b200timg_png_encode(ctx, fb, w, h, rgb24, out, cap, b64, b64_cap);
    }
    const size_t bound = b200timg_png_bound(w, h, rgb24, level), nb = b200timg_base64_size(bound);
    const size_t bytes = (size_t)w * h * 4;
    ctx->resident_fb = nullptr;
    B2_CUDA(ctx, ctx->in_stage.reserve(bytes));
    B2_CUDA(ctx, ctx->out_stage.reserve((bound + 15) / 16 * 16 + nb + 16));
    B2_CUDA(ctx, ctx->offsets.reserve(4 * sizeof(uint64_t)));
    B2_CUDA(ctx, ctx->pinned.reserve(4 * sizeof(uint64_t)));
    B2_CUDA(ctx, cudaMemcpyAsync(ctx->in_stage.p, fb, bytes, cudaMemcpyHostToDevice, ctx->stream));
    uint8_t *d_png = ctx->out_stage.as<uint8_t>();
    char *d_b64 = b64 ? ctx->out_stage.as<char>() + (bound + 15) / 16 * 16 : nullptr;
    uint64_t *d_off = ctx->offsets.as<uint64_t>();
    B2_TRY(launch_png_level(ctx, ctx->in_stage.as<uint8_t>(), w, h, 1, rgb24, level, d_png, bound, d_off, d_b64, nb, d_off + 2));
    uint64_t *h_off = ctx->pinned.as<uint64_t>();
    B2_CUDA(ctx, cudaMemcpyAsync(h_off, d_off, 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const size_t n = (size_t)h_off[1], need_b64 = b200timg_base64_size(n);
    if (png_size) *png_size = n;
    if (cap < n || (b64 && b64_cap < need_b64)) return ctx->fail(B200TIMG_ENOSPC, "png: need %zu (+%zu base64) bytes", n, need_b64);
    B2_CUDA(ctx, cudaMemcpyAsync(out, d_png, n, cudaMemcpyDeviceToHost, ctx->stream));
    if (b64) B2_CUDA(ctx, cudaMemcpyAsync(b64, d_b64, need_b64, cudaMemcpyDeviceToHost, ctx->stream));
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200TIMG_OK;
}

}  // extern "C"
