// p2p_png.cuh - sm_100a PNG encoder for the projected views (SURVEY 8f-2: the encode side, default --output_format).
//
// The reference writes every view with cv2.imwrite (ref app/panorama_to_plane-pitch.py:277); for ".png" (the default,
// ref :400-405) that is libpng + zlib at OpenCV's settings: filter Sub on every row, zlib level 1, strategy Z_RLE,
// memLevel 8, 32 KiB window, IDAT chunks of 8192 bytes.  Everything is deterministic integer work, restated here so the
// file is byte-identical to cv2.imwrite's (oracle/png_model.py is the Python restatement, pinned against zlib and
// cv2.imencode):
//   deflate.c  deflate_rle: greedy matches at distance 1 - a pure function of the maximal byte runs, so the token of
//              every position follows from where its run starts and ends: a forward max-scan and a backward min-scan
//              of the change positions inside 4096-byte tiles, prefix max / prefix sum over the tiles
//   trees.c    one warp per deflate block (16383 symbols), state in shared memory: build_tree / gen_bitlen / gen_codes /
//              scan_tree / send_tree / build_bl_tree exactly (heap order and depth tie-breaks included: lane 0 walks
//              zlib's heap, the lanes share everything else) and the static / dynamic / stored decision
//   emission   one CTA per block: tiles of 1024 positions, prefix sum of code lengths, bits assembled LSB-first in shared
//              memory and written as whole words
//   pngwrite.c Adler-32 (with the first tile pass), 8192-byte IDAT chunks, CRC-32 per chunk (a warp per chunk, staged in
//              shared memory), IHDR / IEND
// Also restated: blocks zlib stores uncompressed (_tr_stored_block: white noise), the window bits libpng writes into the
// zlib header of small images (optimize_cmf, <= 16384 bytes of data), filter type 0 for images one pixel wide, streams
// ending exactly on an IDAT boundary.  sizes[i] = 0 ("fall back to cv2.imwrite") is only left for a stream that would
// not fit its buffer, which the buffer sizing excludes.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace p2ppng {

constexpr int kSymPerBlock = 16383;     // lit_bufsize - 1 with memLevel 8
constexpr int kLCodes = 286, kDCodes = 30, kBlCodes = 19, kHeapSize = 2 * kLCodes + 1, kMaxBits = 15;
constexpr int kHdrWords = 80;           // block header (tree description) capacity in 32-bit words
constexpr int kIdat = 8192;

struct Geom {
    int W, H, n;                 // image size, number of images
    uint32_t row_bytes;          // 1 + 3 W
    uint32_t N;                  // filtered bytes per image = H * row_bytes
    uint32_t Npad;               // per-image stride of the per-position arrays (multiple of 4096)
    uint32_t max_blk;            // per-image stride of the per-block arrays
    size_t img_stride;           // bytes between input images
    size_t z_cap;                // bytes of the zlib stream buffer per image (multiple of 4)
    size_t out_cap;              // bytes of the output file buffer per image
};

struct BlockInfo {
    uint32_t lcode[kLCodes];     // code | len << 16 for literal / length symbols
    uint32_t dcode0;             // code | len << 16 of distance code 0
    uint32_t hdr[kHdrWords];     // header bits, LSB first
    uint32_t hdr_bits;           // 3 block-type bits + tree description
    uint32_t bits;               // whole block: header + symbols + end-of-block
    uint32_t kind;               // 1 static, 2 dynamic, 0 stored
    uint32_t pad;
};

__constant__ uint8_t kExtraL[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint8_t kExtraD[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t kExtraBl[19] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 2, 3, 7};
__constant__ uint8_t kBlOrder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
__constant__ uint16_t kBaseLen[29] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 14, 16, 20, 24, 28, 32, 40, 48, 56, 64, 80, 96, 112, 128,
                                      160, 192, 224, 255};

// trees.c _length_code for lc = match length - 3
__device__ __forceinline__ int length_code(int lc) {
    if (lc == 255) return 28;
    if (lc < 8) return lc;
    const int b = 31 - __clz(lc);          // 3..7
    return 4 * (b - 1) + ((lc >> (b - 2)) & 3);
}

// ---- filter ---------------------------------------------------------------------------------------------------------
// F[y][0] = 1 (Sub), F[y][1 + i] = rgb[i] - rgb[i - 3] (mod 256), RGB order (png_set_bgr).  Images one pixel wide get
// filter type 0: libpng drops Sub / Avg / Paeth for width 1 (same bytes, other type)
__global__ void __launch_bounds__(256)
png_filter_kernel(const uint8_t *__restrict__ bgr, uint8_t *__restrict__ F, const Geom G) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;   // pixel
    const uint32_t y = blockIdx.y;
    const int img = blockIdx.z;
    if (x >= (uint32_t)G.W) return;
    const uint8_t *p = bgr + (size_t)img * G.img_stride + ((size_t)y * G.W + x) * 3;
    uint8_t *o = F + (size_t)img * G.Npad + (size_t)y * G.row_bytes + 1 + (size_t)x * 3;
    int b = p[0], g = p[1], r = p[2];
    if (x > 0) {
        r -= p[-1];
        g -= p[-2];
        b -= p[-3];
    } else {
        o[-1] = (G.W == 1) ? 0 : 1;
    }
    o[0] = (uint8_t)r;
    o[1] = (uint8_t)g;
    o[2] = (uint8_t)b;
}

// ---- tokeniser (zlib deflate_rle) --------------------------------------------------------------------------------------
// With Z_RLE every match has distance 1, so the greedy tokeniser is a pure function of the maximal runs of equal bytes:
// position i with offset j = i - s(i) inside its run (s = the run's first position) and e(i) = the first position behind
// the run is
//     j = 0                              a literal (the byte that starts the run),
//     (j - 1) % 258 = 0                  the start of a chunk of <= 258 bytes: a match of min(258, e - i) bytes if that is
//                                        >= 3, else a literal,
//     (j - 1) % 258 = 1                  covered by the chunk's match if e - i >= 2, else a literal,
//     otherwise                          covered.
// s and e are a forward max-scan and a backward min-scan of the positions where the byte changes.  Tiles of 4096 positions
// (256 threads x 16 bytes, one 16-byte load per thread), three passes over the image instead of round 1's four scan
// launches over a 4-byte-per-position run-start array (1.3 GB of traffic per 12 views, 790 us):
//   png_tile_kernel    last change position per tile (+ the Adler-32 partial sums, the data is in registers anyway)
//   png_tile_scan_kernel<0>   exclusive prefix max over the tiles of an image = the run start every tile inherits
//   png_token_kernel   s, e (the 258 bytes behind the tile come from a short look-ahead), token lengths, tokens per tile
//   png_tile_scan_kernel<1>   exclusive prefix sum = index of every tile's first token, token count of the image
//   png_blockpos_kernel       position of every 16383rd token = start of a deflate block (one warp per block)
// tlen[i]: 0 = no token starts here, 1 = literal, 3..258 = match length.
constexpr uint32_t kTile = 4096;
constexpr int kLookThreads = 18;   // 288 look-ahead bytes >= 258

__device__ __forceinline__ uint32_t byte_of(const uint4 &q, int k) {
    const uint32_t w = (k < 4) ? q.x : (k < 8) ? q.y : (k < 12) ? q.z : q.w;
    return (w >> (8 * (k & 3))) & 0xFFu;
}

// Adler-32 of the filtered data: s1 = 1 + sum F[i], s2 = N + sum (N - i) F[i]  (mod 65521)
__global__ void __launch_bounds__(256)
png_tile_kernel(const uint8_t *__restrict__ F, uint32_t *__restrict__ tile_last, unsigned long long *__restrict__ sums,
                const Geom G) {
    __shared__ uint32_t s_max[8];
    __shared__ unsigned long long s_a[8], s_b[8];
    const int img = blockIdx.y;
    const uint32_t tile = blockIdx.x, n_tiles = G.Npad / kTile, N = G.N;
    const uint8_t *f = F + (size_t)img * G.Npad;
    const uint32_t i0 = tile * kTile + threadIdx.x * 16u;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint4 q = make_uint4(0u, 0u, 0u, 0u);
    if (i0 < N) q = *reinterpret_cast<const uint4 *>(f + i0);
    uint32_t prev = __shfl_up_sync(0xffffffffu, q.w >> 24, 1);
    if (lane == 0) prev = (i0 > 0 && i0 < N) ? f[i0 - 1] : 0u;
    uint32_t last = 0, sv = 0, sk = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const uint32_t i = i0 + k, v = byte_of(q, k);
        if (i < N) {
            if (i > 0 && v != prev) last = i;
            sv += v;
            sk += (uint32_t)k * v;
        }
        prev = v;
    }
    unsigned long long a = sv, b = (i0 < N) ? (unsigned long long)sv * (unsigned long long)(N - i0) - sk : 0ull;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (lane == 0) {
        s_max[warp] = last;
        s_a[warp] = a;
        s_b[warp] = b;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t m = 0;
        unsigned long long ta = 0, tb = 0;   // < 2^64: 4096 bytes of 255 times a weight < 2^31
        for (int w = 0; w < 8; ++w) {
            m = max(m, s_max[w]);
            ta += s_a[w];
            tb += s_b[w];
        }
        tile_last[(size_t)img * n_tiles + tile] = m;
        if (ta) atomicAdd(&sums[2 * img], ta);   // one pair of atomics per tile (per warp they serialise: 196 us per 12 views)
        if (tb) atomicAdd(&sums[2 * img + 1], tb % 65521ull);
    }
}

// exclusive prefix max (MODE 0) / sum (MODE 1) over the tiles of an image; one CTA per image
template <int MODE>
__global__ void __launch_bounds__(1024)
png_tile_scan_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, uint32_t *__restrict__ total, const Geom G) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_carry;
    const int img = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t n_tiles = (G.N + kTile - 1) / kTile, stride = G.Npad / kTile;
    const uint32_t *src = in + (size_t)img * stride;
    uint32_t *dst = out + (size_t)img * stride;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_tiles; base += 1024u) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = (i < n_tiles) ? src[i] : 0u;
        uint32_t inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc = MODE ? inc + u : max(inc, u);
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t u = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w = MODE ? w + u : max(w, u);
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        const uint32_t carry = s_carry;
        uint32_t ex = __shfl_up_sync(0xffffffffu, inc, 1);
        if (lane == 0) ex = 0;
        const uint32_t wb = warp ? s_warp[warp - 1] : 0u;
        ex = MODE ? carry + wb + ex : max(carry, max(wb, ex));
        if (i < n_tiles) dst[i] = ex;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = MODE ? carry + s_warp[31] : max(carry, s_warp[31]);
        __syncthreads();
    }
    if (total && threadIdx.x == 0) total[img] = s_carry;
}

__global__ void __launch_bounds__(256)
png_token_kernel(const uint8_t *__restrict__ F, const uint32_t *__restrict__ tile_carry, uint16_t *__restrict__ tlen,
                 uint32_t *__restrict__ tile_cnt, const Geom G) {
    __shared__ uint32_t s_fwd[8], s_bwd[8], s_cnt[8];
    __shared__ uint32_t s_look, s_lastbyte;
    const int img = blockIdx.y;
    const uint32_t tile = blockIdx.x, n_tiles = G.Npad / kTile, N = G.N;
    const uint32_t base = tile * kTile;
    const uint8_t *f = F + (size_t)img * G.Npad;
    const uint32_t i0 = base + threadIdx.x * 16u;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr uint32_t kInf = 0xFFFFFFFFu;
    uint4 q = make_uint4(0u, 0u, 0u, 0u);
    if (i0 < N) q = *reinterpret_cast<const uint4 *>(f + i0);
    if (threadIdx.x == 255) s_lastbyte = q.w >> 24;
    uint32_t prev0 = __shfl_up_sync(0xffffffffu, q.w >> 24, 1);
    if (lane == 0) prev0 = (i0 > 0 && i0 < N) ? f[i0 - 1] : 0u;
    __syncthreads();
    // look-ahead: the first change among the 288 positions behind the tile (a match is at most 258 long)
    if (warp == 0) {
        const uint32_t l0 = base + kTile + threadIdx.x * 16u;
        uint32_t first = kInf;
        if (threadIdx.x < kLookThreads && l0 < N) {
            const uint4 lq = *reinterpret_cast<const uint4 *>(f + l0);
            const uint32_t pv = threadIdx.x ? (uint32_t)f[l0 - 1] : s_lastbyte;
#pragma unroll
            for (int k = 15; k >= 0; --k) {
                const uint32_t v = byte_of(lq, k), before = k ? byte_of(lq, k - 1) : pv;
                if (l0 + k < N && v != before) first = l0 + k;
            }
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
        if (threadIdx.x == 0) s_look = first;
    }
    // change flags of this thread's 16 positions
    uint32_t chg = 0;
    {
        uint32_t pv = prev0;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const uint32_t v = byte_of(q, k);
            if (i0 + k < N && i0 + k > 0 && v != pv) chg |= 1u << k;
            pv = v;
        }
    }
    const uint32_t my_last = chg ? i0 + (31 - __clz(chg)) : 0u;            // forward aggregate (0 = none)
    const uint32_t my_first = chg ? i0 + (__ffs(chg) - 1) : kInf;         // backward aggregate
    uint32_t fwd = my_last, bwd = my_first;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, fwd, o), d = __shfl_down_sync(0xffffffffu, bwd, o);
        if (lane >= o) fwd = max(fwd, u);
        if (lane + o < 32) bwd = min(bwd, d);
    }
    if (lane == 31) s_fwd[warp] = fwd;
    if (lane == 0) s_bwd[warp] = bwd;
    __syncthreads();
    uint32_t s_before = __shfl_up_sync(0xffffffffu, fwd, 1), e_after = __shfl_down_sync(0xffffffffu, bwd, 1);
    if (lane == 0) s_before = 0u;
    if (lane == 31) e_after = kInf;
    s_before = max(s_before, tile_carry[(size_t)img * n_tiles + tile]);
    e_after = min(e_after, s_look);
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        if (w < warp) s_before = max(s_before, s_fwd[w]);
        if (w > warp) e_after = min(e_after, s_bwd[w]);
    }
    e_after = min(e_after, N);
    // tokens
    uint32_t t[16];
    uint32_t cnt = 0;
    {
        uint32_t e = e_after;
#pragma unroll
        for (int k = 15; k >= 0; --k) {       // e(i): first change behind i
            t[k] = e;
            if ((chg >> k) & 1u) e = i0 + k;
        }
        uint32_t sidx = s_before;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const uint32_t i = i0 + k, e_i = t[k];
            if ((chg >> k) & 1u) sidx = i;
            uint32_t tok = 0;
            if (i < N) {
                const uint32_t j = i - sidx;
                if (j == 0) {
                    tok = 1;
                } else {
                    const uint32_t within = (j - 1u) % 258u, left = e_i - i;
                    if (within == 0) tok = (left >= 3u) ? min(left, 258u) : 1u;
                    else if (within == 1) tok = (left >= 2u) ? 0u : 1u;
                }
            }
            t[k] = tok;
            cnt += tok ? 1u : 0u;
        }
    }
    if (i0 < G.Npad) {
        uint4 o0, o1;
        o0.x = t[0] | (t[1] << 16); o0.y = t[2] | (t[3] << 16); o0.z = t[4] | (t[5] << 16); o0.w = t[6] | (t[7] << 16);
        o1.x = t[8] | (t[9] << 16); o1.y = t[10] | (t[11] << 16); o1.z = t[12] | (t[13] << 16); o1.w = t[14] | (t[15] << 16);
        uint4 *dst = reinterpret_cast<uint4 *>(tlen + (size_t)img * G.Npad + i0);
        dst[0] = o0;
        dst[1] = o1;
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) s_cnt[warp] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t c = 0;
        for (int w = 0; w < 8; ++w) c += s_cnt[w];
        tile_cnt[(size_t)img * n_tiles + tile] = c;
    }
}

// blockpos[b] = position of token b * kSymPerBlock: the tile by binary search over the tiles' first-token indices, the
// position inside the tile by counting.  One warp per deflate block.
__global__ void __launch_bounds__(128)
png_blockpos_kernel(const uint16_t *__restrict__ tlen, const uint32_t *__restrict__ tile_first, const uint32_t *__restrict__ ntok,
                    uint32_t *__restrict__ blockpos, const Geom G) {
    const int img = blockIdx.y, lane = threadIdx.x & 31;
    const uint32_t b = blockIdx.x * 4u + (threadIdx.x >> 5);
    const uint32_t T = ntok[img];
    const unsigned long long target64 = (unsigned long long)b * kSymPerBlock;
    if (b >= G.max_blk || target64 >= T) return;
    const uint32_t target = (uint32_t)target64;
    const uint32_t n_tiles = (G.N + kTile - 1) / kTile, stride = G.Npad / kTile;
    const uint32_t *first = tile_first + (size_t)img * stride;
    uint32_t lo = 0, hi = n_tiles - 1;   // the last tile with first[tile] <= target
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (first[mid] <= target) lo = mid;
        else hi = mid - 1;
    }
    uint32_t r = target - first[lo];     // r-th token of the tile
    const uint16_t *tl = tlen + (size_t)img * G.Npad + (size_t)lo * kTile;
    for (uint32_t it = 0; it < kTile / 256u; ++it) {
        const uint4 v = *reinterpret_cast<const uint4 *>(tl + it * 256u + lane * 8u);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        uint32_t flags = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) if ((w[k >> 1] >> (16 * (k & 1))) & 0xFFFFu) flags |= 1u << k;
        const uint32_t c = __popc(flags);
        uint32_t inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += u;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
        if (r < total) {
            const uint32_t ex = inc - c;
            if (r >= ex && r < inc) {
                uint32_t m = flags, need = r - ex;
                while (need--) m &= m - 1u;      // drop the lowest set bits
                blockpos[(size_t)img * G.max_blk + b] = lo * kTile + it * 256u + lane * 8u + (uint32_t)(__ffs(m) - 1);
            }
            return;
        }
        r -= total;
    }
}

// position range of deflate block b of an image (the last block may be empty)
__device__ __forceinline__ void block_range(const uint32_t *__restrict__ blockpos, uint32_t T, uint32_t N, uint32_t b,
                                            uint32_t &p0, uint32_t &p1) {
    const uint32_t nblk = T / (uint32_t)kSymPerBlock + 1u;
    p0 = (b * (uint32_t)kSymPerBlock < T) ? blockpos[b] : N;
    p1 = (b + 1 < nblk && (b + 1) * (uint32_t)kSymPerBlock < T) ? blockpos[b + 1] : N;
}

// ---- per-block symbol histogram --------------------------------------------------------------------------------------
// One CTA per deflate block; a thread takes 8 consecutive positions per step (one 16-byte load of token lengths, one 8-byte
// load of filtered bytes; the block's range is widened to multiples of 8 and masked).
__global__ void __launch_bounds__(256)
png_hist_kernel(const uint8_t *__restrict__ F, const uint16_t *__restrict__ tlen, const uint32_t *__restrict__ blockpos,
                const uint32_t *__restrict__ ntok, uint32_t *__restrict__ lfreq, const Geom G) {
    __shared__ uint32_t h[kLCodes + 2];   // [kLCodes] = number of matches (distance code 0)
    const int img = blockIdx.y;
    const uint32_t b = blockIdx.x, T = ntok[img];
    if (b >= T / (uint32_t)kSymPerBlock + 1u) return;
    for (int i = threadIdx.x; i < kLCodes + 2; i += blockDim.x) h[i] = 0;
    __syncthreads();
    uint32_t p0, p1;
    block_range(blockpos + (size_t)img * G.max_blk, T, G.N, b, p0, p1);
    const uint8_t *f = F + (size_t)img * G.Npad;
    const uint16_t *tl = tlen + (size_t)img * G.Npad;
    for (uint32_t i0 = (p0 & ~7u) + threadIdx.x * 8u; i0 < p1; i0 += blockDim.x * 8u) {   // (Npad is a multiple of 4096)
        const uint4 tv = *reinterpret_cast<const uint4 *>(tl + i0);
        const uint2 fv = *reinterpret_cast<const uint2 *>(f + i0);
        const uint32_t tw[4] = {tv.x, tv.y, tv.z, tv.w};
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t i = i0 + k;
            const uint32_t t = (tw[k >> 1] >> (16 * (k & 1))) & 0xFFFFu;
            if (i < p0 || i >= p1 || t == 0) continue;
            if (t == 1) {
                atomicAdd(&h[((k < 4 ? fv.x : fv.y) >> (8 * (k & 3))) & 0xFFu], 1u);
            } else {
                atomicAdd(&h[257 + length_code((int)t - 3)], 1u);
                atomicAdd(&h[kLCodes], 1u);
            }
        }
    }
    __syncthreads();
    uint32_t *o = lfreq + ((size_t)img * G.max_blk + b) * (kLCodes + 2);
    for (int i = threadIdx.x; i < kLCodes + 2; i += blockDim.x) o[i] = (i == 256) ? 1u : h[i];   // END_BLOCK once
}

// ---- trees.c, one warp per deflate block ------------------------------------------------------------------------------
// zlib's tree construction is a sequential object: its heap breaks ties between equal (frequency, depth) keys by heap position,
// so the code lengths of equally frequent symbols follow the exact order of its sift-down steps.  What can be done is to make
// that one sequential chain short and everything around it parallel: a warp owns a deflate block, all of its state lives in
// shared memory (7 KB; round 1 ran one THREAD per block with 11 KB of per-thread local memory - 32 lanes indexing 32
// different cache lines per access, ~1 ms per 12 views), lane 0 walks the heap (32-bit entries that carry their own sort key,
// both children fetched at once), the lanes together compact the symbols, set the leaves' lengths, count, sum, assign the
// codes and write the tables; the header bits are assembled in shared memory.
constexpr int kTreeWarps = 4;            // deflate blocks per CTA

struct alignas(16) TreeShared {
    uint32_t heap[kHeapSize + 3];        // heap entries: freq << 16 | depth << 10 | node; below heap_max: node numbers
    uint16_t freq[kHeapSize], dad[kHeapSize];
    uint8_t len[kHeapSize];              // depth of a node while the tree is built (trees.c depth[]), its code length after
    uint32_t bl_count[kMaxBits + 1];
    uint16_t next_code[kMaxBits + 1];
    uint8_t llen[kLCodes];
    uint16_t lcodes[kLCodes];
    uint8_t dlen[kDCodes];
    uint16_t dcodes[kDCodes];
    uint32_t blfreq[kBlCodes];
    uint8_t bllen[kBlCodes];
    uint16_t blcodes[kBlCodes];
    uint32_t hdr[kHdrWords];
};

struct BitAcc {      // LSB-first bit writer into a word array
    uint32_t *w;
    uint32_t nbits;
    __device__ __forceinline__ void send(uint32_t value, int length) {
        const uint32_t i = nbits >> 5, sh = nbits & 31;
        w[i] |= value << sh;
        if (sh + length > 32) w[i + 1] |= value >> (32 - sh);
        nbits += (uint32_t)length;
    }
};

__device__ __forceinline__ uint32_t bi_reverse(uint32_t code, int len) {
    return __brev(code) >> (32 - len);
}

__device__ __forceinline__ int static_l_len(int n) { return n < 144 ? 8 : (n < 256 ? 9 : (n < 280 ? 7 : 8)); }

// build_tree + gen_bitlen + gen_codes for the `elems` symbols whose frequencies sit in t.freq[0 .. elems), called by all
// lanes of the warp.  KIND 0: literal / length tree, 1: distance tree, 2: bit-length tree (no static tree).  Code lengths go
// to lens[], codes to codes[]; returns max_code; opt_len / static_len are updated like in trees.c (warp-uniform values).
template <int KIND>
__device__ int build_tree(TreeShared &t, const int lane, int *opt_len, int *static_len, uint8_t *lens, uint16_t *codes) {
    constexpr int elems = KIND == 0 ? kLCodes : (KIND == 1 ? kDCodes : kBlCodes);
    constexpr int max_length = KIND == 2 ? 7 : kMaxBits;
    auto stree_len = [](int n) { return KIND == 0 ? static_l_len(n) : (KIND == 1 ? 5 : 0); };
    auto xbits_of = [](int n) -> int {
        return KIND == 0 ? (n >= 257 ? (int)kExtraL[n - 257] : 0) : (KIND == 1 ? (int)kExtraD[n] : (int)kExtraBl[n]);
    };
    auto entry = [&](int n) { return ((uint32_t)t.freq[n] << 16) | ((uint32_t)t.len[n] << 10) | (uint32_t)n; };
    const uint32_t lt = (1u << lane) - 1u;
    // the symbols that occur, in symbol order (all lanes)
    int heap_len = 0, max_code = -1;
    for (int base = 0; base < elems; base += 32) {
        const int n = base + lane;
        const bool nz = n < elems && t.freq[n] != 0;
        const uint32_t m = __ballot_sync(0xffffffffu, nz);
        if (nz) {
            t.len[n] = 0;
            t.heap[heap_len + 1 + __popc(m & lt)] = entry(n);
        } else if (n < elems) {
            t.len[n] = 0;
        }
        heap_len += __popc(m);
        if (m) max_code = base + 31 - __clz(m);
    }
    if (lane < kMaxBits + 1) t.bl_count[lane] = 0;
    __syncwarp();
    int heap_max = kHeapSize, last_node = elems, d_opt = 0, d_static = 0;
    if (lane == 0) {
        while (heap_len < 2) {
            const int node = (max_code < 2) ? ++max_code : 0;
            t.freq[node] = 1;
            t.len[node] = 0;
            t.heap[++heap_len] = entry(node);
            d_opt--;
            d_static -= stree_len(node);
        }
        // trees.c pqdownheap, two levels per shared-memory round trip: the children (one 8-byte load) and the four
        // grandchildren (one 16-byte load) of the current node are fetched together - the entries a step can move are the
        // ones above them, so the values are the ones a level-by-level walk would read; index checks come before any use
        // (entries behind heap_len are stale or belong to the sorted region)
        auto pqdownheap = [&](int k) {
            const uint32_t v = t.heap[k];
            const uint32_t vk = v >> 10;
            for (;;) {
                int j = k << 1;
                if (j > heap_len) break;
                const uint2 c = *reinterpret_cast<const uint2 *>(&t.heap[j]);
                uint4 g = make_uint4(0u, 0u, 0u, 0u);
                if ((j << 1) <= heap_len) g = *reinterpret_cast<const uint4 *>(&t.heap[j << 1]);
                uint32_t hj = c.x;
                const bool right = j < heap_len && (c.y >> 10) <= (c.x >> 10);   // smaller(heap[j + 1], heap[j])
                if (right) {
                    hj = c.y;
                    j++;
                }
                if (vk <= (hj >> 10)) break;                                       // smaller(v, heap[j])
                t.heap[k] = hj;
                k = j;
                j = k << 1;
                if (j > heap_len) break;
                const uint32_t a = right ? g.z : g.x, b = right ? g.w : g.y;
                hj = a;
                if (j < heap_len && (b >> 10) <= (a >> 10)) {
                    hj = b;
                    j++;
                }
                if (vk <= (hj >> 10)) break;
                t.heap[k] = hj;
                k = j;
            }
            t.heap[k] = v;
        };
        for (int n = heap_len / 2; n >= 1; --n) pqdownheap(n);
        int node = elems;
        do {
            const int n = (int)(t.heap[1] & 0x3FFu);
            t.heap[1] = t.heap[heap_len--];
            pqdownheap(1);
            const int m = (int)(t.heap[1] & 0x3FFu);
            t.heap[--heap_max] = (uint32_t)n;   // below heap_max only the node numbers are used
            t.heap[--heap_max] = (uint32_t)m;
            t.freq[node] = (uint16_t)(t.freq[n] + t.freq[m]);
            const int dn = t.len[n], dm = t.len[m];
            t.len[node] = (uint8_t)((dn >= dm ? dn : dm) + 1);
            t.dad[n] = t.dad[m] = (uint16_t)node;
            t.heap[1] = entry(node);
            node++;
            pqdownheap(1);
        } while (heap_len >= 2);
        t.heap[--heap_max] = t.heap[1] & 0x3FFu;
        last_node = node;
    }
    heap_max = __shfl_sync(0xffffffffu, heap_max, 0);
    max_code = __shfl_sync(0xffffffffu, max_code, 0);
    last_node = __shfl_sync(0xffffffffu, last_node, 0);
    // gen_bitlen.  trees.c walks the nodes in the order they left the heap, parents before children; any such order gives the
    // same lengths: the internal nodes (a parent has the larger number) on lane 0, then all leaves at once.
    int overflow = 0;
    if (lane == 0) {
        t.len[last_node - 1] = 0;   // the root
        for (int n = last_node - 2; n >= elems; --n) {
            int bits = t.len[t.dad[n]] + 1;
            if (bits > max_length) {
                bits = max_length;
                overflow++;
            }
            t.len[n] = (uint8_t)bits;
        }
    }
    __syncwarp();
    for (int base = 0; base <= max_code; base += 32) {
        const int n = base + lane;
        if (n <= max_code && t.freq[n] != 0) {
            int bits = t.len[t.dad[n]] + 1;
            if (bits > max_length) {
                bits = max_length;
                overflow++;
            }
            t.len[n] = (uint8_t)bits;
            atomicAdd(&t.bl_count[bits], 1u);
            const int xb = xbits_of(n), f = t.freq[n];
            d_opt += f * (bits + xb);
            if (KIND != 2) d_static += f * (stree_len(n) + xb);   // (the bit-length tree has no static counterpart)
        }
    }
    // (d_opt / d_static: every lane sums its own leaves; lane 0 also carries the forced symbols' and the repair's adjustments)
    overflow = __reduce_add_sync(0xffffffffu, overflow);
    __syncwarp();
    if (overflow > 0) {   // rare (a tree deeper than max_length): trees.c's repair, in its heap order, on lane 0
        if (lane == 0) {
            do {
                int bits = max_length - 1;
                while (t.bl_count[bits] == 0) bits--;
                t.bl_count[bits]--;
                t.bl_count[bits + 1] += 2;
                t.bl_count[max_length]--;
                overflow -= 2;
            } while (overflow > 0);
            int h = kHeapSize;
            for (int bits = max_length; bits != 0; --bits) {
                int n = (int)t.bl_count[bits];
                while (n != 0) {
                    const int m = (int)t.heap[--h];
                    if (m > max_code) continue;
                    if (t.len[m] != bits) {
                        d_opt += (bits - (int)t.len[m]) * (int)t.freq[m];
                        t.len[m] = (uint8_t)bits;
                    }
                    n--;
                }
            }
        }
        __syncwarp();
    }
    // gen_codes: canonical codes in symbol order = first code of the length + number of earlier symbols of that length
    if (lane == 0) {
        uint32_t code = 0;
        t.next_code[0] = 0;
        for (int bits = 1; bits <= kMaxBits; ++bits) {
            code = (code + t.bl_count[bits - 1]) << 1;
            t.next_code[bits] = (uint16_t)code;
        }
    }
    __syncwarp();
    for (int base = 0; base < elems; base += 32) {
        const int n = base + lane;
        const int l = (n <= max_code) ? (int)t.len[n] : 0;
        const uint32_t peers = __match_any_sync(0xffffffffu, l ? l : 64 + lane);
        uint32_t code = 0;
        if (l) {
            code = t.next_code[l] + (uint32_t)__popc(peers & lt);
        }
        __syncwarp();
        if (l && (peers >> lane) == 1u) t.next_code[l] = (uint16_t)(t.next_code[l] + __popc(peers));   // the highest lane of the group
        if (n < elems) {
            codes[n] = l ? (uint16_t)bi_reverse(code, l) : (uint16_t)0;
            lens[n] = (uint8_t)l;
        }
        __syncwarp();
    }
    *opt_len += __reduce_add_sync(0xffffffffu, d_opt);
    *static_len += __reduce_add_sync(0xffffffffu, d_static);
    return max_code;
}

// scan_tree (SEND = false: count the code-length symbols) / send_tree (SEND = true: emit them); lane 0
template <bool SEND>
__device__ void walk_tree(const uint8_t *lens, int max_code, uint32_t *blfreq, const uint8_t *bllen, const uint16_t *blcode,
                          BitAcc *out) {
    int prevlen = -1, nextlen = lens[0], count = 0;
    int max_count = 7, min_count = 4;
    if (nextlen == 0) max_count = 138, min_count = 3;
    for (int n = 0; n <= max_code; ++n) {
        const int curlen = nextlen;
        nextlen = (n + 1 <= max_code) ? (int)lens[n + 1] : 0xffff;
        if (++count < max_count && curlen == nextlen) continue;
        if (count < min_count) {
            if (SEND) for (int k = 0; k < count; ++k) out->send(blcode[curlen], bllen[curlen]);
            else blfreq[curlen] += (uint32_t)count;
        } else if (curlen != 0) {
            if (curlen != prevlen) {
                if (SEND) {
                    out->send(blcode[curlen], bllen[curlen]);
                    count--;
                } else {
                    blfreq[curlen]++;
                }
            }
            if (SEND) {
                out->send(blcode[16], bllen[16]);
                out->send((uint32_t)(count - 3), 2);
            } else {
                blfreq[16]++;
            }
        } else if (count <= 10) {
            if (SEND) {
                out->send(blcode[17], bllen[17]);
                out->send((uint32_t)(count - 3), 3);
            } else {
                blfreq[17]++;
            }
        } else {
            if (SEND) {
                out->send(blcode[18], bllen[18]);
                out->send((uint32_t)(count - 11), 7);
            } else {
                blfreq[18]++;
            }
        }
        count = 0;
        prevlen = curlen;
        if (nextlen == 0) max_count = 138, min_count = 3;
        else if (curlen == nextlen) max_count = 6, min_count = 3;
        else max_count = 7, min_count = 4;
    }
}

// _tr_flush_block for one block: trees, static / dynamic decision, header bits, code tables
__global__ void __launch_bounds__(kTreeWarps * 32)
png_tree_kernel(const uint32_t *__restrict__ lfreq, const uint32_t *__restrict__ ntok, const uint32_t *__restrict__ blockpos,
                BlockInfo *__restrict__ info, const Geom G) {
    __shared__ TreeShared s_tree[kTreeWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t b = blockIdx.x * kTreeWarps + warp;
    const int img = blockIdx.y;
    const uint32_t T = ntok[img], nblk = T / (uint32_t)kSymPerBlock + 1u;
    if (b >= nblk) return;
    TreeShared &t = s_tree[warp];
    const uint32_t *fr = lfreq + ((size_t)img * G.max_blk + b) * (kLCodes + 2);
    BlockInfo &bi = info[(size_t)img * G.max_blk + b];
    const uint32_t last = (b + 1 == nblk) ? 1u : 0u;
    int opt_len = 0, static_len = 0;
    // literal / length tree
    for (int n = lane; n < kLCodes; n += 32) t.freq[n] = (uint16_t)fr[n];
    for (int i = lane; i < kHdrWords; i += 32) t.hdr[i] = 0;
    if (lane < kBlCodes) t.blfreq[lane] = 0;
    __syncwarp();
    const int lmax = build_tree<0>(t, lane, &opt_len, &static_len, t.llen, t.lcodes);
    __syncwarp();
    // distance tree (only code 0 can occur: every match has distance 1)
    if (lane < kDCodes) t.freq[lane] = lane == 0 ? (uint16_t)fr[kLCodes] : (uint16_t)0;
    __syncwarp();
    const int dmax = build_tree<1>(t, lane, &opt_len, &static_len, t.dlen, t.dcodes);
    __syncwarp();
    // bit-length tree
    if (lane == 0) {
        walk_tree<false>(t.llen, lmax, t.blfreq, nullptr, nullptr, nullptr);
        walk_tree<false>(t.dlen, dmax, t.blfreq, nullptr, nullptr, nullptr);
    }
    __syncwarp();
    if (lane < kBlCodes) t.freq[lane] = (uint16_t)t.blfreq[lane];
    __syncwarp();
    build_tree<2>(t, lane, &opt_len, &static_len, t.bllen, t.blcodes);
    __syncwarp();
    int max_blindex = kBlCodes - 1;
    while (max_blindex >= 3 && t.bllen[kBlOrder[max_blindex]] == 0) max_blindex--;
    opt_len += 3 * (max_blindex + 1) + 5 + 5 + 4;
    int opt_lenb = (opt_len + 3 + 7) >> 3;
    const int static_lenb = (static_len + 3 + 7) >> 3;
    if (static_lenb <= opt_lenb) opt_lenb = static_lenb;
    uint32_t p0, p1;
    block_range(blockpos + (size_t)img * G.max_blk, T, G.N, b, p0, p1);
    const int stored_len = (int)(p1 - p0);
    BitAcc out;
    out.w = t.hdr;
    out.nbits = 0;
    uint32_t kind, bits;
    if (stored_len + 4 <= opt_lenb) {
        // trees.c _tr_stored_block: 3 header bits, pad to a byte, LEN, ~LEN, the bytes.  (zlib also needs the block's
        // bytes to be still in its window, block_start >= 0: a block chosen here has < 16383 + 1300 bytes - more match
        // bytes and the Huffman form is shorter -, far less than the 32506 that could slide out.)
        kind = 0;
        bits = (uint32_t)stored_len;   // bytes; png_layout_kernel knows the alignment and turns this into bits
        if (lane == 0) out.send((0u << 1) + last, 3);
    } else if (static_lenb == opt_lenb) {
        kind = 1;
        if (lane == 0) out.send((1u << 1) + last, 3);
        // static codes: canonical codes of the fixed lengths (24 codes of 7 bits from 0000000: symbols 256..279; 8 bits from
        // 00110000: 0..143 then 280..287; 9 bits from 110010000: 144..255)
        for (int n = lane; n < kLCodes; n += 32) {
            const int l = static_l_len(n);
            const uint32_t code = n < 144 ? 0x30u + n : (n < 256 ? 0x190u + (n - 144) : (n < 280 ? (uint32_t)(n - 256) : 0xC0u + (n - 280)));
            bi.lcode[n] = bi_reverse(code, l) | ((uint32_t)l << 16);
        }
        if (lane == 0) bi.dcode0 = 0u | (5u << 16);
        bits = (uint32_t)(static_len + 3);
    } else {
        kind = 2;
        if (lane == 0) {
            out.send((2u << 1) + last, 3);
            out.send((uint32_t)(lmax + 1 - 257), 5);
            out.send((uint32_t)(dmax + 1 - 1), 5);
            out.send((uint32_t)(max_blindex + 1 - 4), 4);
            for (int rank = 0; rank <= max_blindex; ++rank) out.send(t.bllen[kBlOrder[rank]], 3);
            walk_tree<true>(t.llen, lmax, nullptr, t.bllen, t.blcodes, &out);
            walk_tree<true>(t.dlen, dmax, nullptr, t.bllen, t.blcodes, &out);
            bi.dcode0 = (uint32_t)t.dcodes[0] | ((uint32_t)t.dlen[0] << 16);
        }
        for (int n = lane; n < kLCodes; n += 32) bi.lcode[n] = (uint32_t)t.lcodes[n] | ((uint32_t)t.llen[n] << 16);
        bits = (uint32_t)(opt_len + 3);
    }
    __syncwarp();
    for (int i = lane; i < kHdrWords; i += 32) bi.hdr[i] = t.hdr[i];
    if (lane == 0) {
        bi.kind = kind;
        bi.bits = bits;
        bi.hdr_bits = out.nbits;
    }
}

// bit offset of every block in the zlib stream (after the 2 header bytes), total length, "handled" flag.  One warp per image.
// A Huffman block of `bits` bits moves the offset by off -> off + bits; a stored block (header, padding to the next byte,
// LEN + ~LEN, data) by off -> roundup8(off + 3) + 32 + 8 * len.  Both are of the form
//     f(off) = align ? roundup8(off + a) + c : off + c,
// and that family is closed under composition (roundup8(x + y) = x + roundup8(y) for x a multiple of 8), so the offsets are
// one prefix "sum" over function composition: every lane composes its contiguous share of the blocks, the warp scans the
// 32 composites, every lane walks its share again from its start offset.  Offsets are 64-bit throughout, blkoff[] included:
// an image of up to 2^31 filtered bytes stored uncompressed makes a stream of more than 2^32 bits (from N > 2^29 bytes of
// noise on), and a 32-bit block offset would put the blocks behind that point at their offset mod 2^32.
struct OffFn {
    uint32_t align;
    unsigned long long a, c;
    __device__ __forceinline__ unsigned long long operator()(unsigned long long off) const {
        return align ? ((off + a + 7ull) & ~7ull) + c : off + c;
    }
};
__device__ __forceinline__ OffFn off_compose(const OffFn &f, const OffFn &g) {   // g after f
    OffFn r;
    if (!g.align) {
        r.align = f.align; r.a = f.a; r.c = f.c + g.c;
    } else if (!f.align) {
        r.align = 1u; r.a = f.c + g.a; r.c = g.c;
    } else {
        r.align = 1u; r.a = f.a; r.c = ((f.c + g.a + 7ull) & ~7ull) + g.c;
    }
    return r;
}
__device__ __forceinline__ OffFn off_of_block(const BlockInfo &bi) {
    OffFn f;
    if (bi.kind == 0) {
        f.align = 1u; f.a = 3ull; f.c = 32ull + 8ull * bi.bits;
    } else {
        f.align = 0u; f.a = 0ull; f.c = bi.bits;
    }
    return f;
}

__global__ void __launch_bounds__(32)
png_layout_kernel(BlockInfo *__restrict__ info, const uint32_t *__restrict__ ntok, unsigned long long *__restrict__ blkoff,
                  unsigned long long *__restrict__ zbits, const Geom G) {
    const int img = blockIdx.x, lane = threadIdx.x;
    const uint32_t nblk = ntok[img] / (uint32_t)kSymPerBlock + 1u;
    const uint32_t per = (nblk + 31u) / 32u;
    const uint32_t b0 = min(nblk, lane * per), b1 = min(nblk, b0 + per);
    BlockInfo *bi = info + (size_t)img * G.max_blk;
    OffFn mine;
    mine.align = 0u; mine.a = 0ull; mine.c = 0ull;
    for (uint32_t b = b0; b < b1; ++b) mine = off_compose(mine, off_of_block(bi[b]));
    OffFn inc = mine;   // inclusive scan over the lanes
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        OffFn u;
        u.align = __shfl_up_sync(0xffffffffu, inc.align, o);
        u.a = __shfl_up_sync(0xffffffffu, inc.a, o);
        u.c = __shfl_up_sync(0xffffffffu, inc.c, o);
        if (lane >= o) inc = off_compose(u, inc);
    }
    OffFn ex;           // everything before this lane's share
    ex.align = __shfl_up_sync(0xffffffffu, inc.align, 1);
    ex.a = __shfl_up_sync(0xffffffffu, inc.a, 1);
    ex.c = __shfl_up_sync(0xffffffffu, inc.c, 1);
    unsigned long long off = lane ? ex(16ull) : 16ull;   // the stream starts after CMF + FLG
    for (uint32_t b = b0; b < b1; ++b) {
        blkoff[(size_t)img * G.max_blk + b] = off;
        const unsigned long long next = off_of_block(bi[b])(off);
        if (bi[b].kind == 0) bi[b].bits = (uint32_t)(next - off);   // 3 + pad + 32 + 8 * len
        off = next;
    }
    const unsigned long long total = __shfl_sync(0xffffffffu, inc(16ull), 31);
    // 0 = not handled (the stream would not fit its buffer)
    if (lane == 0) zbits[img] = (total + 64ull > (unsigned long long)G.z_cap * 8ull) ? 0ull : total;
}

// ---- emission: one CTA per deflate block ------------------------------------------------------------------------------
__device__ __forceinline__ void or_bits(uint32_t *__restrict__ z, unsigned long long pos, unsigned long long value, int length) {
    const uint32_t i = (uint32_t)(pos >> 5), sh = (uint32_t)(pos & 31);
    atomicOr(z + i, (uint32_t)(value << sh));
    if (sh + length > 32) atomicOr(z + i + 1, (uint32_t)(value >> (32 - sh)));
    if (sh + length > 64) atomicOr(z + i + 2, (uint32_t)(value >> (64 - sh)));
}

// A CTA walks its block in tiles of 2048 positions, 8 consecutive positions per thread (one 16-byte load of token lengths,
// one 8-byte load of filtered bytes).  A token is at most two pieces of <= 20 bits - a literal's code, or a match's length
// code with its extra bits followed by the distance code - so everything stays 32-bit arithmetic and a piece touches at
// most two words.  The bits of a tile are assembled in SHARED memory (a prefix sum of the code lengths gives every token
// its place; <= 15 bits per position: 960 words) and leave as whole 32-bit words; only the first and the last word of a
// tile, which it shares with its neighbours, go through an atomicOr in global memory.  (Round 1 issued up to three global
// atomics per token, ~10^8 per 12 views, and three CTA barriers per 256 positions: 452 us.)
constexpr int kEmitPer = 8;
constexpr int kEmitTile = 256 * kEmitPer;
constexpr int kEmitWords = kEmitTile * kMaxBits / 32 + 4;

__global__ void __launch_bounds__(256)
png_emit_kernel(const uint8_t *__restrict__ F, const uint16_t *__restrict__ tlen, const uint32_t *__restrict__ blockpos,
                const uint32_t *__restrict__ ntok, const BlockInfo *__restrict__ info, const unsigned long long *__restrict__ blkoff,
                const unsigned long long *__restrict__ zbits, uint32_t *__restrict__ Z, const Geom G) {
    // the first piece of every possible token, ready to place: bits | length << 24; [0, 256) literal bytes, [256, 512)
    // match lengths 3 .. 258 (length code + extra bits) - one shared-memory look-up per position whatever it holds
    __shared__ uint32_t s_piece[512];
    __shared__ uint32_t s_warp[8];
    __shared__ uint32_t s_bits[kEmitWords];
    const int img = blockIdx.y;
    const uint32_t b = blockIdx.x, T = ntok[img];
    if (b >= T / (uint32_t)kSymPerBlock + 1u || zbits[img] == 0ull) return;
    const BlockInfo &bi = info[(size_t)img * G.max_blk + b];
    {
        const int lc = threadIdx.x, code = length_code(lc);   // blockDim.x == 256
        const uint32_t cl = bi.lcode[lc], cm = bi.lcode[257 + code];
        s_piece[lc] = (cl & 0xFFFFu) | ((cl >> 16) << 24);
        const uint32_t n = cm >> 16;
        s_piece[256 + lc] = ((cm & 0xFFFFu) | ((uint32_t)(lc - (int)kBaseLen[code]) << n)) | ((n + kExtraL[code]) << 24);
    }
    for (int i = threadIdx.x; i < kEmitWords; i += blockDim.x) s_bits[i] = 0;
    uint32_t *z = Z + (size_t)img * (G.z_cap / 4);
    const unsigned long long base = blkoff[(size_t)img * G.max_blk + b];
    // header bits
    for (uint32_t w = threadIdx.x; w * 32 < bi.hdr_bits; w += blockDim.x) {
        const int nb = (bi.hdr_bits - w * 32 < 32) ? (int)(bi.hdr_bits - w * 32) : 32;
        or_bits(z, base + (unsigned long long)w * 32, bi.hdr[w], nb);
    }
    uint32_t p0, p1;
    block_range(blockpos + (size_t)img * G.max_blk, T, G.N, b, p0, p1);
    const uint8_t *f = F + (size_t)img * G.Npad;
    if (bi.kind == 0) {   // stored block: LEN, ~LEN and the filtered bytes themselves, byte aligned
        const unsigned long long data = (base + 3ull + 7ull) & ~7ull;
        const uint32_t len = p1 - p0;
        if (threadIdx.x == 0) or_bits(z, data, (unsigned long long)((len & 0xFFFFu) | ((~len & 0xFFFFu) << 16)), 32);
        for (uint32_t i = threadIdx.x; i < len; i += blockDim.x) or_bits(z, data + 32ull + 8ull * i, f[p0 + i], 8);
        return;
    }
    const uint16_t *tl = tlen + (size_t)img * G.Npad;
    const uint32_t dcode = bi.dcode0 & 0xFFFFu, dlen = bi.dcode0 >> 16;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long at = base + bi.hdr_bits;   // stream position of the tile's first bit
    __syncthreads();
    for (uint32_t t0 = p0 & ~7u; t0 < p1; t0 += kEmitTile) {
        const uint32_t i0 = t0 + threadIdx.x * kEmitPer;
        uint32_t v0[kEmitPer];    // first piece: bits | length << 24 (length 0: no token here)
        uint32_t mine = 0, matches = 0;
        {
            uint4 tv = make_uint4(0u, 0u, 0u, 0u);
            uint2 fv = make_uint2(0u, 0u);
            if (i0 < p1) {   // (Npad is a multiple of 4096: the loads stay inside the image's arrays)
                tv = *reinterpret_cast<const uint4 *>(tl + i0);
                fv = *reinterpret_cast<const uint2 *>(f + i0);
            }
            const uint32_t tw[4] = {tv.x, tv.y, tv.z, tv.w};
#pragma unroll
            for (int k = 0; k < kEmitPer; ++k) {
                const uint32_t i = i0 + k;
                const uint32_t t = (tw[k >> 1] >> (16 * (k & 1))) & 0xFFFFu;
                uint32_t piece = 0;
                if (t != 0 && i >= p0 && i < p1) {
                    const uint32_t byte = ((k < 4 ? fv.x : fv.y) >> (8 * (k & 3))) & 0xFFu;
                    piece = s_piece[t == 1 ? byte : 253u + t];   // 256 + (t - 3)
                    if (t != 1) matches |= 1u << k;
                }
                v0[k] = piece;
                mine += piece >> 24;
            }
            mine += (uint32_t)__popc(matches) * dlen;
        }
        uint32_t inc = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += u;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        uint32_t wsum = 0, tile = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (k < warp) wsum += s_warp[k];
            tile += s_warp[k];
        }
        // place the pieces: bit 0 of s_bits = bit (at & ~31) of the stream
        const uint32_t sh0 = (uint32_t)(at & 31ull);
        // a thread's pieces are one contiguous bit run: gathered in a 64-bit register and handed to shared memory a word at a
        // time (its first and last word are shared with the neighbouring threads: atomicOr throughout)
        {
            const uint32_t pos = sh0 + wsum + (inc - mine);
            uint32_t w = pos >> 5, fill = pos & 31u;
            unsigned long long acc = 0ull;
            auto put = [&](uint32_t v, uint32_t n) {   // n <= 20 bits; fill < 32 on entry
                acc |= (unsigned long long)v << fill;
                fill += n;
                if (fill >= 32u) {
                    atomicOr(&s_bits[w], (uint32_t)acc);
                    acc >>= 32;
                    fill -= 32u;
                    ++w;
                }
            };
#pragma unroll
            for (int k = 0; k < kEmitPer; ++k) {
                const uint32_t n = v0[k] >> 24;
                if (n) {
                    put(v0[k] & 0x00FFFFFFu, n);
                    if ((matches >> k) & 1u) put(dcode, dlen);
                }
            }
            if (acc) atomicOr(&s_bits[w], (uint32_t)acc);
        }
        __syncthreads();
        // flush: words 0 and last are shared with the neighbouring tiles / blocks
        const uint32_t nw = (sh0 + tile + 31u) >> 5;
        uint32_t *zt = z + (uint32_t)(at >> 5);
        for (uint32_t w = threadIdx.x; w < nw; w += blockDim.x) {
            const uint32_t v = s_bits[w];
            s_bits[w] = 0;
            if (w == 0 || w + 1 == nw) {
                if (v) atomicOr(zt + w, v);
            } else {
                zt[w] = v;
            }
        }
        at += tile;
        __syncthreads();
    }
    if (threadIdx.x == 0) {   // END_BLOCK
        const uint32_t c = bi.lcode[256];
        or_bits(z, at, c & 0xFFFFu, (int)(c >> 16));
    }
}

// ---- file assembly ------------------------------------------------------------------------------------------------
// zlib stream = CMF FLG (78 01) | deflate bits | Adler-32 (big endian); PNG = signature | IHDR | IDAT x k (8192 bytes each) | IEND
__device__ __forceinline__ size_t zlib_len(unsigned long long zb) { return (size_t)((zb + 7) >> 3) + 4; }

// CMF (low byte) and FLG (high byte): 78 01, or the smaller window libpng writes into the header of a stream of at most
// 16384 bytes of data (pngwutil.c optimize_cmf); the deflate bits do not depend on it (every match has distance 1)
__device__ __forceinline__ uint32_t zlib_header(uint32_t data_size) {
    uint32_t cinfo = 7, half = 1u << 14;
    if (data_size <= 16384u) {
        do {
            half >>= 1;
            --cinfo;
        } while (cinfo > 0 && data_size <= half);
    }
    const uint32_t cmf = 0x08u | (cinfo << 4);
    const uint32_t flg = 0x1Fu - ((cmf << 8) % 0x1Fu);
    return cmf | (flg << 8);
}

__device__ __forceinline__ uint32_t crc_update(uint32_t crc, uint32_t byte, const uint32_t *__restrict__ table) {
    return table[(crc ^ byte) & 0xFFu] ^ (crc >> 8);
}

// The last step: zlib stream -> file.  One warp per IDAT chunk stages the chunk's 8192 stream bytes in shared memory with
// coalesced 16-byte loads (32 segments of 256 bytes, one padding word per segment so that the lanes' segments start in
// different banks), patches the bytes that are not deflate bits (CMF / FLG in front, the big-endian Adler-32 behind), runs
// the CRC register over one segment per lane from state 0 with the table in shared memory, folds the 32 partial states on
// lane 0 with the linear "advance by 256 zero bytes" operator (crc_table[256 ..] = its 4 byte tables):
//     state(s, A || B) = advance_|B|(state(s, A)) ^ state(0, B),
// and writes length, type, data and CRC into the file buffer - the data as aligned 32-bit words (a chunk's data sits at an
// address = 1 mod 4: every output word is a funnel shift of two staged words).  Warp 0 of the first CTA adds signature, IHDR,
// IEND and the file size.  (Round 1: a byte-per-thread copy kernel, then a CRC kernel whose lanes walked global memory with a
// 256-byte stride and looked the table up in global memory: 64 + 428 us per 12 views.)
__device__ __forceinline__ uint32_t crc_advance256(uint32_t c, const uint32_t *__restrict__ t) {
    return t[256 + (c & 0xFFu)] ^ t[512 + ((c >> 8) & 0xFFu)] ^ t[768 + ((c >> 16) & 0xFFu)] ^ t[1024 + (c >> 24)];
}

constexpr int kFinWarps = 4;
constexpr int kSegWords = 65;   // 64 data words + 1 padding word

__global__ void __launch_bounds__(kFinWarps * 32)
png_finish_kernel(const uint32_t *__restrict__ Z, const unsigned long long *__restrict__ zbits,
                  const unsigned long long *__restrict__ sums, uint8_t *__restrict__ out,
                  const uint32_t *__restrict__ crc_table, unsigned long long *__restrict__ sizes, const Geom G) {
    __shared__ uint32_t s_tab[5 * 256];
    __shared__ uint32_t s_tile[kFinWarps][32 * kSegWords];
    const int img = blockIdx.y;
    const unsigned long long zb = zbits[img];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t c = (size_t)blockIdx.x * kFinWarps + warp;   // chunk = warp
    if (zb == 0ull) {
        if (c == 0 && lane == 0) sizes[img] = 0ull;
        return;
    }
    for (int i = threadIdx.x; i < 5 * 256; i += blockDim.x) s_tab[i] = crc_table[i];
    __syncthreads();
    const size_t L = zlib_len(zb);
    const size_t nchunks = (L + kIdat - 1) / kIdat;
    uint8_t *o = out + (size_t)img * G.out_cap;
    if (c < nchunks) {
        uint32_t *tile = s_tile[warp];
        const uint32_t len = (uint32_t)((c + 1 < nchunks) ? kIdat : L - c * kIdat);
        const uint32_t nwords = (len + 3u) / 4u;
        const uint4 *src = reinterpret_cast<const uint4 *>(Z + (size_t)img * (G.z_cap / 4) + c * (kIdat / 4));
        for (uint32_t q = lane; q * 4u < nwords; q += 32u) {   // (z_cap has 1 KB of slack behind the stream: whole uint4s)
            const uint4 v = src[q];
            const uint32_t w = q * 4u, at = (w >> 6) * kSegWords + (w & 63u);
            tile[at] = v.x; tile[at + 1] = v.y; tile[at + 2] = v.z; tile[at + 3] = v.w;
        }
        __syncwarp();
        uint8_t *tb = reinterpret_cast<uint8_t *>(tile);
        auto at_byte = [](uint32_t i) { return ((i >> 8) * kSegWords) * 4u + (i & 255u); };   // chunk byte -> staged byte
        if (lane == 0) {
            if (c == 0) {
                const uint32_t hd = zlib_header(G.N);
                tb[at_byte(0)] = (uint8_t)hd;
                tb[at_byte(1)] = (uint8_t)(hd >> 8);
            }
            const uint32_t s1 = (uint32_t)((1ull + sums[2 * img]) % 65521ull);
            const uint32_t s2 = (uint32_t)(((unsigned long long)G.N + sums[2 * img + 1]) % 65521ull);
            const uint32_t adler = (s2 << 16) | s1;
            for (int k = 0; k < 4; ++k) {   // the trailer may straddle two chunks
                const size_t i = L - 4 + k;
                if (i >= c * kIdat && i < c * kIdat + len) tb[at_byte((uint32_t)(i - c * kIdat))] = (uint8_t)(adler >> (8 * (3 - k)));
            }
        }
        __syncwarp();
        // CRC over type + data
        const uint32_t nseg = len >> 8;   // full 256-byte segments
        uint32_t r = 0;
        if ((uint32_t)lane < nseg) {
            const uint32_t *seg = tile + lane * kSegWords;
#pragma unroll 4
            for (int k = 0; k < 64; ++k) {
                const uint32_t w = seg[k];
                r = crc_update(r, w, s_tab);
                r = crc_update(r, w >> 8, s_tab);
                r = crc_update(r, w >> 16, s_tab);
                r = crc_update(r, w >> 24, s_tab);
            }
        }
        uint32_t crc = 0xFFFFFFFFu;
        crc = crc_update(crc, 'I', s_tab);
        crc = crc_update(crc, 'D', s_tab);
        crc = crc_update(crc, 'A', s_tab);
        crc = crc_update(crc, 'T', s_tab);
        for (uint32_t k = 0; k < nseg; ++k) {
            const uint32_t rk = __shfl_sync(0xffffffffu, r, (int)k);
            crc = crc_advance256(crc, s_tab) ^ rk;
        }
        if (lane == 0) {
            for (uint32_t i = nseg << 8; i < len; ++i) crc = crc_update(crc, tb[at_byte(i)], s_tab);
            crc ^= 0xFFFFFFFFu;
        }
        crc = __shfl_sync(0xffffffffu, crc, 0);
        // length, type, data, CRC.  ch + 8 = 1 (mod 4): data bytes 3 + 4 j .. 6 + 4 j form the aligned word j
        uint8_t *ch = o + 33 + c * (kIdat + 12);
        auto staged_word = [&](uint32_t w) { return tile[(w >> 6) * kSegWords + (w & 63u)]; };
        const uint32_t n_mid = (len >= 3u) ? (len - 3u) / 4u : 0u;
        uint32_t *dst = reinterpret_cast<uint32_t *>(ch + 8 + 3);
        for (uint32_t j = lane; j < n_mid; j += 32u) {
            const uint32_t lo = staged_word(j), hi = (j + 1u < nwords) ? staged_word(j + 1u) : 0u;
            dst[j] = __funnelshift_r(lo, hi, 24);
        }
        // the ends, bytewise: 8 header bytes + the first 3 data bytes, the last (len - 3) % 4 data bytes + 4 CRC bytes
        if (lane < 8) {
            const uint8_t typ[4] = {'I', 'D', 'A', 'T'};
            ch[lane] = lane < 4 ? (uint8_t)(len >> (8 * (3 - lane))) : typ[lane - 4];
        } else if (lane < 11) {
            const uint32_t i = (uint32_t)lane - 8u;
            if (i < len) ch[8 + i] = tb[at_byte(i)];
        } else if (lane < 14) {
            const uint32_t i = (len >= 3u ? 3u + 4u * n_mid : 3u) + ((uint32_t)lane - 11u);
            if (i >= 3u && i < len) ch[8 + i] = tb[at_byte(i)];
        } else if (lane < 18) {
            ch[8 + len + (lane - 14)] = (uint8_t)(crc >> (8 * (3 - (lane - 14))));
        }
    }
    if (c == 0 && lane == 0) {
        const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
        for (int k = 0; k < 8; ++k) o[k] = sig[k];
        uint8_t *h = o + 8;
        h[0] = 0; h[1] = 0; h[2] = 0; h[3] = 13;
        h[4] = 'I'; h[5] = 'H'; h[6] = 'D'; h[7] = 'R';
        h[8] = (uint8_t)(G.W >> 24); h[9] = (uint8_t)(G.W >> 16); h[10] = (uint8_t)(G.W >> 8); h[11] = (uint8_t)G.W;
        h[12] = (uint8_t)(G.H >> 24); h[13] = (uint8_t)(G.H >> 16); h[14] = (uint8_t)(G.H >> 8); h[15] = (uint8_t)G.H;
        h[16] = 8; h[17] = 2; h[18] = 0; h[19] = 0; h[20] = 0;
        uint32_t crc = 0xFFFFFFFFu;
        for (int k = 4; k < 21; ++k) crc = crc_update(crc, h[k], s_tab);
        crc ^= 0xFFFFFFFFu;
        h[21] = (uint8_t)(crc >> 24); h[22] = (uint8_t)(crc >> 16); h[23] = (uint8_t)(crc >> 8); h[24] = (uint8_t)crc;
        const size_t body = 33 + (nchunks - 1) * (kIdat + 12) + 12 + (L - (nchunks - 1) * kIdat);
        uint8_t *e = o + body;
        const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xAE, 0x42, 0x60, 0x82};
        for (int k = 0; k < 12; ++k) e[k] = iend[k];
        sizes[img] = (unsigned long long)(body + 12);
    }
}

}  // namespace p2ppng
