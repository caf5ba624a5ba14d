// p2p_jpeg.cuh - sm_100a baseline JPEG encoder for the projected views (SURVEY 8f-2: the encode side of the path).
//
// The reference writes every view with cv2.imwrite (ref app/panorama_to_plane-pitch.py:277); with
// --output_format jpg|jpeg (ref :400-405) that is libjpeg-turbo at OpenCV's defaults: quality 95, baseline
// sequential, 4:2:0, Annex K Huffman tables, no restart markers.  Every stage of that encoder is integer
// arithmetic, so the kernels below restate it operation by operation and the produced file is byte-identical
// to cv2.imwrite's (oracle/jpeg_model.py is the NumPy restatement, pinned against cv2.imencode):
//   jccolor.c  rgb_ycc_convert (16-bit fixed point)      jcsample.c  h2v2_downsample (bias 1, 2, 1, 2 ...)
//   jfdctint.c jpeg_fdct_islow                            jcdctmgr.c  round-half-away quantisation by 8 q
//   jccoefct.c dummy edge blocks (zero AC, previous DC)   jchuff.c    Huffman coding, 0xFF stuffing, 1-bit padding
//
// Pipeline (all images of a call in one grid each, blockIdx.y / z = image):
//   jpeg_dct_kernel    BGR tile staged in shared memory -> Y / Cb / Cr MCUs (16 x 16 px) -> FDCT -> quantised coefficients in
//                      zigzag order, stored in scan order (6 blocks per MCU: Y00 Y01 Y10 Y11 Cb Cr)
//   jpeg_size_kernel   bits of every block's Huffman code (DC difference against the previous block of its component)
//   jpeg_scan_kernel   exclusive prefix sum per image -> bit offset of every block
//   jpeg_emit_kernel   every block writes its code bits at its offset (big-endian bit string, 32-bit words,
//                      atomicOr on the two boundary words)
//   jpeg_ffcount_kernel + jpeg_scan_kernel + jpeg_stuff_kernel   0xFF -> 0xFF 0x00 byte stuffing by a second scan
//   jpeg_finish_kernel header (SOI .. SOS), EOI and the file size
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace p2pjpeg {

constexpr int kMcuPerCta = 4;        // jpeg_dct_kernel: 64 threads per MCU
constexpr int kHeaderMax = 640;      // SOI + APP0 + 2 DQT + SOF0 + 4 DHT + SOS = 623 bytes

struct Tables {
    uint16_t div_y[64], div_c[64];   // d = 8 * q, natural order (jcdctmgr.c: the islow FDCT output is scaled by 8)
    uint32_t rcp_y[64], rcp_c[64];   // floor(2^32 / d) + 1: umulhi(n, rcp) == n / d exactly for n < 2^32 / d (n < 2^18 here)
    uint32_t dc[2][16];              // (code << 8) | length, by category
    uint32_t ac[2][256];             // (code << 8) | length, by (run << 4) | size
    uint8_t header[kHeaderMax];
    int header_len;
};

struct Geometry {
    int W, H;
    int mcux, mcuy, n_mcu, n_blocks; // per image
    int blk_stride;                  // n_blocks rounded up to 4: per-image stride of the bits / offsets arrays
    int ybw, ybh;                    // real luma blocks (ceil(W / 8), ceil(H / 8)); chroma blocks are always real
    int cw, ch;                      // chroma plane size (ceil(W / 2), ceil(H / 2))
    size_t img_stride;               // bytes between input images (W * H * 3)
    size_t cap_bits_words;           // 32-bit words of the unstuffed bit string per image
    size_t cap_out;                  // bytes of the output file buffer per image
};

// natural index -> zigzag position, by column: kZigzagCol[c][r] = position of natural index r * 8 + c (one 8-byte load
// per thread of the column pass)
__device__ const uint8_t kZigzagCol[8][8] = {
    {0, 2, 3, 9, 10, 20, 21, 35},
    {1, 4, 8, 11, 19, 22, 34, 36},
    {5, 7, 12, 18, 23, 33, 37, 48},
    {6, 13, 17, 24, 32, 38, 47, 49},
    {14, 16, 25, 31, 39, 46, 50, 57},
    {15, 26, 30, 40, 45, 51, 56, 58},
    {27, 29, 41, 44, 52, 55, 59, 62},
    {28, 42, 43, 53, 54, 60, 61, 63}};

// ---- jfdctint.c: one 8-point pass (exact integers) ---------------------------------------------------------
template <bool FIRST>
__device__ __forceinline__ void fdct_pass(int *d) {
    constexpr int CONST_BITS = 13, PASS1_BITS = 2;
    const int t0 = d[0] + d[7], t7 = d[0] - d[7], t1 = d[1] + d[6], t6 = d[1] - d[6];
    const int t2 = d[2] + d[5], t5 = d[2] - d[5], t3 = d[3] + d[4], t4 = d[3] - d[4];
    const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    constexpr int N = FIRST ? CONST_BITS - PASS1_BITS : CONST_BITS + PASS1_BITS;
    constexpr int RND = 1 << (N - 1);
    if (FIRST) {
        d[0] = (t10 + t11) << PASS1_BITS;
        d[4] = (t10 - t11) << PASS1_BITS;
    } else {
        d[0] = (t10 + t11 + (1 << (PASS1_BITS - 1))) >> PASS1_BITS;
        d[4] = (t10 - t11 + (1 << (PASS1_BITS - 1))) >> PASS1_BITS;
    }
    int z1 = (t12 + t13) * 4433;
    d[2] = (z1 + t13 * 6270 + RND) >> N;
    d[6] = (z1 + t12 * -15137 + RND) >> N;
    z1 = t4 + t7;
    int z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
    const int z5 = (z3 + z4) * 9633;
    const int a4 = t4 * 2446, a5 = t5 * 16819, a6 = t6 * 25172, a7 = t7 * 12299;
    z1 *= -7373;
    z2 *= -20995;
    z3 = z3 * -16069 + z5;
    z4 = z4 * -3196 + z5;
    d[7] = (a4 + z1 + z3 + RND) >> N;
    d[5] = (a5 + z2 + z4 + RND) >> N;
    d[3] = (a6 + z2 + z3 + RND) >> N;
    d[1] = (a7 + z1 + z4 + RND) >> N;
}

// ---- colour conversion + downsample + FDCT + quantisation ----------------------------------------------------
// grid: x = ceil(mcux / kMcuPerCta), y = MCU row, z = image; block: 64 threads per MCU, kMcuPerCta MCUs side by side.
// The CTA first stages its 16 rows x (kMcuPerCta * 16) pixels in shared memory with coalesced word loads (edge
// replication = clamped coordinates on the slow byte path), converts from there, and writes its coefficients -
// contiguous in scan order - with 16-byte stores.
constexpr int kTileBytes = kMcuPerCta * 16 * 3;   // bytes per staged pixel row

__global__ void __launch_bounds__(64 * kMcuPerCta)
jpeg_dct_kernel(const uint8_t *__restrict__ bgr, int16_t *__restrict__ coef, const Tables *__restrict__ T, const Geometry G) {
    __shared__ __align__(16) uint8_t s_px[16][kTileBytes];
    __shared__ int s_blk[kMcuPerCta][6][8 * 9];         // level-shifted samples, then row-pass results; rows padded to 9
                                                        // words: the row / column passes hit 32 different banks
    __shared__ __align__(16) int16_t s_out[kMcuPerCta][6][64];
    const int lm = threadIdx.x >> 6, tid = threadIdx.x & 63;
    const int my = blockIdx.y, img = blockIdx.z;
    const int mx = blockIdx.x * kMcuPerCta + lm;
    const bool live = mx < G.mcux;
    const int mcu = my * G.mcux + mx;
    const uint8_t *src = bgr + (size_t)img * G.img_stride;

    // stage: tile row r = image row min(my * 16 + r, H - 1), tile byte c = pixel x0 + c / 3 (clamped), channel c % 3
    {
        const int x0 = blockIdx.x * kMcuPerCta * 16;
        const bool fast = (x0 + kMcuPerCta * 16 <= G.W) && (((size_t)G.W * 3) % 4 == 0) &&
                          ((reinterpret_cast<uintptr_t>(src) & 3) == 0);
        constexpr int kWords = kTileBytes / 4;
        for (int i = threadIdx.x; i < 16 * kWords; i += blockDim.x) {
            const int r = i / kWords, w = i - r * kWords;
            int y = my * 16 + r;
            y = (y < G.H) ? y : G.H - 1;
            const uint8_t *rowp = src + (size_t)y * G.W * 3;
            uint32_t v;
            if (fast) {
                v = __ldg(reinterpret_cast<const uint32_t *>(rowp + (size_t)x0 * 3) + w);
            } else {
                v = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int c = w * 4 + k;
                    int x = x0 + c / 3;
                    x = (x < G.W) ? x : G.W - 1;
                    v |= (uint32_t)rowp[(size_t)x * 3 + (c % 3)] << (8 * k);
                }
            }
            *reinterpret_cast<uint32_t *>(&s_px[r][w * 4]) = v;
        }
    }
    __syncthreads();

    if (live) {
        // thread = one chroma sample = one 2 x 2 luma quad
        const int qx = tid & 7, qy = tid >> 3;
        const int cx = mx * 8 + qx;
        int cy = my * 8 + qy;                             // chroma row: the DOWNSAMPLED plane is replicated downwards
        cy = (cy < G.ch) ? cy : G.ch - 1;
        const int rc = 2 * cy - my * 16;                  // its two input rows inside the tile (always 0 .. 14)
        int sb = 0, sr = 0;
#pragma unroll
        for (int dy = 0; dy < 2; ++dy) {
#pragma unroll
            for (int dx = 0; dx < 2; ++dx) {
                const int lx = 2 * qx + dx;
                const uint8_t *pc = &s_px[rc + dy][(lm * 16 + lx) * 3];
                const int b = pc[0], g = pc[1], r = pc[2];
                sb += (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16;
                sr += (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16;
                const int ly = 2 * qy + dy;
                const uint8_t *pl = &s_px[ly][(lm * 16 + lx) * 3];
                const int yv = (19595 * (int)pl[2] + 38470 * (int)pl[1] + 7471 * (int)pl[0] + 32768) >> 16;
                s_blk[lm][(ly >> 3) * 2 + (lx >> 3)][(ly & 7) * 9 + (lx & 7)] = yv - 128;
            }
        }
        const int bias = (cx & 1) ? 2 : 1;
        s_blk[lm][4][qy * 9 + qx] = ((sb + bias) >> 2) - 128;
        s_blk[lm][5][qy * 9 + qx] = ((sr + bias) >> 2) - 128;
    }
    __syncthreads();
    const int blk = tid >> 3, lane8 = tid & 7;            // 48 threads: block 0..5, row / column 0..7
    int d[8];
    if (live && blk < 6) {
#pragma unroll
        for (int i = 0; i < 8; ++i) d[i] = s_blk[lm][blk][lane8 * 9 + i];
        fdct_pass<true>(d);
    }
    __syncthreads();
    if (live && blk < 6) {
#pragma unroll
        for (int i = 0; i < 8; ++i) s_blk[lm][blk][lane8 * 9 + i] = d[i];
    }
    __syncthreads();
    if (live && blk < 6) {
#pragma unroll
        for (int i = 0; i < 8; ++i) d[i] = s_blk[lm][blk][i * 9 + lane8];
        fdct_pass<false>(d);
        // real block?  (jccoefct.c: blocks past the real block grid of the component are dummies)
        bool real = true;
        if (blk < 4) real = (mx * 2 + (blk & 1) < G.ybw) && (my * 2 + (blk >> 1) < G.ybh);
        const uint16_t *div = (blk < 4) ? T->div_y : T->div_c;
        const uint32_t *rcp = (blk < 4) ? T->rcp_y : T->rcp_c;
        const uint2 zz2 = __ldg(reinterpret_cast<const uint2 *>(&kZigzagCol[lane8][0]));
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int nat = i * 8 + lane8;
            const int zpos = (int)(((i < 4) ? (zz2.x >> (8 * i)) : (zz2.y >> (8 * (i - 4)))) & 0xFFu);
            const int dv = div[nat];
            const int a = (int)__umulhi((uint32_t)(abs(d[i]) + (dv >> 1)), rcp[nat]);   // (|x| + d / 2) / d
            s_out[lm][blk][zpos] = (int16_t)(real ? ((d[i] < 0) ? -a : a) : 0);
        }
    }
    __syncthreads();
    if (live && tid == 0) {
        // dummy luma blocks carry the DC of the previous block of the MCU buffer
        int prev = s_out[lm][0][0];
        for (int b = 1; b < 4; ++b) {
            const bool real = (mx * 2 + (b & 1) < G.ybw) && (my * 2 + (b >> 1) < G.ybh);
            if (!real) s_out[lm][b][0] = (int16_t)prev;
            else prev = s_out[lm][b][0];
        }
    }
    __syncthreads();
    // the CTA's MCUs are consecutive in scan order: one contiguous run of 768 bytes per MCU
    {
        const int n_live = (G.mcux - blockIdx.x * kMcuPerCta < kMcuPerCta) ? G.mcux - blockIdx.x * kMcuPerCta : kMcuPerCta;
        const int n16 = n_live * 6 * 64 * 2 / 16;
        uint4 *dst = reinterpret_cast<uint4 *>(coef + ((size_t)img * G.n_blocks + (size_t)(my * G.mcux + blockIdx.x * kMcuPerCta) * 6) * 64);
        const uint4 *so = reinterpret_cast<const uint4 *>(&s_out[0][0][0]);
        for (int i = threadIdx.x; i < n16; i += blockDim.x) dst[i] = so[i];
    }
    (void)mcu;
}

// ---- entropy coding ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int nbits_of(int v) { return 32 - __clz(abs(v)); }

// index of the block whose DC is the predictor of block g = mcu * 6 + k (same component, scan order); -1: none
__device__ __forceinline__ int pred_block(int mcu, int k) {
    if (k >= 1 && k <= 3) return mcu * 6 + k - 1;
    if (mcu == 0) return -1;
    return (mcu - 1) * 6 + ((k == 0) ? 3 : k);
}

// thread per block: number of code bits
__global__ void __launch_bounds__(256)
jpeg_size_kernel(const int16_t *__restrict__ coef, uint32_t *__restrict__ bits, const Tables *__restrict__ T, const Geometry G) {
    __shared__ uint32_t s_ac[2][256];
    for (int i = threadIdx.x; i < 512; i += blockDim.x) s_ac[i >> 8][i & 255] = T->ac[i >> 8][i & 255];
    __syncthreads();
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int img = blockIdx.y;
    if (g >= G.n_blocks) return;
    const int mcu = g / 6, k = g - mcu * 6, t = (k < 4) ? 0 : 1;
    const int16_t *c = coef + ((size_t)img * G.n_blocks + g) * 64;
    const int p = pred_block(mcu, k);
    const int pred = (p < 0) ? 0 : coef[((size_t)img * G.n_blocks + p) * 64];
    const uint4 *c4 = reinterpret_cast<const uint4 *>(c);
    uint32_t total = 0;
    int run = 0;
#pragma unroll 1
    for (int w = 0; w < 8; ++w) {
        const uint4 v4 = __ldg(c4 + w);
        const uint32_t ws[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
        for (int h = 0; h < 8; ++h) {
            const int v = (int)(int16_t)(ws[h >> 1] >> ((h & 1) * 16));
            if (w == 0 && h == 0) {
                const int s = nbits_of(v - pred);
                total += (T->dc[t][s] & 0xFF) + s;
                continue;
            }
            if (v == 0) {
                ++run;
                continue;
            }
            total += (uint32_t)(run >> 4) * (s_ac[t][0xF0] & 0xFF);
            const int s = nbits_of(v);
            total += (s_ac[t][((run & 15) << 4) | s] & 0xFF) + s;
            run = 0;
        }
    }
    if (run) total += s_ac[t][0] & 0xFF;
    bits[(size_t)img * G.blk_stride + g] = total;
}

// exclusive prefix sum of n items per image (one CTA per image); out[i] = sum of in[0 .. i), total[img] = sum.
// Tiles of 4096 items: every thread takes 4 consecutive items (one 16-byte load; `stride` and the buffers are
// 16-byte aligned), warp shuffles + one shared-memory hop scan the tile, a running carry links the tiles.
__global__ void __launch_bounds__(1024)
jpeg_scan_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, const uint32_t *__restrict__ n_per_image,
                 uint32_t n_fixed, size_t stride, unsigned long long *__restrict__ total) {
    __shared__ uint32_t s_warp[32];
    __shared__ unsigned long long s_carry;
    const int img = blockIdx.x;
    const uint32_t n = n_per_image ? n_per_image[img] : n_fixed;
    const uint32_t *src = in + (size_t)img * stride;
    uint32_t *dst = out + (size_t)img * stride;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0ull;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 4096u) {
        const uint32_t i0 = base + threadIdx.x * 4u;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (i0 + 3u < n) {
            v = *reinterpret_cast<const uint4 *>(src + i0);
        } else {
            if (i0 < n) v.x = src[i0];
            if (i0 + 1u < n) v.y = src[i0 + 1u];
            if (i0 + 2u < n) v.z = src[i0 + 2u];
        }
        const uint32_t sum = v.x + v.y + v.z + v.w;     // a tile holds < 2^32 (4096 items of < 2^20 each)
        uint32_t inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += u;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t u = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += u;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        const unsigned long long carry = s_carry;
        const uint32_t excl = (uint32_t)carry + (inc - sum) + (warp ? s_warp[warp - 1] : 0u);
        const uint4 o4 = make_uint4(excl, excl + v.x, excl + v.x + v.y, excl + v.x + v.y + v.z);
        if (i0 + 3u < n) {
            *reinterpret_cast<uint4 *>(dst + i0) = o4;
        } else {
            if (i0 < n) dst[i0] = o4.x;
            if (i0 + 1u < n) dst[i0 + 1u] = o4.y;
            if (i0 + 2u < n) dst[i0 + 2u] = o4.z;
        }
        __syncthreads();                                 // everyone has read s_carry and s_warp
        if (threadIdx.x == 0) s_carry = carry + s_warp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) total[img] = s_carry;
}

// The same scan for long arrays in three launches that use the whole GPU instead of one CTA per image:
//   scan_tile_sums_kernel   sum of every 4096-item tile            (grid: tiles x images)
//   jpeg_scan_kernel        exclusive scan of the tile sums        (one CTA per image, a few hundred items)
//   scan_tiles_apply_kernel exclusive scan inside every tile + the tile's offset
// (the DC predictions of an 8192 x 4096 JPEG file are 524,288 differences per luma plane: 153 us in one CTA, ~15 us here)
__global__ void __launch_bounds__(1024)
scan_tile_sums_kernel(const uint32_t *__restrict__ in, const uint32_t *__restrict__ n_per_image, uint32_t n_fixed, size_t stride,
                      uint32_t *__restrict__ tile_sums, size_t tiles_stride) {
    __shared__ uint32_t s_warp[32];
    const int img = blockIdx.y;
    const uint32_t n = n_per_image ? n_per_image[img] : n_fixed;
    const uint32_t *src = in + (size_t)img * stride;
    const uint32_t i0 = blockIdx.x * 4096u + threadIdx.x * 4u;
    uint32_t sum = 0;
    if (i0 + 3u < n) {
        const uint4 v = *reinterpret_cast<const uint4 *>(src + i0);
        sum = v.x + v.y + v.z + v.w;
    } else {
        if (i0 < n) sum += src[i0];
        if (i0 + 1u < n) sum += src[i0 + 1u];
        if (i0 + 2u < n) sum += src[i0 + 2u];
    }
    sum = __reduce_add_sync(0xffffffffu, sum);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x < 32) {
        const uint32_t t = __reduce_add_sync(0xffffffffu, s_warp[threadIdx.x]);
        if (threadIdx.x == 0) tile_sums[(size_t)img * tiles_stride + blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(1024)
scan_tiles_apply_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, const uint32_t *__restrict__ n_per_image,
                        uint32_t n_fixed, size_t stride, const uint32_t *__restrict__ tile_offs, size_t tiles_stride) {
    __shared__ uint32_t s_warp[32];
    const int img = blockIdx.y;
    const uint32_t n = n_per_image ? n_per_image[img] : n_fixed;
    const uint32_t *src = in + (size_t)img * stride;
    uint32_t *dst = out + (size_t)img * stride;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t i0 = blockIdx.x * 4096u + threadIdx.x * 4u;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (i0 + 3u < n) {
        v = *reinterpret_cast<const uint4 *>(src + i0);
    } else {
        if (i0 < n) v.x = src[i0];
        if (i0 + 1u < n) v.y = src[i0 + 1u];
        if (i0 + 2u < n) v.z = src[i0 + 2u];
    }
    const uint32_t sum = v.x + v.y + v.z + v.w;
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += u;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = s_warp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += u;
        }
        s_warp[lane] = w;
    }
    __syncthreads();
    const uint32_t excl = tile_offs[(size_t)img * tiles_stride + blockIdx.x] + (inc - sum) + (warp ? s_warp[warp - 1] : 0u);
    const uint4 o4 = make_uint4(excl, excl + v.x, excl + v.x + v.y, excl + v.x + v.y + v.z);
    if (i0 + 3u < n) {
        *reinterpret_cast<uint4 *>(dst + i0) = o4;
    } else {
        if (i0 < n) dst[i0] = o4.x;
        if (i0 + 1u < n) dst[i0 + 1u] = o4.y;
        if (i0 + 2u < n) dst[i0 + 2u] = o4.z;
    }
}

struct BitSink {
    uint32_t *words;
    unsigned long long acc;   // low `n` bits are pending (the first word starts with the offset's zero bits)
    int n;
    uint32_t widx;
    bool first;
    __device__ __forceinline__ void put(uint32_t code, int size) {
        acc = (acc << size) | code;
        n += size;
        if (n >= 32) {
            const uint32_t w = (uint32_t)(acc >> (n - 32));
            const uint32_t be = __byte_perm(w, 0, 0x0123);
            if (first) atomicOr(words + widx, be);   // shares the word with the previous block
            else words[widx] = be;
            first = false;
            ++widx;
            n -= 32;
        }
    }
    __device__ __forceinline__ void finish() {
        if (n > 0) {
            const uint32_t w = (uint32_t)(acc << (32 - n));  // only the low n bits of acc are pending
            atomicOr(words + widx, __byte_perm(w, 0, 0x0123));
        }
    }
};

// thread per block: write the code bits at the block's bit offset
__global__ void __launch_bounds__(256)
jpeg_emit_kernel(const int16_t *__restrict__ coef, const uint32_t *__restrict__ offs, uint32_t *__restrict__ stream,
                 const Tables *__restrict__ T, const Geometry G, const unsigned long long *__restrict__ total_bits) {
    __shared__ uint32_t s_ac[2][256];
    __shared__ uint32_t s_dc[2][16];
    for (int i = threadIdx.x; i < 512; i += blockDim.x) s_ac[i >> 8][i & 255] = T->ac[i >> 8][i & 255];
    if (threadIdx.x < 32) s_dc[threadIdx.x >> 4][threadIdx.x & 15] = T->dc[threadIdx.x >> 4][threadIdx.x & 15];
    __syncthreads();
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int img = blockIdx.y;
    if (g >= G.n_blocks) return;
    if (total_bits[img] > (unsigned long long)G.cap_bits_words * 32ull) return;  // would not fit: write nothing (size 0)
    const int mcu = g / 6, k = g - mcu * 6, t = (k < 4) ? 0 : 1;
    const int16_t *c = coef + ((size_t)img * G.n_blocks + g) * 64;
    const int p = pred_block(mcu, k);
    const int pred = (p < 0) ? 0 : coef[((size_t)img * G.n_blocks + p) * 64];
    const uint32_t off = offs[(size_t)img * G.blk_stride + g];
    BitSink bs;
    bs.words = stream + (size_t)img * G.cap_bits_words;
    bs.acc = 0;
    bs.n = (int)(off & 31u);
    bs.widx = off >> 5;
    bs.first = true;
    const uint4 *c4 = reinterpret_cast<const uint4 *>(c);
    int run = 0;
#pragma unroll 1
    for (int w = 0; w < 8; ++w) {
        const uint4 v4 = __ldg(c4 + w);
        const uint32_t ws[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
        for (int h = 0; h < 8; ++h) {
            const int v = (int)(int16_t)(ws[h >> 1] >> ((h & 1) * 16));
            if (w == 0 && h == 0) {
                const int diff = v - pred;
                const int s = nbits_of(diff);
                const uint32_t e = s_dc[t][s];
                const uint32_t vb = (uint32_t)((diff < 0) ? diff - 1 : diff) & ((1u << s) - 1u);
                bs.put(((e >> 8) << s) | vb, (int)(e & 0xFF) + s);
                continue;
            }
            if (v == 0) {
                ++run;
                continue;
            }
            while (run > 15) {
                const uint32_t z = s_ac[t][0xF0];
                bs.put(z >> 8, (int)(z & 0xFF));
                run -= 16;
            }
            const int s = nbits_of(v);
            const uint32_t e = s_ac[t][(run << 4) | s];
            const uint32_t vb = (uint32_t)((v < 0) ? v - 1 : v) & ((1u << s) - 1u);
            bs.put(((e >> 8) << s) | vb, (int)(e & 0xFF) + s);
            run = 0;
        }
    }
    if (run) {
        const uint32_t z = s_ac[t][0];
        bs.put(z >> 8, (int)(z & 0xFF));
    }
    bs.finish();
}

// byte i of the unstuffed scan data of an image, with the final partial byte padded with 1-bits (flush_bits)
__device__ __forceinline__ uint32_t scan_byte(const uint8_t *s, unsigned long long i, unsigned long long total_bits) {
    uint32_t b = s[i];
    const unsigned long long last = (total_bits - 1) >> 3;
    const int rem = (int)(total_bits & 7);
    if (i == last && rem) b |= (1u << (8 - rem)) - 1u;
    return b;
}

// thread per 16-byte chunk: number of 0xFF bytes; also the chunk count per image for the scan
__global__ void __launch_bounds__(256)
jpeg_ffcount_kernel(const uint32_t *__restrict__ stream, uint32_t *__restrict__ cnt, uint32_t *__restrict__ n_chunks,
                    const Geometry G, const unsigned long long *__restrict__ total_bits) {
    const int img = blockIdx.y;
    const unsigned long long tb = total_bits[img];
    const unsigned long long nbytes = (tb + 7) >> 3;
    const unsigned long long chunks = (nbytes + 15) >> 4;
    const unsigned long long chunk = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (chunk == 0) n_chunks[img] = (tb > (unsigned long long)G.cap_bits_words * 32ull) ? 0u : (uint32_t)chunks;
    if (chunk >= chunks || tb > (unsigned long long)G.cap_bits_words * 32ull) return;
    const uint8_t *s = reinterpret_cast<const uint8_t *>(stream + (size_t)img * G.cap_bits_words);
    uint32_t n = 0;
    const unsigned long long b0 = chunk << 4;
    for (int i = 0; i < 16; ++i)
        if (b0 + i < nbytes) n += (scan_byte(s, b0 + i, tb) == 0xFFu);
    cnt[(size_t)img * (G.cap_bits_words / 4) + chunk] = n;
}

__global__ void __launch_bounds__(256)
jpeg_stuff_kernel(const uint32_t *__restrict__ stream, const uint32_t *__restrict__ ffoff, uint8_t *__restrict__ out,
                  const Geometry G, const Tables *__restrict__ T, const unsigned long long *__restrict__ total_bits,
                  const unsigned long long *__restrict__ total_ff) {
    const int img = blockIdx.y;
    const unsigned long long tb = total_bits[img];
    if (tb > (unsigned long long)G.cap_bits_words * 32ull) return;
    const unsigned long long nbytes = (tb + 7) >> 3;
    const unsigned long long chunks = (nbytes + 15) >> 4;
    const unsigned long long chunk = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (chunk >= chunks) return;
    if ((unsigned long long)T->header_len + nbytes + total_ff[img] + 2ull > (unsigned long long)G.cap_out) return;
    const uint8_t *s = reinterpret_cast<const uint8_t *>(stream + (size_t)img * G.cap_bits_words);
    const unsigned long long b0 = chunk << 4;
    uint8_t *dst = out + (size_t)img * G.cap_out + T->header_len + b0 + ffoff[(size_t)img * (G.cap_bits_words / 4) + chunk];
    for (int i = 0; i < 16; ++i) {
        if (b0 + i >= nbytes) break;
        const uint32_t b = scan_byte(s, b0 + i, tb);
        *dst++ = (uint8_t)b;
        if (b == 0xFFu) *dst++ = 0;
    }
}

// header, EOI and size of every file (size 0 = did not fit)
__global__ void jpeg_finish_kernel(uint8_t *__restrict__ out, const Geometry G, const Tables *__restrict__ T,
                                   const unsigned long long *__restrict__ total_bits,
                                   const unsigned long long *__restrict__ total_ff, unsigned long long *__restrict__ sizes) {
    const int img = blockIdx.x;
    const unsigned long long tb = total_bits[img];
    const unsigned long long nbytes = (tb + 7) >> 3;
    const unsigned long long size = (unsigned long long)T->header_len + nbytes + total_ff[img] + 2ull;
    const bool fits = tb <= (unsigned long long)G.cap_bits_words * 32ull && size <= (unsigned long long)G.cap_out;
    uint8_t *o = out + (size_t)img * G.cap_out;
    if (fits) {
        for (int i = threadIdx.x; i < T->header_len; i += blockDim.x) o[i] = T->header[i];
        if (threadIdx.x == 0) {
            o[size - 2] = 0xFF;
            o[size - 1] = 0xD9;
        }
    }
    if (threadIdx.x == 0) sizes[img] = fits ? size : 0ull;
}

}  // namespace p2pjpeg
