// p2p_ctx.cuh - contexts, panorama slots and the small helpers every part of the host side uses (included by
// p2p_api.cu only; one translation unit).
#pragma once
#include "p2p.h"
#include "p2p_kernels.cuh"
#include "p2p_jpeg_host.cuh"
#include "p2p_jpegdec.cuh"
#include "p2p_png.cuh"
#include "p2p_pngdec.cuh"

#include <math.h>
#include <stdio.h>
#include <stddef.h>
#include <string.h>

#include <nvtx3/nvToolsExt.h>  // header-only NVTX 3: ranges cost nothing unless a profiler is attached

#include <atomic>
#include <mutex>
#include <new>
#include <string>
#include <vector>

using namespace p2p;

namespace {

// NVTX range over one entry point of the C ABI (per image and stage: upload / decode, project, encode, replicate)
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange &) = delete;
    NvtxRange &operator=(const NvtxRange &) = delete;
};
#define P2P_NVTX(name) NvtxRange nvtx_range_(name)

struct Slot {
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t owned = nullptr;  // created by us, replaced through p2p_set_stream
    uint8_t *d_bgr = nullptr;  // staging copy of the caller's BGR rows
    size_t bgr_cap = 0;
    uint32_t *d_rgba = nullptr;  // packed panorama
    size_t rgba_cap = 0;
    int Wp = 0, Hp = 0, pitch_tex = 0;
    bool valid = false;
    int row0 = 0, row1 = 0;  // packed rows row0 .. row1 (<= Hp, the clamp row) hold data; a full upload has 0 .. Hp
    cudaArray_t arr = nullptr;  // gather-enabled array (sampler 1)
    int arrW = 0, arrH = 0;
    cudaTextureObject_t tex = 0;
    cudaSurfaceObject_t surf = 0;  // the same array, written directly by the pack kernel
    bool tex_current = false;
    // yaw-folded planes (B, G, R) of the quarter-turn sampler, allocated when a panorama renders a quarter-turn group for
    // the second time: (Wp / 4 + 1) x Hp u32 texels each, see fold_kernel
    cudaArray_t farr[3] = {nullptr, nullptr, nullptr};
    int farrW = 0, farrH = 0;
    cudaTextureObject_t ftex[3] = {0, 0, 0};
    cudaSurfaceObject_t fsurf[3] = {0, 0, 0};
    bool fold_current = false;  // the planes hold the panorama of d_rgba (every writer of d_rgba clears it)
    // The panorama of d_rgba has rendered a quarter-turn group from the RGBA texture: the next such launch folds it.  On a
    // B200 the fold costs about one 12-view render (8K: 47 us) and saves ~3 % of every later one, so a panorama rendered
    // once (the files flow, p2p_process_image) never pays it; a resident panorama rendered again and again does.
    bool quarter_seen = false;
    uint8_t *d_out = nullptr;  // device outputs when the caller wants them on the host
    size_t out_cap = 0;
    int32_t *d_tab = nullptr;  // yaw table (ix | fx), 2 * Wp
    size_t tab_cap = 0;
    // JPEG encoder scratch (p2p_encode_jpeg): coefficients, per-block bits / offsets, bit string, stuffed files
    int16_t *j_coef = nullptr;
    size_t j_coef_cap = 0;
    uint32_t *j_bits = nullptr;   // [2][n * n_blocks]: code bits, exclusive offsets
    size_t j_bits_cap = 0;
    uint32_t *j_stream = nullptr;
    size_t j_stream_cap = 0;
    uint32_t *j_cnt = nullptr;    // [2][n * chunks]: 0xFF counts, exclusive offsets
    size_t j_cnt_cap = 0;
    uint8_t *j_out = nullptr;
    size_t j_out_cap = 0;
    unsigned long long *j_tot = nullptr;  // [3][n]: total bits, total 0xFF, n_chunks (as u32 pairs)
    size_t j_tot_cap = 0;
    // PNG encoder scratch (p2p_encode_png)
    uint8_t *pg_F = nullptr;
    size_t pg_F_cap = 0;
    uint16_t *pg_tlen = nullptr;
    size_t pg_tlen_cap = 0;
    uint32_t *pg_blk = nullptr;      // blkoff (64-bit) | blockpos | ntok | lfreq | tile arrays
    size_t pg_blk_cap = 0;
    p2ppng::BlockInfo *pg_info = nullptr;
    size_t pg_info_cap = 0;
    uint32_t *pg_Z = nullptr;
    size_t pg_Z_cap = 0;
    unsigned long long *pg_sums = nullptr;   // [2 n] Adler partial sums | [n] zbits
    size_t pg_sums_cap = 0;
    // JPEG decoder (p2p_upload_pano_jpeg): pinned coefficient staging, device coefficients and component planes
    int16_t *jd_coef_h = nullptr;
    size_t jd_coef_h_cap = 0;
    int16_t *jd_coef_d = nullptr;
    size_t jd_coef_d_cap = 0;
    uint8_t *jd_planes = nullptr;
    size_t jd_planes_cap = 0;
    // device Huffman stage: destuffed scan, subsequence states / block counts, tables, DC differences
    uint32_t *jd_stream = nullptr;
    size_t jd_stream_cap = 0;
    unsigned long long *jd_states = nullptr;  // [2][n_sub]: start, end
    size_t jd_states_cap = 0;
    uint32_t *jd_nblk = nullptr;              // [2][n_sub rounded]: blocks per subsequence, exclusive offsets
    size_t jd_nblk_cap = 0;
    p2pjdec::DevHuff *jd_tables = nullptr;    // [3]
    int32_t *jd_dc = nullptr;                 // [2][3][dc_stride]: DC differences, exclusive sums
    size_t jd_dc_cap = 0;
    uint32_t *jd_tiles = nullptr;             // tile sums / offsets of the three-phase DC scan
    size_t jd_tiles_cap = 0;
    unsigned long long *jd_tot_d = nullptr;   // scan totals (device) [4]
    struct JdFlags { int changed[8]; int bad; int out_of_range; unsigned long long total; int irregular; int gate; } *jd_flags_h = nullptr, *jd_flags_d = nullptr;  // mapped
    uint8_t *jd_raw = nullptr;                // entropy-coded segment as it sits in the file (destuffed on the device)
    size_t jd_raw_cap = 0;
    uint32_t *jd_dcnt = nullptr;              // [2][chunks]: stuffed zeros per 4096-byte chunk, exclusive offsets
    size_t jd_dcnt_cap = 0;
    int *jd_gate_d = nullptr;                 // device copy of the optimistic enqueue's verdict (huff_gate_kernel)
    struct JdRun {                            // the Huffman stage in progress on this slot
        bool pending = false;                 // queued optimistically: the verdict (jd_flags_h->gate) is read after the caller's wait
        bool fast = true;
        p2pjdec::HuffGeom G;
        unsigned sgrid = 0;
        size_t nsub4 = 0;
        p2pjdec::SubSeq *d_sub = nullptr;
        uint32_t *d_ivl_first = nullptr;
        const p2pjdec::SyncLut *d_lut = nullptr;
    } jd_run;
    uint8_t *jd_sub = nullptr;                // subsequence layout + first subsequence of every restart interval
    size_t jd_sub_cap = 0;
    unsigned long long *j_sizes_h = nullptr;  // mapped host memory: file sizes
    unsigned long long *j_sizes_d = nullptr;
    int j_sizes_n = 0;
    // PNG decoder (p2p_upload_pano_png): zlib stream (pinned + device), candidate / block lists, inflated image, history marks
    struct PdCtr { uint32_t n_list, n_cand, n_runs; int bad; unsigned long long sums[2]; };
    uint32_t *pd_zs_h = nullptr;              // pinned: the concatenated zlib stream
    size_t pd_zs_h_cap = 0;
    uint8_t *pd_tab_h = nullptr;              // pinned: CRC segments | candidates read back | blocks of the chain | counters
    size_t pd_tab_h_cap = 0;
    uint32_t *pd_zs = nullptr;
    size_t pd_zs_cap = 0;
    uint8_t *pd_tab = nullptr;                // device: CRC segments | survivor list | candidates | blocks | run starts | counters
    size_t pd_tab_cap = 0;
    uint8_t *pd_raw = nullptr;
    size_t pd_raw_cap = 0;
    uint16_t *pd_ref = nullptr;
    size_t pd_ref_cap = 0;
    p2ppdec::Match *pd_match = nullptr;       // back-references of all blocks (decode pass -> copy pass)
    size_t pd_match_cap = 0;
    cudaEvent_t wait_ev = nullptr;            // blocking-sync event of wait_slot
};

// memoised tap-row range of one view geometry (no yaw, no image: the key of the reference's pitch map cache)
struct RowRange {
    bool valid = false;
    int W = 0, H = 0, Wp = 0, Hp = 0, trig = 0;
    std::vector<p2p_pitch_consts> pc;
    int lo = 0, hi = 0;  // min / max tap row iy over all pixels (the sampler reads rows iy and iy + 1)
};

}  // namespace

struct p2p_ctx {
    int device = 0;
    int n_slots = 0;
    Slot *slots = nullptr;
    std::mutex mu;
    int opt_sampler = 1;
    int opt_warp_w = 32;
    int opt_ny = 4;
    int opt_nb = 1;
    int opt_mirror = 2;        // 2: row-segment kernel (all-word stores, view groups), 1: round-1 mirror kernel, 0: none
    int opt_seg_chunks = 4;    // chunks of 32 pixel pairs a warp of the row-segment kernel walks
    int opt_trig = 0;          // 0: NumPy-exact (SVML) acos / atan2, 1: own minimax fits
    int opt_interp = 0;
    int opt_seam_wrap = 0;     // exact-bilinear mode only: interpolate across the 0 / 360 degree seam instead of clamping
    int opt_partial = 1;       // p2p_process_image transfers only the panorama rows its views can touch
    int opt_gpu_huffman = 1;   // JPEG inputs without restart markers: Huffman decoding on the device
    std::atomic<int> opt_host_wait{0};   // 1: host threads sleep while they wait for a slot's stream (see wait_slot)
    std::atomic<int> opt_png_formats{0}; // PNG decoder subset (parse_png): 0 = 8-bit non-interlaced, 1 = every PNG format
    std::atomic<int> opt_poison{-1};     // P2P_OPT_POISON: byte new buffers are filled with (-1: left as allocated)
    long long gpu_huffman_used = 0, gpu_huffman_fallback = 0;
    std::atomic<long long> png_host_blocks{0};   // dynamic PNG deflate blocks the chain walk measured because the search missed them
    uint32_t *d_crc_table = nullptr;    // CRC-32 table of the PNG encoder
    p2pjpeg::Tables *d_jtab = nullptr;  // JPEG tables + header of (jW, jH, jQ): the entry of jtabs in use
    int jW = 0, jH = 0, jQ = 0;
    struct JTab { int W, H, Q; p2pjpeg::Tables *d; };
    std::vector<JTab> jtabs;            // one device copy per (size, quality) seen: a folder of mixed sizes never waits
    std::vector<RowRange> rows;   // memoised per geometry (the reference's pitch_mapping_cache key, ref :55-73)
    int *d_range = nullptr;
    long long launches = 0;
    uint4 *d_flush = nullptr;
    size_t flush_cap = 0;
};

namespace {

// The last error is kept PER CALLING THREAD (like errno): a context is driven by many host threads at once (one per image
// in flight), several entry points fail before or after they hold the context lock, and a message shared through the
// context could be overwritten - or freed - by another thread between the failing call and p2p_last_error.
thread_local std::string tl_err;
thread_local const p2p_ctx *tl_err_ctx = nullptr;

int fail(p2p_ctx *ctx, int code, const char *what, cudaError_t e = cudaSuccess) {
    if (ctx) {
        tl_err = what;
        if (e != cudaSuccess) {
            tl_err += ": ";
            tl_err += cudaGetErrorString(e);
        }
        tl_err_ctx = ctx;
    }
    return code;
}

#define CK(call)                                                          \
    do {                                                                  \
        cudaError_t e_ = (call);                                          \
        if (e_ != cudaSuccess) {                                          \
            cudaGetLastError();                                           \
            return fail(ctx, (e_ == cudaErrorMemoryAllocation) ? P2P_ERR_NOMEM : P2P_ERR_CUDA, #call, e_); \
        }                                                                 \
    } while (0)

// P2P_OPT_POISON: fill a buffer the context has just allocated with the poison byte.  Device memory: on the legacy stream,
// waited for (the slots' non-blocking streams do not wait for it); a debug facility, so the wait costs nothing that counts.
int poison_new_device(p2p_ctx *ctx, void *p, size_t bytes) {
    const int b = ctx->opt_poison.load(std::memory_order_relaxed);
    if (b < 0) return P2P_OK;
    CK(cudaMemset(p, b, bytes));
    CK(cudaDeviceSynchronize());
    return P2P_OK;
}

void poison_new_host(p2p_ctx *ctx, void *p, size_t bytes) {
    const int b = ctx->opt_poison.load(std::memory_order_relaxed);
    if (b >= 0) memset(p, b, bytes);
}

// every u32 texel of a Wa x Ha array outside rows keep0 .. keep1 := the poison byte (P2P_OPT_POISON, p2p_debug_poison);
// not counted in P2P_OPT_COUNT_LAUNCHES, which must not depend on the poison
int poison_array(p2p_ctx *ctx, cudaSurfaceObject_t surf, int Wa, int Ha, int keep0, int keep1, int byte, cudaStream_t st) {
    if (byte < 0 || Wa <= 0 || Ha <= 0) return P2P_OK;
    poison_surface_kernel<<<dim3((Wa + 255) / 256, Ha), 256, 0, st>>>(surf, Wa, keep0, keep1, 0x01010101u * (uint32_t)byte);
    CK(cudaGetLastError());
    return P2P_OK;
}

template <typename T>
int ensure(p2p_ctx *ctx, T **ptr, size_t *cap, size_t bytes) {
    if (*cap >= bytes && *ptr) return P2P_OK;
    if (*ptr) {
        // a buffer that has to grow (a larger image than this slot has seen) grows with 50 % headroom, and never
        // shrinks: cudaFree / cudaMalloc synchronise the whole device, so a folder of mixed sizes must not pay them per image
        bytes += bytes / 2;
        CK(cudaFree(*ptr));
        *ptr = nullptr;
        *cap = 0;
    }
    void *p = nullptr;
    CK(cudaMalloc(&p, bytes));
    *ptr = static_cast<T *>(p);
    *cap = bytes;
    return poison_new_device(ctx, p, bytes);
}

// for buffers whose size follows the CONTENT of a file (compressed scan length ...): grow with 50 % headroom, so that a
// folder of similar files does not free / allocate (= synchronise the device) on every slightly larger one
template <typename T>
int ensure_grow(p2p_ctx *ctx, T **ptr, size_t *cap, size_t bytes) {
    if (*cap >= bytes && *ptr) return P2P_OK;
    return ensure(ctx, ptr, cap, *ptr ? bytes : bytes + bytes / 2);  // ensure() adds the headroom itself when it regrows
}

// Wait until everything queued on the slot's stream is done.  Default: cudaStreamSynchronize (the CUDA default spins while
// the host has more cores than contexts - lowest latency, one busy core per waiting thread).  P2P_OPT_HOST_WAIT = 1: the
// thread sleeps on a blocking-sync event instead, so that many images in flight (or several ranks on one box) leave the cores
// to the threads that have work: 1.0 instead of 3.7 ms of CPU per image in the files flow, same throughput.
cudaError_t wait_slot(p2p_ctx *ctx, Slot &s) {
    if (!ctx->opt_host_wait.load(std::memory_order_relaxed)) return cudaStreamSynchronize(s.stream);
    if (!s.wait_ev) {
        const cudaError_t e = cudaEventCreateWithFlags(&s.wait_ev, cudaEventBlockingSync | cudaEventDisableTiming);
        if (e != cudaSuccess) return e;
    }
    const cudaError_t e = cudaEventRecord(s.wait_ev, s.stream);
    return e != cudaSuccess ? e : cudaEventSynchronize(s.wait_ev);
}

// the mapped host array the encoders write the sizes of n files to (s.j_sizes_h; the kernels see s.j_sizes_d)
int ensure_file_sizes(p2p_ctx *ctx, Slot &s, int n) {
    if (s.j_sizes_n >= n) return P2P_OK;
    if (s.j_sizes_h) CK(cudaFreeHost(s.j_sizes_h));
    s.j_sizes_h = nullptr;
    CK(cudaHostAlloc(reinterpret_cast<void **>(&s.j_sizes_h), (size_t)n * sizeof(unsigned long long),
                     cudaHostAllocMapped | cudaHostAllocPortable));
    poison_new_host(ctx, s.j_sizes_h, (size_t)n * sizeof(unsigned long long));
    CK(cudaHostGetDevicePointer(reinterpret_cast<void **>(&s.j_sizes_d), s.j_sizes_h, 0));
    s.j_sizes_n = n;
    return P2P_OK;
}

int slot_ok(p2p_ctx *ctx, int slot) { return ctx && slot >= 0 && slot < ctx->n_slots; }

int check_dims(p2p_ctx *ctx, int Wp, int Hp) {
    if (Wp <= 0 || Hp <= 0) return fail(ctx, P2P_ERR_INVALID, "panorama size must be positive");
    // cv::remap asserts every dimension < SHRT_MAX (SURVEY 8b "limits inherited")
    if (Wp >= 32767 || Hp >= 32767) return fail(ctx, P2P_ERR_LIMIT, "panorama dimension >= 32767");
    return P2P_OK;
}

int prepare_slot(p2p_ctx *ctx, Slot &s, int Wp, int Hp) {
    const int pitch_tex = ((Wp + 1) + 31) & ~31;  // 128-byte aligned rows
    const size_t bytes = (size_t)pitch_tex * (size_t)(Hp + 1) * 4;
    int rc = ensure(ctx, &s.d_rgba, &s.rgba_cap, bytes);
    if (rc) return rc;
    s.Wp = Wp;
    s.Hp = Hp;
    s.pitch_tex = pitch_tex;
    s.tex_current = false;
    s.fold_current = false;
    s.quarter_seen = false;
    return P2P_OK;
}

int ensure_array(p2p_ctx *ctx, Slot &s);

}  // namespace
