// p2p_pngdec.cuh - PNG decoder for the input panoramas (SURVEY 8f-2: the decode side of cv2.imread(path), ref :244, for
// .png inputs): inflate, unfilter and the conversion to the BGR staging image on the device.
//
// A deflate stream has no index: block k starts where block k - 1 ends, Huffman codes change per block and every
// back-reference may reach 32 KiB into what earlier blocks produced.  The decoder breaks both chains:
//
//   1. block starts are FOUND, not followed.  Every bit position of the stream is tested for the header of a dynamic
//      Huffman block (pd_quick_kernel: BTYPE = 2, HLIT / HDIST in range, a complete code-length code; pd_full_kernel on the
//      survivors: the 258 .. 316 code lengths decode, an end-of-block code exists, literal / length and distance codes are
//      complete by inflate's own rules).  A random position passes with negligible probability, every true dynamic block
//      passes.
//   2. every candidate is decoded from its header to its end-of-block symbol on its own (pd_measure_kernel, a warp per
//      candidate, tables in shared memory): where it ends, how many bytes it produces.  The host then walks the chain from
//      the first block: a block that ends where a measured candidate starts continues there; stored and fixed-Huffman blocks
//      (no recognisable header) are measured by the same routine on the host when the walk reaches them.  The walk gives
//      every block its output offset.
//   3. the blocks of the chain are decoded in parallel with SYMBOLIC history.  pd_decode_kernel (eight blocks per warp)
//      writes the literals and records the back-references; pd_copy_kernel (a warp per block) executes them in order: a
//      back-reference that reaches in front of its own block cannot be resolved yet, so the byte is recorded as "history
//      byte k before my block" in a 16-bit side array (0 = final byte); copies inside the block copy those marks along.
//   4. the last 32 KiB of every block are made final first (all marks of a block point into the 32 KiB in front of it, i.e.
//      into the last 32 KiB of earlier blocks).  That is a chain through all blocks, cut into ~sqrt(n) GROUPS of consecutive
//      blocks: pd_tails_group_kernel walks every group on its own SM and re-bases what it cannot resolve inside the group to
//      "history byte k before my GROUP"; pd_tails_chain_kernel walks the groups in order and finalises the 32 KiB in front of
//      each; pd_tails_finish_kernel resolves the re-based marks everywhere.  After that every remaining mark anywhere points
//      at a final byte and pd_resolve_kernel finishes the image in one parallel pass.
//   5. Adler-32 of the inflated data and CRC-32 of every chunk are checked (pd_adler_kernel, pd_crc_kernel + host fold):
//      a file libpng would refuse is never decoded differently - it is declined and read by cv2.imread as before.
//   6. pd_unfilter_kernel undoes the scanline filters: a warp per band of 32 rows, lane t one 4-pixel chunk behind lane
//      t - 1 (a skewed wavefront: the reconstructed pixels above arrive through shuffles); a band whose first row needs the
//      row above waits for the band before it (progress flags, 128 pixels at a time); rows filtered None / Sub need nothing.
//      An Adam7 image is seven small images in a row: a launch per non-empty pass, each with its own progress flags.
//   7. pd_bgr_kernel<colour type, bit depth, interlaced> writes the BGR staging image (what cv2.imread(path) with its default
//      flag IMREAD_COLOR returns: gray replicated, alpha dropped, the high byte of 16-bit samples, 1/2/4-bit gray scaled,
//      palette entries looked up), a gather that finds every pixel's Adam7 pass by its position; the usual pack kernel turns
//      it into the packed panorama.
//
// Everything that touches bits (bit reader, header parser, table builder, symbol decoder, block decoder, filters) is
// __host__ __device__ code shared with a serial host model of the same pipeline (p2p_png_decode_host, no GPU: CPU tests
// compare it with cv2.imdecode / zlib on every kind of file before the device sees one).
//
// Subset (parse_png, formats = 0, the default): 8-bit gray / RGB / gray + alpha / RGBA, not interlaced, no APNG, no PLTE, no
// tRNS, no eXIf.  formats = 1 (P2P_OPT_PNG_FORMATS): every colour type and bit depth of the PNG specification, Adam7 too,
// PLTE and tRNS where the specification allows them; still no APNG and no eXIf.  Anything else, any damaged file and any
// stream whose blocks are too long to be worth it (a single huge block, fixed-Huffman-only writers) is declined
// (P2P_ERR_UNSUPPORTED -> the caller uses cv2.imread as before).  The algorithms restated here are zlib's inflate
// (inflate.c / inftrees.c validity rules; RFC 1951), libpng's row filters (pngrutil.c png_read_filter_row; PNG
// specification section 9) and its read transformations png_do_read_interlace, png_do_unpack / png_do_expand,
// png_do_expand_palette and png_do_strip_16 (pngrutil.c, pngrtran.c; PNG specification sections 7, 8.2) - see THIRD_PARTY.md.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <thread>
#include <vector>

namespace p2ppdec {

#define PD_HD __host__ __device__ __forceinline__

constexpr int kLBits = 10;               // primary table of the literal / length code
constexpr int kDBits = 8;                // primary table of the distance code
constexpr uint32_t kMaxSyms = 1u << 20;  // symbols per deflate block a single decoder accepts (bounds its running time)
constexpr uint32_t kWindow = 32768;
enum { PD_OK = 0, PD_BAD = 1, PD_LONG = 2 };

struct Tables {                 // 3264 bytes: one per decoding warp in shared memory, on the stack in the host model
    uint16_t lt[1 << kLBits];   // next kLBits stream bits -> symbol << 4 | code length (0: longer code, or no such code)
    uint16_t dt[1 << kDBits];
    uint16_t lsym[288];         // symbols sorted by (code length, symbol): canonical order
    uint16_t dsym[32];
    uint16_t lcnt[16], dcnt[16];  // codes per length
};

// ---- bit reader: the zlib stream as little-endian 32-bit words (zero padded), LSB first -----------------------------
struct Bits {
    const uint32_t *w;
    uint64_t n_words, wi, buf;   // wi: words taken into buf so far (= index of the word waiting in nextw)
    uint32_t nextw;              // loaded one refill ahead, so that its latency is not on the decoder's dependency chain
    int cnt;
    PD_HD uint32_t word(uint64_t i) const { return i < n_words ? w[i] : 0u; }
    PD_HD void init(const uint32_t *words, uint64_t nw, uint64_t bit) {
        w = words;
        n_words = nw;
        wi = bit >> 5;
        const int sh = (int)(bit & 31);
        buf = (uint64_t)(word(wi) >> sh);
        wi++;
        cnt = 32 - sh;
        nextw = word(wi);
        refill();
    }
    PD_HD void refill() {  // afterwards 33 .. 64 valid bits
        if (cnt <= 32) {
            buf |= (uint64_t)nextw << cnt;
            wi++;
            cnt += 32;
            nextw = word(wi);
        }
    }
    PD_HD uint32_t peek(int n) const { return (uint32_t)(buf & ((1ull << n) - 1ull)); }
    PD_HD void drop(int n) {
        buf >>= n;
        cnt -= n;
    }
    PD_HD uint32_t get(int n) {
        const uint32_t v = peek(n);
        drop(n);
        return v;
    }
    PD_HD uint64_t pos() const { return wi * 32ull - (uint64_t)cnt; }
};

// 64 stream bits starting at `bit`
PD_HD uint64_t window64(const uint32_t *w, uint64_t nw, uint64_t bit) {
    const uint64_t i = bit >> 5;
    const int sh = (int)(bit & 31);
    const uint64_t w0 = i < nw ? w[i] : 0u, w1 = i + 1 < nw ? w[i + 1] : 0u, w2 = i + 2 < nw ? w[i + 2] : 0u;
    const uint64_t lo = w0 | (w1 << 32);
    return sh ? (lo >> sh) | (w2 << (64 - sh)) : lo;
}

// order in which the code-length code's lengths are stored (RFC 1951 3.2.7), 5 bits per entry
PD_HD int cl_order(int i) {
    // 16 17 18 0 8 7 9 6 10 5 11 4 | 12 3 13 2 14 1 15
    const uint64_t lo = 16ull | (17ull << 5) | (18ull << 10) | (0ull << 15) | (8ull << 20) | (7ull << 25) | (9ull << 30) |
                        (6ull << 35) | (10ull << 40) | (5ull << 45) | (11ull << 50) | (4ull << 55);
    const uint64_t hi = 12ull | (3ull << 5) | (13ull << 10) | (2ull << 15) | (14ull << 20) | (1ull << 25) | (15ull << 30);
    return i < 12 ? (int)((lo >> (5 * i)) & 31) : (int)((hi >> (5 * (i - 12))) & 31);
}

PD_HD int popc64(uint64_t v) {
#ifdef __CUDA_ARCH__
    return __popcll(v);
#else
    return __builtin_popcountll(v);
#endif
}

// the first test of a candidate block start: header fields and the Kraft sum of the code-length code (inflate.c: LENLENS
// builds it with type CODES, for which inftrees.c accepts complete codes only).  The up to 19 three-bit lengths are counted
// per value with bit planes and population counts instead of a loop: sum over the lengths l > 0 of 2^(7 - l) must be 128.
PD_HD bool quick_check(uint64_t head, uint64_t lens3) {
    if (((head >> 1) & 3) != 2) return false;
    if (((head >> 3) & 31) > 29 || ((head >> 8) & 31) > 29) return false;  // more than 286 / 30 codes
    const int ncode = (int)((head >> 13) & 15) + 4;
    const uint64_t R = 0x0249249249249249ull;                // bit 0 of each of the 19 fields
    const uint64_t m = lens3 & ((1ull << (3 * ncode)) - 1ull);
    const uint64_t b0 = m & R, b1 = (m >> 1) & R, b2 = (m >> 2) & R;
    const uint64_t n0 = b0 ^ R, n1 = b1 ^ R, n2 = b2 ^ R;
    const uint64_t lo = n2 & n1, l2 = n2 & b1, l4 = b2 & n1, l6 = b2 & b1;
    const int sum = 64 * popc64(lo & b0) + 32 * popc64(l2 & n0) + 16 * popc64(l2 & b0) + 8 * popc64(l4 & n0) + 4 * popc64(l4 & b0) +
                    2 * popc64(l6 & n0) + popc64(l6 & b0);
    return sum == 128;
}

// inftrees.c's test of a set of code lengths (type LENS / DISTS): over-subscribed sets are invalid, incomplete ones too
// unless the set is a single code of length 1; an empty set is accepted (every use of it is an error later)
PD_HD int check_lengths(const uint8_t *lens, int n, uint16_t *cnt) {
    for (int i = 0; i < 16; ++i) cnt[i] = 0;
    for (int s = 0; s < n; ++s) cnt[lens[s]]++;
    int max = 15;
    while (max >= 1 && cnt[max] == 0) --max;
    if (max == 0) return PD_OK;
    int left = 1;
    for (int len = 1; len <= 15; ++len) {
        left <<= 1;
        left -= cnt[len];
        if (left < 0) return PD_BAD;
    }
    if (left > 0 && max != 1) return PD_BAD;
    return PD_OK;
}

// Header of a dynamic block behind its three type bits: the code lengths of the literal / length code (lens[0 .. nlen)) and
// of the distance code (lens[nlen .. nlen + ndist)); every rule of inflate.c states TABLE .. CODELENS.  lens holds 320 bytes.
PD_HD int parse_dynamic_header(Bits &br, uint8_t *lens, int *nlen_out, int *ndist_out) {
    br.refill();
    const int nlen = (int)br.get(5) + 257, ndist = (int)br.get(5) + 1, ncode = (int)br.get(4) + 4;
    if (nlen > 286 || ndist > 30) return PD_BAD;
    uint8_t cl[19];
    for (int i = 0; i < 19; ++i) cl[i] = 0;
    for (int i = 0; i < ncode; ++i) {
        br.refill();
        cl[cl_order(i)] = (uint8_t)br.get(3);
    }
    // the code-length code: complete or invalid; canonical decode structures (count per length, symbols in order)
    uint8_t ccnt[8], csym[19];
    for (int i = 0; i < 8; ++i) ccnt[i] = 0;
    for (int s = 0; s < 19; ++s) ccnt[cl[s]]++;
    int left = 128;
    for (int l = 1; l <= 7; ++l) left -= (int)ccnt[l] * (128 >> l);
    if (left != 0) return PD_BAD;
    {
        uint8_t offs[8];
        offs[1] = 0;
        for (int l = 1; l < 7; ++l) offs[l + 1] = (uint8_t)(offs[l] + ccnt[l]);
        for (int s = 0; s < 19; ++s)
            if (cl[s]) csym[offs[cl[s]]++] = (uint8_t)s;
    }
    const int total = nlen + ndist;
    int i = 0;
    while (i < total) {
        br.refill();
        int code = 0, first = 0, index = 0, sym = -1;
        uint64_t b = br.buf;
        for (int l = 1; l <= 7; ++l) {
            code |= (int)(b & 1);
            b >>= 1;
            const int c = ccnt[l];
            if (code - c < first) {
                sym = csym[index + (code - first)];
                br.drop(l);
                break;
            }
            index += c;
            first += c;
            first <<= 1;
            code <<= 1;
        }
        if (sym < 0) return PD_BAD;
        if (sym < 16) {
            lens[i++] = (uint8_t)sym;
            continue;
        }
        int rep, val = 0;
        if (sym == 16) {
            if (i == 0) return PD_BAD;
            val = lens[i - 1];
            rep = 3 + (int)br.get(2);
        } else if (sym == 17) {
            rep = 3 + (int)br.get(3);
        } else {
            rep = 11 + (int)br.get(7);
        }
        if (i + rep > total) return PD_BAD;
        while (rep--) lens[i++] = (uint8_t)val;
    }
    if (lens[256] == 0) return PD_BAD;  // "invalid code -- missing end-of-block"
    *nlen_out = nlen;
    *ndist_out = ndist;
    return PD_OK;
}

// the full test of a candidate block start at `bit` (pd_full_kernel)
PD_HD bool full_check(const uint32_t *zs, uint64_t n_words, uint64_t bit) {
    Bits br;
    br.init(zs, n_words, bit);
    br.drop(3);
    uint8_t lens[320];
    uint16_t cnt[16];
    int nlen, ndist;
    if (parse_dynamic_header(br, lens, &nlen, &ndist)) return false;
    if (check_lengths(lens, nlen, cnt)) return false;
    if (check_lengths(lens + nlen, ndist, cnt)) return false;
    return true;
}

PD_HD uint32_t bit_reverse(uint32_t v, int n) {
    uint32_t r = 0;
    for (int i = 0; i < n; ++i) {
        r = (r << 1) | (v & 1);
        v >>= 1;
    }
    return r;
}

// decoding tables of one code from its lengths (validity as check_lengths)
PD_HD int build_code(const uint8_t *lens, int n, uint16_t *tab, int tbits, uint16_t *cnt, uint16_t *sym) {
    if (check_lengths(lens, n, cnt)) return PD_BAD;
    cnt[0] = 0;
    uint16_t offs[16];
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = (uint16_t)(offs[l] + cnt[l]);
    for (int s = 0; s < n; ++s)
        if (lens[s]) sym[offs[lens[s]]++] = (uint16_t)s;
    for (int i = 0; i < (1 << tbits); ++i) tab[i] = 0;
    uint32_t code = 0;
    int index = 0;
    for (int l = 1; l <= tbits; ++l) {
        for (int k = 0; k < (int)cnt[l]; ++k, ++code, ++index) {
            const uint16_t e = (uint16_t)((sym[index] << 4) | l);
            for (uint32_t i = bit_reverse(code, l); i < (1u << tbits); i += 1u << l) tab[i] = e;
        }
        code <<= 1;
    }
    return PD_OK;
}

// next symbol of a code: primary table, else the canonical bit-serial walk (codes longer than the table, rare); -1 = no
// such code (inflate's "invalid literal/length code" / "invalid distance code").  Needs 15 valid bits.
PD_HD int decode_sym(Bits &br, const uint16_t *tab, int tbits, const uint16_t *cnt, const uint16_t *sym) {
    const uint32_t e = tab[br.peek(tbits)];
    if (e & 15) {
        br.drop((int)(e & 15));
        return (int)(e >> 4);
    }
    int code = 0, first = 0, index = 0;
    uint64_t b = br.buf;
    for (int l = 1; l <= 15; ++l) {
        code |= (int)(b & 1);
        b >>= 1;
        const int c = cnt[l];
        if (code - c < first) {
            br.drop(l);
            return sym[index + (code - first)];
        }
        index += c;
        first += c;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}

struct BlockOut {
    uint64_t end_bit;
    uint32_t out_len;
    int final_block;
    uint32_t tail_marks;  // WRITE: history marks left in the block's last 32 KiB (0: the tail pass has nothing to do here)
    uint32_t n_matches;   // back-references in the block
};

// Header of the block br stands on: its three type bits, then either the length of a stored block (type 0: *stored_len
// bytes starting at byte *stored_byte0 of the stream) or the decoding tables (fixed or dynamic codes).
PD_HD int block_begin(Bits &br, uint64_t stream_bits, Tables &T, uint8_t *lens, int *final_block, int *type_out, uint32_t *stored_len,
                      uint64_t *stored_byte0) {
    *final_block = (int)br.get(1);
    const int type = (int)br.get(2);
    *type_out = type;
    if (type == 3) return PD_BAD;
    if (type == 0) {
        br.drop((int)((0 - br.pos()) & 7));
        br.refill();
        const uint32_t len = br.get(16);
        br.refill();
        const uint32_t nlen = br.get(16);
        if ((len ^ 0xFFFFu) != nlen) return PD_BAD;
        const uint64_t byte0 = br.pos() >> 3;
        if ((byte0 + len) * 8 > stream_bits) return PD_BAD;
        *stored_len = len;
        *stored_byte0 = byte0;
        return PD_OK;
    }
    int nlen = 288, ndist = 32;
    if (type == 1) {
        for (int s = 0; s < 144; ++s) lens[s] = 8;
        for (int s = 144; s < 256; ++s) lens[s] = 9;
        for (int s = 256; s < 280; ++s) lens[s] = 7;
        for (int s = 280; s < 288; ++s) lens[s] = 8;
        for (int s = 0; s < 32; ++s) lens[288 + s] = 5;
    } else {
        if (parse_dynamic_header(br, lens, &nlen, &ndist)) return PD_BAD;
    }
    if (build_code(lens, nlen, T.lt, kLBits, T.lcnt, T.lsym)) return PD_BAD;
    if (build_code(lens + nlen, ndist, T.dt, kDBits, T.dcnt, T.dsym)) return PD_BAD;
    return PD_OK;
}

// Next token of a Huffman-coded block: 0 = literal (*len = the byte), 1 = match (*len, *dist), 2 = end of block,
// -1 = a code or symbol inflate rejects
PD_HD int next_token(Bits &br, const Tables &T, uint32_t *len, uint32_t *dist) {
    br.refill();
    const int s = decode_sym(br, T.lt, kLBits, T.lcnt, T.lsym);
    if (s < 0) return -1;
    if (s < 256) {
        *len = (uint32_t)s;
        return 0;
    }
    if (s == 256) return 2;
    if (s > 285) return -1;
    const int idx = s - 257;
    if (idx < 8) *len = 3 + idx;
    else if (idx == 28) *len = 258;
    else {
        const int e = (idx >> 2) - 1;
        *len = 3 + ((4 + (idx & 3)) << e) + br.get(e);
    }
    br.refill();
    const int d = decode_sym(br, T.dt, kDBits, T.dcnt, T.dsym);
    if (d < 0 || d > 29) return -1;
    if (d < 4) *dist = 1 + d;
    else {
        const int e = (d >> 1) - 1;
        *dist = 1 + ((2 + (d & 1)) << e) + br.get(e);
    }
    return 1;
}

// One deflate block starting at start_bit.  WRITE = false: only measured (where it ends, how many bytes it produces).
// WRITE = true: bytes go to raw[out_off ..], and ref[] (all zeros before the pass) receives for every byte that is not
// known yet k = 1 .. 32768: it equals the byte k positions in front of this block's first byte.  out_cap: size of the whole
// inflated image; wsize: window of the zlib header.  Distances beyond the data produced so far are invalid ("invalid
// distance too far back").  expect_len (WRITE): the length the block was measured with, which says where its last 32 KiB begin.
template <bool WRITE>
PD_HD int decode_block(const uint32_t *zs, uint64_t n_words, uint64_t stream_bits, uint64_t start_bit, Tables &T,
                       uint8_t *lens, uint8_t *raw, uint16_t *ref, uint64_t out_off, uint64_t out_cap, uint32_t wsize,
                       BlockOut &R, uint32_t expect_len = 0) {
    const uint64_t tail_from = expect_len > kWindow ? expect_len - kWindow : 0;
    uint32_t marks = 0, n_matches = 0;
    R.tail_marks = 0;
    R.n_matches = 0;
    Bits br;
    br.init(zs, n_words, start_bit);
    int type;
    uint32_t slen = 0;
    uint64_t byte0 = 0;
    if (block_begin(br, stream_bits, T, lens, &R.final_block, &type, &slen, &byte0)) return PD_BAD;
    uint64_t o = 0;  // bytes produced by this block
    if (type == 0) {
        if (WRITE) {
            if (out_off + slen > out_cap) return PD_BAD;
            const uint8_t *src = reinterpret_cast<const uint8_t *>(zs) + byte0;
            for (uint32_t i = 0; i < slen; ++i) raw[out_off + i] = src[i];
        }
        R.end_bit = (byte0 + slen) * 8;
        R.out_len = slen;
        return PD_OK;
    }
    const uint64_t room = out_cap > out_off ? out_cap - out_off : 0;
    for (uint32_t n = 0;; ++n) {
        if (n >= kMaxSyms) return PD_LONG;
        uint32_t len = 0, dist = 0;
        const int k = next_token(br, T, &len, &dist);
        if (k < 0) return PD_BAD;
        if (k == 0) {
            if (o >= room) return PD_BAD;
            if (WRITE) raw[out_off + o] = (uint8_t)len;
            ++o;
            continue;
        }
        if (k == 2) break;
        ++n_matches;
        if (dist > wsize) return PD_BAD;
        if (o + len > room) return PD_BAD;
        if (WRITE) {
            if (dist > out_off + o) return PD_BAD;  // in front of the first byte of the image
            const uint64_t at = out_off + o;
            for (uint32_t i = 0; i < len; ++i) {
                const int64_t src = (int64_t)(o + i) - (int64_t)dist;  // relative to the block's first byte
                uint16_t r;
                if (src < 0) {
                    r = (uint16_t)(-src);
                } else {
                    raw[at + i] = raw[out_off + src];
                    r = ref[out_off + src];
                }
                if (r) {
                    ref[at + i] = r;
                    marks += (o + i >= tail_from);
                }
            }
        }
        o += len;
    }
    R.end_bit = br.pos();
    if (R.end_bit > stream_bits) return PD_BAD;
    R.out_len = (uint32_t)o;
    R.tail_marks = marks;
    R.n_matches = n_matches;
    return PD_OK;
}

// ---- scanline filters (PNG specification 9.2; libpng png_read_filter_row) -------------------------------------------
// reconstructed byte from the filtered byte f, filter type ft and the reconstructed neighbours a (left), b (above),
// c (above left)
// (m1 .. m4: all-ones for the row's filter type 1 .. 4, else zero - every predictor is evaluated and masked, so that the
// lanes of a warp, whose rows have different filters, run one instruction stream without branches)
PD_HD uint32_t unfilter_byte_masked(uint32_t f, uint32_t a, uint32_t b, uint32_t c, uint32_t m1, uint32_t m2, uint32_t m3, uint32_t m4) {
    const int da = (int)b - (int)c, db = (int)a - (int)c, dc = da + db;
    const int pa = da < 0 ? -da : da, pb = db < 0 ? -db : db, pc = dc < 0 ? -dc : dc;
    const uint32_t bc = (pb <= pc) ? b : c;
    const uint32_t paeth = ((pa <= pb) & (pa <= pc)) ? a : bc;
    const uint32_t pred = (a & m1) | (b & m2) | (((a + b) >> 1) & m3) | (paeth & m4);
    return (f + pred) & 255u;
}
PD_HD uint32_t unfilter_byte(uint32_t ft, uint32_t f, uint32_t a, uint32_t b, uint32_t c) {
    return unfilter_byte_masked(f, a, b, c, ft == 1 ? ~0u : 0u, ft == 2 ? ~0u : 0u, ft == 3 ? ~0u : 0u, ft >= 4 ? ~0u : 0u);
}

// ---- reconstructed rows -> BGR -------------------------------------------------------------------------------------
// Adam7 (PNG specification 8.2): pass p holds the pixels (x0 + dx i, y0 + dy j), dx = 1 << a7_sx(p), dy = 1 << a7_sy(p)
// (one nibble per pass, pass 0 lowest)
PD_HD int a7_x0(int p) { return (0x0102040 >> (4 * p)) & 15; }
PD_HD int a7_y0(int p) { return (0x1020400 >> (4 * p)) & 15; }
PD_HD int a7_sx(int p) { return (0x0112233 >> (4 * p)) & 15; }
PD_HD int a7_sy(int p) { return (0x1122333 >> (4 * p)) & 15; }
PD_HD int adam7_pass(int x, int y) {
    return (y & 1) ? 6 : (x & 1) ? 5 : (y & 2) ? 4 : (x & 2) ? 3 : (y & 4) ? 2 : (x & 4) ? 1 : 0;
}

// where the conversion finds the reconstructed rows: per pass (one when not interlaced) the offset of its first row and the
// row stride; and the palette (PLTE, RGB triples)
struct Fmt {
    int W, n_plte;
    uint64_t off[7];
    uint32_t stride[7];
    uint8_t plte[768];
};

// the colour type / bit depth pairs the decoder handles (X(colour type, bit depth)); the first four are the default subset
#define PD_FORMATS(X) X(0, 8) X(2, 8) X(4, 8) X(6, 8) X(0, 1) X(0, 2) X(0, 4) X(0, 16) X(2, 16) X(3, 1) X(3, 2) X(3, 4) X(3, 8) \
    X(4, 16) X(6, 16)

// BGR triple of image pixel (x, y), what cv2.imread(path) with flag IMREAD_COLOR returns: gray replicated, alpha dropped,
// 16-bit samples cut to their high byte (libpng png_do_strip_16), 1/2/4-bit gray scaled to 8 bits and sub-byte samples
// unpacked MSB first (png_do_unpack / png_do_expand), palette indices looked up (png_do_expand_palette), the Adam7 pass
// found by position (png_do_read_interlace, as a gather).  false: a palette index without a PLTE entry (bgr = black).
template <int CT, int DEPTH>
PD_HD bool pixel_bgr(const Fmt &F, const uint8_t *recon, bool lace, int x, int y, uint8_t *bgr) {
    int p = 0;
    if (lace) {
        p = adam7_pass(x, y);
        x >>= a7_sx(p);
        y >>= a7_sy(p);
    }
    const uint8_t *row = recon + F.off[p] + (size_t)y * F.stride[p];
    constexpr int CH = CT == 2 ? 3 : CT == 4 ? 2 : CT == 6 ? 4 : 1;
    uint32_t v;
    if (DEPTH < 8) {
        const int bit = x * DEPTH;
        v = ((uint32_t)row[bit >> 3] >> (8 - DEPTH - (bit & 7))) & ((1u << DEPTH) - 1u);
        if (CT == 0) v *= 255u / ((1u << DEPTH) - 1u);
    } else {
        constexpr int SB = DEPTH / 8;   // bytes per sample, the most significant first
        const uint8_t *s = row + (size_t)x * (CH * SB);
        if (CH >= 3) {
            bgr[0] = s[2 * SB];
            bgr[1] = s[SB];
            bgr[2] = s[0];
            return true;
        }
        v = s[0];
    }
    if (CT == 3) {
        if ((int)v >= F.n_plte) {
            bgr[0] = bgr[1] = bgr[2] = 0;
            return false;
        }
        bgr[0] = F.plte[3 * v + 2];
        bgr[1] = F.plte[3 * v + 1];
        bgr[2] = F.plte[3 * v];
        return true;
    }
    bgr[0] = bgr[1] = bgr[2] = (uint8_t)v;
    return true;
}

// One mark of a block's last 32 KiB during the walk through its group (block start bo, group start gs): the history byte
// sits at abs = bo - mark.  Inside the group it has been walked already: final -> copy it; itself re-based -> inherit its
// mark.  In front of the group -> re-base the mark to the group start (still <= 32768: abs >= gs - 32768 because bo >= gs).
PD_HD void tail_step(uint8_t *raw, uint16_t *ref, uint64_t p, uint64_t bo, uint64_t gs) {
    const uint64_t abs = bo - ref[p];
    if (abs >= gs) {
        const uint16_t rt = ref[abs];
        if (rt == 0) raw[p] = raw[abs];
        ref[p] = rt;
    } else {
        ref[p] = (uint16_t)(gs - abs);
    }
}

// ---- CRC-32 (PNG chunk checksums) ----------------------------------------------------------------------------------
// multiplication of two polynomials mod the CRC-32 polynomial, reflected representation (zlib crc32.c multmodp)
inline uint32_t crc_mulmod(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}
// x^(8 n) mod the polynomial
inline uint32_t crc_xpow8n(uint64_t n) {
    uint32_t p = 1u << 31, sq = 1u << 30;  // x^0, x^1
    for (int k = 0; k < 3; ++k) sq = crc_mulmod(sq, sq);  // x^8
    while (n) {
        if (n & 1) p = crc_mulmod(sq, p);
        sq = crc_mulmod(sq, sq);
        n >>= 1;
    }
    return p;
}
// CRC of A || B from the CRCs of A and B (zlib crc32_combine)
inline uint32_t crc_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b) { return crc_mulmod(crc_xpow8n(len_b), crc_a) ^ crc_b; }

inline const uint32_t *crc_table_host() {
    static uint32_t t[256];
    static bool init = false;
    if (!init) {
        for (uint32_t n = 0; n < 256; ++n) {
            uint32_t c = n;
            for (int k = 0; k < 8; ++k) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
            t[n] = c;
        }
        init = true;
    }
    return t;
}
inline uint32_t crc32_host(const uint8_t *p, size_t n, uint32_t crc = 0) {
    const uint32_t *t = crc_table_host();
    crc = ~crc;
    for (size_t i = 0; i < n; ++i) crc = t[(crc ^ p[i]) & 255] ^ (crc >> 8);
    return ~crc;
}

// ---- file structure (host) ---------------------------------------------------------------------------------------
struct Idat {
    size_t file_off;    // of the chunk's data
    uint32_t len;
    size_t stream_off;  // of that data in the concatenated zlib stream
    uint32_t crc;       // stored CRC (over type + data)
};
// a pass of an Adam7 image (a non-interlaced image is one pass: the whole image).  Its rows (filter byte + row_bytes bytes
// each) start at raw_off of the inflated image; an empty pass (w or h = 0) has no rows at all.
struct Pass {
    uint32_t x0, y0, dx, dy, w, h;
    size_t row_bytes, raw_off;
};
struct Info {
    int W = 0, H = 0, color_type = 0, bpp = 0;  // bpp: the filters' byte distance, max(1, bits per pixel / 8)
    int depth = 8, interlace = 0;  // bits per sample; 1 = Adam7
    size_t row_bytes = 0;  // ceil(W * bits per pixel / 8)
    size_t raw_bytes = 0;  // sum over the passes of h * (1 + row_bytes): the inflated image
    int n_pass = 1;
    Pass pass[7] = {};
    int n_plte = 0;        // palette entries (colour type 3)
    uint8_t plte[768] = {};
    uint32_t wsize = 0;    // window of the zlib header
    size_t stream_len = 0; // bytes of the concatenated zlib stream (header and Adler-32 included)
    uint32_t adler = 0;    // stored Adler-32 (read once the end of the deflate data is known)
};
struct Parsed {
    Info info;
    std::vector<Idat> idat;
};

inline uint32_t be32(const uint8_t *p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }

// the passes of the image and the size of the inflated data (W, H, depth, interlace and bits per pixel set)
inline void layout_passes(Info &I, int bits) {
    I.row_bytes = ((size_t)I.W * bits + 7) / 8;
    I.n_pass = I.interlace ? 7 : 1;
    size_t off = 0;
    for (int p = 0; p < I.n_pass; ++p) {
        Pass &q = I.pass[p];
        q.x0 = I.interlace ? a7_x0(p) : 0;
        q.y0 = I.interlace ? a7_y0(p) : 0;
        q.dx = I.interlace ? 1u << a7_sx(p) : 1;
        q.dy = I.interlace ? 1u << a7_sy(p) : 1;
        q.w = (uint32_t)I.W > q.x0 ? ((uint32_t)I.W - q.x0 + q.dx - 1) / q.dx : 0;
        q.h = (uint32_t)I.H > q.y0 ? ((uint32_t)I.H - q.y0 + q.dy - 1) / q.dy : 0;
        if (!q.w) q.h = 0;
        q.row_bytes = ((size_t)q.w * bits + 7) / 8;
        q.raw_off = off;
        off += (size_t)q.h * (1 + q.row_bytes);
    }
    I.raw_bytes = off;
}

// Chunk walk.  0 = inside the subset, 1 = decline.  Checks the CRC of every chunk except IDAT (those are checked on the
// device, or by the host model) - a file libpng rejects or merely warns about is declined.
// formats = 0: 8-bit gray / RGB / gray + alpha / RGBA, not interlaced, no PLTE, no tRNS.  formats = 1: every colour type
// and bit depth of the PNG specification (11.2.2), Adam7 too; PLTE and tRNS where the specification puts them (a tRNS
// key is ignored and the palette's alpha dropped, as cv2.imread's IMREAD_COLOR does), no tRNS on types with alpha.
inline int parse_png(const uint8_t *f, size_t len, Parsed &P, int formats = 0) {
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
    if (len < 8 + 25 + 12 || memcmp(f, sig, 8) != 0) return 1;
    size_t at = 8;
    bool seen_ihdr = false, seen_idat = false, idat_closed = false, seen_iend = false, seen_plte = false, seen_trns = false;
    Info &I = P.info;
    P.idat.clear();
    size_t stream_off = 0;
    while (at + 12 <= len) {
        const uint32_t clen = be32(f + at);
        if (clen > 0x7FFFFFFFu || (size_t)clen + 12 > len - at) return 1;
        const uint8_t *type = f + at + 4, *data = f + at + 8;
        const uint32_t stored = be32(data + clen);
        const bool is_idat = memcmp(type, "IDAT", 4) == 0;
        if (!is_idat && crc32_host(type, (size_t)clen + 4) != stored) return 1;
        if (!seen_ihdr) {
            if (memcmp(type, "IHDR", 4) != 0 || clen != 13) return 1;
            const uint32_t W = be32(data), H = be32(data + 4);
            if (W == 0 || H == 0 || W > 0x7FFFFFFFu || H > 0x7FFFFFFFu) return 1;
            I.color_type = data[9];
            int bits;
            if (!formats) {
                if (data[8] != 8 || data[10] != 0 || data[11] != 0 || data[12] != 0) return 1;  // 8 bit, deflate, adaptive, not interlaced
                I.bpp = I.color_type == 0 ? 1 : I.color_type == 2 ? 3 : I.color_type == 4 ? 2 : I.color_type == 6 ? 4 : 0;
                if (!I.bpp) return 1;  // palette images stay with cv2
                bits = 8 * I.bpp;
            } else {
                const int d = data[8], ct = I.color_type;
                if (data[10] != 0 || data[11] != 0 || data[12] > 1) return 1;   // deflate, adaptive filters, none / Adam7
                const bool ok = ct == 0 ? (d == 1 || d == 2 || d == 4 || d == 8 || d == 16)
                                : ct == 3 ? (d == 1 || d == 2 || d == 4 || d == 8)
                                : (ct == 2 || ct == 4 || ct == 6) && (d == 8 || d == 16);
                if (!ok) return 1;
                I.depth = d;
                I.interlace = data[12];
                bits = d * (ct == 2 ? 3 : ct == 4 ? 2 : ct == 6 ? 4 : 1);
                I.bpp = bits < 8 ? 1 : bits / 8;
            }
            if (W >= 32767 || H >= 32767) return 1;
            I.W = (int)W;
            I.H = (int)H;
            layout_passes(I, bits);
            seen_ihdr = true;
        } else if (is_idat) {
            if (idat_closed) return 1;  // IDAT chunks must be consecutive
            if (I.color_type == 3 && !seen_plte) return 1;
            seen_idat = true;
            if (clen) P.idat.push_back(Idat{at + 8, clen, stream_off, stored});
            else if (crc32_host(type, 4) != stored) return 1;
            stream_off += clen;
        } else {
            if (seen_idat) idat_closed = true;
            if (memcmp(type, "IEND", 4) == 0) {
                if (clen != 0 || !seen_idat) return 1;
                seen_iend = true;
                break;
            }
            if (memcmp(type, "IHDR", 4) == 0) return 1;
            const int ct = I.color_type;
            if (formats && memcmp(type, "PLTE", 4) == 0) {   // one, in front of IDAT; the palette of type 3, a suggestion for 2 / 6
                if (ct == 0 || ct == 4 || seen_plte || seen_idat || clen == 0 || clen % 3 || clen > 768) return 1;
                if (ct == 3 && (int)(clen / 3) > (1 << I.depth)) return 1;
                if (ct == 3) {
                    I.n_plte = (int)(clen / 3);
                    memcpy(I.plte, data, clen);
                }
                seen_plte = true;
                at += (size_t)clen + 12;
                continue;
            }
            if (formats && memcmp(type, "tRNS", 4) == 0) {   // one, in front of IDAT; read by nothing here (IMREAD_COLOR)
                if (seen_trns || seen_idat) return 1;
                const uint32_t lim = I.depth == 16 ? 0xFFFFu : (1u << I.depth) - 1u;
                if (ct == 0) {
                    if (clen != 2 || ((uint32_t)data[0] << 8 | data[1]) > lim) return 1;
                } else if (ct == 2) {
                    if (clen != 6) return 1;
                    for (int k = 0; k < 3; ++k)
                        if (((uint32_t)data[2 * k] << 8 | data[2 * k + 1]) > lim) return 1;
                } else if (ct == 3) {
                    if (!seen_plte || clen == 0 || (int)clen > I.n_plte) return 1;
                } else {
                    return 1;   // types with an alpha channel have no tRNS
                }
                seen_trns = true;
                at += (size_t)clen + 12;
                continue;
            }
            // animation, transparency key, EXIF block, and every critical chunk (PLTE, a suggested palette, included): decline
            if (memcmp(type, "acTL", 4) == 0 || memcmp(type, "fcTL", 4) == 0 || memcmp(type, "fdAT", 4) == 0 ||
                memcmp(type, "tRNS", 4) == 0 || memcmp(type, "eXIf", 4) == 0)  // (cv2.imread rotates by the EXIF orientation)
                return 1;
            if (!(type[0] & 0x20)) return 1;  // critical chunk (PLTE included unless formats = 1)
            for (int k = 0; k < 4; ++k)
                if (!((type[k] >= 'A' && type[k] <= 'Z') || (type[k] >= 'a' && type[k] <= 'z'))) return 1;
        }
        at += (size_t)clen + 12;
    }
    if (!seen_iend || P.idat.empty()) return 1;
    I.stream_len = stream_off;
    if (stream_off < 2 + 1 + 4) return 1;
    // zlib header (may straddle chunks: read through the chunk table)
    uint8_t h[2];
    size_t k = 0;
    for (const Idat &c : P.idat) {
        for (uint32_t i = 0; i < c.len && k < 2; ++i) h[k++] = f[c.file_off + i];
        if (k == 2) break;
    }
    if ((h[0] & 15) != 8 || (h[0] >> 4) > 7 || ((h[0] << 8) | h[1]) % 31 != 0 || (h[1] & 0x20)) return 1;
    I.wsize = 1u << ((h[0] >> 4) + 8);
    return 0;
}

// the concatenated zlib stream, zero padded to whole words plus slack (dst holds stream_words(P) * 4 bytes)
inline size_t stream_words(const Parsed &P) { return (P.info.stream_len + 3) / 4 + 8; }
inline void gather_stream(const uint8_t *f, const Parsed &P, uint8_t *dst) {
    const size_t n = P.idat.size(), total = P.info.stream_len;
    const unsigned parts = total >= (8u << 20) ? 4u : 1u;   // a large file is copied by four threads (chunk ranges of equal size)
    if (parts == 1) {
        for (const Idat &c : P.idat) memcpy(dst + c.stream_off, f + c.file_off, c.len);
    } else {
        std::vector<std::thread> th;
        size_t i0 = 0;
        for (unsigned k = 0; k < parts; ++k) {
            size_t i1 = i0;
            const size_t until = total / parts * (k + 1);
            while (i1 < n && (k + 1 == parts || P.idat[i1].stream_off < until)) ++i1;
            th.emplace_back([&P, f, dst, i0, i1] {
                for (size_t i = i0; i < i1; ++i) memcpy(dst + P.idat[i].stream_off, f + P.idat[i].file_off, P.idat[i].len);
            });
            i0 = i1;
        }
        for (std::thread &t : th) t.join();
    }
    memset(dst + P.info.stream_len, 0, stream_words(P) * 4 - P.info.stream_len);
}

// a measured candidate / a block of the chain
struct Cand {
    uint64_t bit, end_bit;
    uint32_t out_len;
    int32_t status;  // PD_OK | final << 8, or PD_BAD / PD_LONG
    uint32_t n_matches, pad;
};
struct Block {
    uint64_t bit, out_off;
    uint32_t out_len;
    uint32_t tail_marks;  // written by the copy pass
    uint64_t match_off;   // first record of the block in the match list
    uint32_t n_matches, pad;
};
struct Match {            // a back-reference of a block: `len` bytes at offset `o` of the block's output repeat what lies `dist` bytes before
    uint32_t o;
    uint16_t len, dist;
};

// Chain walk (host): from the first block behind the zlib header, through measured candidates where there are any and
// measuring the other blocks (stored, fixed, or dynamic ones the search was not given) with the block decoder itself.
// host_budget bounds the bits the host decodes that way, max_blocks the length of the chain.  0 = ok (blocks filled, *end_bit = end of the deflate data).
// *host_dynamic (optional) grows by the dynamic-Huffman blocks the walk measured itself: blocks the search should have found.
inline int walk_chain(const uint32_t *zs, const Parsed &P, std::vector<Cand> &cands, std::vector<Block> &blocks,
                      uint64_t host_budget, uint64_t *end_bit, size_t max_blocks = (size_t)1 << 24, uint64_t *host_dynamic = nullptr) {
    const Info &I = P.info;
    const uint64_t n_words = stream_words(P), stream_bits = (uint64_t)(I.stream_len - 4) * 8;  // the Adler-32 is not deflate data
    std::sort(cands.begin(), cands.end(), [](const Cand &a, const Cand &b) { return a.bit < b.bit; });
    blocks.clear();
    uint64_t bit = 16, out = 0, spent = 0, n_match_total = 0;
    Tables T;
    uint8_t lens[320];
    for (;;) {
        if (bit + 3 > stream_bits) return 1;
        auto it = std::lower_bound(cands.begin(), cands.end(), bit, [](const Cand &c, uint64_t b) { return c.bit < b; });
        uint64_t end;
        uint32_t out_len, n_matches;
        int fin;
        if (it != cands.end() && it->bit == bit) {
            if ((it->status & 255) != PD_OK) return 1;
            end = it->end_bit;
            out_len = it->out_len;
            n_matches = it->n_matches;
            fin = it->status >> 8;
        } else {
            BlockOut R;
            const uint64_t btype = (window64(zs, n_words, bit) >> 1) & 3;
            const bool stored = btype == 0;   // (a stored block costs nothing to measure)
            if (!stored && spent > host_budget) return 1;
            if (btype == 2 && host_dynamic) ++*host_dynamic;
            if (decode_block<false>(zs, n_words, stream_bits, bit, T, lens, nullptr, nullptr, 0, I.raw_bytes, I.wsize, R)) return 1;
            if (!stored) spent += R.end_bit - bit;
            end = R.end_bit;
            out_len = R.out_len;
            n_matches = R.n_matches;
            fin = R.final_block;
        }
        if (end > stream_bits || out + out_len > I.raw_bytes) return 1;
        if (blocks.size() >= max_blocks) return 1;   // (a stream of millions of empty blocks)
        blocks.push_back(Block{bit, out, out_len, 0, n_match_total, n_matches, 0});
        n_match_total += n_matches;
        out += out_len;
        bit = end;
        if (fin) break;
    }
    if (out != I.raw_bytes) return 1;                         // libpng: "Not enough image data" / "Too much image data"
    if (((bit + 7) >> 3) + 4 != I.stream_len) return 1;      // the Adler-32 follows on the next byte boundary and ends the stream
    *end_bit = bit;
    return 0;
}

// blocks per group of the tail pass: ~sqrt(n), so that the serial walk inside a group and the serial walk over the groups
// are equally long
inline uint32_t group_size(uint32_t n_blocks) {
    uint32_t m = 1;
    while ((uint64_t)m * m < n_blocks) ++m;
    return m;
}

// ---- serial host model of the whole decoder (tests; the product path runs the kernels below) ------------------------
// quick -> full -> measure -> walk -> symbolic decode -> tails -> resolve -> Adler / CRC -> unfilter -> BGR, the same
// routines in the same order, one "thread" after the other.  bgr: H rows of row_stride bytes.  0 = ok, 1 = declined.
// stats (optional, 4 values): positions passing the quick test, candidates, blocks of the chain, blocks measured on the host.
// formats: as parse_png.
inline int decode_host_model(const uint8_t *f, size_t len, uint8_t *bgr, size_t row_stride, uint64_t *stats, int formats = 0) {
    Parsed P;
    if (parse_png(f, len, P, formats)) return 1;
    const Info &I = P.info;
    for (const Idat &c : P.idat) {
        uint32_t crc = crc32_host(reinterpret_cast<const uint8_t *>("IDAT"), 4);
        crc = crc32_host(f + c.file_off, c.len, crc);
        if (crc != c.crc) return 1;
    }
    const uint64_t n_words = stream_words(P);
    std::vector<uint32_t> zsv(n_words);
    gather_stream(f, P, reinterpret_cast<uint8_t *>(zsv.data()));
    const uint32_t *zs = zsv.data();
    const uint64_t stream_bits = (uint64_t)(I.stream_len - 4) * 8;
    std::vector<Cand> cands;
    uint64_t n_quick = 0;
    for (uint64_t bit = 16; bit + 3 <= stream_bits; ++bit) {
        if (!quick_check(window64(zs, n_words, bit), window64(zs, n_words, bit + 17))) continue;
        ++n_quick;
        if (full_check(zs, n_words, bit)) cands.push_back(Cand{bit, 0, 0, 0, 0, 0});
    }
    Tables T;
    uint8_t lens[320];
    for (Cand &c : cands) {
        BlockOut R{0, 0, 0, 0, 0};
        const int rc = decode_block<false>(zs, n_words, stream_bits, c.bit, T, lens, nullptr, nullptr, 0, I.raw_bytes, I.wsize, R);
        c.end_bit = R.end_bit;
        c.out_len = R.out_len;
        c.n_matches = R.n_matches;
        c.status = rc ? rc : (R.final_block << 8);
    }
    std::vector<Block> blocks;
    uint64_t end_bit = 0;
    if (walk_chain(zs, P, cands, blocks, ~0ull, &end_bit)) return 1;
    if (stats) {
        stats[0] = n_quick;
        stats[1] = cands.size();
        stats[2] = blocks.size();
        uint64_t on_host = 0;
        for (const Block &b : blocks) {
            auto it = std::lower_bound(cands.begin(), cands.end(), b.bit, [](const Cand &c, uint64_t x) { return c.bit < x; });
            if (it == cands.end() || it->bit != b.bit) ++on_host;
        }
        stats[3] = on_host;
    }
    std::vector<uint8_t> raw(I.raw_bytes);
    std::vector<uint16_t> ref(I.raw_bytes);
    for (Block &b : blocks) {
        BlockOut R;
        if (decode_block<true>(zs, n_words, stream_bits, b.bit, T, lens, raw.data(), ref.data(), b.out_off, I.raw_bytes, I.wsize, R, b.out_len))
            return 1;
        if (R.out_len != b.out_len) return 1;
        b.tail_marks = R.tail_marks;
    }
    // tails: groups of consecutive blocks (re-base to the group start), the chain over the groups, the re-based marks
    const uint32_t nb = (uint32_t)blocks.size(), per = group_size(nb), ng = (nb + per - 1) / per;
    for (uint32_t g = 0; g < ng; ++g) {
        const uint64_t gs = blocks[(size_t)g * per].out_off;
        for (uint32_t i = g * per; i < std::min(nb, (g + 1) * per); ++i) {
            const Block &b = blocks[i];
            if (!b.tail_marks) continue;
            const uint64_t end = b.out_off + b.out_len, t0 = b.out_len > kWindow ? end - kWindow : b.out_off;
            for (uint64_t p = t0; p < end; ++p)
                if (ref[p]) tail_step(raw.data(), ref.data(), p, b.out_off, gs);
        }
    }
    for (uint32_t g = 1; g + 1 < ng; ++g) {
        const uint64_t gs = blocks[(size_t)g * per].out_off, next = blocks[(size_t)(g + 1) * per].out_off;
        for (uint64_t p = std::max(gs, next > kWindow ? next - kWindow : 0); p < next; ++p)
            if (ref[p]) {
                raw[p] = raw[gs - ref[p]];
                ref[p] = 0;
            }
    }
    for (uint32_t i = per; i < nb; ++i) {
        const Block &b = blocks[i];
        if (!b.tail_marks) continue;
        const uint64_t gs = blocks[(size_t)(i / per) * per].out_off;
        const uint64_t end = b.out_off + b.out_len, t0 = b.out_len > kWindow ? end - kWindow : b.out_off;
        for (uint64_t p = t0; p < end; ++p)
            if (ref[p]) {
                raw[p] = raw[gs - ref[p]];
                ref[p] = 0;
            }
    }
    for (const Block &b : blocks)   // everything else, any order
        for (uint64_t p = b.out_off; p < b.out_off + b.out_len; ++p)
            if (ref[p]) raw[p] = raw[b.out_off - ref[p]];
    {
        uint32_t s1 = 1, s2 = 0;
        for (size_t i = 0; i < raw.size(); ++i) {
            s1 += raw[i];
            if (s1 >= 65521) s1 -= 65521;
            s2 += s1;
            if (s2 >= 65521) s2 -= 65521;
        }
        const uint8_t *tail = reinterpret_cast<const uint8_t *>(zs) + I.stream_len - 4;
        if (((s2 << 16) | s1) != be32(tail)) return 1;
    }
    Fmt F{I.W, I.n_plte, {}, {}, {}};
    memcpy(F.plte, I.plte, sizeof(F.plte));
    for (int p = 0; p < I.n_pass; ++p) {   // every pass filtered on its own, its first row without a row above
        const Pass &q = I.pass[p];
        const size_t stride = 1 + q.row_bytes;
        F.off[p] = q.raw_off + 1;
        F.stride[p] = (uint32_t)stride;
        for (uint32_t y = 0; y < q.h; ++y) {
            uint8_t *row = raw.data() + q.raw_off + (size_t)y * stride;
            const uint8_t *up = y ? row - stride : nullptr;
            const uint32_t ft = row[0];
            if (ft > 4) return 1;
            for (size_t i = 0; i < q.row_bytes; ++i) {
                const uint32_t a = i >= (size_t)I.bpp ? row[1 + i - I.bpp] : 0, b = up ? up[1 + i] : 0,
                               c = (up && i >= (size_t)I.bpp) ? up[1 + i - I.bpp] : 0;
                row[1 + i] = (uint8_t)unfilter_byte(ft, row[1 + i], a, b, c);
            }
        }
    }
    bool ok = true;
    switch (I.color_type * 32 + I.depth) {
#define PD_HOST_BGR(CT, D)                                                                                   \
    case CT * 32 + D:                                                                                        \
        for (int y = 0; y < I.H; ++y)                                                                        \
            for (int x = 0; x < I.W; ++x)                                                                    \
                ok &= pixel_bgr<CT, D>(F, raw.data(), I.interlace != 0, x, y, bgr + (size_t)y * row_stride + 3 * (size_t)x); \
        break;
        PD_FORMATS(PD_HOST_BGR)
#undef PD_HOST_BGR
        default: return 1;
    }
    return ok ? 0 : 1;
}

#ifdef __CUDACC__
// ==== kernels ========================================================================================================

// positions passing the quick test: a thread per stream word (32 bit positions), survivors appended to a list
__global__ void __launch_bounds__(256) pd_quick_kernel(const uint32_t *__restrict__ zs, uint64_t n_words, uint64_t first_bit,
                                                       uint64_t stream_bits, uint64_t *__restrict__ list, uint32_t cap,
                                                       uint32_t *__restrict__ count) {
    const uint64_t wi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (wi * 32 + 3 > stream_bits) return;
    const uint64_t w0 = wi < n_words ? zs[wi] : 0u, w1 = wi + 1 < n_words ? zs[wi + 1] : 0u, w2 = wi + 2 < n_words ? zs[wi + 2] : 0u,
                   w3 = wi + 3 < n_words ? zs[wi + 3] : 0u;
    const uint64_t lo = w0 | (w1 << 32), hi = w2 | (w3 << 32);
    // positions whose type bits say "dynamic Huffman" (bit p + 1 clear, bit p + 2 set): a quarter of them; only those are
    // looked at, so that the lanes of a warp stay busy instead of waiting for the quarter that passes
    uint32_t todo = (uint32_t)(~(lo >> 1) & (lo >> 2));
    while (todo) {
        const int p = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint64_t bit = wi * 32 + p;
        if (bit < first_bit || bit + 3 > stream_bits) continue;
        const uint64_t head = p ? (lo >> p) | (hi << (64 - p)) : lo;
        const int q = p + 17;
        const uint64_t lens3 = (lo >> q) | (hi << (64 - q));
        if (!quick_check(head, lens3)) continue;
        const uint32_t at = atomicAdd(count, 1u);
        if (at < cap) list[at] = bit;
    }
}

// the full header test on the survivors, a thread each; candidates appended to cands[]
__global__ void __launch_bounds__(128) pd_full_kernel(const uint32_t *__restrict__ zs, uint64_t n_words, const uint64_t *__restrict__ list,
                                                      const uint32_t *__restrict__ n_list, uint32_t cap_list, Cand *__restrict__ cands,
                                                      uint32_t cap, uint32_t *__restrict__ count) {
    const uint32_t n = min(*n_list, cap_list);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint64_t bit = list[i];
        if (!full_check(zs, n_words, bit)) continue;
        const uint32_t at = atomicAdd(count, 1u);
        if (at < cap) cands[at].bit = bit;
    }
}

constexpr int kDecoders = 8;  // deflate blocks decoded side by side in one warp (lanes 0 .. 7): 8 x 3264 bytes of tables per CTA

// Every candidate decoded to its end-of-block symbol, nothing written.  One thread per candidate - the chain of dependent
// table look-ups of a Huffman decoder cannot be spread over lanes - and eight of them per warp, each with its tables in
// shared memory: a warp with a single decoding lane spends the same issue slots as one with eight, and with thousands of
// blocks in flight the issue slots, not the latency, bound the pass (measured: one lane per warp 6.0 ms per 8K file).
__global__ void __launch_bounds__(32) pd_measure_kernel(const uint32_t *__restrict__ zs, uint64_t n_words, uint64_t stream_bits,
                                                        Cand *__restrict__ cands, const uint32_t *__restrict__ n_cands, uint32_t cap,
                                                        uint64_t out_cap, uint32_t wsize) {
    __shared__ Tables tabs[kDecoders];
    const uint32_t n = min(*n_cands, cap);
    if (threadIdx.x >= kDecoders) return;
    for (uint32_t i = blockIdx.x * kDecoders + threadIdx.x; i < n; i += gridDim.x * kDecoders) {
        uint8_t lens[320];
        BlockOut R{0, 0, 0, 0, 0};
        const int rc = decode_block<false>(zs, n_words, stream_bits, cands[i].bit, tabs[threadIdx.x], lens, nullptr, nullptr, 0, out_cap, wsize, R);
        cands[i].end_bit = R.end_bit;
        cands[i].out_len = R.out_len;
        cands[i].n_matches = R.n_matches;
        cands[i].status = rc ? rc : (R.final_block << 8);
    }
}

// The blocks of the chain decoded, part 1: eight blocks per warp again, one lane each.  Literals go straight to raw[]; a
// back-reference is only RECORDED (block offset, length, distance) in the block's slice of the match list.  Executing it
// here would make its lane - and with it the seven other decoders of the warp - wait for a read of bytes that were written
// moments ago and sit in L2 (0.7 us each, measured: 11 ms per 8K file with 10 M matches); the copies are the business of
// pd_copy_kernel.  Stored blocks are copied here.  Any failure raises *bad.
__global__ void __launch_bounds__(32) pd_decode_kernel(const uint32_t *__restrict__ zs, uint64_t n_words, uint64_t stream_bits,
                                                       const Block *__restrict__ blocks, uint32_t n_blocks, uint8_t *__restrict__ raw,
                                                       Match *__restrict__ matches, uint64_t out_cap, uint32_t wsize, int *__restrict__ bad) {
    __shared__ Tables tabs[kDecoders];
    if (threadIdx.x >= kDecoders) return;
    const uint32_t i = blockIdx.x * kDecoders + threadIdx.x;
    if (i >= n_blocks) return;
    const Block b = blocks[i];
    const uint64_t room = out_cap > b.out_off ? out_cap - b.out_off : 0;
    Tables &T = tabs[threadIdx.x];
    uint8_t lens[320];
    Bits br;
    br.init(zs, n_words, b.bit);
    int fin, type;
    uint32_t slen = 0;
    uint64_t byte0 = 0;
    if (block_begin(br, stream_bits, T, lens, &fin, &type, &slen, &byte0)) {
        *bad = 1;
        return;
    }
    uint8_t *out = raw + b.out_off;
    if (type == 0) {
        if (slen != b.out_len || slen > room || b.n_matches) {
            *bad = 1;
            return;
        }
        const uint8_t *src = reinterpret_cast<const uint8_t *>(zs) + byte0;
        for (uint32_t k = 0; k < slen; ++k) out[k] = src[k];
        return;
    }
    Match *list = matches + b.match_off;
    uint64_t o = 0;
    uint32_t nm = 0;
    bool ok = false;
    for (uint32_t n = 0; n < kMaxSyms; ++n) {
        uint32_t len = 0, dist = 0;
        const int k = next_token(br, T, &len, &dist);
        if (k == 0) {
            if (o >= room) break;
            out[o++] = (uint8_t)len;
        } else if (k == 1) {
            if (dist > wsize || o + len > room || dist > b.out_off + o || nm >= b.n_matches) break;
            list[nm++] = Match{(uint32_t)o, (uint16_t)len, (uint16_t)dist};   // (a distance of 32768 fits 16 bits)
            o += len;
        } else {
            ok = (k == 2) && br.pos() <= stream_bits;
            break;
        }
    }
    if (!ok || o != b.out_len || nm != b.n_matches) *bad = 1;
}

// part 2: the recorded back-references executed, a warp per block, in order.  The lanes copy the bytes of a match together
// (a match that overlaps its own output repeats its first `dist` bytes, so every byte reads data that existed before the
// match); a byte whose source lies in front of the block becomes a history mark in ref[] (all zeros before the pass), a
// copied mark stays a mark.  With thousands of warps in flight the L2 round trip of every match hides behind the other
// blocks' copies.  Records are fetched 32 at a time.
__global__ void __launch_bounds__(256) pd_copy_kernel(Block *__restrict__ blocks, uint32_t n_blocks, const Match *__restrict__ matches,
                                                      uint8_t *raw, uint16_t *ref) {
    const uint32_t i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n_blocks) return;
    const Block b = blocks[i];
    const Match *list = matches + b.match_off;
    const uint64_t tail_from = b.out_len > kWindow ? b.out_len - kWindow : 0;
    uint8_t *out = raw + b.out_off;
    uint16_t *mark = ref + b.out_off;
    uint32_t marks = 0;
    for (uint32_t m0 = 0; m0 < b.n_matches; m0 += 32) {
        const uint32_t cnt = min(32u, b.n_matches - m0);
        Match mine{0, 0, 1};
        if (lane < cnt) mine = list[m0 + lane];
        for (uint32_t q = 0; q < cnt; ++q) {
            const uint32_t o = __shfl_sync(0xffffffffu, mine.o, q), len = __shfl_sync(0xffffffffu, (uint32_t)mine.len, q);
            const uint32_t dist = __shfl_sync(0xffffffffu, (uint32_t)mine.dist, q);
            // A record is only trusted after it has been checked again: if the decoding pass gave up on this block (it has
            // raised *bad; the file will be declined) the rest of the block's slice holds whatever an earlier file left there.
            if (dist == 0 || (uint64_t)o + len > b.out_len || dist > b.out_off + o) continue;   // (warp-uniform)
            for (uint32_t t = lane; t < len; t += 32) {
                const uint32_t tt = dist >= len ? t : t % dist;
                const int64_t srel = (int64_t)o + tt - (int64_t)dist;   // relative to the block's first byte
                uint16_t r;
                if (srel < 0) {
                    r = (uint16_t)(-srel);
                } else {
                    out[o + t] = out[srel];
                    r = mark[srel];
                }
                if (r) {
                    mark[o + t] = r;
                    marks += (o + t >= tail_from);
                }
            }
            __syncwarp();
        }
    }
    marks = __reduce_add_sync(0xffffffffu, marks);
    if (lane == 0) blocks[i].tail_marks = marks;
}

// Tail pass, part 1: a CTA per group of `per` consecutive blocks walks its blocks in order (tail_step; 1024 threads = 32
// positions per thread: marks first, then the history look-ups, then the stores; blocks without marks in their last 32 KiB
// are skipped)
__global__ void __launch_bounds__(1024) pd_tails_group_kernel(const Block *__restrict__ blocks, uint32_t n_blocks, uint32_t per, uint8_t *raw,
                                                              uint16_t *ref, uint32_t *__restrict__ group_marks) {
    const uint32_t i0 = blockIdx.x * per, i1 = min(n_blocks, i0 + per);
    const uint64_t gs = blocks[i0].out_off;
    for (uint32_t i = i0; i < i1; ++i) {
        const Block b = blocks[i];
        if (b.tail_marks == 0) continue;
        const uint64_t end = b.out_off + b.out_len, t0 = b.out_len > kWindow ? end - kWindow : b.out_off;
        for (int half = 0; half < 2; ++half) {   // 2 x 16 positions per thread (registers)
            uint32_t r[16], rt[16];
            uint8_t v[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const uint64_t p = t0 + threadIdx.x + 1024u * (16 * half + q);
                r[q] = p < end ? ref[p] : 0u;
            }
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const uint64_t abs = b.out_off - r[q];
                const bool inside = r[q] && abs >= gs;
                rt[q] = inside ? ref[abs] : 0u;
                v[q] = inside ? raw[abs] : (uint8_t)0;
            }
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                if (!r[q]) continue;
                const uint64_t p = t0 + threadIdx.x + 1024u * (16 * half + q), abs = b.out_off - r[q];
                if (abs >= gs) {
                    if (rt[q] == 0) raw[p] = v[q];
                    ref[p] = (uint16_t)rt[q];
                } else {
                    ref[p] = (uint16_t)(gs - abs);
                }
            }
        }
        __syncthreads();
    }
    // marks left in the 32 KiB in front of the next group (what pd_tails_chain_kernel has to look at; usually nothing)
    if (i1 < n_blocks) {
        const uint64_t next = blocks[i1].out_off, lo = next > kWindow ? next - kWindow : 0, t0 = lo > gs ? lo : gs;
        int mine = 0;
        for (uint64_t p = t0 + threadIdx.x; p < next; p += 1024) mine |= ref[p] != 0;
        const int any = __syncthreads_or(mine);
        if (threadIdx.x == 0) group_marks[blockIdx.x] = (uint32_t)any;
    }
}

// part 2: the 32 KiB in front of every group made final, group after group (one CTA; marks there are relative to the start
// of the group they sit in, their history is the - already final - 32 KiB in front of that group)
__global__ void __launch_bounds__(1024) pd_tails_chain_kernel(const Block *__restrict__ blocks, uint32_t n_blocks, uint32_t per, uint8_t *raw,
                                                              uint16_t *ref, const uint32_t *__restrict__ group_marks) {
    const uint32_t ng = (n_blocks + per - 1) / per;
    for (uint32_t g = 1; g + 1 < ng; ++g) {
        if (group_marks[g] == 0) continue;
        const uint64_t gs = blocks[g * per].out_off, next = blocks[(g + 1) * per].out_off;
        const uint64_t lo = next > kWindow ? next - kWindow : 0, t0 = lo > gs ? lo : gs;
        uint32_t r[32];
        uint8_t v[32];
#pragma unroll
        for (int q = 0; q < 32; ++q) {
            const uint64_t p = t0 + threadIdx.x + 1024u * q;
            r[q] = p < next ? ref[p] : 0u;
        }
#pragma unroll
        for (int q = 0; q < 32; ++q) v[q] = r[q] ? raw[gs - r[q]] : (uint8_t)0;
#pragma unroll
        for (int q = 0; q < 32; ++q) {
            const uint64_t p = t0 + threadIdx.x + 1024u * q;
            if (r[q]) {
                raw[p] = v[q];
                ref[p] = 0;
            }
        }
        __syncthreads();
    }
}

// part 3: the re-based marks in the last 32 KiB of every block (grid.x = blocks; group 0 has none left)
__global__ void __launch_bounds__(256) pd_tails_finish_kernel(const Block *__restrict__ blocks, uint32_t per, uint8_t *raw, uint16_t *ref) {
    const Block b = blocks[blockIdx.x];
    if (blockIdx.x < per || b.tail_marks == 0) return;
    const uint64_t gs = blocks[(blockIdx.x / per) * per].out_off;
    const uint64_t end = b.out_off + b.out_len, t0 = b.out_len > kWindow ? end - kWindow : b.out_off;
    for (uint64_t p = t0 + threadIdx.x; p < end; p += blockDim.x) {
        const uint32_t r = ref[p];
        if (r) {
            raw[p] = raw[gs - r];
            ref[p] = 0;
        }
    }
}

// every remaining mark points at a final byte: grid.x = blocks of the chain
__global__ void __launch_bounds__(256) pd_resolve_kernel(const Block *__restrict__ blocks, uint8_t *raw, const uint16_t *__restrict__ ref) {
    const Block b = blocks[blockIdx.x];
    const uint64_t end = b.out_off + b.out_len;
    for (uint64_t p = b.out_off + blockIdx.y * blockDim.x + threadIdx.x; p < end; p += (uint64_t)gridDim.y * blockDim.x) {
        const uint32_t r = ref[p];
        if (r) raw[p] = raw[b.out_off - r];
    }
}

// Adler-32 of the inflated image: sums[0] += sum of bytes, sums[1] += sum of ((n - i) mod 65521) * byte[i]
// (s1 = 1 + sums[0], s2 = n + sums[1], both mod 65521); 16 bytes per thread
__global__ void __launch_bounds__(256) pd_adler_kernel(const uint8_t *__restrict__ raw, uint64_t n, unsigned long long *__restrict__ sums) {
    const uint64_t i0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    unsigned long long a = 0, w = 0;
    if (i0 < n) {
        const uint64_t i1 = i0 + 16 < n ? i0 + 16 : n;
        uint32_t wt = (uint32_t)((n - i0) % 65521ull);
        for (uint64_t i = i0; i < i1; ++i) {
            const uint32_t v = raw[i];
            a += v;
            w += (unsigned long long)wt * v;
            wt = wt ? wt - 1 : 65520u;
        }
    }
    for (int d = 16; d; d >>= 1) {
        a += __shfl_down_sync(0xffffffffu, a, d);
        w += __shfl_down_sync(0xffffffffu, w, d);
    }
    __shared__ unsigned long long sa[8], sw[8];
    if ((threadIdx.x & 31) == 0) {
        sa[threadIdx.x >> 5] = a;
        sw[threadIdx.x >> 5] = w;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 8; ++k) {
            a += sa[k];
            w += sw[k];
        }
        atomicAdd(&sums[0], a);
        atomicAdd(&sums[1], w % 65521ull);
    }
}

// CRC-32 of stream segments (a thread per segment, <= 4096 bytes each): the host folds them per IDAT chunk
struct CrcSeg {
    uint64_t off;
    uint32_t len, crc;
};
__global__ void __launch_bounds__(128) pd_crc_kernel(const uint8_t *__restrict__ zs, CrcSeg *__restrict__ segs, uint32_t n_segs,
                                                     const uint32_t *__restrict__ table) {
    __shared__ uint32_t t[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) t[i] = table[i];
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_segs) return;
    const uint8_t *p = zs + segs[i].off;
    const uint32_t n = segs[i].len;
    uint32_t crc = 0xFFFFFFFFu;
    for (uint32_t k = 0; k < n; ++k) crc = t[(crc ^ p[k]) & 255u] ^ (crc >> 8);
    segs[i].crc = ~crc;
}

constexpr int kFetchPx = 128;  // pixels of the row above a band a warp fetches (and a band publishes) at a time

__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// The filters undone: raw (filter byte + filtered bytes per row, stride) -> recon (reconstructed bytes, rows of rstride bytes,
// rstride a multiple of 4).  A warp per BAND of 32 rows (taken in image order through a ticket, so that a band only ever waits
// for a warp that is already running); lane t owns row 32 k + t and works on chunk s - t (CH pixels) at step s: the
// reconstructed chunk above arrives from lane t - 1 through shuffles, one step after that lane finished it (rows filtered
// None / Sub ignore it - a file of such rows, like everything cv2.imwrite produces, is 32 independent rows per warp).  If
// the first row of a band needs the row above (filter Up / Average / Paeth), that is the last row of the band before: that
// band publishes its progress every kFetch chunks (progress[band] = chunks of its last row that are final, release store),
// this one waits for kFetch chunks at a time (acquire load; bounded polling: a wait that does not end raises *bad, it
// cannot hang) and brings them into shared memory with the whole warp.  The filtered bytes of a chunk are loaded (aligned
// words + funnel shift) four steps before they are used.  A filter type above 4 raises *bad.
// CH = pixels a lane reconstructs per step (4 or 8: the chunk is what one row lags behind the row above, so the whole
// image is a chain of H chunk-times; smaller chunks shorten it, larger ones amortise the per-step shuffles and loads).
template <int BPP, int CH>
__global__ void __launch_bounds__(256) pd_unfilter_kernel(const uint8_t *__restrict__ raw, uint8_t *recon, int W, int H, size_t stride, size_t rstride,
                                                          uint32_t *ticket, uint32_t *progress, int *bad) {
    constexpr int kChunkPx = CH, kFetch = kFetchPx / CH;
    constexpr int NW = CH * BPP / 4;       // words per chunk
    constexpr int CB = kChunkPx * BPP;     // bytes per chunk
    __shared__ uint32_t upbuf[8][kFetch * NW];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t k = 0;
    if (lane == 0) k = atomicAdd(ticket, 1u);
    k = __shfl_sync(0xffffffffu, k, 0);
    const int first = (int)k * 32;
    if (first >= H) return;
    const int rows = min(32, H - first);
    const bool active = (int)lane < rows;
    const int row = first + (active ? (int)lane : 0);
    const uint8_t *src = raw + (size_t)row * stride;
    uint8_t *dst = recon + (size_t)row * rstride;
    const uint32_t *up_row = reinterpret_cast<const uint32_t *>(recon + (size_t)(first > 0 ? first - 1 : 0) * rstride);
    const uint32_t ft = active ? src[0] : 0u;
    if (ft > 4) *bad = 1;
    const uint32_t m1 = ft == 1 ? ~0u : 0u, m2 = ft == 2 ? ~0u : 0u, m3 = ft == 3 ? ~0u : 0u, m4 = ft >= 4 ? ~0u : 0u;
    const bool dep = first > 0 && __shfl_sync(0xffffffffu, ft, 0) > 1;                   // this band's first row needs the band above
    const bool next_dep = first + 32 < H && raw[(size_t)(first + 32) * stride] > 1;    // the band below needs this band's last row
    const int row_bytes = W * BPP;
    const int nc = (W + kChunkPx - 1) / kChunkPx;
    // aligned words under this row's filtered bytes
    const uintptr_t addr0 = reinterpret_cast<uintptr_t>(src + 1);
    const uint32_t *wbase = reinterpret_cast<const uint32_t *>(addr0 & ~(uintptr_t)3);
    const int sh = (int)(addr0 & 3) * 8;
    constexpr int PF = 4;   // the filtered bytes of a chunk are loaded PF steps before they are used (a step is shorter than an L2 round trip)
    uint32_t pre[PF][NW + 1], outw[NW], left[BPP], upleft[BPP];
#pragma unroll
    for (int i = 0; i < NW; ++i) outw[i] = 0;
#pragma unroll
    for (int i = 0; i < BPP; ++i) left[i] = upleft[i] = 0;
#pragma unroll
    for (int u = 0; u < PF; ++u) {   // the chunks of this lane's first PF steps
        const int j = u - (int)lane;
#pragma unroll
        for (int i = 0; i <= NW; ++i) pre[u][i] = (active && j >= 0 && j < nc) ? __ldg(wbase + (size_t)j * NW + i) : 0u;
    }
    const int steps = nc + rows - 1;
    for (int s0 = 0; s0 < steps; s0 += PF) {
#pragma unroll
        for (int u = 0; u < PF; ++u) {
            const int s = s0 + u;
            if (s >= steps) break;                 // (warp-uniform)
            const int j = s - (int)lane;           // this lane's chunk at this step
            const bool on = active && j >= 0 && j < nc;
            if (dep && s < nc && (s % kFetch) == 0) {   // (warp-uniform) chunks s .. s + kFetch - 1 of the row above the band
                const uint32_t need = (uint32_t)min(s + kFetch, nc);
                uint32_t spins = 0;
                while (ld_acquire_u32(progress + (k - 1)) < need) {
                    if (++spins > (1u << 22)) {
                        *bad = 1;
                        break;
                    }
                }
                __syncwarp();   // lane 0 has read the chunks fetched before
                for (int w = (int)lane; w < kFetch * NW; w += 32) {
                    const int idx = s * NW + w;
                    upbuf[warp][w] = idx < nc * NW ? __ldcg(up_row + idx) : 0u;
                }
                __syncwarp();
            }
            uint32_t cur[NW];
#pragma unroll
            for (int i = 0; i < NW; ++i) cur[i] = __funnelshift_r(pre[u][i], pre[u][i + 1], sh);
            {   // the filtered bytes this lane needs PF steps from now
                const int jn = j + PF;
                if (active && jn >= 0 && jn < nc) {
#pragma unroll
                    for (int i = 0; i <= NW; ++i) pre[u][i] = __ldg(wbase + (size_t)jn * NW + i);
                }
            }
            // the reconstructed chunk above: from the lane above (its result of the previous step), lane 0 from the fetched chunks
            uint32_t up[NW];
#pragma unroll
            for (int i = 0; i < NW; ++i) up[i] = __shfl_up_sync(0xffffffffu, outw[i], 1);
            if (lane == 0) {
#pragma unroll
                for (int i = 0; i < NW; ++i) up[i] = (dep && on) ? upbuf[warp][(s % kFetch) * NW + i] : 0u;
            }
            if (on) {
#pragma unroll
                for (int px = 0; px < kChunkPx; ++px) {
#pragma unroll
                    for (int c = 0; c < BPP; ++c) {
                        const int byte = px * BPP + c;
                        const uint32_t f = (cur[byte >> 2] >> (8 * (byte & 3))) & 255u;
                        const uint32_t b = (up[byte >> 2] >> (8 * (byte & 3))) & 255u;
                        const uint32_t v = unfilter_byte_masked(f, left[c], b, upleft[c], m1, m2, m3, m4);
                        upleft[c] = b;
                        left[c] = v;
                        if ((byte & 3) == 0) outw[byte >> 2] = v;
                        else outw[byte >> 2] |= v << (8 * (byte & 3));
                    }
                }
                const int nbytes = min(CB, row_bytes - j * CB);
                uint32_t *o = reinterpret_cast<uint32_t *>(dst + (size_t)j * CB);
                if (nbytes == CB) {
#pragma unroll
                    for (int i = 0; i < NW; ++i) o[i] = outw[i];
                } else {
                    for (int i = 0; i < nbytes; ++i) dst[(size_t)j * CB + i] = (uint8_t)(outw[i >> 2] >> (8 * (i & 3)));
                }
                if (next_dep && (int)lane == rows - 1 && (((j + 1) % kFetch) == 0 || j == nc - 1))   // the band's last row, for the band below
                    st_release_u32(progress + k, (uint32_t)(j + 1));
            }
        }
    }
}

// reconstructed rows (per pass: F.off, F.stride) -> BGR staging image (row stride dstride), a thread per image pixel
// (grid.y = image rows).  The palette is a kernel parameter, not a __constant__ symbol: slots decode concurrently.  A palette
// index without a PLTE entry raises *bad.
template <int CT, int DEPTH, bool LACE>
__global__ void __launch_bounds__(256) pd_bgr_kernel(const uint8_t *__restrict__ recon, const __grid_constant__ Fmt F, uint8_t *__restrict__ bgr,
                                                     size_t dstride, int *bad) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= F.W) return;
    uint8_t v[3];
    if (!pixel_bgr<CT, DEPTH>(F, recon, LACE, x, y, v)) *bad = 1;
    uint8_t *o = bgr + (size_t)y * dstride + 3 * (size_t)x;
    o[0] = v[0];
    o[1] = v[1];
    o[2] = v[2];
}
#endif  // __CUDACC__

}  // namespace p2ppdec
