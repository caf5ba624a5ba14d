// p2p_jpegdec.cuh - baseline JPEG decoder for the input panoramas (SURVEY 8f-2: the decode side of the path).
//
// The reference loads every panorama with cv2.imread (ref app/panorama_to_plane-pitch.py:244); for a JPEG file that
// is libjpeg-turbo at its decoder defaults (dct_method = JDCT_ISLOW, do_fancy_upsampling = TRUE).  Everything after
// the entropy decoder is integer arithmetic on independent blocks / pixels, restated here operation by operation
// (oracle/jpeg_decode_model.py is the NumPy restatement, pinned against cv2.imdecode), so the decoded panorama is
// bit-identical to cv2.imread's:
//   device jdhuff.c   Huffman decoding of the single interleaved scan as self-synchronising subsequences (huff_*_kernel);
//   host              the same decoder in C++ (decode_scan) as the fallback when the device stage does not converge
//   device jidctint.c jpeg_idct_islow on dequantised coefficients, + 128, clamp            (jpegdec_idct_kernel)
//          jdsample.c h2v2 / h2v1 fancy upsampling (triangle filters, alternating rounding; replication when the
//                     chroma plane is at most 2 samples wide), jdcolor.c ycc_rgb_convert   (jpegdec_color_kernel)
// Supported: 8-bit, 3 components (YCbCr; 4:4:4 / 4:2:2 / 4:2:0) or 1 (grayscale); SOF0 / SOF1 with one scan and restart
// markers (Huffman stage on the device), SOF2 progressive files (jdphuff.c restated on the host, decode_progressive).
// Any legal Huffman tables, not only the Annex K ones cv2 writes by default: optimised tables, codes of 9 / 10 / 16 bits,
// AC codes whose length + size sits on the 10-bit combined look-up's edge, DC tables of up to 256 entries, size-0 symbols
// other than 0x00 as end of block, table ids 0-3 (tests/jpeg_writer.py writes such files for the tests).
// Anything else (CMYK, RGB-coded files, EXIF orientation != 1, damaged data) is reported as
// unsupported and the caller falls back to cv2.imread, as the reference does for every file.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <thread>
#include <vector>

namespace p2pjdec {

struct Info {
    int W = 0, H = 0;
    int ncomp = 3;                   // 3 = YCbCr; 1 = grayscale: one block per MCU, and the two chroma planes are kept as
                                     // all-zero coefficient planes (= 128 after the IDCT), for which jdcolor.c's YCbCr ->
                                     // RGB gives R = G = B = Y, the same pixels as its gray_rgb_convert
    int hmax = 1, vmax = 1;          // luma sampling factors (chroma is 1 x 1)
    int mcux = 0, mcuy = 0;
    int bw[3] = {0, 0, 0}, bh[3] = {0, 0, 0};   // blocks per row / column of each component plane (MCU padded)
    int cw = 0, ch = 0;              // downsampled_width / height of the chroma components
    uint16_t quant[3][64];           // natural order, per component
    size_t coef_off[3] = {0, 0, 0};  // element offset of each component in the coefficient buffer
    size_t n_coef = 0;
};

// The DCT of 8-bit samples has an L2 norm <= 1024 per block (Parseval), quantisation adds at most 1020: a block of
// dequantised coefficients beyond this norm is damaged data.  libjpeg-turbo's SIMD IDCT (16-bit lanes) wraps on such
// blocks in ways this decoder does not restate, so the file is declined (cv2.imread handles it).
constexpr float kMaxBlockNorm = 2048.f;

// ---- host: markers + Huffman decoding ---------------------------------------------------------------------------
static const uint8_t kNat[64 + 16] = {  // zigzag position -> natural index (+ 16 safety entries like jpeg_natural_order)
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55,
    62, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63};

constexpr int kFastBits = 10;
struct HuffTable {
    bool present = false;
    // AC tables: 10-bit lookahead that resolves code AND value bits at once when both fit:
    // (value << 8) | (run << 4) | total bits, 0 = take the general path
    int32_t fast_ac[1 << kFastBits];
    uint16_t look[512];     // 9-bit lookahead: (length << 8) | symbol, 0 = longer code
    int32_t maxcode[18];    // largest code of each length (-1 if none); [17] = sentinel
    int32_t valoff[18];     // vals index = code + valoff[length]
    uint8_t vals[256];
};

inline bool build_huff(const uint8_t *bits, const uint8_t *vals, int nvals, HuffTable &t) {
    memset(&t, 0, sizeof(t));
    memcpy(t.vals, vals, (size_t)nvals);
    int code = 0, k = 0;
    for (int l = 1; l <= 16; ++l) {
        // jdhuff.c jpeg_make_d_derived_tbl: the codes of a length must fit with the all-ones code left unused
        // (checked before any table write: an over-subscribed length would index past look[])
        if (bits[l - 1] && code + bits[l - 1] >= (1 << l)) return false;
        if (bits[l - 1]) {
            t.valoff[l] = k - code;
            for (int i = 0; i < bits[l - 1]; ++i, ++k, ++code) {
                if (l <= 9) {
                    const int first = code << (9 - l);
                    for (int f = 0; f < (1 << (9 - l)); ++f) t.look[first + f] = (uint16_t)((l << 8) | vals[k]);
                }
            }
            t.maxcode[l] = code - 1;
        } else {
            t.maxcode[l] = -1;
        }
        code <<= 1;
    }
    t.maxcode[17] = 0x7fffffff;
    t.present = (k == nvals);
    // combined code + value lookup (used for AC tables only)
    for (int i = 0; i < (1 << kFastBits); ++i) {
        t.fast_ac[i] = 0;
        const uint16_t e = t.look[i >> (kFastBits - 9)];
        if (!e) continue;
        const int len = e >> 8, rs = e & 0xFF, run = rs >> 4, sz = rs & 15;
        if (sz == 0 || len + sz > kFastBits) continue;
        int v = (i >> (kFastBits - len - sz)) & ((1 << sz) - 1);
        if (v < (1 << (sz - 1))) v += 1 - (1 << sz);
        t.fast_ac[i] = (int32_t)(((uint32_t)v << 8) | (uint32_t)(run << 4) | (uint32_t)(len + sz));
    }
    return t.present;
}

struct BitReader {
    const uint8_t *p, *end;
    uint64_t acc = 0;
    int n = 0;            // valid bits in acc (top-aligned at bit n - 1 .. 0)
    bool marker = false;  // the byte stream hit a marker: zeros are fed from here on
    int zero_bits = 0;    // how many of the bits fed so far were such zeros (consuming one = damaged / truncated data)
    inline void fill() {
        // bulk path: 4 bytes at once when none of them is 0xFF (no stuffing, no marker)
        while (n <= 32 && !marker && p + 4 <= end) {
            const uint32_t w = ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
            const uint32_t v = ~w;
            if ((v - 0x01010101u) & ~v & 0x80808080u) break;   // some byte is 0xFF
            acc = (acc << 32) | w;
            n += 32;
            p += 4;
        }
        while (n <= 56) {
            uint32_t b = 0;
            if (!marker && p < end) {
                b = *p;
                if (b == 0xFF) {
                    if (p + 1 < end && p[1] == 0) {
                        p += 2;
                    } else {
                        marker = true;
                        b = 0;
                        zero_bits += 8;
                    }
                } else {
                    ++p;
                }
            } else {
                marker = true;
                zero_bits += 8;
            }
            acc = (acc << 8) | b;
            n += 8;
        }
    }
    // true if the decoder has consumed bits that were never in the file
    inline bool overran() const { return zero_bits > n; }
    inline uint32_t peek(int k) { return (uint32_t)(acc >> (n - k)) & ((1u << k) - 1u); }
    inline void skip(int k) { n -= k; }
};

// the caller guarantees at least 32 valid bits (one check per coefficient: code <= 16 bits + value <= 15 bits)
inline int decode_sym(BitReader &br, const HuffTable &t) {
    const uint16_t e = t.look[br.peek(9)];
    if (e) {
        br.skip(e >> 8);
        return e & 0xFF;
    }
    const uint32_t w = br.peek(16);
    for (int l = 10; l <= 16; ++l) {
        const int32_t code = (int32_t)(w >> (16 - l));
        if (code <= t.maxcode[l]) {
            br.skip(l);
            return t.vals[(code + t.valoff[l]) & 0xFF];
        }
    }
    return -1;
}

inline int receive_extend(BitReader &br, int s) {
    const int v = (int)br.peek(s);
    br.skip(s);
    return (v < (1 << (s - 1))) ? v - (1 << s) + 1 : v;
}

// EXIF orientation of an APP1 segment (0 = none found)
inline int exif_orientation(const uint8_t *seg, size_t len) {
    if (len < 14 || memcmp(seg, "Exif\0\0", 6) != 0) return 0;
    const uint8_t *t = seg + 6;
    const size_t n = len - 6;
    const bool le = (t[0] == 'I' && t[1] == 'I'), be = (t[0] == 'M' && t[1] == 'M');
    if (!le && !be) return -1;
    auto r16 = [&](size_t o) -> uint32_t { return le ? (uint32_t)(t[o] | (t[o + 1] << 8)) : (uint32_t)((t[o] << 8) | t[o + 1]); };
    auto r32 = [&](size_t o) -> uint32_t {
        return le ? (uint32_t)t[o] | ((uint32_t)t[o + 1] << 8) | ((uint32_t)t[o + 2] << 16) | ((uint32_t)t[o + 3] << 24)
                  : ((uint32_t)t[o] << 24) | ((uint32_t)t[o + 1] << 16) | ((uint32_t)t[o + 2] << 8) | (uint32_t)t[o + 3];
    };
    const size_t ifd = r32(4);
    if (ifd + 2 > n) return -1;
    const uint32_t cnt = r16(ifd);
    for (uint32_t i = 0; i < cnt; ++i) {
        const size_t e = ifd + 2 + 12 * (size_t)i;
        if (e + 12 > n) return -1;
        if (r16(e) == 0x0112) return (int)r16(e + 8);
    }
    return 0;
}

// Parse the headers of a JPEG file.  Returns 0 and fills `info`, the Huffman tables and the scan position if the
// file is in the supported subset, 1 if not.
struct Parsed {
    Info info;
    HuffTable dc[4], ac[4];
    int td[3] = {0, 0, 0}, ta[3] = {0, 0, 0};
    int dri = 0;
    size_t ecs = 0;   // offset of the entropy-coded data (progressive: of the first SOS marker)
    bool progressive = false;   // SOF2: several scans, decoded on the host (decode_progressive)
    int cid[3] = {0, 0, 0};     // component ids of the frame header
};

// one DHT segment into the table sets (jdmarker.c get_dht); 0 = ok.  jdhuff.c jpeg_make_d_derived_tbl checks a table when
// a scan starts to use it, not when it is defined: a table that breaks its rules (an over-subscribed code length, a DC
// symbol above 15) is kept as absent, and a scan that uses it is declined - a progressive file may leave such a table in
// a slot its later scans redefine before they use it.
inline int parse_dht(const uint8_t *seg, size_t sl, HuffTable *dc, HuffTable *ac) {
    size_t j = 0;
    while (j < sl) {
        if (j + 17 > sl) return 1;
        const int tc = seg[j] >> 4, th = seg[j] & 15;
        int nv = 0;
        for (int k = 0; k < 16; ++k) nv += seg[j + 1 + k];
        if (tc > 1 || th > 3 || nv > 256 || j + 17 + nv > sl) return 1;
        HuffTable &t = tc ? ac[th] : dc[th];
        bool ok = build_huff(seg + j + 1, seg + j + 17, nv, t);
        if (!tc)   // DC symbols are categories 0..15
            for (int k = 0; k < nv; ++k) ok = ok && seg[j + 17 + k] <= 15;
        t.present = ok;
        j += 17 + (size_t)nv;
    }
    return 0;
}

inline int parse_headers(const uint8_t *d, size_t len, Parsed &P) {
    if (len < 4 || d[0] != 0xFF || d[1] != 0xD8) return 1;
    size_t i = 2;
    uint16_t qt[4][64];
    bool have_qt[4] = {false, false, false, false};
    bool jfif = false, adobe = false, have_frame = false;
    int adobe_transform = 0;
    int cid[3] = {0, 0, 0}, tq[3] = {0, 0, 0}, hs[3] = {1, 1, 1}, vs[3] = {1, 1, 1};
    Info &I = P.info;
    while (i + 4 <= len) {
        if (d[i] != 0xFF) return 1;
        while (i + 1 < len && d[i + 1] == 0xFF) ++i;
        if (i + 4 > len) return 1;
        const int m = d[i + 1];
        i += 2;
        // only the segments a baseline JFIF / EXIF file is made of; libjpeg rejects or special-cases the rest
        const bool known = (m >= 0xE0 && m <= 0xEF) || m == 0xFE || m == 0xDB || m == 0xC4 || m == 0xC0 || m == 0xC1 ||
                           m == 0xC2 || m == 0xDD || m == 0xDA;
        if (!known) return 1;
        const size_t L = ((size_t)d[i] << 8) | d[i + 1];
        if (L < 2 || i + L > len) return 1;
        const uint8_t *seg = d + i + 2;
        const size_t sl = L - 2;
        i += L;
        if (m == 0xDB) {
            size_t j = 0;
            while (j < sl) {
                const int pq = seg[j] >> 4, t = seg[j] & 15;
                ++j;
                if (t > 3 || pq != 0 || j + 64 > sl) return 1;   // 16-bit tables are not baseline
                for (int k = 0; k < 64; ++k) {
                    qt[t][kNat[k]] = seg[j + k];
                }
                j += 64;
                have_qt[t] = true;
            }
        } else if (m == 0xC4) {
            if (parse_dht(seg, sl, P.dc, P.ac)) return 1;
        } else if (m == 0xC0 || m == 0xC1 || m == 0xC2) {
            P.progressive = (m == 0xC2);
            if (have_frame || sl < 6 || seg[0] != 8 || (seg[5] != 3 && seg[5] != 1) || sl != 6 + 3 * (size_t)seg[5]) return 1;
            I.ncomp = seg[5];
            I.H = (seg[1] << 8) | seg[2];
            I.W = (seg[3] << 8) | seg[4];
            // libjpeg stops at 65500 (JPEG_MAX_DIMENSION); a panorama slot (like cv2.remap's source) at 32766
            if (I.W <= 0 || I.H <= 0 || I.W >= 32767 || I.H >= 32767) return 1;
            for (int k = 0; k < I.ncomp; ++k) {
                cid[k] = seg[6 + 3 * k];
                hs[k] = seg[7 + 3 * k] >> 4;
                vs[k] = seg[7 + 3 * k] & 15;
                tq[k] = seg[8 + 3 * k];
                if (tq[k] > 3 || hs[k] < 1 || hs[k] > 4 || vs[k] < 1 || vs[k] > 4) return 1;
            }
            if (I.ncomp == 3 && (cid[0] == cid[1] || cid[0] == cid[2] || cid[1] == cid[2])) return 1;
            for (int k = 0; k < 3; ++k) P.cid[k] = cid[k];
            have_frame = true;
        } else if (m >= 0xC3 && m <= 0xCF) {
            return 1;  // lossless, arithmetic, hierarchical
        } else if (m == 0xDD) {
            if (sl != 2) return 1;
            P.dri = (seg[0] << 8) | seg[1];
        } else if (m == 0xE0) {
            if (sl >= 14 && memcmp(seg, "JFIF\0", 5) == 0) jfif = true;   // jdmarker.c examine_app0 (APP0_DATA_LEN)
        } else if (m == 0xE1) {
            const int o = exif_orientation(seg, sl);
            if (o > 1 || o < 0) return 1;  // cv2.imread rotates / flips such files; -1 = malformed EXIF: leave it to cv2
        } else if (m == 0xEE) {
            if (sl >= 12 && memcmp(seg, "Adobe", 5) == 0) {   // jdmarker.c examine_app14 (APP14_DATA_LEN)
                adobe = true;
                adobe_transform = seg[11];
            }
        } else if (m == 0xDA) {
            const int nc = I.ncomp;
            if (!have_frame) return 1;
            if (P.progressive) {
                // the scans (their headers, the tables between them) are walked by decode_progressive, from this marker on
                if (sl < 6) return 1;
            } else {
                if (sl != 1 + 2 * (size_t)nc + 3 || seg[0] != nc) return 1;
                for (int k = 0; k < nc; ++k) {
                    if (seg[1 + 2 * k] != cid[k]) return 1;
                    P.td[k] = seg[2 + 2 * k] >> 4;
                    P.ta[k] = seg[2 + 2 * k] & 15;
                    if (P.td[k] > 3 || P.ta[k] > 3 || !P.dc[P.td[k]].present || !P.ac[P.ta[k]].present) return 1;
                }
                if (seg[1 + 2 * nc] != 0 || seg[2 + 2 * nc] != 63 || seg[3 + 2 * nc] != 0) return 1;
            }
            const size_t scan_data = P.progressive ? i - L - 2 : i;   // progressive: the SOS marker itself
            if (nc == 1) {
                // a single-component scan is not interleaved: one block per MCU, ceil(W / 8) x ceil(H / 8) blocks whatever
                // sampling factors the frame header declares; the chroma planes are zero coefficients on the same grid
                I.hmax = I.vmax = 1;
                I.mcux = (I.W + 7) / 8;
                I.mcuy = (I.H + 7) / 8;
                if (!have_qt[tq[0]]) return 1;
                size_t off = 0;
                for (int k = 0; k < 3; ++k) {
                    memcpy(I.quant[k], qt[tq[0]], sizeof(I.quant[k]));
                    I.bw[k] = I.mcux;
                    I.bh[k] = I.mcuy;
                    I.coef_off[k] = off;
                    off += (size_t)I.bw[k] * I.bh[k] * 64;
                    P.td[k] = P.td[0];
                    P.ta[k] = P.ta[0];
                }
                I.n_coef = off;
                I.cw = I.W;
                I.ch = I.H;
                P.ecs = scan_data;
                return 0;
            }
            // colour space as libjpeg guesses it (jdapimin.c default_decompress_parms): JFIF -> YCbCr; else the Adobe
            // marker's transform flag (0 = RGB, anything else YCbCr for 3 components); else by component ids
            if (!jfif) {
                if (adobe) {
                    if (adobe_transform == 0) return 1;
                } else if (cid[0] == 'R' && cid[1] == 'G' && cid[2] == 'B') {
                    return 1;
                }
            }
            if (hs[1] != 1 || vs[1] != 1 || hs[2] != 1 || vs[2] != 1) return 1;
            if (!((hs[0] == 1 && vs[0] == 1) || (hs[0] == 2 && vs[0] == 1) || (hs[0] == 2 && vs[0] == 2))) return 1;
            I.hmax = hs[0];
            I.vmax = vs[0];
            I.mcux = (I.W + 8 * I.hmax - 1) / (8 * I.hmax);
            I.mcuy = (I.H + 8 * I.vmax - 1) / (8 * I.vmax);
            size_t off = 0;
            for (int k = 0; k < 3; ++k) {
                if (!have_qt[tq[k]]) return 1;
                memcpy(I.quant[k], qt[tq[k]], sizeof(I.quant[k]));
                I.bw[k] = I.mcux * (k ? 1 : I.hmax);
                I.bh[k] = I.mcuy * (k ? 1 : I.vmax);
                I.coef_off[k] = off;
                off += (size_t)I.bw[k] * I.bh[k] * 64;
            }
            I.n_coef = off;
            I.cw = (I.W + I.hmax - 1) / I.hmax;
            I.ch = (I.H + I.vmax - 1) / I.vmax;
            P.ecs = scan_data;
            return 0;
        }
    }
    return 1;
}

// Progressive files (SOF2; jdphuff.c): the coefficients arrive in several scans - DC first / DC refinement over one or all
// components, AC bands of ONE component as first pass (with end-of-band runs) or refinement pass (correction bits for the
// coefficients that are already non-zero) - with Huffman tables redefined between them.  Decoded here on the calling
// thread into the same coefficient planes as a baseline scan; inverse DCT, upsampling and colour conversion are the
// device kernels.  The rule for anything libjpeg only warns about stays "declined": scans out of the standard progression
// (a refinement whose Ah is not the previous Al, AC before DC), codes that do not exist, a magnitude other than 1 in a
// refinement pass, restart markers out of sequence, bytes between a scan and the next marker.  A file whose scans do not
// bring every coefficient to full precision is declined too: libjpeg then smooths the blocks from their neighbours'
// DC values (jdcoefct.c decompress_smooth_data), which is not restated.  0 = ok, 1 = declined.
struct ProgScan {
    size_t data = 0, end = 0;    // entropy-coded bytes [data, end): `end` is the marker behind them
    int ns = 0, comp[3] = {0, 0, 0};
    int Ss = 0, Se = 0, Ah = 0, Al = 0, dri = 0;
    HuffTable table[3];          // per scan component: its DC table (first DC scan) or its AC table (AC scans)
};

// the entropy-coded data of one scan (jdphuff.c decode_mcu_DC_first / DC_refine / AC_first / AC_refine)
inline int decode_progressive_scan(const uint8_t *d, const Info &I, const ProgScan &S, int16_t *coef) {
    const int ns = S.ns, Ss = S.Ss, Se = S.Se, Ah = S.Ah, Al = S.Al, dri = S.dri;
    const bool dc_scan = (Ss == 0);
    BitReader br;
    br.p = d + S.data;
    br.end = d + S.end;          // (the reader also stops at the marker itself)
    int pred[3] = {0, 0, 0};
    unsigned eobrun = 0;
    int togo = dri, next_rst = 0;
    const bool interleaved = ns > 1;
    const int c0 = S.comp[0];
    // a single-component scan walks the component's own blocks: ceil(width / 8) x ceil(height / 8)
    const int cw = (c0 == 0 || I.ncomp == 1) ? I.W : I.cw, chh = (c0 == 0 || I.ncomp == 1) ? I.H : I.ch;
    const int nx = interleaved ? I.mcux : (cw + 7) / 8, ny = interleaved ? I.mcuy : (chh + 7) / 8;
    const int p1 = 1 << Al, m1 = -(1 << Al);
    auto get_bit = [&]() -> int {
        if (br.n < 1) br.fill();
        const int b = (int)br.peek(1);
        br.skip(1);
        return b;
    };
    for (int my = 0; my < ny; ++my) {
        for (int mx = 0; mx < nx; ++mx) {
            if (dri) {
                if (togo == 0) {
                    if (br.overran()) return 1;
                    br.acc = 0;
                    br.n = 0;
                    br.marker = false;
                    br.zero_bits = 0;
                    while (br.p + 2 <= br.end && br.p[0] == 0xFF && br.p[1] == 0xFF) ++br.p;   // fill bytes
                    if (br.p + 2 > br.end || br.p[0] != 0xFF || br.p[1] != 0xD0 + next_rst) return 1;
                    next_rst = (next_rst + 1) & 7;
                    br.p += 2;
                    pred[0] = pred[1] = pred[2] = 0;
                    eobrun = 0;
                    togo = dri;
                }
                --togo;
            }
            if (dc_scan) {
                for (int k = 0; k < ns; ++k) {
                    const int c = S.comp[k];
                    const int nb = interleaved ? (c ? 1 : I.hmax * I.vmax) : 1;
                    for (int b = 0; b < nb; ++b) {
                        const int by = interleaved ? (c ? my : my * I.vmax + b / I.hmax) : my;
                        const int bx = interleaved ? (c ? mx : mx * I.hmax + b % I.hmax) : mx;
                        int16_t *blk = coef + I.coef_off[c] + ((size_t)by * I.bw[c] + bx) * 64;
                        if (Ah == 0) {
                            if (br.n < 32) br.fill();
                            const int sz = decode_sym(br, S.table[k]);
                            if (sz < 0 || sz > 11) return 1;
                            if (sz) pred[c] += receive_extend(br, sz);
                            blk[0] = (int16_t)(pred[c] * p1);
                        } else if (get_bit()) {
                            blk[0] = (int16_t)(blk[0] | p1);
                        }
                    }
                }
                continue;
            }
            int16_t *blk = coef + I.coef_off[c0] + ((size_t)my * I.bw[c0] + mx) * 64;
            const HuffTable &act = S.table[0];
            if (Ah == 0) {   // decode_mcu_AC_first
                if (eobrun > 0) {
                    --eobrun;
                    continue;
                }
                for (int k = Ss; k <= Se; ++k) {
                    if (br.n < 32) br.fill();
                    const int rs = decode_sym(br, act);
                    if (rs < 0) return 1;
                    const int r = rs >> 4, sz = rs & 15;
                    if (sz) {
                        k += r;
                        if (k > Se) return 1;
                        blk[kNat[k]] = (int16_t)(receive_extend(br, sz) * p1);
                    } else if (r == 15) {
                        k += 15;
                    } else {
                        eobrun = 1u << r;
                        if (r) {
                            eobrun += br.peek(r);
                            br.skip(r);
                        }
                        --eobrun;
                        break;
                    }
                }
                continue;
            }
            // decode_mcu_AC_refine
            int k = Ss;
            if (eobrun == 0) {
                for (; k <= Se; ++k) {
                    if (br.n < 32) br.fill();
                    const int rs = decode_sym(br, act);
                    if (rs < 0) return 1;
                    int r = rs >> 4, sz = rs & 15, val = 0;
                    if (sz) {
                        if (sz != 1) return 1;
                        val = get_bit() ? p1 : m1;
                    } else if (r != 15) {
                        eobrun = 1u << r;
                        if (r) {
                            eobrun += br.peek(r);
                            br.skip(r);
                        }
                        break;
                    }
                    // over the coefficients that are already non-zero (a correction bit each) and r zero ones
                    do {
                        int16_t *cf = blk + kNat[k];
                        if (*cf != 0) {
                            if (get_bit() && (*cf & p1) == 0) *cf = (int16_t)(*cf + (*cf >= 0 ? p1 : m1));
                        } else if (--r < 0) {
                            break;
                        }
                        ++k;
                    } while (k <= Se);
                    if (val) {
                        if (k > Se) return 1;
                        blk[kNat[k]] = (int16_t)val;
                    }
                }
            }
            if (eobrun > 0) {   // the rest of the band: correction bits only
                for (; k <= Se; ++k) {
                    int16_t *cf = blk + kNat[k];
                    if (*cf != 0 && get_bit() && (*cf & p1) == 0) *cf = (int16_t)(*cf + (*cf >= 0 ? p1 : m1));
                }
                --eobrun;
            }
        }
    }
    if (br.overran()) return 1;
    return (size_t)(br.p - d) == S.end ? 0 : 1;   // the reader must stop in front of the marker that ends the scan
}

inline int decode_progressive(const uint8_t *d, size_t len, const Parsed &P, int16_t *coef, bool check_norm) {
    const Info &I = P.info;
    // ---- pass 1: the scan headers in file order - tables in effect, progression checks, where each scan's data ends
    std::vector<HuffTable> dc(P.dc, P.dc + 4), ac(P.ac, P.ac + 4);
    std::vector<ProgScan> scans;
    int dri = P.dri;
    int cbits[3][64];   // jdphuff.c coef_bits: -1 = not seen yet, else the Al of the last scan that covered the coefficient
    for (int c = 0; c < 3; ++c)
        for (int k = 0; k < 64; ++k) cbits[c][k] = -1;
    size_t i = P.ecs;
    bool eoi = false;
    while (i + 2 <= len) {
        if (d[i] != 0xFF) return 1;
        while (i + 1 < len && d[i + 1] == 0xFF) ++i;
        if (i + 2 > len) return 1;
        const int m = d[i + 1];
        i += 2;
        if (m == 0xD9) {
            eoi = true;
            break;
        }
        if (i + 2 > len) return 1;
        const size_t L = ((size_t)d[i] << 8) | d[i + 1];
        if (L < 2 || i + L > len) return 1;
        const uint8_t *seg = d + i + 2;
        const size_t sl = L - 2;
        i += L;
        if (m == 0xC4) {
            if (parse_dht(seg, sl, dc.data(), ac.data())) return 1;
            continue;
        }
        if (m == 0xDD) {
            if (sl != 2) return 1;
            dri = (seg[0] << 8) | seg[1];
            continue;
        }
        if ((m >= 0xE0 && m <= 0xEF) || m == 0xFE) continue;
        if (m != 0xDA) return 1;
        // scan header (jdmarker.c get_sos, jdphuff.c start_pass_phuff_decoder)
        if (scans.size() >= 64) return 1;
        scans.emplace_back();
        ProgScan &S = scans.back();
        const int ns = sl ? seg[0] : 0;
        if (ns < 1 || ns > I.ncomp || sl != 1 + 2 * (size_t)ns + 3) return 1;
        S.ns = ns;
        S.Ss = seg[1 + 2 * ns];
        S.Se = seg[2 + 2 * ns];
        S.Ah = seg[3 + 2 * ns] >> 4;
        S.Al = seg[3 + 2 * ns] & 15;
        S.dri = dri;
        const bool dc_scan = (S.Ss == 0);
        if (dc_scan ? (S.Se != 0) : (ns != 1 || S.Se < S.Ss || S.Se > 63)) return 1;
        if (S.Al > 13 || (S.Ah != 0 && S.Al != S.Ah - 1)) return 1;
        for (int k = 0; k < ns; ++k) {
            int c = -1;
            for (int q = 0; q < I.ncomp; ++q)
                if (P.cid[q] == seg[1 + 2 * k]) c = q;
            if (c < 0 || (k && c <= S.comp[k - 1])) return 1;
            S.comp[k] = c;
            const int td = seg[2 + 2 * k] >> 4, ta = seg[2 + 2 * k] & 15;
            if (td > 3 || ta > 3) return 1;
            int *cb = cbits[c];
            if (!dc_scan && cb[0] < 0) return 1;                           // AC before DC
            for (int z = S.Ss; z <= S.Se; ++z) {
                if (S.Ah != (cb[z] < 0 ? 0 : cb[z])) return 1;             // not the standard progression
                cb[z] = S.Al;
            }
            if (S.Ah == 0 || !dc_scan) {                                   // (a DC refinement reads raw bits only)
                const HuffTable &t = dc_scan ? dc[td] : ac[ta];
                if (!t.present) return 1;
                S.table[k] = t;
            }
        }
        // the scan's data runs to the next marker that is neither a stuffed zero nor a restart marker; `end` is the first
        // 0xFF in front of that marker, fill bytes included (jdmarker.c next_marker skips them), which is where the bit
        // reader stops
        S.data = i;
        size_t e = i;
        for (;;) {
            const uint8_t *ff = static_cast<const uint8_t *>(memchr(d + e, 0xFF, len - e));
            if (!ff) return 1;                                             // no marker behind the scan: truncated
            e = (size_t)(ff - d);
            size_t f = e;                                                  // the last 0xFF of the run
            while (f + 1 < len && d[f + 1] == 0xFF) ++f;
            if (f + 1 >= len) return 1;
            const uint8_t nx = d[f + 1];
            if (nx == 0x00 || (nx >= 0xD0 && nx <= 0xD7)) e = f + 2;
            else break;
        }
        S.end = e;
        i = e;
    }
    if (!eoi) return 1;
    for (int c = 0; c < I.ncomp; ++c)
        for (int k = 0; k < 64; ++k)
            if (cbits[c][k] != 0) return 1;   // not at full precision: libjpeg would smooth (see above)
    // ---- pass 2: DC scans never touch what AC scans touch, and the AC scans of one component only their own planes: up
    // to four independent chains (DC, AC of Y / Cb / Cr), each decoded in file order on its own thread
    std::vector<int> chain[4];
    for (size_t k = 0; k < scans.size(); ++k) chain[scans[k].Ss == 0 ? 0 : 1 + scans[k].comp[0]].push_back((int)k);
    int failed[4] = {0, 0, 0, 0};
    auto run = [&](int c) {
        // every chain clears what it is about to write: the DC chain nothing (the AC chains clear whole planes and finish
        // clearing before any thread decodes: see the barrier below)
        for (int k : chain[c])
            if (!failed[c] && decode_progressive_scan(d, I, scans[(size_t)k], coef)) failed[c] = 1;
    };
    memset(coef, 0, I.n_coef * sizeof(int16_t));
    {
        std::vector<std::thread> th;
        for (int c = 1; c < 4; ++c)
            if (!chain[c].empty()) th.emplace_back(run, c);
        run(0);
        for (auto &t : th) t.join();
    }
    if (failed[0] | failed[1] | failed[2] | failed[3]) return 1;
    if (!check_norm) return 0;   // (the device IDCT kernel makes the same check on the upload path)
    // damaged data shows as blocks no 8-bit encoder produces (see kMaxBlockNorm): libjpeg's SIMD IDCT wraps on them
    for (int c = 0; c < I.ncomp; ++c) {
        float qf[64];
        for (int k = 0; k < 64; ++k) qf[k] = (float)I.quant[c][k];
        const int16_t *blk = coef + I.coef_off[c];
        for (size_t b = 0, nb = (size_t)I.bw[c] * I.bh[c]; b < nb; ++b, blk += 64) {
            float e = 0.f;
            for (int k = 0; k < 64; ++k) {
                const float v = (float)blk[k] * qf[k];
                e += v * v;
            }
            if (e > kMaxBlockNorm * kMaxBlockNorm) return 1;
        }
    }
    return 0;
}

// Huffman-decode the scan into `coef` (int16, natural order, component planes [by][bx][64]).  0 = ok, 1 = damaged.
inline int decode_scan(const uint8_t *d, size_t len, const Parsed &P, int16_t *coef, bool check_norm = true) {
    if (P.progressive) return decode_progressive(d, len, P, coef, check_norm);
    const Info &I = P.info;
    BitReader br;
    br.p = d + P.ecs;
    br.end = d + len;
    int pred[3] = {0, 0, 0};
    const int nblk[3] = {I.hmax * I.vmax, 1, 1};
    if (I.ncomp == 1) memset(coef + I.coef_off[1], 0, (I.n_coef - I.coef_off[1]) * sizeof(int16_t));   // "chroma" of a gray file
    int togo = P.dri;
    int next_rst = 0;   // restart markers must come in sequence: libjpeg resynchronises by its own heuristics otherwise
    for (int my = 0; my < I.mcuy; ++my) {
        for (int mx = 0; mx < I.mcux; ++mx) {
            if (P.dri) {
                if (togo == 0) {
                    // byte-align, expect RSTn
                    if (br.overran()) return 1;
                    br.acc = 0;
                    br.n = 0;
                    br.marker = false;
                    br.zero_bits = 0;
                    while (br.p + 2 <= br.end && br.p[0] == 0xFF && br.p[1] == 0xFF) ++br.p;   // fill bytes (jdmarker.c next_marker)
                    if (br.p + 2 > br.end || br.p[0] != 0xFF || br.p[1] != 0xD0 + next_rst) return 1;
                    next_rst = (next_rst + 1) & 7;
                    br.p += 2;
                    pred[0] = pred[1] = pred[2] = 0;
                    togo = P.dri;
                }
                --togo;
            }
            for (int c = 0; c < I.ncomp; ++c) {
                const HuffTable &dct = P.dc[P.td[c]], &act = P.ac[P.ta[c]];
                for (int b = 0; b < nblk[c]; ++b) {
                    const int by = c ? my : my * I.vmax + b / I.hmax;
                    const int bx = c ? mx : mx * I.hmax + b % I.hmax;
                    int16_t *blk = coef + I.coef_off[c] + ((size_t)by * I.bw[c] + bx) * 64;
                    memset(blk, 0, 128);
                    if (br.n < 32) br.fill();
                    int s = decode_sym(br, dct);
                    if (s < 0 || s > 11) return 1;
                    if (s) pred[c] += receive_extend(br, s);
                    blk[0] = (int16_t)pred[c];
                    const uint16_t *q = I.quant[c];
                    float e = (float)blk[0] * q[0];   // L2 norm of the dequantised block (see kMaxBlockNorm)
                    e *= e;
                    for (int k = 1; k < 64;) {
                        if (br.n < 32) br.fill();
                        const int32_t fa = act.fast_ac[br.peek(kFastBits)];
                        if (fa) {  // short code + small value: one lookup
                            k += (fa >> 4) & 15;
                            if (k > 63) return 1;
                            br.skip(fa & 15);
                            blk[kNat[k]] = (int16_t)(fa >> 8);
                            const float v = (float)(fa >> 8) * q[kNat[k]];
                            e += v * v;
                            ++k;
                            continue;
                        }
                        const int rs = decode_sym(br, act);
                        if (rs < 0) return 1;
                        const int r = rs >> 4;
                        s = rs & 15;
                        if (s == 0) {
                            if (r != 15) break;
                            k += 16;
                            continue;
                        }
                        k += r;
                        if (k > 63) return 1;
                        blk[kNat[k]] = (int16_t)receive_extend(br, s);
                        const float v = (float)blk[kNat[k]] * q[kNat[k]];
                        e += v * v;
                        ++k;
                    }
                    if (e > kMaxBlockNorm * kMaxBlockNorm) return 1;
                }
            }
        }
    }
    if (br.overran()) return 1;   // truncated or damaged scan: libjpeg has its own recovery, leave the file to it
    return 0;
}

// ---- device Huffman decoding (self-synchronising subsequences) ----------------------------------------------------
// A Huffman stream has no random access, but a decoder started at a wrong bit / block position falls back into step
// with the true decoder after a few code words.  So (Weissenberger & Schmidt, "Massively parallel Huffman decoding on
// GPUs", ICPP 2018, adapted to the JPEG block structure): cut the destuffed scan into subsequences of kSubBits bits,
// let one thread decode each from a guessed state (bit position = start of the subsequence, first block of an MCU,
// DC coefficient), record the state it ends in (bit position, block-in-MCU, zigzag index), then repeat "start
// subsequence i + 1 from the end state of subsequence i" until nothing changes - subsequence 0 starts from the true
// state, so a fixed point is the sequential decoder's trajectory.  A prefix sum over the blocks completed per
// subsequence gives every thread its first output block, the last pass writes the coefficients, a scan per component
// turns the DC differences into DC values.  Typical photographs converge in < 10 rounds, white noise at quality 95
// in about 80; past kMaxSyncRounds the host decoder takes over.  Restart intervals are independent scans: every interval
// starts in a known state, subsequences never span them, DC sums restart with them.
__device__ const uint8_t kNatDev[64 + 16] = {
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55,
    62, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63};

constexpr int kSubBits = 1024;
constexpr int kMaxSyncRounds = 192;
constexpr int kRoundsPerCheck = 4;   // synchronisation rounds enqueued per host-side convergence check

// Symbol lists hold up to 256 entries for DC tables too: libjpeg takes any DHT of <= 256 values, a DC table only has to keep
// every value <= 15 (jdhuff.c jpeg_make_d_derived_tbl), so a DC code of 10 bits or more may sit at index 16 or higher.
constexpr int kHuffVals = 256;

struct DevHuff {                 // one per component: its DC and AC table
    uint16_t dc_look[512];
    int32_t dc_maxcode[18], dc_valoff[18];
    uint8_t dc_vals[kHuffVals];
    int32_t ac_fast[1 << kFastBits];
    uint16_t ac_look[512];
    int32_t ac_maxcode[18], ac_valoff[18];
    uint8_t ac_vals[kHuffVals];
};

// Synchronisation rounds only need to know, per code word, how many bits it consumes (code + value bits) and how far it
// moves the zigzag index: one 16-bit entry per 10-bit window, [component][0 = DC, 1 = AC]: consumed | advance << 5
// (advance: 1 for a DC symbol, run + 1 for a coefficient, 16 for ZRL, 64 = end of block); 0 = the code is longer than 10
// bits (or no code): the general path.  12 KB, staged in shared memory by every CTA: DC and AC symbols, ZRL and EOB then
// take ONE code path - the lanes of a warp sit in different decoder states, and with separate paths per state an iteration
// used to cost the sum of all of them.
struct SyncLut {
    uint16_t e[3][2][1 << kFastBits];
    // the same windows for the write pass, which also needs the code length and the size of the value on their own:
    // length | size << 5 | advance << 9
    uint32_t w[3][2][1 << kFastBits];
};

inline void build_sync_lut(const HuffTable &dc, const HuffTable &ac, uint16_t *dc_out, uint16_t *ac_out, uint32_t *dc_w,
                           uint32_t *ac_w) {
    auto symbol = [](const HuffTable &t, int win10, int &len) -> int {
        const uint16_t e = t.look[win10 >> (kFastBits - 9)];
        if (e) {
            len = e >> 8;
            return e & 0xFF;
        }
        if (win10 <= t.maxcode[10]) {   // jdhuff.c: the first length whose largest code is not below the prefix
            len = 10;
            return t.vals[(win10 + t.valoff[10]) & (kHuffVals - 1)];
        }
        return -1;
    };
    for (int i = 0; i < (1 << kFastBits); ++i) {
        int len = 0;
        int s = symbol(dc, i, len);
        if (s >= 0) {
            s = (s > 15) ? 15 : s;
            dc_out[i] = (uint16_t)((len + s) | (1 << 5));
            dc_w[i] = (uint32_t)len | ((uint32_t)s << 5) | (1u << 9);
        } else {
            dc_out[i] = 0;
            dc_w[i] = 0;
        }
        const int rs = symbol(ac, i, len);
        if (rs >= 0) {
            const int r = rs >> 4, sz = rs & 15;
            const int adv = sz ? r + 1 : (r == 15 ? 16 : 64);
            ac_out[i] = (uint16_t)((len + sz) | (adv << 5));
            ac_w[i] = (uint32_t)len | ((uint32_t)sz << 5) | ((uint32_t)adv << 9);
        } else {
            ac_out[i] = 0;
            ac_w[i] = 0;
        }
    }
}

// Everything the device Huffman stage reads of the file's tables, uploaded as one block: the three per-component tables, then
// the unified look-up of the synchronisation rounds and the write pass.  (p2p_jpeg_device_tables exports the same bytes.)
struct DevTables {
    DevHuff T[3];
    SyncLut L;
};

inline void build_device_tables(const Parsed &P, DevTables &DT) {
    memset(&DT, 0, sizeof(DT));
    for (int c = 0; c < 3; ++c) build_sync_lut(P.dc[P.td[c]], P.ac[P.ta[c]], DT.L.e[c][0], DT.L.e[c][1], DT.L.w[c][0], DT.L.w[c][1]);
    for (int c = 0; c < 3; ++c) {
        const HuffTable &d = P.dc[P.td[c]], &a = P.ac[P.ta[c]];
        DevHuff &T = DT.T[c];
        memcpy(T.dc_look, d.look, sizeof(d.look));
        memcpy(T.dc_maxcode, d.maxcode, sizeof(d.maxcode));
        memcpy(T.dc_valoff, d.valoff, sizeof(d.valoff));
        memcpy(T.dc_vals, d.vals, sizeof(T.dc_vals));
        memcpy(T.ac_fast, a.fast_ac, sizeof(a.fast_ac));
        memcpy(T.ac_look, a.look, sizeof(a.look));
        memcpy(T.ac_maxcode, a.maxcode, sizeof(a.maxcode));
        memcpy(T.ac_valoff, a.valoff, sizeof(a.valoff));
        memcpy(T.ac_vals, a.vals, sizeof(T.ac_vals));
    }
}

struct HuffGeom {
    uint32_t n_bits;             // bits of the destuffed scan
    uint32_t n_sub;              // subsequences
    int nb;                      // blocks per MCU (hmax * vmax + 2; 1 for a grayscale file)
    int n_luma;                  // ... of which belong to component 0 (hmax * vmax)
    int hmax, vmax, mcux;
    uint32_t total_blocks;
    int bw[3];
    size_t coef_off[3];
    uint32_t dc_count[3];        // blocks per component
    uint32_t dc_stride;          // per-component stride of the DC difference arrays (multiple of 4)
    // restart intervals (one interval = the whole scan when the file has no restart markers): an interval starts
    // byte-aligned in the true state (first block of an MCU, DC) with DC predictors 0 and holds ivl_blocks blocks
    uint32_t n_ivl;
    uint32_t ivl_blocks;         // blocks per interval (restart_interval * nb); the last interval may hold fewer
};

// per-subsequence layout built on the host: bit range and restart interval; subsequences never span intervals
struct SubSeq {
    uint32_t begin, end;         // bit positions in the destuffed scan
    uint32_t ivl;                // restart interval
    uint32_t first;              // 1 = first subsequence of its interval (its start state is known)
};

// 32 bits of the stream starting at bit `pos` (words are stored big-endian-swapped: MSB = first bit); two zero
// words follow the data
__device__ __forceinline__ uint32_t window32(const uint32_t *__restrict__ w, uint32_t pos) {
    const uint32_t j = pos >> 5, sh = pos & 31;
    return __funnelshift_l(__ldg(w + j + 1), __ldg(w + j), sh);
}

__device__ __forceinline__ int extend_bits(uint32_t v, int s) {   // jdhuff.c HUFF_EXTEND
    return ((int)v < (1 << (s - 1))) ? (int)v - (1 << s) + 1 : (int)v;
}

// symbol and code length for the code at the top of `win`; -1 = no such code (garbage decoding or damaged data):
// it consumes 16 bits
__device__ __forceinline__ int slow_symbol(uint32_t win, const int32_t *maxcode, const int32_t *valoff,
                                           const uint8_t *vals, int &len) {
    const uint32_t w16 = win >> 16;
    for (int l = 10; l <= 16; ++l) {
        const int32_t code = (int32_t)(w16 >> (16 - l));
        if (code <= maxcode[l]) {
            len = l;
            return vals[(code + valoff[l]) & (kHuffVals - 1)];
        }
    }
    len = 16;
    return -1;
}

struct HState {
    uint32_t pos;
    int b, z;
};
__device__ __forceinline__ unsigned long long pack_state(HState s) {
    return ((unsigned long long)s.pos << 16) | ((unsigned long long)(s.b & 0xFF) << 8) | (unsigned long long)(s.z & 0xFF);
}
__device__ __forceinline__ HState unpack_state(unsigned long long v) {
    HState s;
    s.pos = (uint32_t)(v >> 16);
    s.b = (int)((v >> 8) & 0xFF);
    s.z = (int)(v & 0xFF);
    return s;
}

// Decode from state `st` until the bit position reaches `end`.  WRITE: coefficients (natural order, DC = difference)
// go to their block, starting with scan-order block `blk` and stopping at block `blk_limit`; returns the number of blocks
// completed.  The synchronisation passes decode garbage by design and tolerate everything; the WRITE pass follows the
// true trajectory, so what decode_scan declines (no such code, DC category > 11, a coefficient index past 63) is
// damaged data there too: `damaged` is set and the file is left to libjpeg.
template <bool WRITE>
__device__ __forceinline__ uint32_t huff_decode_range(const uint32_t *__restrict__ w, const DevHuff *__restrict__ T,
                                                      const HuffGeom &G, HState &st, uint32_t end, uint32_t blk,
                                                      uint32_t blk_limit, int16_t *__restrict__ coef,
                                                      int32_t *__restrict__ dcdiff, bool &damaged) {
    uint32_t done = 0;
    int16_t *cur = nullptr;
    int comp = (st.b < G.n_luma) ? 0 : st.b - G.n_luma + 1;
    auto locate = [&]() {   // address of the block being written
        const uint32_t mcu = blk / (uint32_t)G.nb;
        const int k = (int)(blk - mcu * (uint32_t)G.nb);
        const uint32_t my = mcu / (uint32_t)G.mcux, mx = mcu - my * (uint32_t)G.mcux;
        const int c = (k < G.n_luma) ? 0 : k - G.n_luma + 1;
        const uint32_t by = c ? my : my * G.vmax + k / G.hmax, bx = c ? mx : mx * G.hmax + k % G.hmax;
        cur = coef + G.coef_off[c] + ((size_t)by * G.bw[c] + bx) * 64;
    };
    if (WRITE && blk < blk_limit) locate();
    while (st.pos < end) {
        if (WRITE && blk >= blk_limit) break;   // the interval's quota is done: the rest are padding bits
        const DevHuff &H = T[comp];
        const uint32_t win = window32(w, st.pos);
        if (st.z == 0) {
            int len, s;
            const uint16_t e = H.dc_look[win >> 23];
            if (e) {
                len = e >> 8;
                s = e & 0xFF;
            } else {
                s = slow_symbol(win, H.dc_maxcode, H.dc_valoff, H.dc_vals, len);
            }
            if (WRITE && (s < 0 || s > 11)) damaged = true;
            s = (s < 0) ? 0 : (s > 15) ? 15 : s;
            if (WRITE) {
                const int diff = s ? extend_bits((win << len) >> (32 - s), s) : 0;
                const uint32_t mcu = blk / (uint32_t)G.nb;
                const int k = (int)(blk - mcu * (uint32_t)G.nb);
                const uint32_t idx = comp ? mcu : mcu * (uint32_t)G.n_luma + (uint32_t)k;
                dcdiff[(size_t)comp * G.dc_stride + idx] = diff;
            }
            st.pos += (uint32_t)(len + s);
            st.z = 1;
            continue;
        }
        const int32_t fa = H.ac_fast[win >> (32 - kFastBits)];
        if (fa) {
            st.z += (fa >> 4) & 15;
            if (WRITE && st.z > 63) damaged = true;
            if (WRITE && st.z < 64) cur[kNatDev[st.z]] = (int16_t)(fa >> 8);
            st.z += 1;
            st.pos += (uint32_t)(fa & 15);
        } else {
            int len, rs;
            const uint16_t e = H.ac_look[win >> 23];
            if (e) {
                len = e >> 8;
                rs = e & 0xFF;
            } else {
                rs = slow_symbol(win, H.ac_maxcode, H.ac_valoff, H.ac_vals, len);
                if (rs < 0) {
                    if (WRITE) damaged = true;
                    rs = 0;
                }
            }
            const int r = rs >> 4, s = rs & 15;
            if (s == 0) {
                st.z = (r == 15) ? st.z + 16 : 64;
                st.pos += (uint32_t)len;
            } else {
                st.z += r;
                if (WRITE && st.z > 63) damaged = true;
                if (WRITE && st.z < 64) cur[kNatDev[st.z]] = (int16_t)extend_bits((win << len) >> (32 - s), s);
                st.z += 1;
                st.pos += (uint32_t)(len + s);
            }
        }
        if (st.z >= 64) {   // block complete
            st.z = 0;
            st.b = (st.b + 1 == G.nb) ? 0 : st.b + 1;
            comp = (st.b < G.n_luma) ? 0 : st.b - G.n_luma + 1;
            ++done;
            if (WRITE) {
                ++blk;
                if (blk < blk_limit) locate();
            }
        }
    }
    return done;
}

// ---- destuffing on the device (files without restart markers) ----------------------------------------------------
// The entropy-coded segment as it sits in the file: every data byte 0xFF is followed by a stuffed 0x00 (removed here);
// 0xFF followed by anything else is a marker or a fill byte, which a scan without restart intervals must not contain
// before its end: `irregular` is raised and the host pass (which knows libjpeg's rules for those) takes over.
// Chunks of 4096 bytes: one CTA, 16 bytes per thread.
constexpr int kDestuffChunk = 4096;

__device__ __forceinline__ uint32_t destuff_flags16(const uint8_t *__restrict__ raw, uint32_t n, uint32_t i0, int *irregular) {
    // bit j of the result: byte i0 + j is a stuffed zero (to be removed)
    uint32_t rem = 0;
    if (i0 >= n) return 0;
    uint8_t prev = i0 ? raw[i0 - 1] : 0;
    bool bad = false;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const uint32_t i = i0 + j;
        if (i < n) {
            const uint8_t b = raw[i];
            if (prev == 0xFF) {
                if (b == 0x00) rem |= 1u << j;
                else bad = true;
            }
            prev = (prev == 0xFF && b == 0x00) ? 0x01 : b;   // the stuffed zero itself is not data
            if (i + 1 == n && b == 0xFF) bad = true;          // a lone 0xFF at the end: fill byte before the marker
        }
    }
    if (bad) *irregular = 1;
    return rem;
}

__global__ void __launch_bounds__(256)
destuff_count_kernel(const uint8_t *__restrict__ raw, uint32_t n, uint32_t *__restrict__ counts, int *__restrict__ irregular) {
    __shared__ uint32_t s_warp[8];
    const uint32_t i0 = blockIdx.x * (uint32_t)kDestuffChunk + threadIdx.x * 16u;
    uint32_t c = __popc(destuff_flags16(raw, n, i0, irregular));
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < 8; ++w) t += s_warp[w];
        counts[blockIdx.x] = t;
    }
}

// kept byte i of the raw segment -> byte (i - removed before i) of the destuffed stream, stored MSB-first inside 32-bit words
__global__ void __launch_bounds__(256)
destuff_scatter_kernel(const uint8_t *__restrict__ raw, uint32_t n, const uint32_t *__restrict__ chunk_off,
                       uint8_t *__restrict__ out) {
    __shared__ uint32_t s_warp[8];
    int unused = 0;
    const uint32_t i0 = blockIdx.x * (uint32_t)kDestuffChunk + threadIdx.x * 16u;
    const uint32_t rem = destuff_flags16(raw, n, i0, &unused);
    const uint32_t c = __popc(rem);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += u;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint32_t before = chunk_off[blockIdx.x] + (inc - c);
    for (int w = 0; w < warp; ++w) before += s_warp[w];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const uint32_t i = i0 + j;
        if (i < n) {
            if (rem & (1u << j)) {
                ++before;
            } else {
                const uint32_t k = i - before;
                out[(k & ~3u) | (3u - (k & 3u))] = raw[i];
            }
        }
    }
}

// the destuffed scan arrives in file byte order; the decoders read 32-bit windows MSB-first
__global__ void __launch_bounds__(256) bswap_words_kernel(uint32_t *__restrict__ w, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) w[i] = __byte_perm(w[i], 0u, 0x0123);
}

// round 0: every subsequence from its guessed state; later rounds: only where the predecessor's end state moved
__global__ void __launch_bounds__(128)
huff_sync_kernel(const uint32_t *__restrict__ w, const DevHuff *__restrict__ T, const HuffGeom G,
                 const SubSeq *__restrict__ sub, unsigned long long *__restrict__ start,
                 unsigned long long *__restrict__ endst, uint32_t *__restrict__ nblk, int first_round,
                 int *__restrict__ changed) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= G.n_sub) return;
    const SubSeq q = sub[i];
    HState st;
    if (first_round) {
        st.pos = q.begin;
        st.b = 0;
        st.z = 0;
        start[i] = pack_state(st);
    } else {
        if (q.first) return;   // the true state: never moves
        const unsigned long long prev = endst[i - 1];
        if (prev == start[i]) return;
        start[i] = prev;
        st = unpack_state(prev);
        *changed = 1;
    }
    bool unused = false;
    nblk[i] = huff_decode_range<false>(w, T, G, st, q.end, 0u, 0u, nullptr, nullptr, unused);
    endst[i] = pack_state(st);
}

// The same rounds with the stream and the unified look-up staged in shared memory (the default; the kernel above is the
// plain form, kept as the yardstick of the tests).  A CTA owns 128 consecutive subsequences = one contiguous piece of the
// stream (<= 4096 + 3 words, skewed by one word per 32 so that lanes at the same offset of their subsequences hit different
// banks); CTAs in which no subsequence has to move leave before staging anything.
constexpr int kSyncThreads = 128;
constexpr int kSyncWords = kSyncThreads * (kSubBits / 32) + 4;

__global__ void __launch_bounds__(kSyncThreads)
huff_sync_fast_kernel(const uint32_t *__restrict__ w, const DevHuff *__restrict__ T, const SyncLut *__restrict__ lut,
                      const HuffGeom G, const SubSeq *__restrict__ sub, unsigned long long *__restrict__ start,
                      unsigned long long *__restrict__ endst, uint32_t *__restrict__ nblk, int first_round,
                      int *__restrict__ changed) {
    __shared__ uint16_t s_lut[3 * 2 * (1 << kFastBits)];
    __shared__ uint32_t s_w[kSyncWords + kSyncWords / 32 + 2];
    const uint32_t i0 = blockIdx.x * kSyncThreads, i = i0 + threadIdx.x;
    bool active = false;
    SubSeq q;
    q.begin = q.end = q.ivl = q.first = 0;
    HState st;
    st.pos = 0;
    st.b = st.z = 0;
    unsigned long long from = 0;
    if (i < G.n_sub) {
        q = sub[i];
        if (first_round) {
            st.pos = q.begin;
            from = pack_state(st);
            active = true;
        } else if (!q.first) {           // the first subsequence of an interval starts in the true state: never moves
            from = endst[i - 1];
            if (from != start[i]) {
                st = unpack_state(from);
                active = true;
            }
        }
    }
    if (!__syncthreads_or(active)) return;
    // stage the look-up (12 KB) and this CTA's piece of the stream
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(lut);
        uint32_t *dst = reinterpret_cast<uint32_t *>(s_lut);
        for (int k = threadIdx.x; k < 3 * 2 * (1 << kFastBits) / 2; k += kSyncThreads) dst[k] = __ldg(src + k);
    }
    const uint32_t i_last = (i0 + kSyncThreads <= G.n_sub ? i0 + kSyncThreads : G.n_sub) - 1;
    const uint32_t wlo = sub[i0].begin >> 5;
    const uint32_t whi = (sub[i_last].end >> 5) + 3;          // a code word may run 27 bits past the end: two more words
    const uint32_t nw = (whi - wlo < (uint32_t)kSyncWords) ? whi - wlo : (uint32_t)kSyncWords;
    for (uint32_t k = threadIdx.x; k < nw; k += kSyncThreads) s_w[k + (k >> 5)] = __ldg(w + wlo + k);
    __syncthreads();
    if (!active) return;
    uint32_t done = 0;
    int comp = (st.b < G.n_luma) ? 0 : st.b - G.n_luma + 1;
    while (st.pos < q.end) {
        const uint32_t j = (st.pos >> 5) - wlo;
        uint32_t win;
        if (j + 1 < nw) {
            win = __funnelshift_l(s_w[j + 1 + ((j + 1) >> 5)], s_w[j + (j >> 5)], st.pos & 31);
        } else {
            win = window32(w, st.pos);   // (cannot happen for a piece within kSyncWords; kept as a guard)
        }
        const uint32_t e = s_lut[((comp << 1) + (st.z != 0)) * (1 << kFastBits) + (win >> (32 - kFastBits))];
        if (e) {
            st.pos += e & 31u;
            st.z += (int)(e >> 5);
        } else {   // a code longer than 10 bits (or none): the general path, one symbol
            const DevHuff &H = T[comp];
            int len;
            if (st.z == 0) {
                int s = slow_symbol(win, H.dc_maxcode, H.dc_valoff, H.dc_vals, len);
                s = (s < 0) ? 0 : (s > 15) ? 15 : s;
                st.pos += (uint32_t)(len + s);
                st.z = 1;
            } else {
                int rs = slow_symbol(win, H.ac_maxcode, H.ac_valoff, H.ac_vals, len);
                rs = (rs < 0) ? 0 : rs;
                const int r = rs >> 4, s = rs & 15;
                st.z += s ? r + 1 : (r == 15 ? 16 : 64);
                st.pos += (uint32_t)(len + s);
            }
        }
        if (st.z >= 64) {   // block complete
            st.z = 0;
            st.b = (st.b + 1 == G.nb) ? 0 : st.b + 1;
            comp = (st.b < G.n_luma) ? 0 : st.b - G.n_luma + 1;
            ++done;
        }
    }
    start[i] = from;
    nblk[i] = done;
    endst[i] = pack_state(st);
    if (!first_round) *changed = 1;
}

// blkoff = exclusive prefix sum of nblk over ALL subsequences; ivl_first[k] = first subsequence of interval k
// (ivl_first[n_ivl] = n_sub).  An interval must hold at least its quota of blocks (the padding bits at its end may
// decode as a few more).
__global__ void __launch_bounds__(256)
huff_check_kernel(const uint32_t *__restrict__ blkoff, const uint32_t *__restrict__ nblk,
                  const uint32_t *__restrict__ ivl_first, const HuffGeom G, int *__restrict__ bad) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= G.n_ivl) return;
    const uint32_t a = ivl_first[k], b = ivl_first[k + 1];
    const uint32_t got = (b == G.n_sub ? blkoff[b - 1] + nblk[b - 1] : blkoff[b]) - blkoff[a];
    const uint32_t first_blk = k * G.ivl_blocks;
    const uint32_t quota = (first_blk + G.ivl_blocks <= G.total_blocks) ? G.ivl_blocks : G.total_blocks - first_blk;
    if (got < quota || got > quota + 8u) *bad = 1;
}

// Optimistic enqueue: the host queues a fixed number of rounds, the block-count check, the write pass and everything
// after it without waiting for any of them; this one-thread kernel decides on the device whether the write pass may run
// (the last queued round moved nothing = fixed point reached, and every interval holds its quota of blocks) and leaves
// the same verdict where the host finds it after its single wait: 1 = go, 0 = not converged yet (the host queues more
// rounds), -1 = block counts off (the host decoder takes the file).
__global__ void huff_gate_kernel(const int *__restrict__ changed_last, const int *__restrict__ bad, int *__restrict__ gate_dev,
                                 int *__restrict__ gate_host) {
    const int v = *changed_last ? 0 : (*bad ? -1 : 1);
    *gate_dev = (v == 1);
    *gate_host = v;
}

__global__ void __launch_bounds__(128)
huff_write_kernel(const uint32_t *__restrict__ w, const DevHuff *__restrict__ T, const HuffGeom G,
                  const SubSeq *__restrict__ sub, const uint32_t *__restrict__ ivl_first,
                  const unsigned long long *__restrict__ start, const uint32_t *__restrict__ blkoff,
                  int16_t *__restrict__ coef, int32_t *__restrict__ dcdiff, int *__restrict__ damaged_flag,
                  const int *__restrict__ gate) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= G.n_sub) return;
    if (gate && !*gate) return;   // optimistic enqueue: the rounds before did not converge / the block counts are off
    const SubSeq q = sub[i];
    HState st = unpack_state(start[i]);
    // scan-order index of the block in progress: interval base + blocks completed earlier in this interval
    const uint32_t first_blk = q.ivl * G.ivl_blocks;
    const uint32_t blk = first_blk + (blkoff[i] - blkoff[ivl_first[q.ivl]]);
    const uint32_t limit = (first_blk + G.ivl_blocks <= G.total_blocks) ? first_blk + G.ivl_blocks : G.total_blocks;
    bool damaged = false;
    huff_decode_range<true>(w, T, G, st, q.end, blk, limit, coef, dcdiff, damaged);
    // the last block of an interval must end inside it: libjpeg feeds zero bits past a marker, this reader would
    // continue into the next interval
    if (i + 1 == ivl_first[q.ivl + 1] && st.pos > q.end) damaged = true;
    if (damaged) *damaged_flag = 1;
}

// The write pass with the stream and the (length, size, advance) look-up staged in shared memory like the fast rounds.
// Same trajectory, same stores, same "damaged" conditions as huff_decode_range<true>.
__global__ void __launch_bounds__(kSyncThreads)
huff_write_fast_kernel(const uint32_t *__restrict__ w, const DevHuff *__restrict__ T, const SyncLut *__restrict__ lut,
                       const HuffGeom G, const SubSeq *__restrict__ sub, const uint32_t *__restrict__ ivl_first,
                       const unsigned long long *__restrict__ start, const uint32_t *__restrict__ blkoff,
                       int16_t *__restrict__ coef, int32_t *__restrict__ dcdiff, int *__restrict__ damaged_flag,
                       const int *__restrict__ gate) {
    __shared__ uint32_t s_lut[3 * 2 * (1 << kFastBits)];
    __shared__ uint32_t s_w[kSyncWords + kSyncWords / 32 + 2];
    if (gate && !*gate) return;   // optimistic enqueue (see huff_gate_kernel): uniform over the grid
    const uint32_t i0 = blockIdx.x * kSyncThreads, i = i0 + threadIdx.x;
    for (int k = threadIdx.x; k < 3 * 2 * (1 << kFastBits); k += kSyncThreads) s_lut[k] = __ldg(&lut->w[0][0][0] + k);
    const uint32_t i_last = (i0 + kSyncThreads <= G.n_sub ? i0 + kSyncThreads : G.n_sub) - 1;
    const uint32_t wlo = sub[i0].begin >> 5;
    const uint32_t whi = (sub[i_last].end >> 5) + 3;
    const uint32_t nw = (whi - wlo < (uint32_t)kSyncWords) ? whi - wlo : (uint32_t)kSyncWords;
    for (uint32_t k = threadIdx.x; k < nw; k += kSyncThreads) s_w[k + (k >> 5)] = __ldg(w + wlo + k);
    __syncthreads();
    if (i >= G.n_sub) return;
    const SubSeq q = sub[i];
    HState st = unpack_state(start[i]);
    const uint32_t first_blk = q.ivl * G.ivl_blocks;
    uint32_t blk = first_blk + (blkoff[i] - blkoff[ivl_first[q.ivl]]);
    const uint32_t blk_limit = (first_blk + G.ivl_blocks <= G.total_blocks) ? first_blk + G.ivl_blocks : G.total_blocks;
    bool damaged = false;
    int16_t *cur = nullptr;
    int comp = (st.b < G.n_luma) ? 0 : st.b - G.n_luma + 1;
    uint32_t dc_idx = 0;
    auto locate = [&]() {   // address of the block being written, index of its DC difference
        const uint32_t mcu = blk / (uint32_t)G.nb;
        const int k = (int)(blk - mcu * (uint32_t)G.nb);
        const uint32_t my = mcu / (uint32_t)G.mcux, mx = mcu - my * (uint32_t)G.mcux;
        const int c = (k < G.n_luma) ? 0 : k - G.n_luma + 1;
        const uint32_t by = c ? my : my * G.vmax + k / G.hmax, bx = c ? mx : mx * G.hmax + k % G.hmax;
        cur = coef + G.coef_off[c] + ((size_t)by * G.bw[c] + bx) * 64;
        dc_idx = c ? mcu : mcu * (uint32_t)G.n_luma + (uint32_t)k;
    };
    if (blk < blk_limit) locate();
    while (st.pos < q.end) {
        if (blk >= blk_limit) break;   // the interval's quota is done: the rest are padding bits
        const uint32_t j = (st.pos >> 5) - wlo;
        const uint32_t win = (j + 1 < nw) ? __funnelshift_l(s_w[j + 1 + ((j + 1) >> 5)], s_w[j + (j >> 5)], st.pos & 31)
                                          : window32(w, st.pos);
        const uint32_t e = s_lut[((comp << 1) + (st.z != 0)) * (1 << kFastBits) + (win >> (32 - kFastBits))];
        if (e) {
            const int len = (int)(e & 31u), sz = (int)((e >> 5) & 15u), adv = (int)(e >> 9);
            const int val = sz ? extend_bits((win << len) >> (32 - sz), sz) : 0;
            if (st.z == 0) {
                if (sz > 11) damaged = true;
                dcdiff[(size_t)comp * G.dc_stride + dc_idx] = val;
                st.z = 1;
            } else {
                const int zc = st.z + adv - 1;          // zigzag position of this coefficient
                if (sz) {
                    if (zc > 63) damaged = true;
                    else cur[kNatDev[zc]] = (int16_t)val;
                }
                st.z += adv;
            }
            st.pos += (uint32_t)(len + sz);
        } else {   // a code longer than 10 bits (or none): the general path, one symbol
            const DevHuff &H = T[comp];
            int len;
            if (st.z == 0) {
                int s = slow_symbol(win, H.dc_maxcode, H.dc_valoff, H.dc_vals, len);
                if (s < 0 || s > 11) damaged = true;
                s = (s < 0) ? 0 : (s > 15) ? 15 : s;
                dcdiff[(size_t)comp * G.dc_stride + dc_idx] = s ? extend_bits((win << len) >> (32 - s), s) : 0;
                st.pos += (uint32_t)(len + s);
                st.z = 1;
            } else {
                int rs = slow_symbol(win, H.ac_maxcode, H.ac_valoff, H.ac_vals, len);
                if (rs < 0) {
                    damaged = true;
                    rs = 0;
                }
                const int r = rs >> 4, s = rs & 15;
                if (s == 0) {
                    st.z = (r == 15) ? st.z + 16 : 64;
                    st.pos += (uint32_t)len;
                } else {
                    st.z += r;
                    if (st.z > 63) damaged = true;
                    if (st.z < 64) cur[kNatDev[st.z]] = (int16_t)extend_bits((win << len) >> (32 - s), s);
                    st.z += 1;
                    st.pos += (uint32_t)(len + s);
                }
            }
        }
        if (st.z >= 64) {   // block complete
            st.z = 0;
            st.b = (st.b + 1 == G.nb) ? 0 : st.b + 1;
            comp = (st.b < G.n_luma) ? 0 : st.b - G.n_luma + 1;
            ++blk;
            if (blk < blk_limit) locate();
        }
    }
    // the last block of an interval must end inside it (see huff_write_kernel)
    if (i + 1 == ivl_first[q.ivl + 1] && st.pos > q.end) damaged = true;
    if (damaged) *damaged_flag = 1;
}

// DC value of block idx of component c = sum of the differences since the start of its restart interval
// (dcsum holds the exclusive sums over the whole scan)
__global__ void __launch_bounds__(256)
huff_dc_kernel(const int32_t *__restrict__ dcdiff, const uint32_t *__restrict__ dcsum, const HuffGeom G,
               int16_t *__restrict__ coef) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = blockIdx.y;
    if (idx >= G.dc_count[c]) return;
    const uint32_t per = c ? 1u : (uint32_t)G.n_luma;              // blocks of this component per MCU
    const uint32_t seg = (G.ivl_blocks / (uint32_t)G.nb) * per;      // ... and per restart interval
    const uint32_t seg0 = (idx / seg) * seg;
    const size_t base = (size_t)c * G.dc_stride;
    const int dc = (int)(dcsum[base + idx] - dcsum[base + seg0]) + dcdiff[base + idx];
    uint32_t by, bx;
    if (c) {
        by = idx / (uint32_t)G.mcux;
        bx = idx - by * (uint32_t)G.mcux;
    } else {
        const uint32_t mcu = idx / per, k = idx - mcu * per;
        const uint32_t my = mcu / (uint32_t)G.mcux, mx = mcu - my * (uint32_t)G.mcux;
        by = my * G.vmax + k / G.hmax;
        bx = mx * G.hmax + k % G.hmax;
    }
    coef[G.coef_off[c] + ((size_t)by * G.bw[c] + bx) * 64] = (int16_t)dc;
}

// ---- device: IDCT ---------------------------------------------------------------------------------------------------
// jidctint.c: one 8-point pass; `in` are the 8 inputs, outputs descaled by N bits
template <int N>
__device__ __forceinline__ void idct_pass(const int *in, int *out) {
    int z2 = in[2], z3 = in[6];
    int z1 = (z2 + z3) * 4433;
    int tmp2 = z1 + z3 * -15137;
    int tmp3 = z1 + z2 * 6270;
    z2 = in[0];
    z3 = in[4];
    int tmp0 = (z2 + z3) << 13, tmp1 = (z2 - z3) << 13;
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    tmp0 = in[7];
    tmp1 = in[5];
    tmp2 = in[3];
    tmp3 = in[1];
    z1 = tmp0 + tmp3;
    z2 = tmp1 + tmp2;
    z3 = tmp0 + tmp2;
    int z4 = tmp1 + tmp3;
    const int z5 = (z3 + z4) * 9633;
    tmp0 *= 2446;
    tmp1 *= 16819;
    tmp2 *= 25172;
    tmp3 *= 12299;
    z1 *= -7373;
    z2 *= -20995;
    z3 = z3 * -16069 + z5;
    z4 = z4 * -3196 + z5;
    tmp0 += z1 + z3;
    tmp1 += z2 + z4;
    tmp2 += z2 + z3;
    tmp3 += z1 + z4;
    constexpr int R = 1 << (N - 1);
    out[0] = (tmp10 + tmp3 + R) >> N;
    out[7] = (tmp10 - tmp3 + R) >> N;
    out[1] = (tmp11 + tmp2 + R) >> N;
    out[6] = (tmp11 - tmp2 + R) >> N;
    out[2] = (tmp12 + tmp1 + R) >> N;
    out[5] = (tmp12 - tmp1 + R) >> N;
    out[3] = (tmp13 + tmp0 + R) >> N;
    out[4] = (tmp13 - tmp0 + R) >> N;
}

struct Quant {
    uint16_t q[64];
};

// 8 threads per block, 32 blocks per CTA; plane[(by * 8 + r) * pitch + bx * 8 + c]
__global__ void __launch_bounds__(256)
jpegdec_idct_kernel(const int16_t *__restrict__ coef, uint8_t *__restrict__ plane, const __grid_constant__ Quant Q,
                    int n_blocks, int bw, int pitch, int *__restrict__ out_of_range) {
    __shared__ int ws[32][8][9];
    const int lb = threadIdx.x >> 3, l8 = threadIdx.x & 7;
    const int blk = blockIdx.x * 32 + lb;
    const bool live = blk < n_blocks;
    int in[8], out[8];
    if (live) {
        const int16_t *c = coef + (size_t)blk * 64;
#pragma unroll
        for (int k = 0; k < 8; ++k) in[k] = (int)c[k * 8 + l8] * (int)Q.q[k * 8 + l8];   // column l8
        // damaged data check (kMaxBlockNorm)
        float e = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) e += (float)in[k] * (float)in[k];
        const unsigned group = 0xFFu << (threadIdx.x & 24);   // the 8 lanes of this block
        e += __shfl_xor_sync(group, e, 1);
        e += __shfl_xor_sync(group, e, 2);
        e += __shfl_xor_sync(group, e, 4);
        if (l8 == 0 && e > kMaxBlockNorm * kMaxBlockNorm) *out_of_range = 1;
        idct_pass<13 - 2>(in, out);
#pragma unroll
        for (int k = 0; k < 8; ++k) ws[lb][k][l8] = out[k];
    }
    __syncthreads();
    if (live) {
#pragma unroll
        for (int k = 0; k < 8; ++k) in[k] = ws[lb][l8][k];                                 // row l8
        idct_pass<13 + 2 + 3>(in, out);
        uint32_t lo = 0, hi = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            lo |= (uint32_t)min(max(out[k] + 128, 0), 255) << (8 * k);
            hi |= (uint32_t)min(max(out[k + 4] + 128, 0), 255) << (8 * k);
        }
        const int by = blk / bw, bx = blk - by * bw;
        *reinterpret_cast<uint2 *>(plane + (size_t)(by * 8 + l8) * pitch + bx * 8) = make_uint2(lo, hi);
    }
}

// ---- device: upsampling + colour conversion -------------------------------------------------------------------------
struct ColorParams {
    const uint8_t *y, *cb, *cr;   // component planes (pitch = blocks per row * 8)
    int pitch_y, pitch_c;
    int W, H, hmax, vmax, cw, ch;
    uint8_t *bgr;                 // output rows (PACKED = false)
    size_t stride;
    // PACKED = true: straight into the slot's panorama layout (what pack_kernel makes of a BGR image): RGBA-packed texels,
    // pitch_tex per row, column W repeats column 0, row H repeats row H - 1, and the gather array through its surface
    uint32_t *rgba;
    int pitch_tex;
    cudaSurfaceObject_t surf;
};

// chroma sample of output pixel (x, y): jdsample.c fancy upsampling (or replication for planes <= 2 samples wide)
__device__ __forceinline__ int chroma_at(const uint8_t *__restrict__ c, int pitch, int x, int y, const ColorParams &P) {
    if (P.hmax == 1) return c[(size_t)y * pitch + x];
    const int cx = x >> 1;
    if (P.cw <= 2) {  // h2v1_upsample / h2v2_upsample: plain replication
        const int cy = (P.vmax == 2) ? (y >> 1) : y;
        return c[(size_t)cy * pitch + cx];
    }
    if (P.vmax == 1) {  // h2v1_fancy_upsample
        const uint8_t *r = c + (size_t)y * pitch;
        const int v = r[cx];
        if (x & 1) return (cx == P.cw - 1) ? v : (3 * v + r[cx + 1] + 2) >> 2;
        return (cx == 0) ? v : (3 * v + r[cx - 1] + 1) >> 2;
    }
    // h2v2_fancy_upsample: nearer row weighs 3, the other 1; context rows replicate at the image edges
    const int cy = y >> 1;
    int fy = (y & 1) ? cy + 1 : cy - 1;
    fy = min(max(fy, 0), P.ch - 1);
    const uint8_t *r0 = c + (size_t)cy * pitch, *r1 = c + (size_t)fy * pitch;
    const int cs = 3 * r0[cx] + r1[cx];
    if (x & 1) {
        if (cx == P.cw - 1) return (cs * 4 + 7) >> 4;
        return (cs * 3 + (3 * r0[cx + 1] + r1[cx + 1]) + 7) >> 4;
    }
    if (cx == 0) return (cs * 4 + 8) >> 4;
    return (cs * 3 + (3 * r0[cx - 1] + r1[cx - 1]) + 8) >> 4;
}

// thread per 4 output pixels of a row: 12 bytes = 3 words when the row can take word stores; PACKED: one 16-byte store
// of packed texels (+ the surface write), the staging image and the pack kernel are skipped (100 MB written and read
// again per 8K file)
template <bool PACKED>
__global__ void __launch_bounds__(256)
jpegdec_color_kernel(const __grid_constant__ ColorParams P) {
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int y = blockIdx.y;
    if (x0 >= P.W) return;
    uint32_t px[4] = {0u, 0u, 0u, 0u};
    const int n = (P.W - x0 < 4) ? P.W - x0 : 4;
    for (int i = 0; i < n; ++i) {
        const int x = x0 + i;
        const int yy = P.y[(size_t)y * P.pitch_y + x];
        const int cb = chroma_at(P.cb, P.pitch_c, x, y, P) - 128, cr = chroma_at(P.cr, P.pitch_c, x, y, P) - 128;
        // jdcolor.c build_ycc_rgb_table / ycc_rgb_convert
        const int r = yy + ((91881 * cr + 32768) >> 16);
        const int b = yy + ((116130 * cb + 32768) >> 16);
        const int g = yy + ((-22554 * cb + 32768 - 46802 * cr) >> 16);
        px[i] = (uint32_t)min(max(b, 0), 255) | ((uint32_t)min(max(g, 0), 255) << 8) | ((uint32_t)min(max(r, 0), 255) << 16);
    }
    if (PACKED) {
        uint32_t *drow = P.rgba + (size_t)y * P.pitch_tex;
        const bool last_row = (y == P.H - 1);   // the clamp row below the image repeats it
        if (n == 4) {
            const uint4 o = make_uint4(px[0], px[1], px[2], px[3]);
            *reinterpret_cast<uint4 *>(drow + x0) = o;
            if (last_row) *reinterpret_cast<uint4 *>(drow + P.pitch_tex + x0) = o;
            if (P.surf != 0) surf2Dwrite(o, P.surf, x0 * 4, y);
        } else {
            for (int i = 0; i < n; ++i) {
                drow[x0 + i] = px[i];
                if (last_row) drow[P.pitch_tex + x0 + i] = px[i];
                if (P.surf != 0) surf2Dwrite(px[i], P.surf, (x0 + i) * 4, y);
            }
        }
        if (x0 == 0) {                          // the wrap column behind the row repeats column 0
            drow[P.W] = px[0];
            if (last_row) drow[P.pitch_tex + P.W] = px[0];
        }
        return;
    }
    uint8_t *o = P.bgr + (size_t)y * P.stride + (size_t)x0 * 3;
    if (n == 4 && (P.stride & 3) == 0) {
        uint32_t *w = reinterpret_cast<uint32_t *>(o);
        w[0] = px[0] | (px[1] << 24);
        w[1] = (px[1] >> 8) | (px[2] << 16);
        w[2] = (px[2] >> 16) | (px[3] << 8);
    } else {
        for (int i = 0; i < n; ++i) {
            o[3 * i] = (uint8_t)px[i];
            o[3 * i + 1] = (uint8_t)(px[i] >> 8);
            o[3 * i + 2] = (uint8_t)(px[i] >> 16);
        }
    }
}

}  // namespace p2pjdec
