// jpeg.cu — see jpeg.h.  Host: JFIF marker parse + baseline Huffman decode (ITU-T T.81 Annex B, F.2.2).  Device:
// the sample reconstruction exactly as libjpeg / libjpeg-turbo does it with the defaults PIL leaves in place
// (reference server/detector.py:128-133 reaches them through Image.open + np.array):
//   * jpeg_idct_islow    (jidctint.c)  13-bit fixed-point Loeffler-Ligtenberg-Moschytz IDCT, two passes
//   * h2v1 / h2v2 "fancy" upsampling (jdsample.c)  3:1 triangle filter, edge columns/rows replicated
//   * ycc_rgb_convert    (jdcolor.c)   16.16 fixed-point tables, G built from the two chroma products summed
//                                      before the shift
// libjpeg is a dependency of PIL, not part of the reference tree; the test oracle (ref_jpeg) restates the same
// published algorithm in numpy and both are pinned against PIL's output in tests/test_jpeg.py.
#include "jpeg.h"

#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

namespace fd {

// ------------------------------------------------------------------------------------------- host: parse
namespace {

const uint8_t kNatural[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                              41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                              30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

int say(int status, char* why, size_t cap, const char* fmt, ...) {
    if (why && cap) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(why, cap, fmt, ap);
        va_end(ap);
    }
    return status;
}

// T.81 Annex C (code generation) + F.2.2.3 (decoder tables)
bool derive(HuffTable& h, bool is_ac) {
    int total = 0;
    for (int l = 1; l <= 16; ++l) total += h.bits[l];
    if (total > 256) return false;
    memset(h.lut, 0, sizeof(h.lut));
    unsigned code = 0;
    int p = 0, longest = 0;
    for (int l = 1; l <= 16; ++l)
        if (h.bits[l]) longest = l;
    for (int l = 1; l <= 16; ++l) {
        h.valoffset[l] = p - static_cast<int>(code);
        for (int i = 0; i < h.bits[l]; ++i, ++p, ++code) {
            if (code >= (1u << l)) return false;  // more codes than the length can hold
            if (l <= 9) {
                const unsigned first = code << (9 - l), count = 1u << (9 - l);
                for (unsigned k = 0; k < count; ++k) h.lut[first + k] = static_cast<uint16_t>((l << 8) | h.vals[p]);
            }
        }
        // libjpeg (jpeg_make_d_derived_tbl) also rejects a length whose codes use up the whole code space, all-ones
        // code included: "Bogus Huffman table definition", which PIL reports as a broken data stream
        if (l <= longest && code >= (1u << l)) return false;
        h.maxcode[l] = h.bits[l] ? static_cast<int>(code) - 1 : -1;
        code <<= 1;
    }
    h.maxcode[17] = 0x7fffffff;
    // AC shortcut: where code + magnitude bits fit in the look-ahead, precompute (value << 8) | (run << 4) | total bits
    for (unsigned i = 0; is_ac && i < 512; ++i) {
        const unsigned e = h.lut[i];
        if (!e) continue;
        const int len = e >> 8, run = (e >> 4) & 15, mag = e & 15;
        if (mag == 0 || len + mag > 9) continue;
        int v = static_cast<int>((i >> (9 - len - mag)) & ((1u << mag) - 1));
        if (v < (1 << (mag - 1))) v += -(1 << mag) + 1;
        if (v >= -128 && v <= 127) h.fast_ac[i] = static_cast<int16_t>(v * 256 + run * 16 + len + mag);
    }
    return true;
}

inline unsigned be16(const uint8_t* p) { return (unsigned(p[0]) << 8) | p[1]; }

}  // namespace

int jpeg_parse(const uint8_t* d, size_t len, JpegInfo* info, char* why, size_t cap) {
    if (!d || len < 4 || d[0] != 0xFF || d[1] != 0xD8) return say(JPEG_NOT_JPEG, why, cap, "no SOI marker");
    JpegInfo& J = *info;
    memset(&J, 0, sizeof(J));
    uint16_t qt[4][64];
    bool have_qt[4] = {false, false, false, false};
    int comp_id[3] = {0, 0, 0}, comp_tq[3] = {0, 0, 0}, comp_h[3] = {0, 0, 0}, comp_v[3] = {0, 0, 0};
    bool have_sof = false, jfif = false, adobe = false;
    int adobe_transform = -1;
    size_t pos = 2;
    while (true) {
        if (pos + 2 > len) return say(JPEG_CORRUPT, why, cap, "ran out of data before SOS");
        if (d[pos] != 0xFF) return say(JPEG_CORRUPT, why, cap, "expected a marker at byte %zu", pos);
        while (pos < len && d[pos] == 0xFF) ++pos;  // fill bytes
        if (pos >= len) return say(JPEG_CORRUPT, why, cap, "ran out of data before SOS");
        const int m = d[pos++];
        if (m == 0x01 || m == 0x00) return say(JPEG_CORRUPT, why, cap, "unexpected marker 0x%02x", m);
        if (m >= 0xD0 && m <= 0xD7) return say(JPEG_CORRUPT, why, cap, "restart marker outside a scan");
        if (m == 0xD8) return say(JPEG_CORRUPT, why, cap, "second SOI");
        if (m == 0xD9) return say(JPEG_CORRUPT, why, cap, "EOI before any scan");
        if (pos + 2 > len) return say(JPEG_CORRUPT, why, cap, "truncated marker segment");
        const size_t L = be16(d + pos);
        if (L < 2 || pos + L > len) return say(JPEG_CORRUPT, why, cap, "marker 0x%02x: bad segment length", m);
        const uint8_t* s = d + pos + 2;
        const size_t n = L - 2;
        pos += L;
        if (m == 0xC0 || m == 0xC1) {  // baseline / extended-sequential Huffman
            if (have_sof) return say(JPEG_CORRUPT, why, cap, "second SOF");
            if (n < 6) return say(JPEG_CORRUPT, why, cap, "short SOF");
            if (s[0] != 8) return say(JPEG_UNSUPPORTED, why, cap, "%d-bit samples", s[0]);
            J.height = be16(s + 1);
            J.width = be16(s + 3);
            J.ncomp = s[5];
            if (J.height == 0) return say(JPEG_UNSUPPORTED, why, cap, "height given by a DNL marker");
            if (J.width == 0) return say(JPEG_CORRUPT, why, cap, "zero width");
            if (J.ncomp != 3) return say(JPEG_UNSUPPORTED, why, cap, "%d components (only 3-component YCbCr on the device)", J.ncomp);
            if (n != size_t(6 + 3 * J.ncomp)) return say(JPEG_CORRUPT, why, cap, "SOF length");
            for (int c = 0; c < 3; ++c) {
                comp_id[c] = s[6 + 3 * c];
                comp_h[c] = s[7 + 3 * c] >> 4;
                comp_v[c] = s[7 + 3 * c] & 15;
                comp_tq[c] = s[8 + 3 * c];
                if (comp_tq[c] > 3) return say(JPEG_CORRUPT, why, cap, "quantisation table id %d", comp_tq[c]);
            }
            have_sof = true;
        } else if ((m >= 0xC2 && m <= 0xCF) && m != 0xC4 && m != 0xC8 && m != 0xCC) {
            return say(JPEG_UNSUPPORTED, why, cap, "SOF%d (progressive / lossless / arithmetic)", m - 0xC0);
        } else if (m == 0xCC) {
            return say(JPEG_UNSUPPORTED, why, cap, "arithmetic coding");
        } else if (m == 0xDB) {  // DQT
            size_t o = 0;
            while (o < n) {
                const int pq = s[o] >> 4, tq = s[o] & 15;
                if (tq > 3 || pq > 1) return say(JPEG_CORRUPT, why, cap, "DQT header");
                const size_t need = 1 + 64 * size_t(pq + 1);
                if (o + need > n) return say(JPEG_CORRUPT, why, cap, "short DQT");
                for (int z = 0; z < 64; ++z)
                    qt[tq][kNatural[z]] = pq ? static_cast<uint16_t>(be16(s + o + 1 + 2 * z)) : s[o + 1 + z];
                have_qt[tq] = true;
                o += need;
            }
        } else if (m == 0xC4) {  // DHT
            size_t o = 0;
            while (o < n) {
                if (o + 17 > n) return say(JPEG_CORRUPT, why, cap, "short DHT");
                const int tc = s[o] >> 4, th = s[o] & 15;
                if (tc > 1 || th > 3) return say(JPEG_CORRUPT, why, cap, "DHT header");
                HuffTable& H = tc ? J.ac[th] : J.dc[th];
                memset(&H, 0, sizeof(H));
                int total = 0;
                for (int l = 1; l <= 16; ++l) { H.bits[l] = s[o + l]; total += H.bits[l]; }
                if (total > 256 || o + 17 + total > n) return say(JPEG_CORRUPT, why, cap, "DHT counts");
                memcpy(H.vals, s + o + 17, total);
                if (!derive(H, tc == 1)) return say(JPEG_CORRUPT, why, cap, "DHT codes do not fit");
                H.present = true;
                o += 17 + total;
            }
        } else if (m == 0xDD) {
            if (n != 2) return say(JPEG_CORRUPT, why, cap, "DRI length");
            J.restart_interval = be16(s);
        } else if (m == 0xE0) {
            if (n >= 5 && !memcmp(s, "JFIF\0", 5)) {
                if (n < 14) return say(JPEG_UNSUPPORTED, why, cap, "short JFIF segment");  // PIL reads version, units and density
                jfif = true;
            }
        } else if (m == 0xEE) {
            if (n >= 12 && !memcmp(s, "Adobe", 5)) { adobe = true; adobe_transform = s[11]; }
        } else if (m == 0xDA) {  // SOS
            if (!have_sof) return say(JPEG_CORRUPT, why, cap, "SOS before SOF");
            if (n < 1) return say(JPEG_CORRUPT, why, cap, "short SOS");
            const int ns = s[0];
            if (ns != 3) return say(JPEG_UNSUPPORTED, why, cap, "non-interleaved scan (%d of 3 components)", ns);
            if (n != size_t(4 + 2 * ns)) return say(JPEG_CORRUPT, why, cap, "SOS length");
            for (int c = 0; c < 3; ++c) {
                if (s[1 + 2 * c] != comp_id[c]) return say(JPEG_UNSUPPORTED, why, cap, "scan component order differs from the frame's");
                J.dc_tbl[c] = s[2 + 2 * c] >> 4;
                J.ac_tbl[c] = s[2 + 2 * c] & 15;
                if (J.dc_tbl[c] > 3 || J.ac_tbl[c] > 3) return say(JPEG_CORRUPT, why, cap, "SOS table id");
                if (!J.dc[J.dc_tbl[c]].present || !J.ac[J.ac_tbl[c]].present) return say(JPEG_CORRUPT, why, cap, "scan uses an undefined Huffman table");
                {   // libjpeg validates the DC symbols of the tables a scan uses when the scan starts
                    const HuffTable& D = J.dc[J.dc_tbl[c]];
                    int total = 0;
                    for (int l = 1; l <= 16; ++l) total += D.bits[l];
                    for (int i = 0; i < total; ++i)
                        if (D.vals[i] > 15) return say(JPEG_CORRUPT, why, cap, "DC Huffman table holds a category above 15");
                }
                if (!have_qt[comp_tq[c]]) return say(JPEG_CORRUPT, why, cap, "component uses an undefined quantisation table");
                memcpy(J.q[c], qt[comp_tq[c]], sizeof(J.q[c]));
            }
            if (s[1 + 2 * ns] != 0 || s[2 + 2 * ns] != 63 || s[3 + 2 * ns] != 0) return say(JPEG_UNSUPPORTED, why, cap, "spectral selection / successive approximation in a sequential scan");
            // colour space as libjpeg guesses it (jdapimin.c default_decompress_parms)
            bool ycc = true;
            if (jfif) ycc = true;
            else if (adobe) ycc = adobe_transform == 1;
            else if (comp_id[0] == 'R' && comp_id[1] == 'G' && comp_id[2] == 'B') ycc = false;
            if (!ycc) return say(JPEG_UNSUPPORTED, why, cap, "RGB-coded JPEG");
            if (comp_h[1] != 1 || comp_v[1] != 1 || comp_h[2] != 1 || comp_v[2] != 1 ||
                !((comp_h[0] == 1 && comp_v[0] == 1) || (comp_h[0] == 2 && comp_v[0] == 1) || (comp_h[0] == 2 && comp_v[0] == 2)))
                return say(JPEG_UNSUPPORTED, why, cap, "sampling %dx%d,%dx%d,%dx%d (device path: 4:4:4, 4:2:2, 4:2:0)", comp_h[0], comp_v[0],
                           comp_h[1], comp_v[1], comp_h[2], comp_v[2]);
            J.hs = comp_h[0];
            J.vs = comp_v[0];
            // libjpeg switches the fancy filter off for components 1 or 2 samples wide (jdsample.c)
            if (J.hs == 2 && (J.width + 1) / 2 <= 2) return say(JPEG_UNSUPPORTED, why, cap, "image too narrow for the fancy upsampler");
            J.mcus_x = (J.width + 8 * J.hs - 1) / (8 * J.hs);
            J.mcus_y = (J.height + 8 * J.vs - 1) / (8 * J.vs);
            J.bw[0] = J.mcus_x * J.hs; J.bh[0] = J.mcus_y * J.vs;
            J.bw[1] = J.bw[2] = J.mcus_x; J.bh[1] = J.bh[2] = J.mcus_y;
            J.scan_off = pos;
            return JPEG_OK;
        }
        else if (!((m >= 0xE0 && m <= 0xEF) || m == 0xFE)) {
            // only APPn and COM are skipped: PIL's marker loop and libjpeg both give up on the reserved / extension ones
            return say(JPEG_UNSUPPORTED, why, cap, "marker 0x%02x", m);
        }
    }
}

size_t jpeg_coef_count(const JpegInfo& J) {
    size_t blocks = 0;
    for (int c = 0; c < 3; ++c) blocks += size_t(J.bw[c]) * J.bh[c];
    return blocks * 64;
}

size_t jpeg_frame_stride(int width, int height) {
    // 4:4:4 on a 16-pixel grid: at least the coefficients of 4:2:2 and 4:2:0, whose planes are padded to 16-pixel MCUs
    return size_t((width + 15) / 16) * ((height + 15) / 16) * 4 * 3 * 64 * sizeof(int16_t);
}

void jpeg_frame_desc(const JpegInfo& J, size_t coef_index, JpegFrameDev* F) {
    memset(F, 0, sizeof(*F));
    memcpy(F->q, J.q, sizeof(F->q));
    size_t co = coef_index, po = 0;
    for (int c = 0; c < 3; ++c) {
        F->coef_off[c] = static_cast<uint32_t>(co);
        F->plane_off[c] = static_cast<uint32_t>(po);
        F->bw[c] = static_cast<uint16_t>(J.bw[c]);
        F->bh[c] = static_cast<uint16_t>(J.bh[c]);
        co += size_t(J.bw[c]) * J.bh[c] * 64;
        po += size_t(J.bw[c]) * J.bh[c] * 64;
    }
    F->hs = static_cast<uint16_t>(J.hs);
    F->vs = static_cast<uint16_t>(J.vs);
}

// ------------------------------------------------------------------------------------------- host: entropy decode
namespace {

struct BitReader {
    const uint8_t* p;
    const uint8_t* end;
    uint64_t acc = 0;   // left-aligned
    int cnt = 0;        // valid bits in acc
    int pad = 0;        // zero bits appended after the data ran into a marker / the end
    int marker = -1;    // marker the reader stopped at (p points at its 0xFF)
    bool at_end = false;

    // byte-at-a-time path: 0xFF00 un-stuffing, fill bytes, markers, end of buffer
    __attribute__((noinline)) void refill_slow() {
        while (cnt <= 56) {
            unsigned b = 0;
            if (marker < 0 && !at_end) {
                if (p >= end) {
                    at_end = true;
                } else if (*p != 0xFF) {
                    b = *p++;
                } else {
                    const uint8_t* q = p + 1;
                    while (q < end && *q == 0xFF) ++q;  // fill bytes
                    if (q >= end) {
                        at_end = true;
                    } else if (*q == 0x00 && q == p + 1) {
                        b = 0xFF;
                        p += 2;
                    } else if (*q == 0x00) {
                        at_end = true;  // FF FF 00: not a shape libjpeg decodes quietly
                    } else {
                        marker = *q;
                        p = q - 1;
                    }
                }
            }
            if (marker >= 0 || at_end) pad += 8;
            acc |= static_cast<uint64_t>(b) << (56 - cnt);
            cnt += 8;
        }
    }
    // common case: the next 8 bytes hold no 0xFF, so whole bytes can be appended with one load
    inline void refill() {
        if (end - p >= 8 && marker < 0) {
            uint64_t w;
            memcpy(&w, p, 8);
            w = __builtin_bswap64(w);
            const uint64_t v = ~w;
            if (((v - 0x0101010101010101ull) & ~v & 0x8080808080808080ull) == 0) {
                const int bytes = (64 - cnt) >> 3;
                if (bytes) {
                    const int now = cnt + 8 * bytes;
                    const uint64_t keep = now == 64 ? ~0ull : ~(~0ull >> now);
                    acc |= (w >> cnt) & keep;
                    p += bytes;
                    cnt = now;
                }
                return;
            }
        }
        refill_slow();
    }
    inline unsigned peek(int n) const { return static_cast<unsigned>(acc >> (64 - n)); }
    inline void drop(int n) { acc <<= n; cnt -= n; }
    inline bool overran() const { return cnt < pad; }  // consumed bits that were never in the stream
};

inline int extend(int v, int s) { return v < (1 << (s - 1)) ? v - (1 << s) + 1 : v; }  // T.81 Figure F.12

// slow half of a symbol decode: codes longer than the 9-bit look-ahead
inline int huff_long(BitReader& br, const HuffTable& h) {
    const unsigned code16 = br.peek(16);
    for (int l = 10; l <= 16; ++l) {
        const int c = static_cast<int>(code16 >> (16 - l));
        if (c <= h.maxcode[l]) {
            br.drop(l);
            return h.vals[(c + h.valoffset[l]) & 255];
        }
    }
    return -1;
}

// One 8x8 block (T.81 F.2.2).  The reader always holds >= 32 bits before a symbol: 16 for the longest code plus 15
// (in practice <= 11) magnitude bits.
// A finished block leaves the core with streaming stores.  The destination is the pinned buffer the GPU's DMA engine
// reads next: lines left dirty in sixteen cores' private caches made that copy crawl at 7 GB/s (55 GB/s once the data
// bypasses the caches); it also spares zero-filling the whole buffer first.
inline void store_block(int16_t* dst, const int16_t* blk) {
#if defined(__SSE2__)
    if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
        for (int i = 0; i < 8; ++i)
            _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + i, _mm_load_si128(reinterpret_cast<const __m128i*>(blk) + i));
        return;
    }
#endif
    memcpy(dst, blk, 128);
}

inline bool decode_block(BitReader& br, const HuffTable& dc, const HuffTable& ac, int& pred, int16_t* dst) {
    alignas(64) int16_t blk[64];
    memset(blk, 0, sizeof(blk));
    if (br.cnt < 32) br.refill();
    unsigned e = dc.lut[br.peek(9)];
    int s;
    if (e) { br.drop(e >> 8); s = e & 255; } else { s = huff_long(br, dc); }
    if (s < 0 || s > 15) return false;
    if (s) {
        pred += extend(static_cast<int>(br.peek(s)), s);
        br.drop(s);
    }
    blk[0] = static_cast<int16_t>(pred);
    for (int k = 1; k < 64;) {
        if (br.cnt < 32) br.refill();
        const unsigned look = br.peek(9);
        const int f = ac.fast_ac[look];
        if (f) {  // code and magnitude bits both inside the look-ahead: run, length and value in one lookup
            k += (f >> 4) & 15;
            if (k > 63) return false;
            br.drop(f & 15);
            blk[kNatural[k++]] = static_cast<int16_t>(f >> 8);
            continue;
        }
        e = ac.lut[look];
        int rs;
        if (e) { br.drop(e >> 8); rs = e & 255; } else { rs = huff_long(br, ac); }
        if (rs < 0) return false;
        const int r = rs >> 4;
        s = rs & 15;
        if (s == 0) {
            if (r != 15) break;  // EOB
            k += 16;
            continue;
        }
        k += r;
        if (k > 63) return false;
        blk[kNatural[k++]] = static_cast<int16_t>(extend(static_cast<int>(br.peek(s)), s));
        br.drop(s);
    }
    store_block(dst, blk);
    return true;
}

}  // namespace

int jpeg_decode_coefficients(const uint8_t* d, size_t len, const JpegInfo& J, int16_t* out, char* why, size_t cap) {
    int16_t* plane[3];
    plane[0] = out;
    plane[1] = plane[0] + size_t(J.bw[0]) * J.bh[0] * 64;
    plane[2] = plane[1] + size_t(J.bw[1]) * J.bh[1] * 64;
    BitReader br;
    br.p = d + J.scan_off;
    br.end = d + len;
    int pred[3] = {0, 0, 0};
    const int total = J.mcus_x * J.mcus_y;
    int until_restart = J.restart_interval ? J.restart_interval : total;
    int next_rst = 0;
    const HuffTable* dct[3] = {&J.dc[J.dc_tbl[0]], &J.dc[J.dc_tbl[1]], &J.dc[J.dc_tbl[2]]};
    const HuffTable* act[3] = {&J.ac[J.ac_tbl[0]], &J.ac[J.ac_tbl[1]], &J.ac[J.ac_tbl[2]]};
    for (int my = 0, mcu = 0; my < J.mcus_y; ++my) {
        for (int mx = 0; mx < J.mcus_x; ++mx, ++mcu) {
            if (until_restart == 0) {  // T.81 E.2.4: byte-align, RSTn, reset the predictors
                br.drop(br.cnt & 7);
                br.refill();
                if (br.overran() || br.cnt != br.pad || br.marker != 0xD0 + next_rst)
                    return say(JPEG_CORRUPT, why, cap, "restart marker RST%d missing before MCU %d", next_rst, mcu);
                br.p += 2;
                br.acc = 0; br.cnt = 0; br.pad = 0; br.marker = -1;
                next_rst = (next_rst + 1) & 7;
                pred[0] = pred[1] = pred[2] = 0;
                until_restart = J.restart_interval;
            }
            for (int v = 0; v < J.vs; ++v)
                for (int h = 0; h < J.hs; ++h) {
                    int16_t* blk = plane[0] + (size_t(my * J.vs + v) * J.bw[0] + (mx * J.hs + h)) * 64;
                    if (!decode_block(br, *dct[0], *act[0], pred[0], blk)) return say(JPEG_CORRUPT, why, cap, "bad Huffman code in MCU %d", mcu);
                }
            for (int c = 1; c < 3; ++c) {
                int16_t* blk = plane[c] + (size_t(my) * J.bw[c] + mx) * 64;
                if (!decode_block(br, *dct[c], *act[c], pred[c], blk)) return say(JPEG_CORRUPT, why, cap, "bad Huffman code in MCU %d", mcu);
            }
            if (br.overran()) return say(JPEG_CORRUPT, why, cap, "entropy-coded data ends inside MCU %d", mcu);
            --until_restart;
        }
    }
    br.drop(br.cnt & 7);
    br.refill();
    if (br.overran() || br.cnt != br.pad) return say(JPEG_CORRUPT, why, cap, "extra bytes after the last MCU");
    if (br.marker != 0xD9) return say(JPEG_CORRUPT, why, cap, "no EOI after the last MCU");
#if defined(__SSE2__)
    _mm_sfence();  // the streaming stores are globally visible before the caller hands the buffer to the copy engine
#endif
    return JPEG_OK;
}

// ------------------------------------------------------------------------------------------- host: thread pool
JpegPool::JpegPool(int threads) {
    for (int i = 1; i < threads; ++i) workers_.emplace_back([this] { worker(); });
}

JpegPool::~JpegPool() {
    {
        std::lock_guard<std::mutex> g(mu_);
        stop_ = true;
    }
    cv_work_.notify_all();
    for (std::thread& t : workers_) t.join();
}

void JpegPool::worker() {
    unsigned long seen = 0;
    std::unique_lock<std::mutex> lk(mu_);
    while (true) {
        cv_work_.wait(lk, [&] { return stop_ || (generation_ != seen && next_ < tasks_); });
        if (stop_) return;
        seen = generation_;
        ++running_;
        while (next_ < tasks_) {
            const int i = next_++;
            lk.unlock();
            (*fn_)(i);
            lk.lock();
        }
        if (--running_ == 0) cv_done_.notify_all();
    }
}

void JpegPool::run(int tasks, const std::function<void(int)>& fn) {
    if (tasks <= 0) return;
    if (tasks == 1 || workers_.empty()) {  // nothing to share: do not wake the pool (batch-1 latency)
        for (int i = 0; i < tasks; ++i) fn(i);
        return;
    }
    std::unique_lock<std::mutex> lk(mu_);
    fn_ = &fn;
    tasks_ = tasks;
    next_ = 0;
    ++generation_;
    ++running_;  // the calling thread works too
    lk.unlock();
    cv_work_.notify_all();
    lk.lock();
    while (next_ < tasks_) {
        const int i = next_++;
        lk.unlock();
        fn(i);
        lk.lock();
    }
    --running_;
    cv_done_.wait(lk, [&] { return running_ == 0; });
    fn_ = nullptr;
    tasks_ = 0;
}

// ------------------------------------------------------------------------------------------- device: IDCT
namespace {

constexpr int CONST_BITS = 13, PASS1_BITS = 2;
constexpr int F_0_298 = 2446, F_0_390 = 3196, F_0_541 = 4433, F_0_765 = 6270, F_0_899 = 7373, F_1_175 = 9633,
              F_1_501 = 12299, F_1_847 = 15137, F_1_961 = 16069, F_2_053 = 16819, F_2_562 = 20995, F_3_072 = 25172;

// One 8-point pass of jpeg_idct_islow; the caller applies the pass-specific descale.  Inputs are 16-bit values.  For
// the streams a sane encoder writes this is jidctint.c to the letter; outside that range it follows the SIMD versions
// libjpeg-turbo actually runs (jidctint-sse2/avx2: 16-bit paddw/psubw for in0 +- in4 and for z3, z4; 32-bit lanes that
// wrap; saturating packs after each pass), because that is what PIL returns for a damaged-but-decodable stream.
__device__ __forceinline__ int wrap16(int v) { return static_cast<int>(static_cast<short>(v)); }
__device__ __forceinline__ int sat16(int v) { return min(max(v, -32768), 32767); }

__device__ __forceinline__ void idct8(const int (&in)[8], int (&out)[8]) {
    int z2 = in[2], z3 = in[6];
    int z1 = (z2 + z3) * F_0_541;
    const int e2 = z1 + z3 * (-F_1_847);
    const int e3 = z1 + z2 * F_0_765;
    z2 = in[0];
    z3 = in[4];
    const int e0 = wrap16(z2 + z3) << CONST_BITS;
    const int e1 = wrap16(z2 - z3) << CONST_BITS;
    const int t10 = e0 + e3, t13 = e0 - e3, t11 = e1 + e2, t12 = e1 - e2;
    int o0 = in[7], o1 = in[5], o2 = in[3], o3 = in[1];
    z1 = o0 + o3;
    z2 = o1 + o2;
    z3 = wrap16(o0 + o2);
    int z4 = wrap16(o1 + o3);
    const int z5 = (z3 + z4) * F_1_175;
    o0 *= F_0_298;
    o1 *= F_2_053;
    o2 *= F_3_072;
    o3 *= F_1_501;
    z1 *= -F_0_899;
    z2 *= -F_2_562;
    z3 *= -F_1_961;
    z4 *= -F_0_390;
    z3 += z5;
    z4 += z5;
    o0 += z1 + z3;
    o1 += z2 + z4;
    o2 += z2 + z3;
    o3 += z1 + z4;
    out[0] = t10 + o3; out[7] = t10 - o3;
    out[1] = t11 + o2; out[6] = t11 - o2;
    out[2] = t12 + o1; out[5] = t12 - o1;
    out[3] = t13 + o0; out[4] = t13 - o0;
}

// final range limit: clamp(x + 128) — the C code's table look-up for every value a valid stream produces, and the
// saturating packs of the SIMD code (not the table's wrap-around) beyond
__device__ __forceinline__ unsigned range_limit_idct(int x) { return static_cast<unsigned>(min(max(x, -128), 127) + 128); }

constexpr int IDCT_BLOCKS = 32, WS_PITCH = 72;

__global__ void __launch_bounds__(IDCT_BLOCKS * 8)
jpeg_idct_kernel(const int16_t* __restrict__ coefs, const JpegFrameDev* __restrict__ frames, uint8_t* __restrict__ planes,
                 size_t plane_stride) {
    __shared__ int ws[IDCT_BLOCKS][WS_PITCH];
    const JpegFrameDev& F = frames[blockIdx.y];
    const int t = threadIdx.x & 7, lb = threadIdx.x >> 3;
    const int b = blockIdx.x * IDCT_BLOCKS + lb;
    const int n0 = F.bw[0] * F.bh[0], n1 = F.bw[1] * F.bh[1], n2 = F.bw[2] * F.bh[2];
    const bool live = b < n0 + n1 + n2;
    const int c = !live ? 0 : (b >= n0) + (b >= n0 + n1);
    const int bc = !live ? 0 : b - (c > 0 ? n0 : 0) - (c > 1 ? n1 : 0);
    int v[8], o[8];
    bool row_nonzero = false;
    const int lane_in_warp = threadIdx.x & 31;
    if (live) {  // row t of the block: 8 coefficients x 8 quantiser steps (DEQUANTIZE in jidctint.c)
        const int4 raw = __ldg(reinterpret_cast<const int4*>(coefs + F.coef_off[c] + size_t(bc) * 64 + t * 8));
        row_nonzero = (raw.x | raw.y | raw.z | raw.w) != 0;
        const int4 qv = __ldg(reinterpret_cast<const int4*>(F.q[c] + t * 8));
        const int r[4] = {raw.x, raw.y, raw.z, raw.w};
        const int q[4] = {qv.x, qv.y, qv.z, qv.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            // (pmullw: the product is kept to 16 bits)
            ws[lb][t * 8 + 2 * j] = wrap16(static_cast<int>(static_cast<short>(r[j] & 0xffff)) * (q[j] & 0xffff));
            ws[lb][t * 8 + 2 * j + 1] = wrap16((r[j] >> 16) * static_cast<int>(static_cast<unsigned>(q[j]) >> 16));
        }
    }
    // the SIMD code's shortcut for a block whose rows 1..7 are all zero: every column is its DC term shifted left in a
    // 16-bit lane (psllw wraps where the full column pass would saturate)
    const unsigned ac_rows = __ballot_sync(0xffffffffu, live && t > 0 && row_nonzero);
    const bool dc_only = ((ac_rows >> (8 * (lane_in_warp >> 3))) & 0xffu) == 0u;
    __syncwarp();
    if (live) {  // pass 1: column t
#pragma unroll
        for (int r = 0; r < 8; ++r) v[r] = ws[lb][r * 8 + t];
        idct8(v, o);
    }
    __syncwarp();
    if (live) {
#pragma unroll
        for (int r = 0; r < 8; ++r)
            ws[lb][r * 8 + t] = dc_only ? wrap16(v[0] << PASS1_BITS)
                                        : sat16((o[r] + (1 << (CONST_BITS - PASS1_BITS - 1))) >> (CONST_BITS - PASS1_BITS));
    }
    __syncwarp();
    if (live) {  // pass 2: row t
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = ws[lb][t * 8 + j];
        idct8(v, o);
        unsigned px[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
            px[j] = range_limit_idct((o[j] + (1 << (CONST_BITS + PASS1_BITS + 2))) >> (CONST_BITS + PASS1_BITS + 3));
        const int bwc = F.bw[c];
        const int by = bc / bwc, bx = bc - by * bwc;
        uint2 w;
        w.x = px[0] | (px[1] << 8) | (px[2] << 16) | (px[3] << 24);
        w.y = px[4] | (px[5] << 8) | (px[6] << 16) | (px[7] << 24);
        uint8_t* dst = planes + blockIdx.y * plane_stride + F.plane_off[c] + (size_t(by) * 8 + t) * (bwc * 8) + bx * 8;
        *reinterpret_cast<uint2*>(dst) = w;
    }
}

// ------------------------------------------------------------------------------------------- device: upsample + colour
__device__ __forceinline__ int clamp255(int x) { return min(max(x, 0), 255); }

__device__ __forceinline__ void ycc_to_rgb(int y, int cb, int cr, uint8_t* dst) {  // jdcolor.c build_ycc_rgb_table + ycc_rgb_convert
    const int cbx = cb - 128, crx = cr - 128;
    dst[0] = static_cast<uint8_t>(clamp255(y + ((91881 * crx + 32768) >> 16)));
    dst[1] = static_cast<uint8_t>(clamp255(y + ((-22554 * cbx + 32768 - 46802 * crx) >> 16)));
    dst[2] = static_cast<uint8_t>(clamp255(y + ((116130 * cbx + 32768) >> 16)));
}

// one thread per horizontal pixel pair (2i, 2i+1): they share chroma column i in the subsampled layouts
__global__ void __launch_bounds__(256)
jpeg_rgb_kernel(const uint8_t* __restrict__ planes, size_t plane_stride, const JpegFrameDev* __restrict__ frames,
                uint8_t* __restrict__ rgb, int h, int w) {
    const int i = blockIdx.x * 64 + (threadIdx.x & 63);
    const int y = blockIdx.y * 4 + (threadIdx.x >> 6);
    const int f = blockIdx.z;
    const int x = 2 * i;
    if (y >= h || x >= w) return;
    const JpegFrameDev& F = frames[f];
    const uint8_t* base = planes + f * plane_stride;
    const uint8_t* Y = base + F.plane_off[0] + size_t(y) * (F.bw[0] * 8);
    const int pc = F.bw[1] * 8;
    const uint8_t* CB = base + F.plane_off[1];
    const uint8_t* CR = base + F.plane_off[2];
    const bool second = x + 1 < w;
    const int y0 = Y[x], y1 = second ? Y[x + 1] : 0;
    int cb0, cb1, cr0, cr1;
    if (F.hs == 1) {  // fullsize_upsample
        cb0 = CB[size_t(y) * pc + x]; cr0 = CR[size_t(y) * pc + x];
        cb1 = second ? CB[size_t(y) * pc + x + 1] : 0; cr1 = second ? CR[size_t(y) * pc + x + 1] : 0;
    } else {
        const int cw = (w + 1) >> 1;  // downsampled_width
        const int il = max(i - 1, 0), ir = min(i + 1, cw - 1);
        if (F.vs == 1) {  // h2v1_fancy_upsample: 3/4 nearer + 1/4 further, edge columns copied
            const uint8_t* rb = CB + size_t(y) * pc;
            const uint8_t* rr = CR + size_t(y) * pc;
            const int b = rb[i], r = rr[i];
            cb0 = i == 0 ? b : (3 * b + rb[il] + 1) >> 2;
            cr0 = i == 0 ? r : (3 * r + rr[il] + 1) >> 2;
            cb1 = i == cw - 1 ? b : (3 * b + rb[ir] + 2) >> 2;
            cr1 = i == cw - 1 ? r : (3 * r + rr[ir] + 2) >> 2;
        } else {  // h2v2_fancy_upsample: 9/16, 3/16, 3/16, 1/16; the context row beyond the image is the edge row
            const int ch = (h + 1) >> 1;
            const int cy = y >> 1;
            const int fy = (y & 1) ? min(cy + 1, ch - 1) : max(cy - 1, 0);
            const uint8_t* nb = CB + size_t(cy) * pc;
            const uint8_t* fb = CB + size_t(fy) * pc;
            const uint8_t* nr = CR + size_t(cy) * pc;
            const uint8_t* fr = CR + size_t(fy) * pc;
            const int sb = 3 * nb[i] + fb[i], sbl = 3 * nb[il] + fb[il], sbr = 3 * nb[ir] + fb[ir];
            const int sr = 3 * nr[i] + fr[i], srl = 3 * nr[il] + fr[il], srr = 3 * nr[ir] + fr[ir];
            cb0 = i == 0 ? (sb * 4 + 8) >> 4 : (sb * 3 + sbl + 8) >> 4;
            cr0 = i == 0 ? (sr * 4 + 8) >> 4 : (sr * 3 + srl + 8) >> 4;
            cb1 = i == cw - 1 ? (sb * 4 + 7) >> 4 : (sb * 3 + sbr + 7) >> 4;
            cr1 = i == cw - 1 ? (sr * 4 + 7) >> 4 : (sr * 3 + srr + 7) >> 4;
        }
    }
    uint8_t* dst = rgb + ((size_t(f) * h + y) * w + x) * 3;
    ycc_to_rgb(y0, cb0, cr0, dst);
    if (second) ycc_to_rgb(y1, cb1, cr1, dst + 3);
}

}  // namespace

int launch_jpeg_idct(const int16_t* coefs, const JpegFrameDev* frames, uint8_t* planes, size_t plane_stride, int n,
                     int max_blocks, cudaStream_t s) {
    if (n < 1 || max_blocks < 1) return -1;
    const dim3 grid((max_blocks + IDCT_BLOCKS - 1) / IDCT_BLOCKS, n);
    jpeg_idct_kernel<<<grid, IDCT_BLOCKS * 8, 0, s>>>(coefs, frames, planes, plane_stride);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

int launch_jpeg_rgb(const uint8_t* planes, size_t plane_stride, const JpegFrameDev* frames, uint8_t* rgb, int n, int h,
                    int w, cudaStream_t s) {
    if (n < 1) return -1;
    const int pairs = (w + 1) / 2;
    const dim3 grid((pairs + 63) / 64, (h + 3) / 4, n);
    jpeg_rgb_kernel<<<grid, 256, 0, s>>>(planes, plane_stride, frames, rgb, h, w);
    return cudaPeekAtLastError() == cudaSuccess ? 0 : -1;  // (peek: the caller reports the reason)
}

}  // namespace fd
