// Baseline JPEG (the frames of an MJPG video) decoded on the device, bit for bit what libjpeg-turbo's default
// decompression gives -- the decoder behind cv2.imdecode(packet, cv2.IMREAD_COLOR):
//   * Huffman decoding as jdhuff.c (canonical tables, the Annex K tables where a packet carries no DHT);
//   * dequantisation + ISLOW IDCT as jidctint.c (CONST_BITS 13, PASS1_BITS 2, 64-bit intermediates, the range-limit
//     table with its RANGE_MASK wrap);
//   * h2v1 / h2v2 "fancy" upsampling as jdsample.c (edge columns and the replicated context rows);
//   * YCbCr -> BGR as jdcolor.c (SCALEBITS 16 tables).
// The host parses the markers, removes the FF00 byte stuffing and splits the scan at its restart markers; the
// per-block and per-pixel arithmetic below is written once and runs in the kernels and in the host entry
// (jpeg_decode_host), so the whole decoder can be checked against cv2.imdecode without a GPU.
//
// Supported: SOF0 / SOF1, 8-bit samples and quantisation tables, one scan holding every component, grey or YCbCr with
// luma sampling 1x1, 2x1 or 2x2 and chroma 1x1.  Anything else is reported as kJpegFallback (the caller decodes it
// with cv2.imdecode); headers that libjpeg itself rejects raise OPB_ERR_INVALID.
#include "jpeg.cuh"
#include <algorithm>

namespace opb {
namespace {

constexpr int kLutBits = 9;                 // codes of up to 9 bits are decoded by one table lookup
constexpr int kLutSize = 1 << kLutBits;
constexpr int kTables = 8;                  // DC 0-3, AC 0-3

struct HuffTable {                          // canonical form of jdhuff.c's d_derived_tbl
    int maxcode[18];                        // [l]: largest code of length l, -1 if none
    int valoff[17];                         // [l]: index in vals of the first code of length l, minus that code
    uint8_t vals[256];
};

struct Comp {
    int h, v, tq, td, ta;
    int bw, bh;                             // coefficient block grid
    int dw, dh;                             // libjpeg's downsampled_width / downsampled_height
    int coef;                               // first block of the component, relative to the frame
    int plane;                              // first sample byte of the component, relative to the frame
};

struct Frame {
    int width, height, ncomp, hmax, vmax, mcux, mcus, restart;
    int nscan, scan[3];                     // component indices in scan order
    int x0, y0;                             // ROI origin
    int skip;                               // not decoded here (fallback or corrupt at parse)
    int blocks;
    long long coef_base;                    // first block of the frame in the batch's coefficient buffer
    long long plane_base;                   // first byte of the frame's sample planes
    Comp comp[3];
    uint16_t qt[4][64];                     // natural order
    HuffTable huff[kTables];
};

struct Segment {                            // one entropy-coded segment: the scan, or one restart interval
    int frame, mcu_first, mcu_count, pad;
    long long begin, end;                   // byte range in the destuffed data
};

// jpeg_natural_order (jutils.c)
#define OPB_ZIGZAG                                                                                                     \
    {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,     \
     7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46,    \
     53, 60, 61, 54, 47, 55, 62, 63}
__constant__ uint8_t kZigzagDev[64] = OPB_ZIGZAG;
const uint8_t kZigzagHost[64] = OPB_ZIGZAG;

__host__ __device__ inline int zigzag(int k) {
#ifdef __CUDA_ARCH__
    return kZigzagDev[k];
#else
    return kZigzagHost[k];
#endif
}

// ---- entropy decoding ------------------------------------------------------------------------------------------------
struct Bits {
    const uint8_t* p;
    long long next, end;                    // next byte to load, end of the segment
    unsigned long long acc;                 // next bit at bit 63
    int cnt;                                // valid bits in acc
};

__host__ __device__ inline void fill(Bits& b) {
    while (b.cnt <= 56) {                   // past the segment's end the stream reads as zeros
        const unsigned long long byte = b.next < b.end ? b.p[b.next] : 0;
        ++b.next;
        b.acc |= byte << (56 - b.cnt);
        b.cnt += 8;
    }
}

__host__ __device__ inline int take(Bits& b, int n) {     // 1 <= n <= 16, n <= cnt
    const int v = (int)(b.acc >> (64 - n));
    b.acc <<= n;
    b.cnt -= n;
    return v;
}

__host__ __device__ inline int extend(int x, int s) {     // HUFF_EXTEND
    return x < (1 << (s - 1)) ? x - (1 << s) + 1 : x;
}

// entry i of the 9-bit lookup table: (length << 8) | symbol, 0 when no code of up to 9 bits is a prefix of i
__host__ __device__ inline uint16_t lut_entry(const HuffTable& t, int i) {
    for (int l = 1; l <= kLutBits; ++l) {
        const int code = i >> (kLutBits - l);
        if (code <= t.maxcode[l]) return (uint16_t)((l << 8) | t.vals[(code + t.valoff[l]) & 255]);
    }
    return 0;
}

// one symbol (cnt >= 16); -1 on a bad code
__host__ __device__ inline int huff_decode(Bits& b, const uint16_t* lut, const HuffTable& t) {
    const int e = lut[b.acc >> (64 - kLutBits)];
    if (e) {
        b.acc <<= e >> 8;
        b.cnt -= e >> 8;
        return e & 255;
    }
    for (int l = kLutBits + 1; l <= 16; ++l) {
        const int code = (int)(b.acc >> (64 - l));
        if (code <= t.maxcode[l]) {
            b.acc <<= l;
            b.cnt -= l;
            return t.vals[(code + t.valoff[l]) & 255];
        }
    }
    return -1;
}

// one block into coef (zeroed by the caller), natural order; false on a bad code
__host__ __device__ inline bool decode_block(Bits& b, const uint16_t* luts, const Frame& f, const Comp& c, int& pred,
                                             short* coef) {
    fill(b);
    int s = huff_decode(b, luts + c.td * kLutSize, f.huff[c.td]);
    if (s < 0) return false;
    if (s) pred += extend(take(b, s), s);
    coef[0] = (short)pred;
    const uint16_t* aclut = luts + (4 + c.ta) * kLutSize;
    const HuffTable& act = f.huff[4 + c.ta];
    for (int k = 1; k < 64; ++k) {
        fill(b);
        const int rs = huff_decode(b, aclut, act);
        if (rs < 0) return false;
        const int r = rs >> 4;
        s = rs & 15;
        if (s) {
            k += r;                         // past 63: jpeg_natural_order's padding entries all point at 63
            coef[k > 63 ? 63 : zigzag(k)] = (short)extend(take(b, s), s);
        } else {
            if (r != 15) break;
            k += 15;
        }
    }
    return true;
}

// MCUs [mcu_first, mcu_first + mcu_count) of one frame; false when a code is bad, the data runs out, or more than the
// final byte's padding is left over
__host__ __device__ inline bool decode_segment(const Frame& f, const uint8_t* data, long long begin, long long end,
                                               int mcu_first, int mcu_count, const uint16_t* luts, short* coefs) {
    Bits b{data, begin, end, 0ull, 0};
    int pred[3] = {0, 0, 0};
    short* base = coefs + f.coef_base * 64;
    for (int m = mcu_first; m < mcu_first + mcu_count; ++m) {
        if (f.nscan == 1) {                 // non-interleaved: an MCU is one block
            const Comp& c = f.comp[f.scan[0]];
            if (!decode_block(b, luts, f, c, pred[0], base + ((long long)c.coef + m) * 64)) return false;
            continue;
        }
        const int mx = m % f.mcux, my = m / f.mcux;
        for (int k = 0; k < f.nscan; ++k) {
            const Comp& c = f.comp[f.scan[k]];
            for (int v = 0; v < c.v; ++v)
                for (int h = 0; h < c.h; ++h) {
                    const long long blk = c.coef + (long long)(my * c.v + v) * c.bw + mx * c.h + h;
                    if (!decode_block(b, luts, f, c, pred[k], base + blk * 64)) return false;
                }
        }
    }
    const long long left = (end - begin) * 8 - ((b.next - begin) * 8 - b.cnt);
    return left >= 0 && left < 8;
}

// ---- jidctint.c: jpeg_idct_islow ------------------------------------------------------------------------------------
__host__ __device__ inline uint8_t idct_range_limit(int x) {    // range_limit[x & RANGE_MASK]
    const int y = ((x & 1023) ^ 512) - 512;                     // the table wraps at 1024
    return (uint8_t)min(max(y + 128, 0), 255);
}

__host__ __device__ inline void idct_islow(const short* in, const uint16_t* q, uint8_t* out, int stride) {
    typedef long long L;
    const int CB = 13, P1 = 2;
    int ws[64];
    for (int c = 0; c < 8; ++c) {
        L z2 = (L)in[16 + c] * q[16 + c], z3 = (L)in[48 + c] * q[48 + c];
        L z1 = (z2 + z3) * 4433;
        L tmp2 = z1 + z3 * -15137, tmp3 = z1 + z2 * 6270;
        z2 = (L)in[c] * q[c];
        z3 = (L)in[32 + c] * q[32 + c];
        L tmp0 = (z2 + z3) * 8192, tmp1 = (z2 - z3) * 8192;
        const L tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
        tmp0 = (L)in[56 + c] * q[56 + c];
        tmp1 = (L)in[40 + c] * q[40 + c];
        tmp2 = (L)in[24 + c] * q[24 + c];
        tmp3 = (L)in[8 + c] * q[8 + c];
        z1 = tmp0 + tmp3;
        z2 = tmp1 + tmp2;
        z3 = tmp0 + tmp2;
        L z4 = tmp1 + tmp3;
        const L z5 = (z3 + z4) * 9633;
        tmp0 *= 2446; tmp1 *= 16819; tmp2 *= 25172; tmp3 *= 12299;
        z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;
        z3 += z5; z4 += z5;
        tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
        const int sh = CB - P1;
        const L r = (L)1 << (sh - 1);
        ws[c] = (int)((tmp10 + tmp3 + r) >> sh);
        ws[56 + c] = (int)((tmp10 - tmp3 + r) >> sh);
        ws[8 + c] = (int)((tmp11 + tmp2 + r) >> sh);
        ws[48 + c] = (int)((tmp11 - tmp2 + r) >> sh);
        ws[16 + c] = (int)((tmp12 + tmp1 + r) >> sh);
        ws[40 + c] = (int)((tmp12 - tmp1 + r) >> sh);
        ws[24 + c] = (int)((tmp13 + tmp0 + r) >> sh);
        ws[32 + c] = (int)((tmp13 - tmp0 + r) >> sh);
    }
    for (int rr = 0; rr < 8; ++rr) {
        const int* w = ws + rr * 8;
        L z2 = w[2], z3 = w[6];
        L z1 = (z2 + z3) * 4433;
        L tmp2 = z1 + z3 * -15137, tmp3 = z1 + z2 * 6270;
        L tmp0 = ((L)w[0] + w[4]) * 8192, tmp1 = ((L)w[0] - w[4]) * 8192;
        const L tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
        tmp0 = w[7]; tmp1 = w[5]; tmp2 = w[3]; tmp3 = w[1];
        z1 = tmp0 + tmp3;
        z2 = tmp1 + tmp2;
        z3 = tmp0 + tmp2;
        L z4 = tmp1 + tmp3;
        const L z5 = (z3 + z4) * 9633;
        tmp0 *= 2446; tmp1 *= 16819; tmp2 *= 25172; tmp3 *= 12299;
        z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;
        z3 += z5; z4 += z5;
        tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
        const int sh = CB + P1 + 3;
        const L r = (L)1 << (sh - 1);
        uint8_t* o = out + (size_t)rr * stride;
        o[0] = idct_range_limit((int)((tmp10 + tmp3 + r) >> sh));
        o[7] = idct_range_limit((int)((tmp10 - tmp3 + r) >> sh));
        o[1] = idct_range_limit((int)((tmp11 + tmp2 + r) >> sh));
        o[6] = idct_range_limit((int)((tmp11 - tmp2 + r) >> sh));
        o[2] = idct_range_limit((int)((tmp12 + tmp1 + r) >> sh));
        o[5] = idct_range_limit((int)((tmp12 - tmp1 + r) >> sh));
        o[3] = idct_range_limit((int)((tmp13 + tmp0 + r) >> sh));
        o[4] = idct_range_limit((int)((tmp13 - tmp0 + r) >> sh));
    }
}

// block b of a frame: its coefficients and where its samples go
__host__ __device__ inline void idct_block(const Frame& f, int b, const short* coefs, uint8_t* planes) {
    int ci = f.ncomp - 1;
    while (ci > 0 && b < f.comp[ci].coef) --ci;
    const Comp& c = f.comp[ci];
    const int local = b - c.coef, bx = local % c.bw, by = local / c.bw, stride = c.bw * 8;
    idct_islow(coefs + (f.coef_base + b) * 64, f.qt[c.tq],
               planes + f.plane_base + c.plane + (size_t)by * 8 * stride + bx * 8, stride);
}

// ---- jdsample.c fancy upsampling + jdcolor.c ------------------------------------------------------------------------
// sample of component ci at full-resolution position (y, x)
__host__ __device__ inline int upsampled(const Frame& f, const uint8_t* planes, int ci, int y, int x) {
    const Comp& c = f.comp[ci];
    const uint8_t* p = planes + c.plane;
    const int st = c.bw * 8;
    if (c.h == f.hmax && c.v == f.vmax) return p[(size_t)y * st + x];
    const int cx = x >> 1;
    // the column beyond the edge is the edge column itself (jdsample.c's first / last column cases)
    const int side = (x & 1) ? min(cx + 1, c.dw - 1) : max(cx - 1, 0);
    if (c.v == f.vmax) {                                   // h2v1_fancy_upsample
        const uint8_t* r = p + (size_t)y * st;
        return (3 * r[cx] + r[side] + 1 + (x & 1)) >> 2;
    }
    // h2v2_fancy_upsample: the nearer row and the next nearer one, replicated at the top and bottom (jdmainct.c)
    const int row = y >> 1, other = (y & 1) ? min(row + 1, c.dh - 1) : max(row - 1, 0);
    const uint8_t* r0 = p + (size_t)row * st;
    const uint8_t* r1 = p + (size_t)other * st;
    const int here = 3 * r0[cx] + r1[cx], there = 3 * r0[side] + r1[side];
    return (3 * here + there + 8 - (x & 1)) >> 4;
}

__host__ __device__ inline uint8_t clamp255(int v) { return (uint8_t)min(max(v, 0), 255); }

// BGR of the full-resolution pixel (y, x)
__host__ __device__ inline void bgr_pixel(const Frame& f, const uint8_t* planes, int y, int x, uint8_t* o) {
    const int Y = upsampled(f, planes, 0, y, x);
    if (f.ncomp == 1) {
        o[0] = o[1] = o[2] = (uint8_t)Y;
        return;
    }
    const int cb = upsampled(f, planes, 1, y, x) - 128, cr = upsampled(f, planes, 2, y, x) - 128;
    const int half = 1 << 15;
    o[0] = clamp255(Y + ((116130 * cb + half) >> 16));                 // Cb_b_tab
    o[1] = clamp255(Y + ((-22554 * cb + half - 46802 * cr) >> 16));    // Cb_g_tab + Cr_g_tab
    o[2] = clamp255(Y + ((91881 * cr + half) >> 16));                  // Cr_r_tab
}

// ---- host parser -----------------------------------------------------------------------------------------------------
// Annex K tables (jstdhuff.c): used for slots 0 and 1 that a packet leaves undefined, like Motion-JPEG decoders do
const uint8_t kStdBits[4][17] = {
    {0, 0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0},          // DC luma
    {0, 0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0},          // DC chroma
    {0, 0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d},       // AC luma
    {0, 0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}};      // AC chroma
const uint8_t kStdDcVals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
const uint8_t kStdAcLuma[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14,
    0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09,
    0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a,
    0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65,
    0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88,
    0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9,
    0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca,
    0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea,
    0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
const uint8_t kStdAcChroma[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32,
    0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16,
    0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39,
    0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64,
    0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86,
    0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7,
    0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8,
    0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9,
    0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};

[[noreturn]] void invalid(const char* what) { throw Error(OPB_ERR_INVALID, std::string("jpeg: ") + what); }

// jpeg_make_d_derived_tbl's checks and canonical codes; bits[1..16]
void derive(const uint8_t* bits, const uint8_t* vals, bool dc, HuffTable& t) {
    int count = 0;
    for (int l = 1; l <= 16; ++l) count += bits[l];
    if (count > 256) invalid("bad Huffman table");
    int code = 0, p = 0, last = 0;
    for (int l = 1; l <= 16; ++l)
        if (bits[l]) last = l;
    for (int l = 1; l <= 16; ++l) {
        if (bits[l]) {
            t.valoff[l] = p - code;
            t.maxcode[l] = code + bits[l] - 1;
        } else {
            t.valoff[l] = 0;
            t.maxcode[l] = -1;
        }
        p += bits[l];
        code += bits[l];
        if (l <= last && code >= (1 << l)) invalid("bad Huffman table");
        code <<= 1;
    }
    t.maxcode[0] = -1;
    t.maxcode[17] = 0xFFFFF;
    t.valoff[0] = 0;
    memset(t.vals, 0, sizeof(t.vals));
    for (int i = 0; i < count; ++i) {
        if (dc && vals[i] > 15) invalid("bad Huffman table");
        t.vals[i] = vals[i];
    }
}

struct Parse {
    int status = 0;                         // 0, kJpegFallback or kJpegCorrupt
    int width = 0, height = 0;              // 0 until a frame header has been read
};

// EXIF orientation of an APP1 payload; 1 when absent
int exif_orientation(const uint8_t* p, size_t n) {
    if (n < 14 || memcmp(p, "Exif\0\0", 6) != 0) return 1;
    const uint8_t* t = p + 6;
    const size_t tn = n - 6;
    const bool le = t[0] == 'I' && t[1] == 'I';
    if (!le && !(t[0] == 'M' && t[1] == 'M')) return 0;
    auto u16 = [&](size_t o) -> unsigned { return le ? t[o] | t[o + 1] << 8 : t[o] << 8 | t[o + 1]; };
    auto u32 = [&](size_t o) -> size_t { return le ? (size_t)u16(o) | (size_t)u16(o + 2) << 16
                                                   : (size_t)u16(o) << 16 | u16(o + 2); };
    const size_t ifd = u32(4);
    if (ifd + 2 > tn) return 0;
    const unsigned entries = u16(ifd);
    for (unsigned e = 0; e < entries; ++e) {
        const size_t o = ifd + 2 + 12 * (size_t)e;
        if (o + 12 > tn) return 0;
        if (u16(o) == 0x0112) return (int)u16(o + 8);
    }
    return 1;
}

// Parses one packet into f (tables, geometry, ROI left to the caller), appending its destuffed entropy data at
// data[*used] and its segments to segs.  Throws OPB_ERR_INVALID where libjpeg raises an error.
Parse parse(const uint8_t* p, size_t n, int fi, Frame& f, uint8_t* data, size_t* used, std::vector<Segment>& segs) {
    Parse r;
    memset(&f, 0, sizeof(f));
    if (n < 4 || p[0] != 0xFF || p[1] != 0xD8) invalid("not a JPEG packet (no SOI)");
    bool have_q[4] = {}, have_h[kTables] = {}, sof = false, jfif = false, rgb_ids = false;
    uint8_t bits[kTables][17] = {}, vals[kTables][256] = {};
    int ids[3] = {};
    size_t i = 2;
    const size_t seg_start = segs.size();
    auto fallback = [&]() { r.status = kJpegFallback; return r; };
    while (true) {
        while (i < n && p[i] != 0xFF) ++i;                  // garbage between markers: libjpeg skips it too
        while (i < n && p[i] == 0xFF) ++i;
        if (i >= n) invalid("packet ends before the scan");
        const int m = p[i++];
        if (m == 0xD9) invalid("EOI before the scan");
        if (m == 0x01 || (m >= 0xD0 && m <= 0xD7)) continue;
        if (i + 2 > n) invalid("truncated marker");
        const size_t len = (size_t)p[i] << 8 | p[i + 1];
        if (len < 2 || i + len > n) invalid("truncated marker segment");
        const uint8_t* q = p + i + 2;
        const size_t ql = len - 2;
        i += len;
        if (m == 0xC0 || m == 0xC1) {                        // baseline / extended sequential, Huffman
            if (sof) invalid("two frame headers");
            if (ql < 6) invalid("bad SOF");
            sof = true;
            r.height = q[1] << 8 | q[2];
            r.width = q[3] << 8 | q[4];
            const int nc = q[5];
            if (r.width <= 0 || nc <= 0 || ql != 6 + 3 * (size_t)nc) invalid("bad SOF");
            if (q[0] != 8 || r.height == 0 || (nc != 1 && nc != 3)) return fallback();
            f.width = r.width;
            f.height = r.height;
            f.ncomp = nc;
            for (int c = 0; c < nc; ++c) {
                ids[c] = q[6 + 3 * c];
                f.comp[c].h = q[7 + 3 * c] >> 4;
                f.comp[c].v = q[7 + 3 * c] & 15;
                f.comp[c].tq = q[8 + 3 * c];
                if (f.comp[c].h < 1 || f.comp[c].h > 4 || f.comp[c].v < 1 || f.comp[c].v > 4 || f.comp[c].tq > 3)
                    invalid("bad component in SOF");
                f.hmax = std::max(f.hmax, f.comp[c].h);
                f.vmax = std::max(f.vmax, f.comp[c].v);
            }
            rgb_ids = nc == 3 && ids[0] == 'R' && ids[1] == 'G' && ids[2] == 'B';
        } else if ((m >= 0xC2 && m <= 0xCB && m != 0xC4 && m != 0xC8) || (m >= 0xCD && m <= 0xCF)) {
            if (ql >= 5) {                                   // progressive, lossless, arithmetic: dims only
                r.height = q[1] << 8 | q[2];
                r.width = q[3] << 8 | q[4];
            }
            return fallback();
        } else if (m == 0xC4) {                              // DHT
            size_t o = 0;
            while (o < ql) {
                if (o + 17 > ql) invalid("bad DHT");
                const int tc = q[o] >> 4, th = q[o] & 15;
                if (tc > 1 || th > 3) invalid("bad DHT class or slot");
                int count = 0;
                for (int l = 1; l <= 16; ++l) count += q[o + l];
                if (count > 256 || o + 17 + count > ql) invalid("bad DHT");
                const int t = tc * 4 + th;
                bits[t][0] = 0;
                memcpy(bits[t] + 1, q + o + 1, 16);
                memcpy(vals[t], q + o + 17, count);
                have_h[t] = true;
                o += 17 + count;
            }
        } else if (m == 0xDB) {                              // DQT
            size_t o = 0;
            while (o < ql) {
                const int pq = q[o] >> 4, tq = q[o] & 15;
                if (tq > 3 || pq > 1) invalid("bad DQT");
                if (o + 1 + 64 * (pq + 1) > ql) invalid("bad DQT");
                if (pq) return fallback();                   // 16-bit table
                for (int k = 0; k < 64; ++k) f.qt[tq][kZigzagHost[k]] = q[o + 1 + k];
                have_q[tq] = true;
                o += 65;
            }
        } else if (m == 0xDD) {                              // DRI
            if (ql != 2) invalid("bad DRI");
            f.restart = q[0] << 8 | q[1];
        } else if (m == 0xE0) {
            if (ql >= 5 && memcmp(q, "JFIF\0", 5) == 0) jfif = true;
        } else if (m == 0xE1) {
            if (exif_orientation(q, ql) != 1) return fallback();   // cv2.IMREAD_COLOR would rotate the picture
        } else if (m == 0xEE) {
            if (ql >= 5 && memcmp(q, "Adobe", 5) == 0) return fallback();  // colour transform chosen by the marker
        } else if (m == 0xCC || m == 0xDC) {                 // DAC, DNL
            return fallback();
        } else if (m == 0xDA) {                              // SOS: the scan follows
            if (!sof) invalid("scan before the frame header");
            if (ql < 1) invalid("bad SOS");
            const int ns = q[0];
            if (ql != 4 + 2 * (size_t)ns || ns < 1 || ns > f.ncomp) invalid("bad SOS");
            if (ns != f.ncomp) return fallback();           // multi-scan
            bool used_c[3] = {};
            for (int k = 0; k < ns; ++k) {
                int c = 0;
                while (c < f.ncomp && ids[c] != q[1 + 2 * k]) ++c;
                if (c == f.ncomp || used_c[c]) invalid("bad component in SOS");
                used_c[c] = true;
                f.scan[k] = c;
                f.comp[c].td = q[2 + 2 * k] >> 4;
                f.comp[c].ta = q[2 + 2 * k] & 15;
                if (f.comp[c].td > 3 || f.comp[c].ta > 3) invalid("bad table in SOS");
            }
            f.nscan = ns;
            const int ss = q[1 + 2 * ns], se = q[2 + 2 * ns], ah = q[3 + 2 * ns];
            if (ss != 0 || se != 63 || ah != 0) invalid("bad spectral selection for a sequential scan");
            if (rgb_ids && !jfif) return fallback();
            if (f.ncomp == 3) {                              // YCbCr: luma 1x1, 2x1 or 2x2; chroma 1x1
                const Comp& y = f.comp[0];
                if (!((y.h == 1 && y.v == 1) || (y.h == 2 && y.v == 1) || (y.h == 2 && y.v == 2))) return fallback();
                for (int c = 1; c < 3; ++c)
                    if (f.comp[c].h != 1 || f.comp[c].v != 1) return fallback();
            }
            for (int c = 0; c < f.ncomp; ++c) {
                if (!have_q[f.comp[c].tq]) invalid("quantisation table not defined");
                for (int t : {f.comp[c].td, 4 + f.comp[c].ta}) {
                    if (have_h[t]) continue;
                    const int slot = t & 3, ac = t >> 2;
                    if (slot > 1) invalid("Huffman table not defined");
                    memcpy(bits[t], kStdBits[ac * 2 + slot], 17);
                    const uint8_t* v = ac ? (slot ? kStdAcChroma : kStdAcLuma) : kStdDcVals;
                    memcpy(vals[t], v, ac ? 162 : 12);
                    have_h[t] = true;
                }
            }
            for (int t = 0; t < kTables; ++t) {
                if (have_h[t]) derive(bits[t], vals[t], t < 4, f.huff[t]);
                else {
                    for (int l = 0; l < 18; ++l) f.huff[t].maxcode[l] = -1;
                    f.huff[t].maxcode[17] = 0xFFFFF;
                }
            }
            // geometry (jdinput.c initial_setup / per_scan_setup)
            int blocks = 0, plane = 0;
            for (int c = 0; c < f.ncomp; ++c) {
                Comp& k = f.comp[c];
                k.dw = (int)(((long long)f.width * k.h + f.hmax - 1) / f.hmax);
                k.dh = (int)(((long long)f.height * k.v + f.vmax - 1) / f.vmax);
            }
            if (f.ncomp == 1) {
                Comp& k = f.comp[0];
                k.bw = (k.dw + 7) / 8;
                k.bh = (k.dh + 7) / 8;
                f.mcux = k.bw;
                f.mcus = k.bw * k.bh;
            } else {
                f.mcux = (f.width + 8 * f.hmax - 1) / (8 * f.hmax);
                const int mcuy = (f.height + 8 * f.vmax - 1) / (8 * f.vmax);
                f.mcus = f.mcux * mcuy;
                for (int c = 0; c < f.ncomp; ++c) {
                    f.comp[c].bw = f.mcux * f.comp[c].h;
                    f.comp[c].bh = mcuy * f.comp[c].v;
                }
            }
            for (int c = 0; c < f.ncomp; ++c) {
                f.comp[c].coef = blocks;
                f.comp[c].plane = plane;
                blocks += f.comp[c].bw * f.comp[c].bh;
                plane += f.comp[c].bw * f.comp[c].bh * 64;
            }
            f.blocks = blocks;
            // entropy-coded data: destuff, split at RSTn, stop at any other marker or the packet's end
            const int per = f.restart ? f.restart : f.mcus;
            const int expected = (f.mcus + per - 1) / per;
            int found = 0;
            bool bad_rst = false;
            long long begin = (long long)*used;
            auto close = [&]() {
                if (found < expected) {
                    const int first = found * per;
                    segs.push_back(Segment{fi, first, std::min(per, f.mcus - first), 0, begin, (long long)*used});
                }
                ++found;
                begin = (long long)*used;
            };
            while (i < n) {
                const uint8_t b = p[i];
                if (b != 0xFF) {
                    data[(*used)++] = b;
                    ++i;
                    continue;
                }
                size_t j = i + 1;
                while (j < n && p[j] == 0xFF) ++j;           // fill bytes
                if (j >= n) { i = n; break; }
                if (p[j] == 0x00) {
                    data[(*used)++] = 0xFF;
                    i = j + 1;
                    continue;
                }
                if (p[j] >= 0xD0 && p[j] <= 0xD7) {
                    if (p[j] != 0xD0 + (found & 7)) bad_rst = true;
                    close();
                    i = j + 1;
                    continue;
                }
                break;                                       // EOI or another marker: the scan ends
            }
            close();
            if (found != expected || bad_rst) {
                segs.resize(seg_start);
                r.status = kJpegCorrupt;
            }
            return r;                                        // whatever follows the scan does not change this frame
        }
        // APPn, COM and other markers: skipped
    }
}

void apply_roi(const int* roi, int W, int H, int& x0, int& y0, int& w, int& h) {
    auto idx = [](int v, int dim) {                          // one end of a Python slice, step 1
        if (v < 0) v = std::max(v + dim, 0);
        return std::min(v, dim);
    };
    x0 = 0; y0 = 0; w = W; h = H;
    if (!roi) return;
    x0 = idx(roi[0], W);
    y0 = idx(roi[1], H);
    w = std::max(idx(roi[2], W) - x0, 0);
    h = std::max(idx(roi[3], H) - y0, 0);
}

// ---- kernels ---------------------------------------------------------------------------------------------------------
// the lookup tables of every frame, once per frame (a frame with restart markers has many segments)
__global__ void jpeg_lut_kernel(const Frame* frames, uint16_t* luts) {
    const Frame& f = frames[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (f.skip || i >= kTables * kLutSize) return;
    luts[(size_t)blockIdx.y * kTables * kLutSize + i] = lut_entry(f.huff[i / kLutSize], i % kLutSize);
}

// one segment per block; its MCUs are sequential, so one thread decodes them
__global__ void jpeg_entropy_kernel(const Frame* frames, const Segment* segs, const uint8_t* data,
                                    const uint16_t* luts, short* coefs, int* flags) {
    const Segment s = segs[blockIdx.x];
    const uint16_t* lut = luts + (size_t)s.frame * kTables * kLutSize;
    if (!decode_segment(frames[s.frame], data, s.begin, s.end, s.mcu_first, s.mcu_count, lut, coefs))
        atomicOr(flags + s.frame, kJpegCorrupt);
}

__global__ void jpeg_idct_kernel(const Frame* frames, const short* coefs, uint8_t* planes) {
    const Frame& f = frames[blockIdx.y];
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (f.skip || b >= f.blocks) return;
    idct_block(f, b, coefs, planes);
}

__global__ void jpeg_color_kernel(const Frame* frames, const uint8_t* planes, uint8_t* out, int h, int w) {
    const Frame& f = frames[blockIdx.y];
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (f.skip || pix >= h * w) return;
    const int oy = pix / w, ox = pix - oy * w;
    bgr_pixel(f, planes + f.plane_base, f.y0 + oy, f.x0 + ox, out + ((size_t)blockIdx.y * h * w + pix) * 3);
}

template <typename T>
void grow_pinned(T*& p, size_t& cap, size_t need) {
    if (cap >= need) return;
    if (p) cudaFreeHost(p);
    p = nullptr;
    OPB_CUDA(cudaMallocHost((void**)&p, need * sizeof(T)));
    cap = need;
}

template <typename T>
bool grow_dev(T*& p, size_t& cap, size_t need, cudaStream_t st) {
    if (cap >= need) return false;
    OPB_CUDA(cudaStreamSynchronize(st));           // the previous batch may still read it
    if (p) cudaFree(p);
    p = nullptr;
    OPB_CUDA(cudaMalloc((void**)&p, need * sizeof(T)));
    cap = need;
    return true;
}

}  // namespace

struct JpegBatch {
    // pinned host side, reused once the upload of the previous batch has finished (`uploaded`)
    Frame* frames_h = nullptr;
    Segment* segs_h = nullptr;
    uint8_t* data_h = nullptr;
    int* flags_dev_h = nullptr;                     // device flags of the last batch, copied back behind its kernels
    size_t frames_hcap = 0, segs_hcap = 0, data_hcap = 0, flags_hcap = 0;
    std::vector<int> flags_host;                    // flags found at submit
    std::vector<Segment> segs;
    // device side
    Frame* frames_d = nullptr;
    Segment* segs_d = nullptr;
    uint8_t* data_d = nullptr;
    uint16_t* luts = nullptr;                       // [frames][kTables][kLutSize]
    short* coefs = nullptr;
    uint8_t* planes = nullptr;
    uint8_t* out = nullptr;
    int* flags_d = nullptr;
    size_t frames_dcap = 0, segs_dcap = 0, data_dcap = 0, luts_cap = 0, coefs_cap = 0, planes_cap = 0, out_cap = 0, flags_dcap = 0;
    cudaEvent_t uploaded = nullptr, flags_ready = nullptr;
    int n = 0, h = 0, w = 0;
    ~JpegBatch() {
        for (void* p : {(void*)frames_h, (void*)segs_h, (void*)data_h, (void*)flags_dev_h})
            if (p) cudaFreeHost(p);
        for (void* p : {(void*)frames_d, (void*)segs_d, (void*)data_d, (void*)luts, (void*)coefs, (void*)planes, (void*)out,
                        (void*)flags_d})
            if (p) cudaFree(p);
        if (uploaded) cudaEventDestroy(uploaded);
        if (flags_ready) cudaEventDestroy(flags_ready);
    }
};

void jpeg_batch_free(JpegBatch* jb) { delete jb; }

int jpeg_submit(JpegBatch*& jb, int device, cudaStream_t st, const uint8_t* packed, const int64_t* offsets, int n,
                const int* roi, int* flags, uint8_t** dev, int* h, int* w) {
    OPB_REQUIRE(n > 0 && packed && offsets && flags && dev && h && w, "jpeg submit: bad arguments");
    for (int i = 0; i < n; ++i) OPB_REQUIRE(offsets[i] >= 0 && offsets[i] <= offsets[i + 1], "jpeg submit: bad offsets");
    OPB_CUDA(cudaSetDevice(device));
    if (!jb) {
        jb = new JpegBatch();
        OPB_CUDA(cudaEventCreateWithFlags(&jb->uploaded, cudaEventDisableTiming));
        OPB_CUDA(cudaEventCreateWithFlags(&jb->flags_ready, cudaEventDisableTiming));
    } else {
        OPB_CUDA(cudaEventSynchronize(jb->uploaded));        // the pinned buffers still feed the previous upload
    }
    JpegBatch& b = *jb;
    const size_t bytes = (size_t)(offsets[n] - offsets[0]);
    grow_pinned(b.frames_h, b.frames_hcap, (size_t)n);
    grow_pinned(b.data_h, b.data_hcap, bytes + 8);
    b.segs.clear();
    b.flags_host.assign(n, 0);
    size_t used = 0;
    int H = -1, W = -1, first = -1;
    for (int i = 0; i < n; ++i) {
        Frame& f = b.frames_h[i];
        const size_t mark = used, nseg = b.segs.size();
        Parse r;
        try {
            r = parse(packed + offsets[i], (size_t)(offsets[i + 1] - offsets[i]), i, f, b.data_h, &used, b.segs);
        } catch (const Error&) {                              // the host decodes it (and reports what it finds)
            r.status = kJpegFallback;
        }
        if (r.status) {
            used = mark;
            b.segs.resize(nseg);
            f.skip = 1;
            f.blocks = 0;
            b.flags_host[i] = r.status;
        }
        if (r.width > 0 && r.height > 0) {
            if (first < 0) {
                first = i;
                H = r.height;
                W = r.width;
            }
            OPB_REQUIRE(r.width == W && r.height == H, "jpeg submit: packet " + std::to_string(i) + " is " +
                        std::to_string(r.width) + "x" + std::to_string(r.height) + ", packet " + std::to_string(first) +
                        " is " + std::to_string(W) + "x" + std::to_string(H) + ": a batch holds frames of one size");
        }
    }
    OPB_REQUIRE(first >= 0, "jpeg submit: no packet of the batch has a readable frame header");
    int x0, y0, ow, oh;
    apply_roi(roi, W, H, x0, y0, ow, oh);
    OPB_REQUIRE(ow > 0 && oh > 0, "jpeg submit: the ROI is empty");
    long long coef = 0, plane = 0;
    for (int i = 0; i < n; ++i) {
        Frame& f = b.frames_h[i];
        f.x0 = x0;
        f.y0 = y0;
        f.coef_base = coef;
        f.plane_base = plane;
        coef += f.blocks;
        plane += (long long)f.blocks * 64;
    }
    const size_t nseg = b.segs.size();
    grow_pinned(b.segs_h, b.segs_hcap, std::max<size_t>(nseg, 1));
    if (nseg) memcpy(b.segs_h, b.segs.data(), nseg * sizeof(Segment));
    if (b.flags_hcap < (size_t)n) {
        OPB_CUDA(cudaEventSynchronize(b.flags_ready));       // the previous batch's flags may still be copied there
        grow_pinned(b.flags_dev_h, b.flags_hcap, (size_t)n);
    }

    grow_dev(b.frames_d, b.frames_dcap, (size_t)n, st);
    grow_dev(b.segs_d, b.segs_dcap, std::max<size_t>(nseg, 1), st);
    grow_dev(b.data_d, b.data_dcap, used + 8, st);
    grow_dev(b.luts, b.luts_cap, (size_t)n * kTables * kLutSize, st);
    grow_dev(b.coefs, b.coefs_cap, (size_t)std::max<long long>(coef, 1) * 64, st);
    grow_dev(b.planes, b.planes_cap, (size_t)std::max<long long>(plane, 1), st);
    grow_dev(b.out, b.out_cap, (size_t)n * oh * ow * 3, st);
    grow_dev(b.flags_d, b.flags_dcap, (size_t)n, st);

    OPB_CUDA(cudaMemcpyAsync(b.frames_d, b.frames_h, (size_t)n * sizeof(Frame), cudaMemcpyHostToDevice, st));
    if (nseg) OPB_CUDA(cudaMemcpyAsync(b.segs_d, b.segs_h, nseg * sizeof(Segment), cudaMemcpyHostToDevice, st));
    if (used) OPB_CUDA(cudaMemcpyAsync(b.data_d, b.data_h, used, cudaMemcpyHostToDevice, st));
    OPB_CUDA(cudaEventRecord(b.uploaded, st));
    OPB_CUDA(cudaMemsetAsync(b.flags_d, 0, (size_t)n * sizeof(int), st));
    int launches = 0;
    if (coef) {
        OPB_CUDA(cudaMemsetAsync(b.coefs, 0, (size_t)coef * 64 * sizeof(short), st));
        int max_blocks = 0;
        for (int i = 0; i < n; ++i) max_blocks = std::max(max_blocks, b.frames_h[i].blocks);
        jpeg_lut_kernel<<<dim3((unsigned)cdiv(kTables * kLutSize, 256), (unsigned)n), 256, 0, st>>>(b.frames_d, b.luts);
        jpeg_entropy_kernel<<<(unsigned)nseg, 32, 0, st>>>(b.frames_d, b.segs_d, b.data_d, b.luts, b.coefs, b.flags_d);
        jpeg_idct_kernel<<<dim3((unsigned)cdiv(max_blocks, 128), (unsigned)n), 128, 0, st>>>(b.frames_d, b.coefs,
                                                                                              b.planes);
        jpeg_color_kernel<<<dim3((unsigned)cdiv(oh * ow, 256), (unsigned)n), 256, 0, st>>>(b.frames_d, b.planes, b.out,
                                                                                            oh, ow);
        OPB_CUDA(cudaGetLastError());
        launches = 4;
    }
    OPB_CUDA(cudaMemcpyAsync(b.flags_dev_h, b.flags_d, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, st));
    OPB_CUDA(cudaEventRecord(b.flags_ready, st));
    b.n = n;
    b.h = oh;
    b.w = ow;
    for (int i = 0; i < n; ++i) flags[i] = b.flags_host[i];
    *dev = b.out;
    *h = oh;
    *w = ow;
    return launches;
}

void jpeg_upload(JpegBatch* jb, cudaStream_t st, int index, const uint8_t* frame) {
    OPB_REQUIRE(jb && jb->n > 0, "jpeg upload: no batch submitted");
    OPB_REQUIRE(index >= 0 && index < jb->n && frame, "jpeg upload: bad frame index");
    const size_t bytes = (size_t)jb->h * jb->w * 3;
    OPB_CUDA(cudaMemcpyAsync(jb->out + bytes * index, frame, bytes, cudaMemcpyHostToDevice, st));
}

void jpeg_fetch(JpegBatch* jb, cudaStream_t st, uint8_t* host) {
    OPB_REQUIRE(jb && jb->n > 0 && host, "jpeg fetch: no batch submitted");
    OPB_CUDA(cudaMemcpyAsync(host, jb->out, (size_t)jb->n * jb->h * jb->w * 3, cudaMemcpyDeviceToHost, st));
    OPB_CUDA(cudaStreamSynchronize(st));
}

void jpeg_status(JpegBatch* jb, int* flags) {
    OPB_REQUIRE(jb && jb->n > 0 && flags, "jpeg status: no batch submitted");
    OPB_CUDA(cudaEventSynchronize(jb->flags_ready));
    for (int i = 0; i < jb->n; ++i) flags[i] = jb->flags_host[i] | jb->flags_dev_h[i];
}

void jpeg_decode_host(const uint8_t* packet, int64_t size, const int* roi, uint8_t* out, int64_t out_bytes, int* h,
                      int* w, int* status) {
    OPB_REQUIRE(packet && size >= 0 && h && w && status, "jpeg decode: bad arguments");
    std::unique_ptr<Frame> fp(new Frame());
    Frame& f = *fp;
    std::vector<uint8_t> data((size_t)size + 8);
    std::vector<Segment> segs;
    size_t used = 0;
    const Parse r = parse(packet, (size_t)size, 0, f, data.data(), &used, segs);
    int x0 = 0, y0 = 0, ow = 0, oh = 0;
    if (r.width > 0 && r.height > 0) apply_roi(roi, r.width, r.height, x0, y0, ow, oh);
    *h = oh;
    *w = ow;
    *status = r.status;
    if (r.status || !out) return;
    if (out_bytes < (int64_t)oh * ow * 3)
        throw Error(OPB_ERR_CAPACITY, "jpeg decode: the output holds " + std::to_string(out_bytes) + " bytes, the frame needs " +
                    std::to_string((int64_t)oh * ow * 3));
    std::vector<uint16_t> luts(kTables * kLutSize);
    for (int i = 0; i < kTables * kLutSize; ++i) luts[i] = lut_entry(f.huff[i / kLutSize], i % kLutSize);
    std::vector<short> coefs((size_t)f.blocks * 64, 0);
    std::vector<uint8_t> planes((size_t)f.blocks * 64);
    for (const Segment& s : segs)
        if (!decode_segment(f, data.data(), s.begin, s.end, s.mcu_first, s.mcu_count, luts.data(), coefs.data()))
            *status = kJpegCorrupt;
    for (int b = 0; b < f.blocks; ++b) idct_block(f, b, coefs.data(), planes.data());
    for (int y = 0; y < oh; ++y)
        for (int x = 0; x < ow; ++x) bgr_pixel(f, planes.data(), y0 + y, x0 + x, out + ((size_t)y * ow + x) * 3);
}

}  // namespace opb
