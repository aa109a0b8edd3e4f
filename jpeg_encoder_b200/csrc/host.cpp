// Host-side planner: see host.h. Citations are into /root/reference/src.
#include "host.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>

namespace jpgb {

// Figure A.6 zig-zag sequence (writer.rs:64-68): natural index of zig-zag position i
const uint8_t kZigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,
                             12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,  7,  14, 21, 28,
                             35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
                             58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

int bytes_per_pixel(uint8_t ct) { // encoder.rs:101-111
    if (ct == JPGB_LUMA) return 1;
    if (ct == JPGB_RGB || ct == JPGB_BGR || ct == JPGB_YCBCR) return 3;
    return 4;
}
int num_components(uint8_t ct) { // adaptors' get_jpeg_color_type + encoder.rs:55-65
    if (ct == JPGB_LUMA) return 1;
    if (ct <= JPGB_YCBCR) return 3;
    return 4;
}

// ---- quantization tables (quantization.rs:62-183, mozjpeg jcparam.c families) ------------------
namespace {
// index order = QuantizationTableType::index(). Rows: luma then chroma for each family.
const uint16_t kBaseTables[9][2][64] = {
    {{16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
      14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
      49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99},
     {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99,
      47, 66, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
      99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99}},
    {{16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16,
      16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16,
      16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16},
     {16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16,
      16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16,
      16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 16}},
    {{12, 17, 20, 21, 30, 34, 56, 63, 18, 20, 20, 26, 28, 51, 61, 55, 19, 20, 21, 26, 33, 58, 69, 55,
      26, 26, 26, 30, 46, 87, 86, 66, 31, 33, 36, 40, 46, 96, 100, 73, 40, 35, 46, 62, 81, 100, 111, 91,
      46, 66, 76, 86, 102, 121, 120, 101, 68, 90, 90, 96, 113, 102, 105, 103},
     {8, 12, 15, 15, 86, 96, 96, 98, 13, 13, 15, 26, 90, 96, 99, 98, 12, 15, 18, 96, 99, 99, 99, 99,
      17, 16, 90, 96, 99, 99, 99, 99, 96, 96, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
      99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99}},
    {{9, 10, 12, 14, 27, 32, 51, 62, 11, 12, 14, 19, 27, 44, 59, 73, 12, 14, 18, 25, 42, 59, 79, 78,
      17, 18, 25, 42, 61, 92, 87, 92, 23, 28, 42, 75, 79, 112, 112, 99, 40, 42, 59, 84, 88, 124, 132, 111,
      42, 64, 78, 95, 105, 126, 125, 99, 70, 75, 100, 102, 116, 100, 107, 98},
     {9, 10, 17, 19, 62, 89, 91, 97, 12, 13, 18, 29, 84, 91, 88, 98, 14, 19, 29, 93, 95, 95, 98, 97,
      20, 26, 84, 88, 95, 95, 98, 94, 26, 86, 91, 93, 97, 99, 98, 99, 99, 100, 98, 99, 99, 99, 99, 99,
      99, 99, 99, 99, 99, 99, 99, 99, 97, 97, 99, 99, 99, 99, 97, 99}},
    {{16, 16, 16, 18, 25, 37, 56, 85, 16, 17, 20, 27, 34, 40, 53, 75, 16, 20, 24, 31, 43, 62, 91, 135,
      18, 27, 31, 40, 53, 74, 106, 156, 25, 34, 43, 53, 69, 94, 131, 189, 37, 40, 62, 74, 94, 124, 169, 238,
      56, 53, 91, 106, 131, 169, 226, 311, 85, 75, 135, 156, 189, 238, 311, 418},
     {16, 16, 16, 18, 25, 37, 56, 85, 16, 17, 20, 27, 34, 40, 53, 75, 16, 20, 24, 31, 43, 62, 91, 135,
      18, 27, 31, 40, 53, 74, 106, 156, 25, 34, 43, 53, 69, 94, 131, 189, 37, 40, 62, 74, 94, 124, 169, 238,
      56, 53, 91, 106, 131, 169, 226, 311, 85, 75, 135, 156, 189, 238, 311, 418}},
    {{10, 12, 14, 19, 26, 38, 57, 86, 12, 18, 21, 28, 35, 41, 54, 76, 14, 21, 25, 32, 44, 63, 92, 136,
      19, 28, 32, 41, 54, 75, 107, 157, 26, 35, 44, 54, 70, 95, 132, 190, 38, 41, 63, 75, 95, 125, 170, 239,
      57, 54, 92, 107, 132, 170, 227, 312, 86, 76, 136, 157, 190, 239, 312, 419},
     {10, 12, 14, 19, 26, 38, 57, 86, 12, 18, 21, 28, 35, 41, 54, 76, 14, 21, 25, 32, 44, 63, 92, 136,
      19, 28, 32, 41, 54, 75, 107, 157, 26, 35, 44, 54, 70, 95, 132, 190, 38, 41, 63, 75, 95, 125, 170, 239,
      57, 54, 92, 107, 132, 170, 227, 312, 86, 76, 136, 157, 190, 239, 312, 419}},
    {{7, 8, 10, 14, 23, 44, 95, 241, 8, 8, 11, 15, 25, 47, 102, 255, 10, 11, 13, 19, 31, 58, 127, 255,
      14, 15, 19, 27, 44, 83, 181, 255, 23, 25, 31, 44, 72, 136, 255, 255, 44, 47, 58, 83, 136, 255, 255, 255,
      95, 102, 127, 181, 255, 255, 255, 255, 241, 255, 255, 255, 255, 255, 255, 255},
     {7, 8, 10, 14, 23, 44, 95, 241, 8, 8, 11, 15, 25, 47, 102, 255, 10, 11, 13, 19, 31, 58, 127, 255,
      14, 15, 19, 27, 44, 83, 181, 255, 23, 25, 31, 44, 72, 136, 255, 255, 44, 47, 58, 83, 136, 255, 255, 255,
      95, 102, 127, 181, 255, 255, 255, 255, 241, 255, 255, 255, 255, 255, 255, 255}},
    {{15, 11, 11, 12, 15, 19, 25, 32, 11, 13, 10, 10, 12, 15, 19, 24, 11, 10, 14, 14, 16, 18, 22, 27,
      12, 10, 14, 18, 21, 24, 28, 33, 15, 12, 16, 21, 26, 31, 36, 42, 19, 15, 18, 24, 31, 38, 45, 53,
      25, 19, 22, 28, 36, 45, 55, 65, 32, 24, 27, 33, 42, 53, 65, 77},
     {15, 11, 11, 12, 15, 19, 25, 32, 11, 13, 10, 10, 12, 15, 19, 24, 11, 10, 14, 14, 16, 18, 22, 27,
      12, 10, 14, 18, 21, 24, 28, 33, 15, 12, 16, 21, 26, 31, 36, 42, 19, 15, 18, 24, 31, 38, 45, 53,
      25, 19, 22, 28, 36, 45, 55, 65, 32, 24, 27, 33, 42, 53, 65, 77}},
    {{14, 10, 11, 14, 19, 25, 34, 45, 10, 11, 11, 12, 15, 20, 26, 33, 11, 11, 15, 18, 21, 25, 31, 38,
      14, 12, 18, 24, 28, 33, 39, 47, 19, 15, 21, 28, 36, 43, 51, 59, 25, 20, 25, 33, 43, 54, 64, 74,
      34, 26, 31, 39, 51, 64, 77, 91, 45, 33, 38, 47, 59, 74, 91, 108},
     {14, 10, 11, 14, 19, 25, 34, 45, 10, 11, 11, 12, 15, 20, 26, 33, 11, 11, 15, 18, 21, 25, 31, 38,
      14, 12, 18, 24, 28, 33, 39, 47, 19, 15, 21, 28, 36, 43, 51, 59, 25, 20, 25, 33, 43, 54, 64, 74,
      34, 26, 31, 39, 51, 64, 77, 91, 45, 33, 38, 47, 59, 74, 91, 108}},
};

// quantization.rs:187-207: 15-bit reciprocal with rounding correction
void reciprocal_for(uint32_t divisor, int32_t &recip, int32_t &corr) {
    if (divisor <= 1) {
        recip = 1;
        corr = 0;
        return;
    }
    uint32_t r = 32768u / divisor, frac = 32768u % divisor, c = divisor / 2;
    if (frac != 0) {
        if (frac <= c) ++c;
        else ++r;
    }
    recip = (int32_t)r;
    corr = (int32_t)c;
}

// QuantizationTable::new_with_quality, quantization.rs:216-283
void make_quant_table(uint8_t kind, const uint16_t custom[64], uint8_t quality, bool luma, QuantTable &t) {
    if (kind == JPGB_QT_CUSTOM) {
        for (int i = 0; i < 64; ++i) {
            uint16_t v = std::min<uint16_t>(std::max<uint16_t>(custom[i], 1), 2 << 10);
            t.value[i] = (uint16_t)(v << 3);
        }
    } else {
        uint32_t q = std::min<uint32_t>(std::max<uint32_t>(quality, 1), 100);
        uint32_t scale = q < 50 ? 5000 / q : 200 - 2 * q;
        const uint16_t *base = kBaseTables[kind][luma ? 0 : 1];
        for (int i = 0; i < 64; ++i) {
            uint32_t v = (base[i] * scale + 50) / 100;
            v = std::min<uint32_t>(std::max<uint32_t>(v, 1), 255);
            t.value[i] = (uint16_t)(v << 3);
        }
    }
    for (int i = 0; i < 64; ++i) reciprocal_for(t.value[i], t.recip[i], t.corr[i]);
}

void put16(std::vector<uint8_t> &o, uint32_t v) {
    o.push_back((uint8_t)(v >> 8));
    o.push_back((uint8_t)v);
}
void put_marker(std::vector<uint8_t> &o, uint8_t m) {
    o.push_back(0xFF);
    o.push_back(m);
}
void put_segment(std::vector<uint8_t> &o, uint8_t marker, const uint8_t *data, size_t n) { // writer.rs:208-214
    put_marker(o, marker);
    put16(o, (uint32_t)n + 2);
    o.insert(o.end(), data, data + n);
}
} // namespace

// ---- Huffman tables (huffman.rs) -----------------------------------------------------------------
bool HuffTable::device_words(bool ac, uint32_t out[256]) const {
    for (int s = 0; s < 256; ++s) {
        const uint32_t len = lookup[s] >> 16, code = lookup[s] & 0xFFFFu;
        const uint32_t z = ac ? (uint32_t)(s & 15) : (uint32_t)s;
        if (!ac && s > 15) {
            out[s] = 0; // DC categories are 0..15
            continue;
        }
        if (len && (len + z > 31 || ((uint64_t)code << z) >> 27)) return false;
        out[s] = ((len + z) << 27) | (code << z);
    }
    return true;
}

void HuffTable::set(const uint8_t len[16], const uint8_t *vals, size_t n) {
    std::memcpy(length, len, 16);
    values.assign(vals, vals + n);
    // Figures C.1-C.3 (huffman.rs:240-288): canonical codes in order of `values`
    std::memset(lookup, 0, sizeof(lookup));
    uint32_t code = 0;
    size_t k = 0;
    for (int bits = 1; bits <= 16; ++bits) {
        for (int j = 0; j < length[bits - 1] && k < n; ++j, ++k) {
            lookup[values[k]] = ((uint32_t)bits << 16) | (code & 0xFFFF);
            ++code;
        }
        code <<= 1;
    }
}

bool HuffTable::set_optimized(const uint32_t freq_in[257]) {
    uint32_t freq[257];
    int others[257];
    uint32_t codesize[257];
    std::memcpy(freq, freq_in, sizeof(freq));
    std::fill(others, others + 257, -1);
    std::fill(codesize, codesize + 257, 0u);
    for (;;) { // Figure K.1; ties go to the largest index (`<=` while scanning upward)
        int v1 = -1, v2 = -1;
        uint32_t m1 = UINT32_MAX, m2 = UINT32_MAX;
        for (int i = 0; i < 257; ++i)
            if (freq[i] && freq[i] <= m1) m1 = freq[i], v1 = i;
        if (v1 < 0) break;
        for (int i = 0; i < 257; ++i)
            if (freq[i] && freq[i] <= m2 && i != v1) m2 = freq[i], v2 = i;
        if (v2 < 0) break;
        freq[v1] += freq[v2];
        freq[v2] = 0;
        for (++codesize[v1]; others[v1] >= 0;) v1 = others[v1], ++codesize[v1];
        others[v1] = v2;
        for (++codesize[v2]; others[v2] >= 0;) v2 = others[v2], ++codesize[v2];
    }
    uint8_t bits[33] = {0}; // Figure K.2
    bool any = false;
    for (int i = 0; i < 257; ++i) {
        if (codesize[i] > 32) return false;
        if (codesize[i]) ++bits[codesize[i]], any = true;
    }
    if (!any) return false; // nothing but the reserved code point: the reference indexes out of bounds and panics
    int i = 32; // Figure K.3
    for (; i > 16; --i)
        while (bits[i] > 0) {
            int j = i - 2;
            while (bits[j] == 0) --j;
            bits[i] -= 2;
            bits[i - 1] += 1;
            bits[j + 1] += 2;
            bits[j] -= 1;
        }
    while (bits[i] == 0) --i;
    --bits[i]; // drop the reserved all-ones code point
    uint8_t vals[256]; // Figure K.4: by code size, then symbol value
    size_t k = 0;
    for (uint32_t sz = 1; sz <= 32; ++sz)
        for (int j = 0; j < 256; ++j)
            if (codesize[j] == sz) vals[k++] = (uint8_t)j;
    uint8_t len[16];
    for (int l = 0; l < 16; ++l) len[l] = bits[l + 1];
    set(len, vals, k);
    return true;
}

void default_huffman_tables(HuffTable huff[2][2]) {
    static const uint8_t dc_vals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
    static const uint8_t luma_dc_len[16] = {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0};
    static const uint8_t chroma_dc_len[16] = {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0};
    static const uint8_t luma_ac_len[16] = {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7D};
    static const uint8_t chroma_ac_len[16] = {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77};
    static const uint8_t luma_ac_vals[162] = {
        0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71,
        0x14, 0x32, 0x81, 0x91, 0xA1, 0x08, 0x23, 0x42, 0xB1, 0xC1, 0x15, 0x52, 0xD1, 0xF0, 0x24, 0x33, 0x62, 0x72,
        0x82, 0x09, 0x0A, 0x16, 0x17, 0x18, 0x19, 0x1A, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2A, 0x34, 0x35, 0x36, 0x37,
        0x38, 0x39, 0x3A, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4A, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
        0x5A, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6A, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7A, 0x83,
        0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8A, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9A, 0xA2, 0xA3,
        0xA4, 0xA5, 0xA6, 0xA7, 0xA8, 0xA9, 0xAA, 0xB2, 0xB3, 0xB4, 0xB5, 0xB6, 0xB7, 0xB8, 0xB9, 0xBA, 0xC2, 0xC3,
        0xC4, 0xC5, 0xC6, 0xC7, 0xC8, 0xC9, 0xCA, 0xD2, 0xD3, 0xD4, 0xD5, 0xD6, 0xD7, 0xD8, 0xD9, 0xDA, 0xE1, 0xE2,
        0xE3, 0xE4, 0xE5, 0xE6, 0xE7, 0xE8, 0xE9, 0xEA, 0xF1, 0xF2, 0xF3, 0xF4, 0xF5, 0xF6, 0xF7, 0xF8, 0xF9, 0xFA};
    static const uint8_t chroma_ac_vals[162] = {
        0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22,
        0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xA1, 0xB1, 0xC1, 0x09, 0x23, 0x33, 0x52, 0xF0, 0x15, 0x62, 0x72, 0xD1,
        0x0A, 0x16, 0x24, 0x34, 0xE1, 0x25, 0xF1, 0x17, 0x18, 0x19, 0x1A, 0x26, 0x27, 0x28, 0x29, 0x2A, 0x35, 0x36,
        0x37, 0x38, 0x39, 0x3A, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4A, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
        0x59, 0x5A, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6A, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7A,
        0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8A, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9A,
        0xA2, 0xA3, 0xA4, 0xA5, 0xA6, 0xA7, 0xA8, 0xA9, 0xAA, 0xB2, 0xB3, 0xB4, 0xB5, 0xB6, 0xB7, 0xB8, 0xB9, 0xBA,
        0xC2, 0xC3, 0xC4, 0xC5, 0xC6, 0xC7, 0xC8, 0xC9, 0xCA, 0xD2, 0xD3, 0xD4, 0xD5, 0xD6, 0xD7, 0xD8, 0xD9, 0xDA,
        0xE2, 0xE3, 0xE4, 0xE5, 0xE6, 0xE7, 0xE8, 0xE9, 0xEA, 0xF2, 0xF3, 0xF4, 0xF5, 0xF6, 0xF7, 0xF8, 0xF9, 0xFA};
    huff[0][0].set(luma_dc_len, dc_vals, 12);
    huff[0][1].set(luma_ac_len, luma_ac_vals, 162);
    huff[1][0].set(chroma_dc_len, dc_vals, 12);
    huff[1][1].set(chroma_ac_len, chroma_ac_vals, 162);
}

// ---- plan ---------------------------------------------------------------------------------------
int Plan::build(const jpgb_params &params, const jpgb_strip *st) {
    p = params;
    is_strip = st != nullptr;
    if (st) {
        strip = *st;
        p.height = st->rows; // geometry below is the strip's; the SOF carries strip.full_height
    }
    if (p.color_type > JPGB_YCCK) return JPGB_ERR_BAD_PARAMS;
    const int sh = (p.sampling >> 4) & 0x07, sv = p.sampling & 0x0f; // get_sampling_factors, encoder.rs:173-176
    auto pow2 = [](int f) { return f == 1 || f == 2 || f == 4; };
    if (!pow2(sh) || !pow2(sv) || (sh == 4 && sv == 4)) return JPGB_ERR_BAD_PARAMS; // the 8 SamplingFactor variants
    if (p.progressive_scans == 1 || p.progressive_scans > 64) return JPGB_ERR_BAD_PARAMS; // encoder.rs:329-333
    if (p.qtable_kind[0] > JPGB_QT_CUSTOM || p.qtable_kind[1] > JPGB_QT_CUSTOM) return JPGB_ERR_BAD_PARAMS;
    for (uint32_t i = 0; i < p.n_app; ++i) { // encoder.rs:374-383
        if (p.apps[i].nr == 0 || p.apps[i].nr > 15) return JPGB_ERR_INVALID_APP_SEGMENT;
        if (p.apps[i].len > 65533) return JPGB_ERR_APP_SEGMENT_TOO_LARGE;
    }
    if (p.width == 0 || p.height == 0) return JPGB_ERR_ZERO_DIMENSIONS;

    bpp = bytes_per_pixel(p.color_type);
    ncomp = num_components(p.color_type);

    // init_components, encoder.rs:569-619: the sampling factor applies to luma (and K)
    auto comp = [](uint8_t id, uint8_t tbl, int h, int v) { return Component{id, tbl, tbl, tbl, (uint8_t)h, (uint8_t)v}; };
    if (ncomp == 1) {
        comps[0] = comp(0, 0, 1, 1);
    } else if (ncomp == 3) {
        comps[0] = comp(0, 0, sh, sv);
        comps[1] = comp(1, 1, 1, 1);
        comps[2] = comp(2, 1, 1, 1);
    } else if (p.color_type == JPGB_CMYK) {
        comps[0] = comp(0, 1, 1, 1);
        comps[1] = comp(1, 1, 1, 1);
        comps[2] = comp(2, 1, 1, 1);
        comps[3] = comp(3, 0, sh, sv);
    } else {
        comps[0] = comp(0, 0, sh, sv);
        comps[1] = comp(1, 1, 1, 1);
        comps[2] = comp(2, 1, 1, 1);
        comps[3] = comp(3, 0, sh, sv);
    }
    hmax = vmax = 1;
    for (int c = 0; c < ncomp; ++c) hmax = std::max<int>(hmax, comps[c].h), vmax = std::max<int>(vmax, comps[c].v);

    mcu_cols = (p.width + 8 * hmax - 1) / (8 * hmax); // encoder.rs:713-714
    mcu_rows = (p.height + 8 * vmax - 1) / (8 * vmax);
    const uint32_t bw = (p.width + 7) / 8, bh = (p.height + 7) / 8; // encoder.rs:1012-1013
    for (int c = 0; c < ncomp; ++c) {
        pad_w[c] = mcu_cols * comps[c].h;
        pad_h[c] = mcu_rows * comps[c].v;
        const uint32_t hs = hmax / comps[c].h, vs = vmax / comps[c].v; // encoder.rs:1021-1025
        true_w[c] = (bw + hs - 1) / hs;
        true_h[c] = (bh + vs - 1) / vs;
    }
    for (int c = ncomp; c < 4; ++c) pad_w[c] = pad_h[c] = true_w[c] = true_h[c] = 0, block_off[c] = 0;

    make_quant_table(p.qtable_kind[0], p.qtable_custom[0], p.quality, true, q[0]);  // encoder.rs:528-531
    make_quant_table(p.qtable_kind[1], p.qtable_custom[1], p.quality, false, q[1]);

    // mode switch, encoder.rs:556-562 (supports_interleaved: factors 1 and 2 only, :178-187)
    const bool interleavable = sh <= 2 && sv <= 2;
    if (p.progressive_scans) mode = Mode::Progressive;
    else if (p.optimize_huffman || !interleavable) mode = Mode::Sequential;
    else mode = Mode::Interleaved;

    // coefficient layout follows the scan order of the mode, so that a scan reads its blocks linearly
    blocks_per_image = 0;
    bpu_interleaved = 0;
    for (int c = 0; c < ncomp; ++c) {
        slot_base[c] = bpu_interleaved;
        bpu_interleaved += comps[c].h * comps[c].v;
    }
    if (mode == Mode::Interleaved) {
        for (int c = 0; c < ncomp; ++c) block_off[c] = 0;
        blocks_per_image = (uint64_t)mcu_cols * mcu_rows * bpu_interleaved;
    } else {
        for (int c = 0; c < ncomp; ++c) {
            block_off[c] = blocks_per_image;
            blocks_per_image += (uint64_t)true_w[c] * true_h[c];
        }
    }

    // scans, with their SOS segments (writer.rs:424-452; Ah/Al always 0)
    scans.clear();
    auto sos_for = [&](int c, int ss, int se) {
        std::vector<uint8_t> s;
        put_marker(s, 0xDA);
        const int n = c < 0 ? ncomp : 1;
        put16(s, 2 + 1 + n * 2 + 3);
        s.push_back((uint8_t)n);
        for (int i = 0; i < ncomp; ++i)
            if (c < 0 || c == i) {
                s.push_back(comps[i].id);
                s.push_back((uint8_t)((comps[i].dc_table << 4) | comps[i].ac_table));
            }
        s.push_back((uint8_t)ss);
        s.push_back((uint8_t)se);
        s.push_back(0);
        return s;
    };
    auto add_scan = [&](int c, int ss, int se) {
        Scan s;
        s.comp = c;
        s.ss = ss;
        s.se = se;
        if (c < 0) {
            s.n_units = mcu_cols * mcu_rows;
            s.blocks_per_unit = 0;
            for (int i = 0; i < ncomp; ++i) s.blocks_per_unit += comps[i].h * comps[i].v;
        } else {
            s.n_units = true_w[c] * true_h[c];
            s.blocks_per_unit = 1;
        }
        s.sos = sos_for(c, ss, se);
        scans.push_back(std::move(s));
    };
    if (mode == Mode::Interleaved) {
        add_scan(-1, 0, 63);
    } else if (mode == Mode::Sequential) {
        for (int c = 0; c < ncomp; ++c) add_scan(c, 0, 63);
    } else { // encoder.rs:885-972
        for (int c = 0; c < ncomp; ++c) add_scan(c, 0, 0);
        const int bands = p.progressive_scans - 1, per = 64 / bands;
        for (int b = 0; b < bands; ++b) {
            const int start = std::max(b * per, 1), end = b == bands - 1 ? 64 : (b + 1) * per;
            for (int c = 0; c < ncomp; ++c) add_scan(c, start, end - 1);
        }
    }
    if (is_strip) {
        if ((p.restart_interval == 0) != contiguous) return JPGB_ERR_BAD_PARAMS;
        if (strip.n_strips == 0 || strip.strip_index >= strip.n_strips || strip.rows == 0) return JPGB_ERR_BAD_PARAMS;
        if (strip.first_row % (8 * vmax) != 0 || (uint32_t)strip.first_row + strip.rows > strip.full_height) return JPGB_ERR_BAD_PARAMS;
        if (strip.strip_index + 1 < strip.n_strips && strip.rows % (8 * vmax) != 0) return JPGB_ERR_BAD_PARAMS;
        const uint32_t mcu_row0 = strip.first_row / (8 * vmax);
        for (Scan &s : scans) {
            if (contiguous) break;
            const uint64_t first_unit = s.comp < 0 ? (uint64_t)mcu_row0 * mcu_cols : (uint64_t)mcu_row0 * comps[s.comp].v * true_w[s.comp];
            if (first_unit % p.restart_interval != 0) return JPGB_ERR_BAD_PARAMS;
            s.rst_base = (uint32_t)(first_unit / p.restart_interval);
        }
    }
    visits_per_image = 0;
    segs_per_image = 0;
    for (Scan &s : scans) {
        s.visit_base = visits_per_image;
        s.seg_base = segs_per_image;
        s.n_segs = p.restart_interval ? (s.n_units + p.restart_interval - 1) / p.restart_interval : 1;
        visits_per_image += (uint64_t)s.n_units * s.blocks_per_unit;
        segs_per_image += s.n_segs;
    }

    // ---- coding chunks ----
    n_groups = mode == Mode::Interleaved ? 1 : (uint32_t)ncomp;
    scans_per_group = (uint32_t)scans.size() / n_groups;
    uint64_t sv_max = 0;
    for (uint32_t g = 0; g < n_groups; ++g) {
        const Scan &s0 = scans[g];
        Group &G = groups[g];
        G.comp = s0.comp;
        G.bpu = s0.blocks_per_unit;
        G.n_visits = (uint64_t)s0.n_units * s0.blocks_per_unit;
        G.block_base = s0.comp < 0 ? 0 : block_off[s0.comp];
        const uint64_t sv = p.restart_interval ? std::min<uint64_t>((uint64_t)p.restart_interval * G.bpu, G.n_visits) : G.n_visits;
        G.seg_visits = (uint32_t)(p.restart_interval ? (uint64_t)p.restart_interval * G.bpu : G.n_visits);
        G.n_segs = s0.n_segs;
        sv_max = std::max(sv_max, sv);
    }
    {   // the largest CTA size whose chunks are filled nearly as well as the best size fills them. 128 is the largest
        // used by default: measured on B200 (1080p 4:2:0 batch) the coding kernel is 8 % faster with 128 than with
        // 256 visits per CTA -- fewer warps wait at each barrier for the warp that drew the chunk's busiest blocks.
        uint32_t cap = 128;
        if (const char *e = std::getenv("JPGB_CHUNK_T")) { // tuning hook
            const uint32_t v = (uint32_t)std::atoi(e);
            if (v == 32 || v == 64 || v == 128 || v == 256) cap = v;
        }
        auto eff = [&](uint32_t T) { return (double)sv_max / (double)((sv_max + T - 1) / T * T); };
        double best = 0;
        for (uint32_t T : {256u, 128u, 64u, 32u})
            if (T <= cap) best = std::max(best, eff(T));
        chunk_T = 32;
        for (uint32_t T : {256u, 128u, 64u, 32u})
            if (T <= cap && eff(T) >= 0.8 * best) {
                chunk_T = T;
                break;
            }
    }
    items_per_image = 0;
    for (uint32_t g = 0; g < n_groups; ++g) {
        Group &G = groups[g];
        const uint64_t sv = std::min<uint64_t>(G.seg_visits, G.n_visits);
        G.cps = (uint32_t)((sv + chunk_T - 1) / chunk_T);
        G.item_base = items_per_image;
        items_per_image += G.n_segs * G.cps;
    }
    chunks_per_image = 0;
    for (size_t k = 0; k < scans.size(); ++k) {
        const Group &G = groups[k % n_groups];
        scans[k].chunk_base = chunks_per_image;
        chunks_per_image += G.n_segs * G.cps;
    }

    // SOI, JFIF APP0, [Adobe APP14], user APPn  (encoder.rs:536-554, writer.rs:216-239)
    prefix.clear();
    put_marker(prefix, 0xD8);
    put_marker(prefix, 0xE0);
    put16(prefix, 16);
    const uint8_t jfif[7] = {'J', 'F', 'I', 'F', 0, 0x01, 0x02};
    prefix.insert(prefix.end(), jfif, jfif + 7);
    prefix.push_back(p.density_unit == 1 ? 1 : (p.density_unit == 2 ? 2 : 0));
    put16(prefix, p.density_x);
    put16(prefix, p.density_y);
    prefix.push_back(0);
    prefix.push_back(0);
    if (ncomp == 4) {
        uint8_t adobe[12] = {'A', 'd', 'o', 'b', 'e', 0, 0, 0, 0, 0, 0, 0};
        adobe[11] = p.color_type == JPGB_CMYK ? 0 : 2;
        put_segment(prefix, 0xEE, adobe, 12);
    }
    for (uint32_t i = 0; i < p.n_app; ++i) put_segment(prefix, (uint8_t)(0xE0 + p.apps[i].nr), p.apps[i].data, p.apps[i].len);
    return JPGB_OK;
}

void Plan::join(uint32_t world) {
    join_world = world;
    for (size_t k = 0; k < scans.size(); ++k) scans[k].chunk_base = (uint32_t)(k * world);
    for (uint32_t g = 0; g < n_groups; ++g) groups[g].cps = world;
    chunks_per_image = (uint32_t)scans.size() * world;
}

void Plan::frame_header(const HuffTable huff[2][2], std::vector<uint8_t> &o) const {
    put_marker(o, p.progressive_scans ? 0xC2 : 0xC0); // writer.rs:390-422
    put16(o, 2 + 1 + 2 + 2 + 1 + ncomp * 3);
    o.push_back(8);
    put16(o, is_strip ? strip.full_height : p.height);
    put16(o, p.width);
    o.push_back((uint8_t)ncomp);
    for (int c = 0; c < ncomp; ++c) {
        o.push_back(comps[c].id);
        o.push_back((uint8_t)((comps[c].h << 4) | comps[c].v));
        o.push_back(comps[c].qtable);
    }
    for (int t = 0; t < 2; ++t) { // both DQT always, 8-bit precision, truncated value (Q10)  writer.rs:283-300
        put_marker(o, 0xDB);
        put16(o, 2 + 1 + 64);
        o.push_back((uint8_t)t);
        for (int i = 0; i < 64; ++i) o.push_back(q[t].dqt_byte(kZigzag[i]));
    }
    const int n_tables = ncomp >= 3 ? 2 : 1; // encoder.rs:648-660
    for (int t = 0; t < n_tables; ++t)
        for (int cls = 0; cls < 2; ++cls) { // writer.rs:253-269
            const HuffTable &h = huff[t][cls];
            put_marker(o, 0xC4);
            put16(o, 2 + 1 + 16 + (uint32_t)h.values.size());
            o.push_back((uint8_t)((cls << 4) | t));
            o.insert(o.end(), h.length, h.length + 16);
            o.insert(o.end(), h.values.begin(), h.values.end());
        }
    if (p.restart_interval) { // writer.rs:302-306
        put_marker(o, 0xDD);
        put16(o, 4);
        put16(o, p.restart_interval);
    }
}

void Plan::fill_device_plan(DevPlan &d) const {
    std::memset(&d, 0, sizeof(d));
    d.n_scans = (int)scans.size();
    d.ncomp = ncomp;
    d.restart = p.restart_interval;
    d.n_groups = (int)n_groups;
    d.spg = (int)scans_per_group;
    d.chunk_T = (int)chunk_T;
    d.mcu_order = mode == Mode::Interleaved;
    d.mcu_cols = mcu_cols;
    d.blocks_per_image = blocks_per_image;
    d.segs_per_image = segs_per_image;
    d.chunks_per_image = chunks_per_image;
    d.items_per_image = items_per_image;
    d.div_items = make_fastdiv(items_per_image);
    d.has_eoi = !is_strip || (!contiguous && strip.strip_index + 1 == strip.n_strips);
    d.bare = contiguous;
    int n = 0;
    for (int c = 0; c < ncomp; ++c) {
        d.comp_tbl[c] = comps[c].dc_table;
        const int per_mcu = comps[c].h * comps[c].v;
        for (int i = 0; i < per_mcu; ++i) { // MCU order: component, then v outer, h inner (encoder.rs:759-761)
            d.slot_comp[n] = (int8_t)c;
            d.slot_first[n] = i == 0;
            // the DC predecessor is the previous block of the component: the slot before, or the component's last slot of the MCU before
            d.slot_back[n] = (uint8_t)(i == 0 ? bpu_interleaved - (per_mcu - 1) : 1);
            ++n;
        }
    }
    d.n_slots = n;
    for (uint32_t g = 0; g < n_groups; ++g) {
        const Group &G = groups[g];
        DevGroup &D = d.groups[g];
        D.comp = G.comp;
        D.bpu = G.bpu;
        D.n_visits = G.n_visits;
        D.block_base = G.block_base;
        D.seg_visits = G.seg_visits;
        D.n_segs = G.n_segs;
        D.cps = G.cps;
        D.item_base = G.item_base;
        D.div_cps = make_fastdiv(G.cps);
        D.div_bpu = make_fastdiv(G.bpu);
    }
    unsigned blob = 0;
    for (size_t k = 0; k < scans.size(); ++k) {
        const Scan &s = scans[k];
        DevScan &ds = d.scans[k];
        ds.comp = s.comp;
        ds.ss = s.ss;
        ds.se = s.se;
        ds.n_units = s.n_units;
        ds.bpu = s.blocks_per_unit;
        ds.seg_base = s.seg_base;
        ds.n_segs = s.n_segs;
        ds.chunk_base = s.chunk_base;
        ds.rst_base = s.rst_base;
        ds.sos_off = blob;
        ds.sos_len = 0;
        if (k > 0) { // scan 0's SOS travels with the per-image file header
            ds.sos_len = (unsigned)s.sos.size();
            std::memcpy(d.blob + blob, s.sos.data(), s.sos.size());
            blob += ds.sos_len;
        }
    }
}

void Plan::fill_stage_a(StageAParams &a, const jpgb_device_images &im, int16_t *coef) const {
    std::memset(&a, 0, sizeof(a));
    a.pixels = static_cast<const uint8_t *>(im.data);
    a.coef = coef;
    a.image_stride = im.image_stride;
    a.blocks_per_image = blocks_per_image;
    a.width = p.width;
    a.height = p.height;
    a.bpp = bpp;
    a.color_type = p.color_type;
    a.ncomp = ncomp;
    a.hmax = hmax;
    a.vmax = vmax;
    a.mcu_cols = (int)mcu_cols;
    a.mcu_rows = (int)mcu_rows;
    a.mcu_order = mode == Mode::Interleaved;
    a.bpu = (int)bpu_interleaved;
    for (int c = 0; c < ncomp; ++c) {
        a.comp_h[c] = comps[c].h;
        a.comp_v[c] = comps[c].v;
        a.comp_qt[c] = comps[c].qtable;
        a.comp_pw[c] = (int)pad_w[c];
        a.comp_off[c] = block_off[c];
        a.comp_tw[c] = (int)true_w[c];
        a.comp_th[c] = (int)true_h[c];
        a.slot_base[c] = (int)slot_base[c];
    }
    // every ColorType, sampling factor and planar input has a warp-kernel instantiation; the generic kernel stays as
    // the cross-check of the tests
    const char *fg = std::getenv("JPGB_FORCE_GENERIC_STAGE_A");
    a.use_fast = !(fg && fg[0] == '1');
    a.planar = planar ? 1 : 0;
    a.row_stride = im.row_stride;
    // Channel-planar pixels of a packed ColorType are staged by the kernels with byte k of a pixel taken from plane
    // plane_of[k]: Bgr, Rgba and Bgra are the Rgb kernels with their R, G, B planes in that order (the alpha plane is
    // not read). Packed pixels leave plane_stride 0: no kernel reads it for them.
    if (planar) {
        a.bpp = 1;
        a.plane_stride = im.plane_stride;
    } else if (im.plane_stride && ncomp > 1) {
        const uint8_t ct = p.color_type;
        const bool bgr = ct == JPGB_BGR || ct == JPGB_BGRA;
        a.channel_planar = 1;
        a.plane_stride = im.plane_stride;
        for (int k = 0; k < 4; ++k) a.plane_of[k] = (bgr && k < 3) ? 2 - k : k;
        if (ct == JPGB_BGR || ct == JPGB_RGBA || ct == JPGB_BGRA) {
            a.color_type = JPGB_RGB;
            a.bpp = 3;
        }
    }
    for (int t = 0; t < 2; ++t)
        for (int i = 0; i < 64; ++i) {
            const int32_t c = q[t].corr[i] * q[t].recip[i];
            a.q[t].mul[i] = 2 * q[t].recip[i];
            a.q[t].add_pos[i] = 2 * c;
            a.q[t].add_neg[i] = 2 * (32767 - c);
        }
}

} // namespace jpgb
