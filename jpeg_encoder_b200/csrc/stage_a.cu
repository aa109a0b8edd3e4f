// Stage A: packed pixels -> quantized zig-zag coefficients, one fused kernel.
//
// Replaces, bit for bit, the reference's per-block numeric chain
//   ImageBuffer::fill_buffers (colour conversion)       src/image_buffer.rs:9-38, 100-313
//   row padding (replicate last sample / last row)       src/encoder.rs:732-745, 998-1010
//   get_block (strided gather = point decimation, -128)  src/encoder.rs:1222-1242
//   fdct (jfdctint islow, i32, x8 scaled)                src/fdct.rs:107-238
//   Operations::quantize_block (reciprocal, zig-zag)     src/encoder.rs:1265-1271, quantization.rs:291-307
//
// Work decomposition (stage_a_warp_kernel, the path of every BASELINE configuration): persistent and
// warp-autonomous. Each warp owns a private shared-memory tile of 32 full-resolution blocks (256 pixels) x one or
// more MCU rows, fetched by TMA (cp.async near image edges, which are replicated while staging), and walks warp
// tiles on its own -- no CTA barrier. A *warp task* is 32 consecutive blocks of one component block row: each
// lane owns one whole 8x8 block in registers, so both DCT passes, the transpose between them and the zig-zag
// permutation are register renaming -- no shuffles, no shared-memory round trip, no divergence. Each lane then
// writes its 128-byte block with 256-bit stores. stage_a_kernel<CT> is the generic CTA-tile variant for what the
// warp kernel does not instantiate.
//
// All arithmetic is 32-bit integer; tensor cores are not used (the DCT must be bit-exact).
#include <cuda.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <utility>

#include "kernels.h"

namespace jpgb {

namespace {

__device__ __forceinline__ int clamp_u8_formula_y(int r, int g, int b) {
    return (19595 * r + 38470 * g + 7471 * b + 0x7FFF) >> 16; // image_buffer.rs:22,26
}
__device__ __forceinline__ int formula_cb(int r, int g, int b) {
    return (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 0x7FFF) >> 16; // :23,27
}
__device__ __forceinline__ int formula_cr(int r, int g, int b) {
    return (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 0x7FFF) >> 16; // :24,28
}

// One sample of component `comp` from the pixel at `px` (shared memory), unshifted 0..255.
constexpr int kPlanar = 9; // internal: one full-resolution plane per component (the ImageBuffer path)

template <int CT>
__device__ __forceinline__ int sample(const uint8_t *px, int comp) {
    if (CT == JPGB_LUMA || CT == kPlanar) return px[0];
    if (CT == JPGB_YCBCR || CT == JPGB_YCCK) return px[comp];
    if (CT == JPGB_CMYK) return 255 - px[comp];
    int r, g, b;
    if (CT == JPGB_BGR || CT == JPGB_BGRA) {
        r = px[2]; g = px[1]; b = px[0];
    } else {
        r = px[0]; g = px[1]; b = px[2];
    }
    if (CT == JPGB_CMYK_AS_YCCK && comp == 3) return 255 - px[3];
    if (comp == 0) return clamp_u8_formula_y(r, g, b);
    if (comp == 1) return formula_cb(r, g, b);
    return formula_cr(r, g, b);
}

// 1-D 8-point LL&M forward DCT (fdct.rs:116-171 for PASS 1, :178-237 for PASS 2).
// PASS 1 takes *unshifted* samples 0..255: the -128 level shift (encoder.rs:1237) only moves the
// DC term of the row by -128*8 << PASS1_BITS, every other output is a function of differences.
template <int PASS>
__device__ __forceinline__ void dct8(int &d0, int &d1, int &d2, int &d3, int &d4, int &d5, int &d6, int &d7) {
    constexpr int N = PASS == 1 ? 11 : 15; // CONST_BITS -/+ PASS1_BITS
    constexpr int RND = 1 << (N - 1);
    const int tmp0 = d0 + d7, tmp7 = d0 - d7;
    const int tmp1 = d1 + d6, tmp6 = d1 - d6;
    const int tmp2 = d2 + d5, tmp5 = d2 - d5;
    const int tmp3 = d3 + d4, tmp4 = d3 - d4;
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3;
    const int tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    if (PASS == 1) {
        d0 = (tmp10 + tmp11 - 1024) << 2;
        d4 = (tmp10 - tmp11) << 2;
    } else {
        d0 = (tmp10 + tmp11 + 2) >> 2;
        d4 = (tmp10 - tmp11 + 2) >> 2;
    }
    const int z1e = (tmp12 + tmp13) * 4433 + RND;      // FIX_0_541196100
    d2 = (z1e + tmp13 * 6270) >> N;                    // FIX_0_765366865
    d6 = (z1e - tmp12 * 15137) >> N;                   // FIX_1_847759065
    // Odd part with the constants combined per input (the integer sums are identical to fdct.rs:149-170
    // term by term -- multiplication distributes exactly in two's complement):
    //   z3' = z3*(c3 - c3c5) + z4*c3,  z4' = z3*c3 + z4*(c3 - c5c3)            [FIX_1_175875602 etc.]
    //   out7 = tmp4*(0.298631336 - 0.899976223) - tmp7*0.899976223 + z3'   and so on.
    const int z3 = tmp4 + tmp6, z4 = tmp5 + tmp7;
    const int z3m = z3 * (9633 - 16069) + (z4 * 9633 + RND);
    const int z4m = z3 * 9633 + (z4 * (9633 - 3196) + RND);
    d7 = (tmp4 * (2446 - 7373) + (tmp7 * -7373 + z3m)) >> N;
    d5 = (tmp5 * (16819 - 20995) + (tmp6 * -20995 + z4m)) >> N;
    d3 = (tmp6 * (25172 - 20995) + (tmp5 * -20995 + z3m)) >> N;
    d1 = (tmp7 * (12299 - 7373) + (tmp4 * -7373 + z4m)) >> N;
}

// 2-D DCT of one block in registers, natural order: the rows (pass 1), then the columns (pass 2)
__device__ __forceinline__ void dct_2d(int (&v)[64]) {
#pragma unroll
    for (int y = 0; y < 8; ++y)
        dct8<1>(v[y * 8 + 0], v[y * 8 + 1], v[y * 8 + 2], v[y * 8 + 3], v[y * 8 + 4], v[y * 8 + 5], v[y * 8 + 6], v[y * 8 + 7]);
#pragma unroll
    for (int x = 0; x < 8; ++x)
        dct8<2>(v[x], v[8 + x], v[16 + x], v[24 + x], v[32 + x], v[40 + x], v[48 + x], v[56 + x]);
}

struct ZZ {
    int v[64];
};
__host__ __device__ constexpr ZZ make_zz() {
    return ZZ{{0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
               41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
               30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63}};
}

// quantize natural-order coefficient n with table T: the upper half of the 32-bit result is the
// quantized value (see QuantConsts in device_types.h)
template <int T>
__device__ __forceinline__ int quant32(const StageAParams &p, int v, int n) {
    const int add = v < 0 ? p.q[T].add_neg[n] : p.q[T].add_pos[n];
    return v * p.q[T].mul[n] + add;
}

__device__ __forceinline__ void store256(void *dst, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t a4,
                                         uint32_t a5, uint32_t a6, uint32_t a7) {
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst), "r"(a0), "r"(a1), "r"(a2), "r"(a3),
                 "r"(a4), "r"(a5), "r"(a6), "r"(a7)
                 : "memory");
}

// the quantized block in zig-zag order -> its 128 bytes at `dst` (32-byte aligned), four 256-bit stores
template <int T>
__device__ __forceinline__ void quantize_store256(const StageAParams &p, const int (&v)[64], int16_t *dst) {
    constexpr ZZ zz = make_zz();
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        uint32_t r[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int i0 = w * 16 + k * 2, i1 = i0 + 1;
            const int a = quant32<T>(p, v[zz.v[i0]], zz.v[i0]);
            const int b = quant32<T>(p, v[zz.v[i1]], zz.v[i1]);
            r[k] = __byte_perm((uint32_t)a, (uint32_t)b, 0x7632); // {hi16(a), hi16(b)}
        }
        store256(dst + w * 16, r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7]);
    }
}

// Byte-wise fill of one 16-byte chunk with the row's last pixel replicated (Q4). Cold path, kept out of line.
template <int BPP>
__device__ __noinline__ void stage_edge_chunk(uint8_t *dst, const uint8_t *row, int cb, int valid_px) {
    for (int b = 0; b < 16; ++b) {
        const int byte = cb + b;
        const int px = byte / BPP, ch = byte - px * BPP;
        dst[cb + b] = row[min(px, valid_px - 1) * BPP + ch];
    }
}

// The same chunk of packed pixels gathered from channel planes: byte ch of a pixel comes from plane plane_of[ch].
// `row` is the row's first pixel in plane 0.
template <int BPP>
__device__ __noinline__ void stage_planes_chunk(uint8_t *dst, const uint8_t *row, unsigned long long plane_stride, const int *plane_of,
                                                int cb, int valid_px) {
    for (int b = 0; b < 16; ++b) {
        const int byte = cb + b;
        const int px = byte / BPP, ch = byte - px * BPP;
        dst[cb + b] = row[(size_t)plane_of[ch] * plane_stride + min(px, valid_px - 1)];
    }
}

// ---- samples of a wider element type (jpgb_sample_format), turned into the 8-bit samples of the tile while staging ----
// Colour types that take them: Luma and the RGB family (Bgr, Rgba and Bgra planes are Rgb planes in another order)
__host__ __device__ constexpr bool converts(int ct) {
    return ct == JPGB_LUMA || ct == JPGB_RGB || ct == JPGB_BGR || ct == JPGB_RGBA || ct == JPGB_BGRA;
}
__host__ __device__ constexpr int element_size(int type) { return type == JPGB_SAMPLE_F32 ? 4 : 2; }

// The conversion of jpgb_encode_batch_device_samples: y = fadd_rn(fmul_rn(x, scale), offset) -- the intrinsics keep
// nvcc from contracting them into an FMA -- then NaN -> 0, else clamp(rint(y), 0, 255). cvt.rni.sat.u8.f32 is that last
// step: round to nearest even, saturate to 0..255, NaN to 0. The result is read through its low byte only.
__device__ __forceinline__ uint32_t to_sample(float x, const jpgb_sample_format &f) {
    const float y = __fadd_rn(__fmul_rn(x, f.scale), f.offset);
    uint32_t r;
    asm("cvt.rni.sat.u8.f32 %0, %1;" : "=r"(r) : "f"(y));
    return r;
}
// element `bits` (the low 16 bits for the 16-bit types) of type T widened to fp32: exact for every type
template <int T>
__device__ __forceinline__ float widen(uint32_t bits) {
    if constexpr (T == JPGB_SAMPLE_U16) return (float)(bits & 0xFFFFu);
    else if constexpr (T == JPGB_SAMPLE_F16) return __half2float(__ushort_as_half((unsigned short)bits));
    else if constexpr (T == JPGB_SAMPLE_BF16) return __uint_as_float(bits << 16);
    else return __uint_as_float(bits);
}
__device__ __forceinline__ float load_element(const uint8_t *src, int type) {
    if (type == JPGB_SAMPLE_F32) return widen<JPGB_SAMPLE_F32>(__ldg(reinterpret_cast<const unsigned *>(src)));
    const uint32_t b = __ldg(reinterpret_cast<const unsigned short *>(src));
    if (type == JPGB_SAMPLE_U16) return widen<JPGB_SAMPLE_U16>(b);
    if (type == JPGB_SAMPLE_F16) return widen<JPGB_SAMPLE_F16>(b);
    return widen<JPGB_SAMPLE_BF16>(b);
}

// The converting counterpart of stage_edge_chunk / stage_planes_chunk, element by element: tile bytes e0 .. e0 + n - 1 of
// a row whose pixels have `pxe` samples, the row's last valid pixel replicated (Q4). Sample ch of pixel px lies at
// row + (px * pxe + ch) * es, or with `plane_of` at row + plane_of[ch] * plane_stride + px * es. A fourth (alpha) sample
// of packed pixels is not read: its tile byte is 0. Cold path (image edges, rows not 16-byte aligned), kept out of line.
__device__ __noinline__ void stage_convert_edge(uint8_t *dst, const uint8_t *row, int e0, int n, int pxe, int valid_px,
                                                const jpgb_sample_format f, const int *plane_of, unsigned long long plane_stride) {
    const int es = element_size((int)f.type);
    for (int e = e0; e < e0 + n; ++e) {
        const int px = e / pxe, ch = e - px * pxe, sx = min(px, valid_px - 1);
        uint32_t s = 0;
        if (plane_of) s = to_sample(load_element(row + (size_t)plane_of[ch] * plane_stride + (size_t)sx * es, (int)f.type), f);
        else if (!(pxe == 4 && ch == 3)) s = to_sample(load_element(row + ((size_t)sx * pxe + ch) * es, (int)f.type), f);
        dst[e] = (uint8_t)s;
    }
}

// 8 consecutive elements of type T at a 16-byte aligned address -> their 8 tile bytes. ALPHA: packed 4-sample pixels
// (the unit starts on a pixel); their alpha sample is not converted and its byte is 0.
template <int T>
__device__ __forceinline__ void load_unit(const uint8_t *g, uint4 (&a)[2]) {
    a[0] = __ldg(reinterpret_cast<const uint4 *>(g));
    if constexpr (element_size(T) == 4) a[1] = __ldg(reinterpret_cast<const uint4 *>(g) + 1);
}
template <int T, bool ALPHA>
__device__ __forceinline__ uint2 convert_unit(const uint4 (&a)[2], const jpgb_sample_format &f) {
    const uint32_t w[8] = {a[0].x, a[0].y, a[0].z, a[0].w, a[1].x, a[1].y, a[1].z, a[1].w};
    uint32_t s[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint32_t bits = element_size(T) == 4 ? w[j] : (j & 1 ? w[j >> 1] >> 16 : w[j >> 1]);
        s[j] = (ALPHA && (j & 3) == 3) ? 0u : to_sample(widen<T>(bits), f);
    }
    auto pack4 = [](uint32_t b0, uint32_t b1, uint32_t b2, uint32_t b3) {
        return __byte_perm(__byte_perm(b0, b1, 0x0040), __byte_perm(b2, b3, 0x0040), 0x5410);
    };
    return make_uint2(pack4(s[0], s[1], s[2], s[3]), pack4(s[4], s[5], s[6], s[7]));
}

// A warp tile of LINES lines of 256 * PXB samples (packed rows, or ROWS rows of each plane read) converted into the u8
// tile, line i at tile + i * PITCH. Line i is row min(py0 + i % ROWS, height - 1) of plane i / ROWS, from
// src = image + px0 * PXB * es (+ plane * plane_stride). Interior tiles: every lane converts its 8-element units with
// 16-byte loads, U units (U or 2U loads) in flight. Elsewhere a unit inside the row's valid samples takes the same
// path when the row is 16-byte aligned, and stage_convert_edge otherwise.
template <int T, int PXB, int ROWS, int LINES, bool ALPHA>
__device__ __forceinline__ void stage_convert_tile(uint8_t *tile, const uint8_t *src, const StageAParams &p, const jpgb_sample_format &f,
                                                   int py0, int valid_px, int needed_px, bool interior, int lane) {
    constexpr int ES = element_size(T), UPL = 32 * PXB, PITCH = 256 * PXB, U = 4;
    const size_t row_stride = p.row_stride;
    if (interior) {
        static_assert((LINES * PXB) % U == 0, "whole batches of units per lane");
#pragma unroll 1
        for (int u0 = lane; u0 < LINES * UPL; u0 += 32 * U) {
            uint4 a[U][2];
#pragma unroll
            for (int j = 0; j < U; ++j) {
                const int u = u0 + 32 * j, i = u / UPL, k = i / ROWS, ry = i - k * ROWS;
                load_unit<T>(src + (size_t)k * p.plane_stride + (size_t)(py0 + ry) * row_stride + (size_t)(u - i * UPL) * 8 * ES, a[j]);
            }
#pragma unroll
            for (int j = 0; j < U; ++j) {
                const int u = u0 + 32 * j, i = u / UPL;
                *reinterpret_cast<uint2 *>(tile + i * PITCH + (u - i * UPL) * 8) = convert_unit<T, ALPHA>(a[j], f);
            }
        }
        return;
    }
    const int valid = valid_px * PXB, needed = needed_px * PXB;
#pragma unroll 1
    for (int i = 0; i < LINES; ++i) {
        const int k = i / ROWS, ry = i - k * ROWS;
        const uint8_t *row = src + (size_t)k * p.plane_stride + (size_t)min(py0 + ry, p.height - 1) * row_stride;
        uint8_t *dst = tile + i * PITCH;
        const bool aligned = (reinterpret_cast<uintptr_t>(row) & 15) == 0;
#pragma unroll 1
        for (int e0 = lane * 8; e0 < needed; e0 += 32 * 8) {
            if (aligned && e0 + 8 <= valid) {
                uint4 a[2];
                load_unit<T>(row + (size_t)e0 * ES, a);
                *reinterpret_cast<uint2 *>(dst + e0) = convert_unit<T, ALPHA>(a, f);
            } else {
                stage_convert_edge(dst, row, e0, 8, PXB, valid_px, f, nullptr, 0);
            }
        }
    }
}

// The generic kernel's body: a CTA tile of `groups` x 32 MCUs x one MCU row. CONV: the samples are elements of
// fmt.type, converted while staging. FRAME (CT == kPlanar): the planes are those of `frame`, subsampled, staged
// upsampled to full resolution with byte loads.
template <int CT, bool CONV, bool FRAME = false>
__device__ __forceinline__ void generic_tile(const StageAParams &p, const jpgb_sample_format &fmt, const jpgb_device_ycbcr &frame = {}) {
    extern __shared__ __align__(128) uint8_t tile[];
    constexpr int BPP = (CT == JPGB_LUMA || CT == kPlanar) ? 1 : ((CT == JPGB_RGB || CT == JPGB_BGR || CT == JPGB_YCBCR) ? 3 : 4);
    constexpr bool PLANAR = CT == kPlanar;

    const int tile_x = blockIdx.x, mcu_y = blockIdx.y, img = blockIdx.z;
    const int mcu_x0 = tile_x * 32 * p.groups;
    const int px0 = mcu_x0 * 8 * p.hmax, py0 = mcu_y * 8 * p.vmax;
    const uint8_t *src = p.pixels + (size_t)img * p.image_stride;
    const int px_bytes = (p.channel_planar ? 1 : BPP) * (CONV ? element_size((int)fmt.type) : 1); // of one pixel in one input row

    // ---- stage the tile: 16-byte chunks, edges replicated (Q4) ----
    const int chunks_per_row = p.tile_pitch / 16;
    const int n_chunks = chunks_per_row * p.tile_h_px;
    const int valid_px = min(p.tile_w_px, p.width - px0);  // > 0 by construction
    const int valid_bytes = valid_px * BPP;
    const int plane_tile = p.tile_pitch * p.tile_h_px; // planar: one such tile per component, back to back
    const int n_planes = PLANAR ? p.ncomp : 1;
    for (int c = threadIdx.x; c < n_chunks * n_planes; c += blockDim.x) {
        const int plane = c / n_chunks, cc = c - plane * n_chunks;
        const int ry = cc / chunks_per_row, cb = (cc - ry * chunks_per_row) * 16;
        const int sy = min(py0 + ry, p.height - 1);
        const uint8_t *row = src + (size_t)plane * p.plane_stride + (size_t)sy * p.row_stride + (size_t)px0 * px_bytes;
        uint8_t *dst = tile + plane * plane_tile + ry * p.tile_pitch;
        if constexpr (FRAME) { // the mapping of jpgb_device_ycbcr restated: plane row sy / c_v, column (px / c_h) * c_sample_stride
            const int sh = plane ? frame.c_h : 1, sv = plane ? frame.c_v : 1, ss = plane ? (int)frame.c_sample_stride : 1;
            const uint8_t *fr = static_cast<const uint8_t *>(plane == 0 ? frame.y : (plane == 1 ? frame.cb : frame.cr)) +
                                (size_t)img * (plane ? frame.c_image_stride : frame.y_image_stride) +
                                (size_t)(sy / sv) * (plane ? frame.c_row_stride : frame.y_row_stride);
            for (int b = 0; b < 16; ++b) dst[cb + b] = fr[(size_t)((px0 + min(cb + b, valid_px - 1)) / sh) * ss];
            continue;
        }
        if (CONV) stage_convert_edge(dst, row, cb, 16, BPP, valid_px, fmt, p.channel_planar ? p.plane_of : nullptr, p.plane_stride);
        else if (p.channel_planar) stage_planes_chunk<BPP>(dst, row, p.plane_stride, p.plane_of, cb, valid_px);
        else if (cb + 16 <= valid_bytes && ((reinterpret_cast<uintptr_t>(row + cb) & 15) == 0))
            *reinterpret_cast<uint4 *>(dst + cb) = __ldg(reinterpret_cast<const uint4 *>(row + cb));
        else stage_edge_chunk<BPP>(dst, row, cb, valid_px);
    }
    __syncthreads();

    // ---- warp tasks ----
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const int n_tasks = p.groups * p.tasks_per_group;
    for (int task = warp; task < n_tasks; task += n_warps) {
        const int group = task / p.tasks_per_group, slot = task - group * p.tasks_per_group;
        const int comp = p.task_comp[slot], bv = p.task_v[slot], bh = p.task_h[slot];
        const int mcu_local = group * 32 + lane;
        const int mcu_x = mcu_x0 + mcu_local;
        if (mcu_x >= p.mcu_cols) continue;
        // get_block arguments, encoder.rs:762-769: start = mcu*8*max + offset*8, stride = max/factor
        const int sx = p.hmax / p.comp_h[comp], sy = p.vmax / p.comp_v[comp];
        const int x0 = mcu_local * 8 * p.hmax + bh * 8, y0 = bv * 8;
        const uint8_t *base = tile + (PLANAR ? comp * plane_tile : 0) + y0 * p.tile_pitch + x0 * BPP;
        const int step_x = sx * BPP, step_y = sy * p.tile_pitch;

        int v[64];
#pragma unroll
        for (int y = 0; y < 8; ++y)
#pragma unroll
            for (int x = 0; x < 8; ++x) v[y * 8 + x] = sample<CT>(base + y * step_y + x * step_x, comp);
        dct_2d(v);

        size_t blk = (size_t)img * p.blocks_per_image;
        const int gy = mcu_y + p.mcu_row0; // MCU row inside the whole image (this launch may cover a slice of it)
        if (p.mcu_order) { // the order the interleaved scan codes them (encoder.rs:747-791)
            blk += ((size_t)gy * p.mcu_cols + mcu_x) * p.bpu + p.slot_base[comp] + bv * p.comp_h[comp] + bh;
        } else {           // raster of the component's true grid (encoder.rs:1012-1031); MCU padding blocks are not stored
            const int by = gy * p.comp_v[comp] + bv, bx = mcu_x * p.comp_h[comp] + bh;
            if (bx >= p.comp_tw[comp] || by >= p.comp_th[comp]) continue;
            blk += p.comp_off[comp] + (size_t)by * p.comp_tw[comp] + bx;
        }
        int16_t *dst = p.coef + blk * 64;
        if (p.comp_qt[comp] == 0) quantize_store256<0>(p, v, dst);
        else quantize_store256<1>(p, v, dst);
    }
}

template <int CT>
__global__ void __launch_bounds__(256) stage_a_kernel(const __grid_constant__ StageAParams p) {
    generic_tile<CT, false>(p, jpgb_sample_format{});
}
template <int CT>
__global__ void __launch_bounds__(256) stage_a_convert_kernel(const __grid_constant__ StageAParams p, const __grid_constant__ jpgb_sample_format fmt) {
    generic_tile<CT, true>(p, fmt);
}
// the cross-check of jpgb_encode_batch_device_ycbcr (JPGB_FORCE_GENERIC_STAGE_A=1)
__global__ void __launch_bounds__(256) stage_a_frame_generic_kernel(const __grid_constant__ StageAParams p,
                                                                    const __grid_constant__ jpgb_device_ycbcr frame) {
    generic_tile<kPlanar, false, true>(p, jpgb_sample_format{}, frame);
}


// =================================================================================================
// Fast path (the BASELINE configurations): Luma, the RGB family and CmykAsYcck at luma sampling
// 1x1 / 2x1 / 1x2 / 2x2. Same one-block-per-lane decomposition as the generic kernel, but
//   * a task is 32 *consecutive blocks of one component block row*, so the 32 lanes read
//     adjacent 8-pixel spans (bank-conflict-free 64/128-bit shared loads) and write one contiguous
//     4 KB run of coefficients with 256-bit stores;
//   * colour conversion runs on packed pixel words with IDP.2A (dp2a: two 16-bit coefficients x
//     two pixel bytes + accumulator per instruction), measured on B200 at the same 64 lanes/clk/SM
//     as IMAD (profiles/r1_int_pipe_microbench.txt): 2 IDP + 1 shift per Y sample, no byte
//     extraction. The arithmetic is the reference's: the same integer sum, + 0x7FFF, >> 16.
// =================================================================================================

// acc + CA * byte(2*HI) + CB * byte(2*HI+1) of w, exactly, for compile-time coefficients.
template <int CA, int CB, bool HI>
__device__ __forceinline__ int idp2(int acc, uint32_t w) {
    constexpr bool fits_u = CA >= 0 && CB >= 0 && CA <= 65535 && CB <= 65535;
    constexpr bool fits_s = CA >= -32768 && CA <= 32767 && CB >= -32768 && CB <= 32767;
    if constexpr (CA == 0 && CB == 0) {
        return acc;
    } else if constexpr (fits_u) {
        constexpr uint32_t c = (uint32_t)CA | ((uint32_t)CB << 16);
        int r;
        if constexpr (HI) asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(c), "r"(w), "r"(acc));
        else asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(c), "r"(w), "r"(acc));
        return r;
    } else if constexpr (fits_s) {
        constexpr uint32_t c = ((uint32_t)CA & 0xFFFFu) | (((uint32_t)CB & 0xFFFFu) << 16);
        int r;
        if constexpr (HI) asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(c), "r"(w), "r"(acc));
        else asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(c), "r"(w), "r"(acc));
        return r;
    } else { // one coefficient needs the signed, the other the unsigned 16-bit range: two instructions
        return idp2<CA, 0, HI>(idp2<0, CB, HI>(acc, w), w);
    }
}

// K + M0*b[O] + M1*b[O+1] + M2*b[O+2] where b[] are the bytes of the word array w (register
// resident, compile-time indices). Three consecutive bytes always straddle exactly two byte pairs.
template <int O, int M0, int M1, int M2, int K, int NW>
__device__ __forceinline__ int dot3(const uint32_t (&w)[NW]) {
    constexpr int P0 = O >> 1, P1 = (O + 2) >> 1; // byte-pair indices
    constexpr int A0 = (2 * P0 == O) ? M0 : 0;    // coefficient of pair P0 slot 0
    constexpr int B0 = (2 * P0 + 1 == O) ? M0 : ((2 * P0 + 1 == O + 1) ? M1 : 0);
    constexpr int A1 = (2 * P1 == O + 1) ? M1 : ((2 * P1 == O + 2) ? M2 : 0);
    constexpr int B1 = (2 * P1 + 1 == O + 2) ? M2 : 0;
    int acc = K;
    acc = idp2<A0, B0, (P0 & 1) != 0>(acc, w[P0 >> 1]);
    acc = idp2<A1, B1, (P1 & 1) != 0>(acc, w[P1 >> 1]);
    return acc;
}

enum Role { ROLE_Y = 0, ROLE_CB = 1, ROLE_CR = 2, ROLE_K = 3, ROLE_RAW = 4, ROLE_CBCR = 5 };
struct ChromaConsts;

template <int CT>
__host__ __device__ constexpr bool is_bgr() { return CT == JPGB_BGR || CT == JPGB_BGRA; }

template <int CT>
struct Fmt {
    static constexpr int BPP = CT == JPGB_LUMA ? 1 : ((CT == JPGB_RGB || CT == JPGB_BGR || CT == JPGB_YCBCR) ? 3 : 4);
    // formats whose samples are pixel bytes taken verbatim (Ycbcr, Ycck) or inverted (Cmyk): image_buffer.rs:206-257, 288-313
    static constexpr bool BYTES = CT == JPGB_YCBCR || CT == JPGB_YCCK || CT == JPGB_CMYK;
    static constexpr int NCOMP = CT == JPGB_LUMA ? 1 : ((CT == JPGB_CMYK_AS_YCCK || CT == JPGB_YCCK || CT == JPGB_CMYK) ? 4 : 3);
    // components that carry the sampling factor (luma, and K; for Cmyk only K -- encoder.rs:569-619) and the 1x1 ones
    static constexpr int NFULL = (CT == JPGB_CMYK_AS_YCCK || CT == JPGB_YCCK) ? 2 : 1;
    static constexpr int NSUB = NCOMP == 1 ? 0 : (CT == JPGB_CMYK ? 3 : 2);
    __host__ __device__ static constexpr int full_comp(int i) { return CT == JPGB_CMYK ? 3 : (i == 0 ? 0 : 3); }
    __host__ __device__ static constexpr int sub_comp(int i) { return CT == JPGB_CMYK ? i : 1 + i; }
};

// sample I of a block row from the row's pixel words (compile-time I: every byte offset is static)
template <int CT, int ROLE, int SX, int I, int NW>
__device__ __forceinline__ int sample_at(const uint32_t (&w)[NW]) {
    constexpr int BPP = Fmt<CT>::BPP;
    constexpr int RND = 0x7FFF, MID = (128 << 16) + 0x7FFF;
    constexpr int O = I * SX * BPP; // byte offset of the pixel inside w
    if constexpr (ROLE == ROLE_RAW) {
        return (int)__byte_perm(w[O >> 2], 0, 0x4440 + (O & 3));
    } else if constexpr (ROLE == ROLE_K) { // 255 - k, image_buffer.rs:35-38
        return (int)__byte_perm(~w[(O + 3) >> 2], 0, 0x4440 + ((O + 3) & 3));
    } else if constexpr (ROLE == ROLE_Y) {
        // Y = (19595 R + 38470 G + 7471 B + 0x7FFF) >> 16            image_buffer.rs:22,26
        if constexpr (is_bgr<CT>()) return dot3<O, 7471, 38470, 19595, RND>(w) >> 16;
        else return dot3<O, 19595, 38470, 7471, RND>(w) >> 16;
    } else if constexpr (ROLE == ROLE_CB) {
        // Cb = (-11059 R - 21709 G + 32768 B + (128 << 16) + 0x7FFF) >> 16   :23,27
        if constexpr (is_bgr<CT>()) return dot3<O, 32768, -21709, -11059, MID>(w) >> 16;
        else return dot3<O, -11059, -21709, 32768, MID>(w) >> 16;
    } else {
        // Cr = (32768 R - 27439 G - 5329 B + (128 << 16) + 0x7FFF) >> 16     :24,28
        if constexpr (is_bgr<CT>()) return dot3<O, -5329, -27439, 32768, MID>(w) >> 16;
        else return dot3<O, 32768, -27439, -5329, MID>(w) >> 16;
    }
}
template <int CT, int ROLE, int SX, int NW, int... Is>
__device__ __forceinline__ void sample_row(const uint32_t (&w)[NW], int *s, std::integer_sequence<int, Is...>) {
    ((s[Is] = sample_at<CT, ROLE, SX, Is, NW>(w)), ...);
}

// ---- Cb and Cr in one instruction stream (horizontally decimated chroma) -------------------------
// In the warp-autonomous kernel lanes 0..15 produce Cb blocks and lanes 16..31 Cr blocks of the same
// pixels. Both are  MID + M0*b[O] + M1*b[O+1] + M2*b[O+2]  with different coefficients, so the
// coefficients travel in per-lane registers and every lane runs the same four IDP.2A: two in signed
// 16-bit mode for the negative coefficients, two in unsigned mode for the +32768 one (which fits
// neither s16 nor, together with a negative neighbour, u16). Pixels sit at even byte offsets here
// (O = 2*BPP*i), so pair 0 holds (M0, M1) and pair 1 holds (M2, -).
struct ChromaConsts {
    uint32_t sA, sB, uA, uB; // signed pair 0 / pair 1, unsigned pair 0 / pair 1
};
template <int CT>
__device__ __forceinline__ ChromaConsts chroma_consts(bool cr) {
    auto pk = [](int a, int b) { return ((uint32_t)a & 0xFFFFu) | (((uint32_t)b & 0xFFFFu) << 16); };
    ChromaConsts c;
    if (!is_bgr<CT>()) { // memory order R, G, B
        if (!cr) { c.sA = pk(-11059, -21709); c.sB = 0; c.uA = 0; c.uB = pk(32768, 0); }
        else { c.sA = pk(0, -27439); c.sB = pk(-5329, 0); c.uA = pk(32768, 0); c.uB = 0; }
    } else {             // memory order B, G, R
        if (!cr) { c.sA = pk(0, -21709); c.sB = pk(-11059, 0); c.uA = pk(32768, 0); c.uB = 0; }
        else { c.sA = pk(-5329, -27439); c.sB = 0; c.uA = 0; c.uB = pk(32768, 0); }
    }
    return c;
}
template <bool HI, bool SIGNED>
__device__ __forceinline__ int idp2r(int acc, uint32_t coef, uint32_t w) {
    int r;
    if constexpr (HI && SIGNED) asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(coef), "r"(w), "r"(acc));
    else if constexpr (HI) asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(coef), "r"(w), "r"(acc));
    else if constexpr (SIGNED) asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(coef), "r"(w), "r"(acc));
    else asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(coef), "r"(w), "r"(acc));
    return r;
}
template <int O, int NW>
__device__ __forceinline__ int chroma_at(const uint32_t (&w)[NW], const ChromaConsts &c) {
    static_assert((O & 1) == 0, "decimated chroma pixels start at even byte offsets");
    constexpr int P0 = O >> 1, P1 = P0 + 1;
    int acc = (128 << 16) + 0x7FFF;
    acc = idp2r<(P0 & 1) != 0, true>(acc, c.sA, w[P0 >> 1]);
    acc = idp2r<(P1 & 1) != 0, true>(acc, c.sB, w[P1 >> 1]);
    acc = idp2r<(P0 & 1) != 0, false>(acc, c.uA, w[P0 >> 1]);
    acc = idp2r<(P1 & 1) != 0, false>(acc, c.uB, w[P1 >> 1]);
    return acc >> 16;
}
template <int CT, int SX, int NW, int... Is>
__device__ __forceinline__ void chroma_row(const uint32_t (&w)[NW], int *s, const ChromaConsts &c, std::integer_sequence<int, Is...>) {
    ((s[Is] = chroma_at<Is * SX * Fmt<CT>::BPP, NW>(w, c)), ...);
}

// The pixel words of one block row: the 8 * SX pixels from `row` (shared tile) on, as few wide loads as the
// alignment allows. With 4 bytes per pixel and SX > 1 only every SX-th pixel is read; the words between are 0.
template <int BPP, int SX>
__host__ __device__ constexpr int row_words() { return (((7 * SX + 1) * BPP) + 3) / 4; }
template <int BPP, int SX, int NW>
__device__ __forceinline__ void load_words(const uint8_t *row, uint32_t (&w)[NW]) {
    static_assert(NW == row_words<BPP, SX>(), "words spanned by the block row");
    if constexpr (BPP == 4 && SX > 1) {
        const uint32_t *r = reinterpret_cast<const uint32_t *>(row);
#pragma unroll
        for (int i = 0; i < NW; ++i) w[i] = (i % SX) ? 0u : r[i];
    } else if constexpr ((SX * BPP) % 2 != 0) { // a block is 8 or 24 bytes wide: 8-byte aligned
        const uint2 *r = reinterpret_cast<const uint2 *>(row);
#pragma unroll
        for (int i = 0; i < NW / 2; ++i) {
            const uint2 a = r[i];
            w[2 * i] = a.x;
            w[2 * i + 1] = a.y;
        }
    } else { // a block is a multiple of 16 bytes wide: 16-byte aligned
        const uint4 *r = reinterpret_cast<const uint4 *>(row);
#pragma unroll
        for (int i = 0; i < (NW + 3) / 4; ++i) {
            const uint4 a = r[i];
            w[4 * i] = a.x;
            if (4 * i + 1 < NW) w[4 * i + 1] = a.y;
            if (4 * i + 2 < NW) w[4 * i + 2] = a.z;
            if (4 * i + 3 < NW) w[4 * i + 3] = a.w;
        }
    }
}

// ---- channel-planar tiles ([plane][rows][256]): the same pixel words, interleaved from one word per plane ----
// Byte t of packed word M is byte (4M + t) % BPP (the channel) of pixel (4M + t) / BPP. It is taken from word
// pixel / 4 of that channel's plane. A packed word draws on at most four plane words: one PRMT merges the first
// two, one more each further source.
struct WordSrc {
    int n, ch[4], j[4], sel[3];
};
template <int BPP>
__host__ __device__ constexpr WordSrc word_src(int m) {
    WordSrc r{};
    int src[4] = {}, byte[4] = {};
    for (int t = 0; t < 4; ++t) {
        const int q = (4 * m + t) / BPP, ch = (4 * m + t) % BPP, j = q >> 2;
        int k = 0;
        while (k < r.n && !(r.ch[k] == ch && r.j[k] == j)) ++k;
        if (k == r.n) r.ch[r.n] = ch, r.j[r.n] = j, ++r.n;
        src[t] = k;
        byte[t] = q & 3;
    }
    for (int t = 0; t < 4; ++t) {
        r.sel[0] |= (src[t] == 0 ? byte[t] : (src[t] == 1 ? 4 + byte[t] : 0)) << (4 * t);
        r.sel[1] |= (src[t] == 2 ? 4 + byte[t] : t) << (4 * t);
        r.sel[2] |= (src[t] == 3 ? 4 + byte[t] : t) << (4 * t);
    }
    return r;
}
template <int BPP, int M, int NPW>
__device__ __forceinline__ uint32_t packed_word(const uint32_t (&pw)[BPP][NPW]) {
    constexpr WordSrc s = word_src<BPP>(M);
    static_assert(s.j[0] < NPW && s.j[1] < NPW && s.j[2] < NPW && s.j[3] < NPW, "pixels of the block row");
    uint32_t acc = __byte_perm(pw[s.ch[0]][s.j[0]], pw[s.ch[1]][s.j[1]], s.sel[0]);
    if constexpr (s.n > 2) acc = __byte_perm(acc, pw[s.ch[2]][s.j[2]], s.sel[1]);
    if constexpr (s.n > 3) acc = __byte_perm(acc, pw[s.ch[3]][s.j[3]], s.sel[2]);
    return acc;
}
template <int BPP, int SX, int NW, int NPW, int... Ms>
__device__ __forceinline__ void interleave_words(const uint32_t (&pw)[BPP][NPW], uint32_t (&w)[NW], std::integer_sequence<int, Ms...>) {
    ((w[Ms] = (BPP == 4 && SX > 1 && Ms % SX) ? 0u : packed_word<BPP, Ms, NPW>(pw)), ...); // the words load_words leaves 0
}
// load_words for a channel-planar tile: `row` is the block row's first pixel in tile plane 0, plane offsets in `choff`
// (byte k of a pixel lies choff[k] further). A block row starts at a multiple of 8 * SX pixels.
template <int BPP, int SX, int NW>
__device__ __forceinline__ void load_words_planes(const uint8_t *row, const int *choff, uint32_t (&w)[NW]) {
    constexpr int NPW = 2 * SX; // words of one plane under the 8 * SX pixels
    uint32_t pw[BPP][NPW];
#pragma unroll
    for (int k = 0; k < BPP; ++k) {
        if constexpr (SX == 1) {
            const uint2 a = *reinterpret_cast<const uint2 *>(row + choff[k]);
            pw[k][0] = a.x;
            pw[k][1] = a.y;
        } else {
#pragma unroll
            for (int i = 0; i < NPW / 4; ++i) {
                const uint4 a = reinterpret_cast<const uint4 *>(row + choff[k])[i];
                pw[k][4 * i] = a.x;
                pw[k][4 * i + 1] = a.y;
                pw[k][4 * i + 2] = a.z;
                pw[k][4 * i + 3] = a.w;
            }
        }
    }
    interleave_words<BPP, SX, NW, NPW>(pw, w, std::make_integer_sequence<int, NW>{});
}
template <int BPP, int SX, bool PL, int NW>
__device__ __forceinline__ void load_tile_words(const uint8_t *row, const int *choff, uint32_t (&w)[NW]) {
    if constexpr (PL) load_words_planes<BPP, SX>(row, choff, w);
    else load_words<BPP, SX>(row, w);
}

// 8 samples (unshifted, 0..255) of one block row. `row` points at the first pixel of the row in the
// shared tile; the pixels used are 0, SX, 2*SX, ... (point decimation, encoder.rs:1222-1242).
// PL: a channel-planar tile, plane offsets in `choff`.
template <int CT, int ROLE, int SX, bool PL = false>
__device__ __forceinline__ void load_row(const uint8_t *row, int *s, const ChromaConsts *cc = nullptr, const int *choff = nullptr) {
    constexpr int NW = row_words<Fmt<CT>::BPP, SX>();
    uint32_t w[NW];
    load_tile_words<Fmt<CT>::BPP, SX, PL>(row, choff, w);
    if constexpr (ROLE == ROLE_CBCR) chroma_row<CT, SX, NW>(w, s, *cc, std::make_integer_sequence<int, 8>{});
    else sample_row<CT, ROLE, SX, NW>(w, s, std::make_integer_sequence<int, 8>{});
}

// ---- verbatim / inverted byte formats: sample = byte `coff` of the pixel, xor `xorv` (0xFF inverts: 255 - x) ----
// coff may differ between the lanes of a warp (two components share a task when chroma is horizontally decimated):
// the byte is picked with PRMT on a register selector out of the pixel's word and the word behind it.
template <int BPP, int SX, int I, int NW>
__device__ __forceinline__ int byte_at(const uint32_t (&w)[NW], unsigned coff, unsigned xorv) {
    constexpr int O = I * SX * BPP;
    constexpr int W0 = O >> 2, W1 = (W0 + 1 < NW) ? W0 + 1 : W0;
    return (int)((__byte_perm(w[W0], w[W1], (O & 3) + coff) ^ xorv) & 0xFFu);
}
template <int BPP, int SX, int NW, int... Is>
__device__ __forceinline__ void byte_row(const uint32_t (&w)[NW], int *s, unsigned coff, unsigned xorv, std::integer_sequence<int, Is...>) {
    ((s[Is] = byte_at<BPP, SX, Is, NW>(w, coff, xorv)), ...);
}
template <int BPP, int SX, bool PL>
__device__ __forceinline__ void load_row_bytes(const uint8_t *row, int *s, unsigned coff, unsigned xorv, const int *choff) {
    constexpr int NW = row_words<BPP, SX>();
    uint32_t w[NW];
    load_tile_words<BPP, SX, PL>(row, choff, w);
    byte_row<BPP, SX, NW>(w, s, coff, xorv, std::make_integer_sequence<int, 8>{});
}
template <int BPP, int SX, int SY, bool PL = false>
__device__ __forceinline__ void load_block_bytes(const uint8_t *base, int pitch, int (&v)[64], unsigned coff, unsigned xorv,
                                                 const int *choff = nullptr) {
#pragma unroll
    for (int y = 0; y < 8; ++y) load_row_bytes<BPP, SX, PL>(base + y * SY * pitch, &v[y * 8], coff, xorv, choff);
}

template <int CT, int ROLE, int SX, int SY, bool PL = false>
__device__ __forceinline__ void load_block(const uint8_t *base, int pitch, int (&v)[64], const ChromaConsts *cc = nullptr,
                                           const int *choff = nullptr) {
#pragma unroll
    for (int y = 0; y < 8; ++y) load_row<CT, ROLE, SX, PL>(base + y * SY * pitch, &v[y * 8], cc, choff);
}

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- TMA (cp.async.bulk.tensor) + mbarrier, one barrier per warp --------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned phase) {
    const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(a), "r"(phase) : "memory");
}
// one 3-D box (x in 4-byte elements, y in pixel rows, z = image) -> shared memory, completion on `bar`
__device__ __forceinline__ void tma_load_3d(void *smem_dst, const CUtensorMap *map, uint64_t *bar, int x, int y, int z) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(map), "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(x), "r"(y), "r"(z)
                 : "memory");
}
// the same for a 4-D box (x in 4-byte elements, y in rows, z = plane, w = image)
__device__ __forceinline__ void tma_load_4d(void *smem_dst, const CUtensorMap *map, uint64_t *bar, int x, int y, int z, int w) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(map), "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(x), "r"(y), "r"(z),
                 "r"(w)
                 : "memory");
}

// MCU rows per warp tile: formats whose one-MCU-row tile is small (grayscale: 2 KB, one task) take several
// rows per tile so that the staging and bookkeeping are amortised over more blocks.
template <int CT, int HS, int VS>
__host__ __device__ constexpr int warp_tile_mcu_rows() {
    constexpr int bytes = 256 * Fmt<CT>::BPP * 8 * VS;
    return bytes <= 2048 ? 4 : (bytes <= 6144 ? 2 : 1);
}

// =================================================================================================
// Warp-autonomous variant. Every warp owns a private shared-memory tile of 32 full-resolution blocks
// (256 pixels) x one MCU row and walks warp tiles on its own: cp.async its pixel rows, wait with
// __syncwarp only, then run its tasks -- the luma (and K) block rows and one chroma task in which
// lanes 0..15 take Cb and lanes 16..31 Cr when chroma is horizontally decimated. No CTA barrier, no
// role imbalance between warps; the other resident warps hide a warp's load latency.
// PL (channel-planar input, p.channel_planar): the tile holds the BPP planes read, [plane][ROWS][256] in the planes'
// memory order -- the same bytes per tile -- and the row loader interleaves them into the packed pixel words, so the
// arithmetic behind it is the packed kernel's. Byte k of a pixel comes from tile plane p.plane_of[k].
// =================================================================================================
// The body is shared as text (stage_a_warp_body.inc) rather than through an inline function: with the parameters
// passed to a function, the compiler schedules the uint8 kernels' instructions differently.
template <int CT, int HS, int VS, bool PL>
__global__ void __launch_bounds__(128, 4) stage_a_warp_kernel(const __grid_constant__ StageAParams p,
                                                              const __grid_constant__ CUtensorMap tmap, const int use_tma) {
    constexpr bool CONV = false;
    [[maybe_unused]] const jpgb_sample_format fmt{};
#include "stage_a_warp_body.inc"
}
// CONV: the samples are elements of fmt.type, converted while staging; no TMA (tmap and use_tma are placeholders)
template <int CT, int HS, int VS, bool PL>
__global__ void __launch_bounds__(128, 4) stage_a_warp_convert_kernel(const __grid_constant__ StageAParams p,
                                                                      const __grid_constant__ jpgb_sample_format fmt) {
    constexpr bool CONV = true;
    [[maybe_unused]] const CUtensorMap tmap{};
    const int use_tma = 0;
#include "stage_a_warp_body.inc"
}

// =================================================================================================
// Planar input (the ImageBuffer path, encoder.rs:506-515: full-resolution planes of samples taken verbatim).
// One launch per component: a plane is a one-byte-per-sample image whose blocks cover 8*SX x 8*SY samples
// (SX, SY = the component's decimation, point sampling as everywhere). Same warp-autonomous scheme as above:
// a warp tile is 32 blocks of the component x MR block rows; only the sampled rows are staged (cp.async).
// =================================================================================================
template <int SX>
__host__ __device__ constexpr int plane_tile_block_rows() { return SX == 1 ? 4 : (SX == 2 ? 2 : 1); } // 8 KB per warp tile

template <int SX, int SY>
__global__ void __launch_bounds__(128, 4) stage_a_plane_kernel(const __grid_constant__ StageAParams p, const int comp) {
    extern __shared__ __align__(128) uint8_t smem[];
    constexpr int MR = plane_tile_block_rows<SX>();
    constexpr int PITCH = 256 * SX, ROWS = 8 * MR, TILE_BYTES = PITCH * ROWS;
    const int lane = threadIdx.x & 31;
    const unsigned warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned n_warps_total = (gridDim.x * blockDim.x) >> 5;
    uint8_t *tile = smem + (threadIdx.x >> 5) * TILE_BYTES;
    const int H = p.comp_h[comp], V = p.comp_v[comp];
    // block columns and block rows this launch produces (the interleaved layout also holds the MCU padding)
    const int tw = p.mcu_order ? p.comp_pw[comp] : p.comp_tw[comp];
    const int th = p.mcu_order ? p.mcu_rows * V : min(p.mcu_rows * V, p.comp_th[comp] - p.mcu_row0 * V);
    if (th <= 0) return;
    const unsigned tiles_per_row = ((unsigned)tw + 31) / 32, tile_rows = ((unsigned)th + MR - 1) / MR;
    const unsigned n_tiles = tiles_per_row * tile_rows * p.n_images;
    const uint8_t *plane = p.pixels + (size_t)comp * p.plane_stride;
    const int needed_total = tw * 8 * SX; // bytes of a row the blocks read (beyond `width`: the last sample repeated, Q4)

    for (unsigned t = warp_global; t < n_tiles; t += n_warps_total) {
        const unsigned tx = t % tiles_per_row, r = t / tiles_per_row;
        const int by0 = (int)(r % tile_rows) * MR, img = (int)(r / tile_rows);
        const int bx0 = (int)tx * 32;
        const int px0 = bx0 * 8 * SX, py0 = by0 * 8 * SY;
        const uint8_t *src = plane + (size_t)img * p.image_stride;
        const int valid_px = min(PITCH, p.width - px0);
        const int needed_bytes = min(PITCH, needed_total - px0);
        __syncwarp(); // all lanes are done reading the previous tile
        const bool interior = px0 + PITCH <= p.width && py0 + (ROWS - 1) * SY < p.height && (p.row_stride & 15) == 0 &&
                              ((reinterpret_cast<uintptr_t>(src) + (size_t)px0) & 15) == 0;
        if (interior) {
            const uint8_t *g = src + (size_t)py0 * p.row_stride + px0 + lane * 16;
            uint8_t *d = tile + lane * 16;
#pragma unroll 4
            for (int ry = 0; ry < ROWS; ++ry) {
#pragma unroll
                for (int c = 0; c < (PITCH + 511) / 512; ++c)
                    if (c * 512 + 512 <= PITCH || lane * 16 + c * 512 < PITCH) cp_async16(d + c * 512, g + c * 512);
                g += (size_t)SY * p.row_stride;
                d += PITCH;
            }
        } else {
#pragma unroll 1
            for (int ry = 0; ry < ROWS; ++ry) {
                const int sy = min(py0 + ry * SY, p.height - 1);
                const uint8_t *row = src + (size_t)sy * p.row_stride + px0;
                uint8_t *dst = tile + ry * PITCH;
                const bool aligned = (reinterpret_cast<uintptr_t>(row) & 15) == 0;
#pragma unroll 1
                for (int cb = lane * 16; cb < needed_bytes; cb += 32 * 16) {
                    if (aligned && cb + 16 <= valid_px) cp_async16(dst + cb, row + cb);
                    else stage_edge_chunk<1>(dst, row, cb, valid_px);
                }
            }
        }
        cp_async_commit();
        cp_async_wait<0>();
        __syncwarp();
#pragma unroll 1
        for (int mr = 0; mr < MR; ++mr) {
            const int by = by0 + mr, bx = bx0 + lane;
            if (by >= th) break;
            if (bx >= tw) continue;
            const uint8_t *base = tile + mr * 8 * PITCH + lane * 8 * SX;
            int v[64];
            load_block<JPGB_LUMA, ROLE_RAW, SX, 1>(base, PITCH, v);
            dct_2d(v);
            const int gby = by + p.mcu_row0 * V; // block row inside the whole image
            size_t blk = (size_t)img * p.blocks_per_image;
            if (p.mcu_order) {
                const int mcu_x = bx / H, bh = bx - mcu_x * H, gy = gby / V, bv = gby - gy * V;
                blk += ((size_t)gy * p.mcu_cols + mcu_x) * p.bpu + p.slot_base[comp] + bv * H + bh;
            } else {
                blk += p.comp_off[comp] + (size_t)gby * p.comp_tw[comp] + bx;
            }
            int16_t *dst = p.coef + blk * 64;
            if (p.comp_qt[comp] == 0) quantize_store256<0>(p, v, dst);
            else quantize_store256<1>(p, v, dst);
        }
    }
}

// =================================================================================================
// Subsampled YCbCr frames (jpgb_encode_batch_device_ycbcr): one launch per component, each reading its own plane.
// A frame means the full-resolution image whose chroma repeats every plane sample c_h x c_v times. Its block sample at
// full-resolution column X = bx*8*sx + k*sx (sx: the component's decimation) reads column min(X, w-1), which is plane
// column min(X / c_h, cw - 1): the plane is read at its own resolution and clamped at its own edge, rows alike.
// With sx >= c_h and sy >= c_v and one byte per sample, that is stage_a_plane_kernel<sx / c_h, sy / c_v> on the plane
// (its launch's pixels, width and height describe the plane). stage_a_frame_kernel covers the rest:
//   NX, NY: the step between block samples in half plane samples (1, 2, 4, 8). Step 1 (sx = 1 < c_h = 2): each plane
//           sample feeds two block samples; block sample k reads plane sample (k * NX) / 2 of the block's span.
//   BPP:    bytes between horizontally adjacent samples (2: interleaved Cb/Cr). The channel read is byte `coff` of a
//           pair; p.pixels is the pair's first byte, so the edge clamp lands on the same channel's last sample.
//           n_comp = 2 (Cb and Cr in the two bytes of the same pairs, NV12 / NV21): one launch codes components comp and
//           comp + 1, the second from byte coff ^ 1, so the interleaved plane is staged once for both.
// A warp tile is 32 blocks x MR block rows; only the plane rows the blocks read are staged (cp.async).
// =================================================================================================
template <int NX, int NY, int BPP>
struct FrameTile {
    static constexpr int SPAN = 4 * NX;             // plane samples under a block row
    static constexpr int PITCH = 32 * SPAN * BPP;   // bytes of a staged row
    static constexpr int R = NY == 1 ? 4 : 8;       // plane rows under a block
    static constexpr int YSTEP = NY == 1 ? 1 : NY / 2;
    static constexpr int FIT = 8192 / (PITCH * R);  // block rows in about 8 KB
    static constexpr int MR = FIT < 1 ? 1 : (FIT > 8 ? 8 : FIT);
    static constexpr int ROWS = R * MR, TILE_BYTES = PITCH * ROWS;
};

// One 16-byte chunk of a staged frame row, byte by byte, the row's last valid sample of each channel replicated.
// coff >= 0: only byte coff of a pair is read, and the pair's other byte gets that channel's sample too (it is never
// read); coff < 0: both channels. Cold path, kept out of line.
template <int BPP>
__device__ __noinline__ void stage_frame_edge_chunk(uint8_t *dst, const uint8_t *row, int cb, int valid_px, int coff) {
    for (int b = 0; b < 16; ++b) dst[cb + b] = row[(coff < 0 ? (cb + b) % BPP : coff) + min((cb + b) / BPP, valid_px - 1) * BPP];
}

template <int NX, int BPP, int I, int NW>
__device__ __forceinline__ int frame_sample_at(const uint32_t (&w)[NW], unsigned coff) {
    constexpr int O = (I * NX / 2) * BPP;
    return (int)__byte_perm(w[O >> 2], 0, 0x4440 + (O & 3) + (BPP == 1 ? 0u : coff));
}
template <int NX, int BPP, int NW, int... Is>
__device__ __forceinline__ void frame_row(const uint32_t (&w)[NW], int *s, unsigned coff, std::integer_sequence<int, Is...>) {
    ((s[Is] = frame_sample_at<NX, BPP, Is, NW>(w, coff)), ...);
}
// the 8 samples of a block row: the words under its 4 * NX samples (row: 4 * NX * BPP-byte aligned), then the bytes
template <int NX, int BPP>
__device__ __forceinline__ void load_frame_row(const uint8_t *row, int *s, unsigned coff) {
    constexpr int NW = NX * BPP;
    uint32_t w[NW];
    if constexpr (NW % 4 == 0) {
#pragma unroll
        for (int i = 0; i < NW / 4; ++i) {
            const uint4 a = reinterpret_cast<const uint4 *>(row)[i];
            w[4 * i] = a.x;
            w[4 * i + 1] = a.y;
            w[4 * i + 2] = a.z;
            w[4 * i + 3] = a.w;
        }
    } else if constexpr (NW == 2) {
        const uint2 a = *reinterpret_cast<const uint2 *>(row);
        w[0] = a.x;
        w[1] = a.y;
    } else {
        w[0] = *reinterpret_cast<const uint32_t *>(row);
    }
    frame_row<NX, BPP, NW>(w, s, coff, std::make_integer_sequence<int, 8>{});
}

template <int NX, int NY, int BPP>
__global__ void __launch_bounds__(128, 4) stage_a_frame_kernel(const __grid_constant__ StageAParams p, const int comp, const int coff,
                                                                       const int n_comp) {
    extern __shared__ __align__(128) uint8_t smem[];
    using T = FrameTile<NX, NY, BPP>;
    constexpr int SPAN = T::SPAN, PITCH = T::PITCH, R = T::R, YSTEP = T::YSTEP, MR = T::MR, ROWS = T::ROWS;
    const int lane = threadIdx.x & 31;
    const unsigned warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned n_warps_total = (gridDim.x * blockDim.x) >> 5;
    uint8_t *tile = smem + (threadIdx.x >> 5) * T::TILE_BYTES;
    const int H = p.comp_h[comp], V = p.comp_v[comp];
    const int tw = p.mcu_order ? p.comp_pw[comp] : p.comp_tw[comp];
    const int th = p.mcu_order ? p.mcu_rows * V : min(p.mcu_rows * V, p.comp_th[comp] - p.mcu_row0 * V);
    if (th <= 0) return;
    const unsigned tiles_per_row = ((unsigned)tw + 31) / 32, tile_rows = ((unsigned)th + MR - 1) / MR;
    const unsigned n_tiles = tiles_per_row * tile_rows * p.n_images;
    const int needed_total = tw * SPAN * BPP; // bytes of a row the blocks read (beyond the plane: its last sample repeated)

    for (unsigned t = warp_global; t < n_tiles; t += n_warps_total) {
        const unsigned tx = t % tiles_per_row, r = t / tiles_per_row;
        const int by0 = (int)(r % tile_rows) * MR, img = (int)(r / tile_rows);
        const int bx0 = (int)tx * 32;
        const int px0 = bx0 * SPAN, py0 = by0 * 4 * NY; // in plane samples and rows
        const uint8_t *src = p.pixels + (size_t)img * p.image_stride + (size_t)px0 * BPP;
        const int valid_px = p.width - px0;                     // > 0: a tile starts inside the image
        const int valid_bytes = n_comp == 2 ? valid_px * BPP : coff + (valid_px - 1) * BPP + 1; // up to the channel's last sample
        const int needed_bytes = min(PITCH, needed_total - px0 * BPP);
        __syncwarp(); // all lanes are done reading the previous tile
        const bool interior = PITCH <= valid_bytes && py0 + (ROWS - 1) * YSTEP < p.height && (p.row_stride & 15) == 0 &&
                              (reinterpret_cast<uintptr_t>(src) & 15) == 0;
        if (interior) {
            const uint8_t *g = src + (size_t)py0 * p.row_stride + lane * 16;
            uint8_t *d = tile + lane * 16;
#pragma unroll 4
            for (int ry = 0; ry < ROWS; ++ry) {
#pragma unroll
                for (int c = 0; c < (PITCH + 511) / 512; ++c)
                    if (c * 512 + 512 <= PITCH || lane * 16 + c * 512 < PITCH) cp_async16(d + c * 512, g + c * 512);
                g += (size_t)YSTEP * p.row_stride;
                d += PITCH;
            }
        } else {
#pragma unroll 1
            for (int ry = 0; ry < ROWS; ++ry) {
                const uint8_t *row = src + (size_t)min(py0 + ry * YSTEP, p.height - 1) * p.row_stride;
                uint8_t *dst = tile + ry * PITCH;
                const bool aligned = (reinterpret_cast<uintptr_t>(row) & 15) == 0;
#pragma unroll 1
                for (int cb = lane * 16; cb < needed_bytes; cb += 32 * 16) {
                    if (aligned && cb + 16 <= valid_bytes) cp_async16(dst + cb, row + cb);
                    else stage_frame_edge_chunk<BPP>(dst, row, cb, valid_px, n_comp == 2 ? -1 : coff);
                }
            }
        }
        cp_async_commit();
        cp_async_wait<0>();
        __syncwarp();
#pragma unroll 1
        for (int mr = 0; mr < MR; ++mr) {
            const int by = by0 + mr, bx = bx0 + lane;
            if (by >= th) break;
            if (bx >= tw) continue;
            const uint8_t *base = tile + mr * R * PITCH + lane * SPAN * BPP;
            const int gby = by + p.mcu_row0 * V; // block row inside the whole image
#pragma unroll 1
            for (int k = 0; k < (BPP == 2 ? n_comp : 1); ++k) { // the components share their sampling factors
                const int c = comp + k;
                int v[64];
#pragma unroll
                for (int y = 0; y < 8; ++y) load_frame_row<NX, BPP>(base + (NY == 1 ? y / 2 : y) * PITCH, &v[y * 8], (unsigned)(coff ^ k));
                dct_2d(v);
                size_t blk = (size_t)img * p.blocks_per_image;
                if (p.mcu_order) {
                    const int mcu_x = bx / H, bh = bx - mcu_x * H, gy = gby / V, bv = gby - gy * V;
                    blk += ((size_t)gy * p.mcu_cols + mcu_x) * p.bpu + p.slot_base[c] + bv * H + bh;
                } else {
                    blk += p.comp_off[c] + (size_t)gby * p.comp_tw[c] + bx;
                }
                int16_t *dst = p.coef + blk * 64;
                if (p.comp_qt[c] == 0) quantize_store256<0>(p, v, dst);
                else quantize_store256<1>(p, v, dst);
            }
        }
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) f = nullptr;
        return reinterpret_cast<EncodeTiledFn>(f);
    }();
    return fn;
}

// The image stride a tensor map is given: the caller's, or for a single image one that cannot matter (every box has
// image coordinate 0). 0: no map (several images at the same address).
inline unsigned long long tma_image_stride(const StageAParams &p) {
    if (p.image_stride || p.n_images > 1) return p.image_stride;
    return (unsigned long long)p.height * p.row_stride;
}

// Tensor map of the packed pixels as a 3-D tensor of 4-byte elements: (row bytes / 4, rows, images), box =
// one warp tile. Needs 16-byte aligned base, row pitch and image pitch; otherwise the kernel stages with cp.async.
// The extent of a row ends at its last pixel: boxes never reach into the pitch.
inline bool make_pixel_tensor_map(CUtensorMap &map, const StageAParams &p, int bpp, int pitch_bytes, int rows) {
    const unsigned long long row_bytes = (unsigned long long)p.width * bpp, image_stride = tma_image_stride(p);
    if (std::getenv("JPGB_NO_TMA")) return false;
    if ((reinterpret_cast<uintptr_t>(p.pixels) & 15) || (p.row_stride & 15) || (image_stride & 15) || !image_stride || p.width < 256 ||
        p.height < rows)
        return false;
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    const cuuint64_t dims[3] = {row_bytes / 4, (cuuint64_t)p.height, (cuuint64_t)p.n_images};
    const cuuint64_t strides[2] = {p.row_stride, image_stride};
    const cuuint32_t box[3] = {(cuuint32_t)(pitch_bytes / 4), (cuuint32_t)rows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    return fn(&map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<uint8_t *>(p.pixels), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Channel-planar pixels as a 4-D tensor of 4-byte elements: (width / 4, rows, planes, images), box = one warp tile of
// the `planes` planes read (the first ones in memory order). Needs width % 16 == 0 and 16-byte aligned base and strides.
inline bool make_plane_tensor_map(CUtensorMap &map, const StageAParams &p, int planes, int rows) {
    const unsigned long long image_stride = tma_image_stride(p);
    if (std::getenv("JPGB_NO_TMA")) return false;
    if ((reinterpret_cast<uintptr_t>(p.pixels) & 15) || (p.row_stride & 15) || (p.plane_stride & 15) || (image_stride & 15) || !image_stride ||
        (p.width & 15) || p.width < 256 || p.height < rows)
        return false;
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)p.width / 4, (cuuint64_t)p.height, (cuuint64_t)planes, (cuuint64_t)p.n_images};
    const cuuint64_t strides[3] = {p.row_stride, p.plane_stride, image_stride};
    const cuuint32_t box[4] = {64, (cuuint32_t)rows, (cuuint32_t)planes, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    return fn(&map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 4, const_cast<uint8_t *>(p.pixels), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Grid of a persistent warp-kernel launch: the CTAs that fit at once, but no more than the warp tiles need
template <auto Kernel, int CT, int HS, int VS>
cudaError_t warp_grid(const StageAParams &p, size_t smem, unsigned &grid) {
    constexpr int MR = warp_tile_mcu_rows<CT, HS, VS>(), MCUS = 32 / HS;
    unsigned long long ctas = 0;
    const cudaError_t e = resident_ctas<Kernel>(128, smem, ctas);
    if (e != cudaSuccess) return e;
    const unsigned long long n_tiles = (unsigned long long)((p.mcu_cols + MCUS - 1) / MCUS) * ((p.mcu_rows + MR - 1) / MR) * p.n_images;
    if (ctas * 4 > n_tiles) ctas = (n_tiles + 3) / 4;
    grid = (unsigned)ctas;
    return cudaSuccess;
}

template <int CT, int HS, int VS, bool PL>
cudaError_t launch_warp_variant(const StageAParams &p, const jpgb_sample_format &fmt, cudaStream_t stream) {
    constexpr int BPP = Fmt<CT>::BPP;
    constexpr int MR = warp_tile_mcu_rows<CT, HS, VS>();
    constexpr int TILE = 256 * BPP * 8 * VS * MR;
    constexpr size_t smem = (size_t)4 * TILE + 4 * sizeof(uint64_t); // 4 warps per CTA: one private tile and one mbarrier each
    unsigned grid = 0;
    cudaError_t e;
    if constexpr (converts(CT)) {
        if (fmt.type) {
            if ((e = warp_grid<stage_a_warp_convert_kernel<CT, HS, VS, PL>, CT, HS, VS>(p, smem, grid)) != cudaSuccess) return e;
            stage_a_warp_convert_kernel<CT, HS, VS, PL><<<grid, 128, smem, stream>>>(p, fmt);
            return cudaGetLastError();
        }
    }
    if ((e = warp_grid<stage_a_warp_kernel<CT, HS, VS, PL>, CT, HS, VS>(p, smem, grid)) != cudaSuccess) return e;
    CUtensorMap tmap;
    std::memset(&tmap, 0, sizeof(tmap));
    const bool tma = PL ? make_plane_tensor_map(tmap, p, BPP, 8 * VS * MR) : make_pixel_tensor_map(tmap, p, BPP, 256 * BPP, 8 * VS * MR);
    stage_a_warp_kernel<CT, HS, VS, PL><<<grid, 128, smem, stream>>>(p, tmap, tma ? 1 : 0);
    return cudaGetLastError();
}

// the warp kernel instantiated for the luma sampling factors (a single component is always sampled 1x1)
template <int CT, bool PL>
cudaError_t launch_warp(const StageAParams &p, const jpgb_sample_format &fmt, cudaStream_t stream) {
    if constexpr (Fmt<CT>::NCOMP == 1) {
        return launch_warp_variant<CT, 1, 1, PL>(p, fmt, stream);
    } else {
        if (p.hmax == 1 && p.vmax == 1) return launch_warp_variant<CT, 1, 1, PL>(p, fmt, stream);
        if (p.hmax == 2 && p.vmax == 1) return launch_warp_variant<CT, 2, 1, PL>(p, fmt, stream);
        if (p.hmax == 1 && p.vmax == 2) return launch_warp_variant<CT, 1, 2, PL>(p, fmt, stream);
        if (p.hmax == 2 && p.vmax == 2) return launch_warp_variant<CT, 2, 2, PL>(p, fmt, stream);
        if (p.hmax == 4 && p.vmax == 1) return launch_warp_variant<CT, 4, 1, PL>(p, fmt, stream);
        if (p.hmax == 4 && p.vmax == 2) return launch_warp_variant<CT, 4, 2, PL>(p, fmt, stream);
        if (p.hmax == 1 && p.vmax == 4) return launch_warp_variant<CT, 1, 4, PL>(p, fmt, stream);
        return launch_warp_variant<CT, 2, 4, PL>(p, fmt, stream);
    }
}

template <int SX, int SY>
cudaError_t launch_plane_variant(const StageAParams &p, int comp, cudaStream_t stream) {
    constexpr int MR = plane_tile_block_rows<SX>();
    constexpr size_t smem = (size_t)4 * 256 * SX * 8 * MR;
    unsigned long long grid = 0;
    const cudaError_t e = resident_ctas<stage_a_plane_kernel<SX, SY>>(128, smem, grid);
    if (e != cudaSuccess) return e;
    const int tw = p.mcu_order ? p.comp_pw[comp] : p.comp_tw[comp], th = p.mcu_rows * p.comp_v[comp];
    const unsigned long long n_tiles = (unsigned long long)((tw + 31) / 32) * ((th + MR - 1) / MR) * p.n_images;
    if (grid * 4 > n_tiles) grid = (n_tiles + 3) / 4;
    stage_a_plane_kernel<SX, SY><<<(unsigned)grid, 128, smem, stream>>>(p, comp);
    return cudaGetLastError();
}

// planar input: one launch per component with the component's own decimation
cudaError_t launch_planes(const StageAParams &p, cudaStream_t stream) {
    for (int c = 0; c < p.ncomp; ++c) {
        const int sx = p.hmax / p.comp_h[c], sy = p.vmax / p.comp_v[c];
        cudaError_t e = cudaErrorInvalidValue;
#define JPGB_PLANE(X, Y) \
    if (sx == X && sy == Y) e = launch_plane_variant<X, Y>(p, c, stream);
        JPGB_PLANE(1, 1) JPGB_PLANE(2, 1) JPGB_PLANE(1, 2) JPGB_PLANE(2, 2)
        JPGB_PLANE(4, 1) JPGB_PLANE(4, 2) JPGB_PLANE(1, 4) JPGB_PLANE(2, 4) JPGB_PLANE(4, 4)
#undef JPGB_PLANE
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

template <int NX, int NY, int BPP>
cudaError_t launch_frame_variant(const StageAParams &p, int comp, int coff, int n_comp, cudaStream_t stream) {
    using T = FrameTile<NX, NY, BPP>;
    constexpr size_t smem = (size_t)4 * T::TILE_BYTES;
    unsigned long long grid = 0;
    const cudaError_t e = resident_ctas<stage_a_frame_kernel<NX, NY, BPP>>(128, smem, grid);
    if (e != cudaSuccess) return e;
    const int tw = p.mcu_order ? p.comp_pw[comp] : p.comp_tw[comp], th = p.mcu_rows * p.comp_v[comp];
    const unsigned long long n_tiles = (unsigned long long)((tw + 31) / 32) * ((th + T::MR - 1) / T::MR) * p.n_images;
    if (grid * 4 > n_tiles) grid = (n_tiles + 3) / 4;
    stage_a_frame_kernel<NX, NY, BPP><<<(unsigned)grid, 128, smem, stream>>>(p, comp, coff, n_comp);
    return cudaGetLastError();
}

// subsampled YCbCr frames: one launch per component, each with its own plane as p.pixels, width, height, row_stride
// and image_stride; the block geometry and coefficient destinations stay the image's. Cb and Cr in the two bytes of the
// same pairs (NV12, NV21) share one launch: the interleaved plane is read once.
cudaError_t launch_frames(const StageAParams &p, const jpgb_device_ycbcr &f, cudaStream_t stream) {
    const uint8_t *cb = static_cast<const uint8_t *>(f.cb), *cr = static_cast<const uint8_t *>(f.cr);
    const bool pairs = f.c_sample_stride == 2 && (cr == cb + 1 || cb == cr + 1);
    for (int c = 0; c < 3; c += (c == 1 && pairs) ? 2 : 1) {
        const int ch = c ? f.c_h : 1, cv = c ? f.c_v : 1, bpp = c ? (int)f.c_sample_stride : 1;
        const int n_comp = (c == 1 && pairs) ? 2 : 1;
        const uint8_t *plane = c == 0 ? static_cast<const uint8_t *>(f.y) : (c == 1 ? cb : cr);
        const int coff = n_comp == 2 ? (cb > cr ? 1 : 0) : (bpp == 2 ? (int)(reinterpret_cast<uintptr_t>(plane) & 1) : 0); // the channel's byte in its pair
        StageAParams q = p;
        q.pixels = plane - coff;
        q.width = (p.width + ch - 1) / ch;
        q.height = (p.height + cv - 1) / cv;
        q.row_stride = c ? f.c_row_stride : f.y_row_stride;
        q.image_stride = c ? f.c_image_stride : f.y_image_stride;
        q.plane_stride = 0;
        const int nx = 2 * (p.hmax / p.comp_h[c]) / ch, ny = 2 * (p.vmax / p.comp_v[c]) / cv; // steps in half samples
        cudaError_t e = cudaErrorInvalidValue;
        if (bpp == 1 && nx >= 2 && ny >= 2) {
#define JPGB_PLANE(X, Y) \
    if (nx == 2 * X && ny == 2 * Y) e = launch_plane_variant<X, Y>(q, c, stream);
            JPGB_PLANE(1, 1) JPGB_PLANE(2, 1) JPGB_PLANE(1, 2) JPGB_PLANE(2, 2)
            JPGB_PLANE(4, 1) JPGB_PLANE(4, 2) JPGB_PLANE(1, 4) JPGB_PLANE(2, 4) JPGB_PLANE(4, 4)
#undef JPGB_PLANE
        } else {
#define JPGB_FRAME(X, Y, B) \
    if (nx == X && ny == Y && bpp == B) e = launch_frame_variant<X, Y, B>(q, c, coff, n_comp, stream);
            // one byte per sample: only the steps of half a sample
            JPGB_FRAME(1, 1, 1) JPGB_FRAME(1, 2, 1) JPGB_FRAME(1, 4, 1) JPGB_FRAME(1, 8, 1)
            JPGB_FRAME(2, 1, 1) JPGB_FRAME(4, 1, 1) JPGB_FRAME(8, 1, 1)
            // interleaved: every step the 8 JPEG samplings and the 4 chroma subsamplings give
            JPGB_FRAME(1, 1, 2) JPGB_FRAME(1, 2, 2) JPGB_FRAME(1, 4, 2) JPGB_FRAME(1, 8, 2)
            JPGB_FRAME(2, 1, 2) JPGB_FRAME(2, 2, 2) JPGB_FRAME(2, 4, 2) JPGB_FRAME(2, 8, 2)
            JPGB_FRAME(4, 1, 2) JPGB_FRAME(4, 2, 2) JPGB_FRAME(4, 4, 2) JPGB_FRAME(4, 8, 2)
            JPGB_FRAME(8, 1, 2) JPGB_FRAME(8, 2, 2) JPGB_FRAME(8, 4, 2)
#undef JPGB_FRAME
        }
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// The generic kernel's CTA tile: `groups` x 32 MCUs wide, one MCU row high, ~24 KB of pixels in shared memory. A warp
// task is one block position of the MCU (component, v, h) in one group. `frame`: the planes of a subsampled YCbCr
// frame batch (CT == kPlanar)
template <int CT>
cudaError_t launch_generic(StageAParams p, const jpgb_sample_format &fmt, cudaStream_t stream, const jpgb_device_ycbcr *frame = nullptr) {
    const int group_bytes = 32 * 8 * p.hmax * 8 * p.vmax * (p.planar ? p.ncomp : p.bpp);
    const int g = std::min({std::max(1, 24576 / group_bytes), 8, (p.mcu_cols + 31) / 32});
    p.groups = g;
    p.tiles_per_row = (p.mcu_cols + 32 * g - 1) / (32 * g);
    p.tile_w_px = 32 * g * 8 * p.hmax;
    p.tile_h_px = 8 * p.vmax;
    p.tile_pitch = p.tile_w_px * p.bpp; // planar input: one byte per sample
    int n = 0;
    for (int c = 0; c < p.ncomp; ++c)
        for (int v = 0; v < p.comp_v[c]; ++v)
            for (int h = 0; h < p.comp_h[c]; ++h, ++n) {
                p.task_comp[n] = (int8_t)c;
                p.task_v[n] = (int8_t)v;
                p.task_h[n] = (int8_t)h;
            }
    p.tasks_per_group = n;
    const size_t smem = (size_t)p.tile_pitch * p.tile_h_px * (p.planar ? p.ncomp : 1);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(stage_a_kernel<CT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if constexpr (converts(CT))
            if (e == cudaSuccess) e = cudaFuncSetAttribute(stage_a_convert_kernel<CT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (frame && e == cudaSuccess) e = cudaFuncSetAttribute(stage_a_frame_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const int warps = std::min(g * n, 8);
    // grid.z carries the image index and is limited to 65535: larger batches go in several launches
    const unsigned n_images = (unsigned)p.n_images;
    for (unsigned i0 = 0; i0 < n_images; i0 += 65535) {
        StageAParams q = p;
        q.pixels = p.pixels + (size_t)i0 * p.image_stride;
        q.coef = p.coef + (size_t)i0 * p.blocks_per_image * 64;
        q.n_images = (int)std::min(n_images - i0, 65535u);
        const dim3 grid(p.tiles_per_row, p.mcu_rows, q.n_images);
        if (frame) {
            jpgb_device_ycbcr f = *frame;
            f.y = static_cast<const uint8_t *>(f.y) + (size_t)i0 * f.y_image_stride;
            f.cb = static_cast<const uint8_t *>(f.cb) + (size_t)i0 * f.c_image_stride;
            f.cr = static_cast<const uint8_t *>(f.cr) + (size_t)i0 * f.c_image_stride;
            stage_a_frame_generic_kernel<<<grid, warps * 32, smem, stream>>>(q, f);
            continue;
        }
        if constexpr (converts(CT))
            if (fmt.type) {
                stage_a_convert_kernel<CT><<<grid, warps * 32, smem, stream>>>(q, fmt);
                continue;
            }
        stage_a_kernel<CT><<<grid, warps * 32, smem, stream>>>(q);
    }
    return cudaGetLastError();
}

// packed pixels: the warp kernel, or the generic one when JPGB_FORCE_GENERIC_STAGE_A asks for the cross-check.
// Channel-planar pixels take the warp kernel's planar staging, instantiated for Rgb (Bgr, Rgba and Bgra are Rgb with
// their planes in another order), Cmyk and CmykAsYcck. Samples of a wider type: the converting kernels, instantiated
// for the colour types that take them (converts()).
template <int CT>
cudaError_t launch_packed(const StageAParams &p, const jpgb_sample_format &fmt, cudaStream_t stream) {
    if (fmt.type && !converts(CT)) return cudaErrorInvalidValue;
    if (!p.use_fast) return launch_generic<CT>(p, fmt, stream);
    if (!p.channel_planar) return launch_warp<CT, false>(p, fmt, stream);
    if constexpr (CT == JPGB_RGB || CT == JPGB_CMYK || CT == JPGB_CMYK_AS_YCCK) return launch_warp<CT, true>(p, fmt, stream);
    return cudaErrorInvalidValue;
}

} // namespace

cudaError_t launch_stage_a(const StageAParams &p_in, uint32_t n_images, const jpgb_sample_format &fmt, cudaStream_t stream) {
    StageAParams p = p_in;
    p.n_images = (int)n_images;
    if (p.planar) {
        if (fmt.type) return cudaErrorInvalidValue;
        return p.use_fast ? launch_planes(p, stream) : launch_generic<kPlanar>(p, fmt, stream);
    }
    switch (p.color_type) {
    case JPGB_LUMA: return launch_packed<JPGB_LUMA>(p, fmt, stream);
    case JPGB_RGB: return launch_packed<JPGB_RGB>(p, fmt, stream);
    case JPGB_RGBA: return launch_packed<JPGB_RGBA>(p, fmt, stream);
    case JPGB_BGR: return launch_packed<JPGB_BGR>(p, fmt, stream);
    case JPGB_BGRA: return launch_packed<JPGB_BGRA>(p, fmt, stream);
    case JPGB_CMYK_AS_YCCK: return launch_packed<JPGB_CMYK_AS_YCCK>(p, fmt, stream);
    case JPGB_YCBCR: return launch_packed<JPGB_YCBCR>(p, fmt, stream);
    case JPGB_YCCK: return launch_packed<JPGB_YCCK>(p, fmt, stream);
    case JPGB_CMYK: return launch_packed<JPGB_CMYK>(p, fmt, stream);
    default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_stage_a_frames(const StageAParams &p_in, uint32_t n_images, const jpgb_device_ycbcr &frame, cudaStream_t stream) {
    StageAParams p = p_in;
    p.n_images = (int)n_images;
    if (!p.planar || p.ncomp != 3) return cudaErrorInvalidValue;
    return p.use_fast ? launch_frames(p, frame, stream) : launch_generic<kPlanar>(p, jpgb_sample_format{}, stream, &frame);
}

} // namespace jpgb
