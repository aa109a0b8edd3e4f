// Plain structs shared between the host planner and the kernels.
#pragma once
#include <cstdint>

namespace jpgb {

constexpr int kMaxScans = 256;  // 4 components x 64 progressive scans
constexpr int kMaxSlots = 20;   // blocks per MCU-sized unit: YCCK at F_4_2 / F_2_4 has 8 + 1 + 1 + 8 = 18

// n / d for 32-bit n and a divisor fixed per launch: one multiply-high and one correction step instead of the
// ~20-instruction divide. m = floor(2^32 / d) (2^32 - 1 for d = 1) under-estimates the quotient by at most one.
struct FastDiv {
    unsigned d, m;
};
inline FastDiv make_fastdiv(unsigned d) {
    FastDiv f;
    f.d = d;
    f.m = d <= 1 ? 0xFFFFFFFFu : (unsigned)((1ull << 32) / d);
    return f;
}
#ifdef __CUDACC__
__device__ __forceinline__ void divmod(unsigned n, const FastDiv f, unsigned &q, unsigned &r) {
    q = __umulhi(n, f.m);
    r = n - q * f.d;
    if (r >= f.d) {
        ++q;
        r -= f.d;
    }
}
#endif

// Quantizer constants per table, natural order. q = (v*mul + (v < 0 ? add_neg : add_pos)) >> 16
// reproduces `((abs(v) + corr) * recip) >> 15` with the sign re-applied (src/quantization.rs:291-307):
// mul = 2*recip, add_pos = 2*corr*recip, add_neg = 2*(32767 - corr*recip).
struct QuantConsts {
    int32_t mul[64];
    int32_t add_pos[64];
    int32_t add_neg[64];
};

struct StageAParams {
    const uint8_t *pixels;
    int16_t *coef;
    unsigned long long image_stride;     // bytes between images
    unsigned long long blocks_per_image;
    int width, height, bpp, color_type, ncomp;
    int hmax, vmax;
    int mcu_cols, mcu_rows;
    // groups .. tile_pitch and task_*: the CTA tiling of the generic kernel, filled by its launcher
    int groups;            // 32-MCU groups per CTA tile
    int tiles_per_row;
    int tasks_per_group;   // warp tasks per group = sum over components of H_c*V_c
    int tile_w_px, tile_h_px, tile_pitch; // pitch in bytes
    int n_images;
    int planar;            // 1: pixels = ncomp full-resolution planes of width*height bytes (plane_stride apart)
    unsigned long long plane_stride;
    unsigned long long row_stride; // bytes between pixel rows (of a plane when planar / channel_planar)
    // 1: the packed ColorType's pixels come as planes, byte k of a pixel from plane plane_of[k] (plane_stride apart);
    // the kernels interleave them while staging
    int channel_planar;
    int plane_of[4];
    int use_fast;          // 1: stage_a_warp_kernel / stage_a_plane_kernel, 0: stage_a_kernel
    // Coefficient layout (DESIGN.md section 3). mcu_order = 1 (interleaved scan): blocks in the order the scan codes
    // them, block = (mcu * bpu + slot). mcu_order = 0: per component the raster of its TRUE grid (comp_tw x comp_th,
    // the one encode_blocks walks), components back to back; blocks of the MCU padding are not stored.
    int mcu_order, bpu;
    int mcu_row0;          // a horizontal slice of the image: its first MCU row inside the whole image (destination rows are global)
    int slot_base[4];      // first slot of the component inside the MCU (mcu_order)
    int comp_tw[4], comp_th[4];
    // per warp task inside a group of the generic kernel: component and block position inside the MCU
    int8_t task_comp[kMaxSlots], task_v[kMaxSlots], task_h[kMaxSlots];
    int comp_h[4], comp_v[4], comp_qt[4], comp_pw[4];
    unsigned long long comp_off[4];
    QuantConsts q[2];
};

struct DevScan {
    int comp, ss, se;
    unsigned n_units, bpu;
    unsigned seg_base, n_segs;
    unsigned chunk_base;        // first chunk of this scan inside one image
    unsigned sos_off, sos_len;  // into DevPlan::blob
    unsigned rst_base;          // restart segments of this scan that lie before this strip (0 for a whole image)
};

// Scans that code the same blocks in the same order: the single interleaved scan, or all scans of one component
// (one in sequential mode; the DC scan and every AC band in progressive mode). A coding CTA stages the blocks of
// one *chunk* once and codes them for every scan of the group.
struct DevGroup {
    int comp;                       // -1: interleaved
    unsigned bpu;                   // blocks per unit (MCU): 1 unless interleaved
    unsigned long long n_visits;    // blocks the group walks = n_units * bpu
    unsigned long long block_base;  // first block of the group in one image's coefficient buffer
    unsigned seg_visits;            // visits per restart segment (n_visits when restarts are off)
    unsigned n_segs, cps;           // segments, chunks per segment
    unsigned item_base;             // first work item of the group inside one image
    FastDiv div_cps, div_bpu;
};

struct DevPlan {
    int n_scans, ncomp, n_slots, restart;   // restart interval in units (0 = off)
    int n_groups, spg;                      // groups, scans per group: scan index = group + j * n_groups
    int chunk_T;                            // visits per chunk = threads of the coding CTA (32 / 64 / 128 / 256)
    int mcu_order;
    unsigned mcu_cols;
    unsigned long long blocks_per_image;
    unsigned segs_per_image, chunks_per_image, items_per_image;
    FastDiv div_items;      // by items_per_image (tickets below 2^32; beyond that the kernel divides in 64 bits)
    int has_eoi;            // 0 for every strip but the last
    // 1: a strip without restart intervals. Its part of each scan is a bare bit string: no lead, no pad bits, no EOI,
    // and the scan's segment is rounded up to 16 bytes so that the next one starts on a 128-bit word
    int bare;
    int8_t slot_comp[kMaxSlots];
    uint8_t slot_back[kMaxSlots];   // interleaved: distance (in blocks of the MCU-ordered buffer) to the DC predecessor
    uint8_t slot_first[kMaxSlots];  // 1: first block of its component inside the MCU (predictor resets at restarts)
    int comp_tbl[4];
    DevGroup groups[4];
    DevScan scans[kMaxScans];
    unsigned char blob[kMaxScans * 10]; // SOS segments of scans 1.. (10 bytes each: single component)
};

} // namespace jpgb
