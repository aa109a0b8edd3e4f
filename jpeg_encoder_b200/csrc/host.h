// Host-side model of the reference's encoder state: components, quantization tables, Huffman
// tables, scan plan and container segments. Everything here is tiny and runs on the CPU, exactly
// where the reference does it once per encode (SURVEY.md section 8a: "negligible (host-side in new
// build)"). The per-pixel / per-block / per-bit work lives in the .cu files.
#pragma once

#include <cstdint>
#include <string>
#include <vector>

#include "../../include/jpegenc_b200.h"
#include "device_types.h"

namespace jpgb {

// src/encoder.rs:190-197
struct Component {
    uint8_t id, qtable, dc_table, ac_table, h, v;
};

// src/quantization.rs:209-213; `value` is the table entry already multiplied by 8
struct QuantTable {
    uint16_t value[64];
    int32_t recip[64], corr[64];
    uint8_t dqt_byte(int natural_index) const { return (uint8_t)(value[natural_index] >> 3); }
};

// src/huffman.rs:66-70; lookup packed as (size << 16) | code, 0 for a symbol without a code (Q18)
struct HuffTable {
    uint8_t length[16];
    std::vector<uint8_t> values;
    uint32_t lookup[256];
    void set(const uint8_t len[16], const uint8_t *vals, size_t n);
    // HuffmanTable::new_optimized (Annex K.2), src/huffman.rs:99-221. false if a code would exceed 32 bits.
    bool set_optimized(const uint32_t freq[257]);
    // What the entropy kernel reads: for symbol s with value size z (s itself for a DC table, s & 15 for an AC
    // table) the word (code_length + z) << 27 | code << z, i.e. everything of huffman_encode_value's write_bits
    // argument (src/writer.rs:320-329) except the value bits. false if a coded symbol does not fit
    // (code_length + z > 31 or code << z beyond 27 bits: impossible for 8-bit samples, where z <= 11).
    bool device_words(bool ac, uint32_t out[256]) const;
};

enum class Mode { Interleaved, Sequential, Progressive };

struct Scan {
    int comp;        // component index, or -1 for the interleaved scan over all components
    int ss, se;      // spectral selection, inclusive
    uint32_t n_units, blocks_per_unit;
    uint64_t visit_base;   // first block visit of this scan inside one image
    uint32_t seg_base, n_segs;
    uint32_t chunk_base = 0; // first coding chunk of this scan inside one image
    uint32_t rst_base = 0; // restart segments of this scan before this strip
    std::vector<uint8_t> sos; // SOS segment bytes (marker included)
};

// Everything derived from jpgb_params that does not depend on pixel values.
struct Plan {
    jpgb_params p;       // copy (apps pointer not owned)
    int bpp, ncomp;
    Component comps[4];
    int hmax, vmax;
    uint32_t mcu_cols, mcu_rows;
    uint32_t pad_w[4], pad_h[4];   // MCU-padded block grid per component
    uint32_t true_w[4], true_h[4]; // grid walked by encode_blocks (src/encoder.rs:1012-1025)
    // Coefficient buffer of one image (DESIGN.md section 3). Interleaved mode: blocks in MCU order (block = mcu * bpu + slot),
    // block_off unused. Other modes: per component the raster of its true grid, components back to back at block_off[c].
    uint64_t block_off[4], blocks_per_image;
    uint32_t bpu_interleaved = 0;   // blocks per MCU
    uint32_t slot_base[4] = {};     // first slot of component c inside the MCU
    // Coding chunks: a chunk is <= chunk_T consecutive visits of one restart segment of one scan; scans that walk the
    // same blocks (a component's DC scan and AC bands) form a group whose chunks are coded by the same CTA.
    uint32_t chunk_T = 256, n_groups = 1, scans_per_group = 1;
    struct Group {
        int comp;
        uint32_t bpu, seg_visits, n_segs, cps, item_base;
        uint64_t n_visits, block_base;
    } groups[4];
    uint32_t chunks_per_image = 0, items_per_image = 0;
    QuantTable q[2];
    Mode mode;
    std::vector<Scan> scans;
    uint64_t visits_per_image;
    uint32_t segs_per_image;
    std::vector<uint8_t> prefix; // SOI, APP0, [APP14], user APPn  (src/encoder.rs:536-554)

    // strip mode (strip != nullptr): geometry of the strip, header of the whole image
    bool planar = false; // ImageBuffer path: one plane per component, samples taken verbatim
    bool is_strip = false;
    jpgb_strip strip{};
    int build(const jpgb_params &params, const jpgb_strip *strip = nullptr); // returns JPGB_* code
    // SOF, DQT x2, DHT x2|4, [DRI] (Encoder::write_frame_header, src/encoder.rs:633-667)
    void frame_header(const HuffTable huff[2][2], std::vector<uint8_t> &out) const;
    void fill_device_plan(DevPlan &d) const;
    void fill_stage_a(StageAParams &a) const;
};

void default_huffman_tables(HuffTable huff[2][2]); // Annex K.3, src/huffman.rs:14-64
int bytes_per_pixel(uint8_t color_type);
int num_components(uint8_t color_type);
extern const uint8_t kZigzag[64];

} // namespace jpgb
