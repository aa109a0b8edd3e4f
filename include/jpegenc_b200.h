/*
 * jpegenc_b200.h -- C ABI of the B200-native JPEG encode path (drop-in for the encode path of
 * vstroebel/jpeg-encoder v0.7.0). Plain pointers and sizes only; no CUDA or torch types.
 *
 * The reference has no FFI of its own (SURVEY.md section 8b). The cut is made at
 * `Encoder::encode_image_internal` (/root/reference/src/encoder.rs:517-567): everything between
 * "packed pixels in" and "JFIF bytes out". A Rust `Encoder<W>` shim keeps the crate's public API
 * (Encoder::new, the setters, encode) and forwards to these entry points; the binding a maintainer
 * would add is shown in INTEGRATION.md. include/jpeg_encoder.hpp is the same mirror in C++ and
 * jpeg_encoder_b200/encoder.py in Python (ctypes).
 *
 * Output bytes are identical to the reference's for the same input and settings. There is no CPU
 * fallback: every entry point fails with JPGB_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef JPEGENC_B200_H
#define JPEGENC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ColorType -- /root/reference/src/encoder.rs:72-99 (same order) */
enum {
    JPGB_LUMA = 0, JPGB_RGB = 1, JPGB_RGBA = 2, JPGB_BGR = 3, JPGB_BGRA = 4,
    JPGB_YCBCR = 5, JPGB_CMYK = 6, JPGB_CMYK_AS_YCCK = 7, JPGB_YCCK = 8
};

/* QuantizationTableType -- src/quantization.rs:8-59 (index() order), 9 = Custom(Box<[u16;64]>) */
enum {
    JPGB_QT_DEFAULT = 0, JPGB_QT_FLAT = 1, JPGB_QT_CUSTOM_MS_SSIM = 2, JPGB_QT_CUSTOM_PSNR_HVS = 3,
    JPGB_QT_IMAGE_MAGICK = 4, JPGB_QT_KLEIN_SILVERSTEIN_CARNEY = 5, JPGB_QT_DENTAL_XRAYS = 6,
    JPGB_QT_VISUAL_DETECTION_MODEL = 7, JPGB_QT_IMPROVED_DETECTION_MODEL = 8, JPGB_QT_CUSTOM = 9
};

/* EncodingError -- src/error.rs:6-28, plus the CUDA failure the reference cannot have */
enum {
    JPGB_OK = 0,
    JPGB_ERR_BAD_IMAGE_DATA = 1,     /* BadImageData { length, required }   src/encoder.rs:447-454 */
    JPGB_ERR_ZERO_DIMENSIONS = 2,    /* ZeroImageDimensions                 src/encoder.rs:521-526 */
    JPGB_ERR_INVALID_APP_SEGMENT = 3,/* InvalidAppSegment(nr)               src/encoder.rs:375-376 */
    JPGB_ERR_APP_SEGMENT_TOO_LARGE = 4, /* AppSegmentTooLarge(len)          src/encoder.rs:377-378 */
    JPGB_ERR_BAD_PARAMS = 5,         /* what the reference rejects by panic/assert (scan count, sampling) */
    JPGB_ERR_SINK = 6,               /* IoError / Write: the sink callback returned non-zero */
    JPGB_ERR_NOMEM = 7,
    JPGB_ERR_CUDA = 8,               /* no usable sm_100 device, or a CUDA call failed */
    JPGB_ERR_HUFFMAN = 9             /* optimized code longer than 32 bits (the reference panics) */
};

/* one `add_app_segment(nr, data)` entry, src/encoder.rs:374-383. ICC/EXIF are expanded into
 * these by the caller exactly as add_icc_profile / add_exif_metadata do (:392-435). */
typedef struct jpgb_app_segment {
    uint8_t nr;            /* 1..15 */
    const uint8_t *data;
    uint32_t len;          /* <= 65533 */
} jpgb_app_segment;

/* The state of an `Encoder<W>` at the moment `encode` is called (src/encoder.rs:213-231).
 * Caller-owned, read-only during the call. */
typedef struct jpgb_params {
    uint16_t width, height;        /* encode(data, width, height, ..)                  :440-446 */
    uint8_t color_type;            /* JPGB_LUMA .. JPGB_YCCK                            :72-99  */
    uint8_t quality;               /* Encoder::new(w, quality); clamped 1..=100         :239    */
    uint8_t sampling;              /* SamplingFactor as (h<<4)|v; alias bit 0x80 ignored :120-176 */
    uint8_t qtable_kind[2];        /* [luma, chroma] JPGB_QT_*                          :300-306 */
    uint16_t qtable_custom[2][64]; /* natural (row-major) order, used when kind == JPGB_QT_CUSTOM */
    uint8_t progressive_scans;     /* 0 = baseline; 2..=64 = set_progressive_scans      :317-335 */
    uint8_t optimize_huffman;      /* set_optimized_huffman_tables                      :357-359 */
    uint16_t restart_interval;     /* 0 = off; set_restart_interval                     :345-347 */
    uint8_t density_unit;          /* 0 PixelAspectRatio, 1 Inches, 2 Centimeters  src/writer.rs:16-59 */
    uint16_t density_x, density_y; /* default (1,1) with unit 0 */
    uint32_t n_app;
    const jpgb_app_segment *apps;  /* insertion order */
} jpgb_params;

/* Fill `p` with what `Encoder::new(w, quality)` sets (src/encoder.rs:239-275): default tables,
 * F_2_2 below quality 90 else F_1_1, density (1,1) unit 0, everything else off. */
void jpgb_params_default(jpgb_params *p, uint8_t quality);

/* An encoder context bound to one CUDA device: its stream, scratch buffers and pinned staging.
 * Not thread-safe; create one per host thread (the reference's Encoder is likewise single-owner).
 * `cuda_stream` may be NULL (the context creates its own) or a cudaStream_t the work is queued on. */
typedef struct jpgb_encoder jpgb_encoder;
int jpgb_encoder_create(int device, void *cuda_stream, jpgb_encoder **out);
void jpgb_encoder_destroy(jpgb_encoder *enc);
const char *jpgb_last_error(const jpgb_encoder *enc); /* text of the last failure on this context */

/* Encoder::encode (src/encoder.rs:440-503): host pixels in, complete JFIF file out.
 * `pixels` is packed, row stride width*bpp; bytes past width*height*bpp are ignored (Q22).
 * On success *out is a library-owned buffer (release with jpgb_free). */
int jpgb_encode(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *pixels, size_t len,
                uint8_t **out, size_t *out_len);
void jpgb_free(void *buf);

/* Same, delivering the bytes through a JfifWrite::write_all-style callback
 * (src/writer.rs:76-82). A non-zero return from `write_all` aborts with JPGB_ERR_SINK. The callback is
 * invoked once, on the context's pinned download buffer (no intermediate copy). `pixels` may be pageable
 * (it is staged through pinned buffers of the context) or pinned / registered (copied directly). */
typedef int (*jpgb_write_all_fn)(void *user, const uint8_t *buf, size_t len);
int jpgb_encode_to_sink(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *pixels, size_t len,
                        jpgb_write_all_fn write_all, void *user);

/* Encoder::encode_image<I: ImageBuffer> (src/encoder.rs:506-515, trait at src/image_buffer.rs:86-98):
 * the caller has already produced the component samples (what `fill_buffers` appends row by row).
 * `p->color_type` names the JPEG colour type: JPGB_LUMA (1 plane), JPGB_YCBCR (3), JPGB_CMYK or
 * JPGB_YCCK (4). planes[c] holds width*height samples of component c, taken verbatim. */
int jpgb_encode_planar(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *const planes[4], size_t plane_len,
                       uint8_t **out, size_t *out_len);
/* Same, delivering the bytes to a JfifWrite::write_all-style callback (what `Encoder<W>::encode_image` binds). */
int jpgb_encode_planar_to_sink(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *const planes[4], size_t plane_len,
                               jpgb_write_all_fn write_all, void *user);

/* Batch of `n` images of identical geometry and settings (BASELINE config 3; no reference
 * equivalent -- the crate is called once per image). Host memory in and out.
 * pixels[i] points at image i. outs[i]/out_lens[i] receive library-owned buffers (jpgb_free). */
int jpgb_encode_batch(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *const *pixels,
                      size_t len_each, uint32_t n, uint8_t **outs, size_t *out_lens);

/* Same, without the per-file copies: the n files are left back to back in pinned host memory owned by
 * the context (*files), file i at [offsets[i], offsets[i+1]) (host array of n + 1). Valid until the
 * next call on this context. Uploads, encoding and downloads of consecutive chunks overlap. */
int jpgb_encode_batch_pinned(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *const *pixels,
                             size_t len_each, uint32_t n, const uint8_t **files, uint64_t *offsets);

/* Device-resident batch: `d_pixels` is device memory holding n images `image_stride` bytes apart.
 * The n files are written back to back into device memory owned by the context; on return
 * *d_files points at it and offsets[0..n] (host array of n+1) delimits file i as
 * [offsets[i], offsets[i+1]). The buffer stays valid until the next call on this context.
 * This is the path bench.py times for the device-resident `value`. */
int jpgb_encode_batch_device(jpgb_encoder *enc, const jpgb_params *p, const void *d_pixels,
                             size_t image_stride, uint32_t n, const void **d_files, uint64_t *offsets);

/* Device images in any row pitch, packed or channel-planar (crops and views of a tensor, pitched allocations,
 * (N, C, H, W) tensors), read where they lie. Sample ch of pixel (x, y) of image i is at
 *   packed (plane_stride == 0): data + i*image_stride + y*row_stride + x*bpp + ch
 *   planar (plane_stride > 0):  data + i*image_stride + ch*plane_stride + y*row_stride + x
 * with ch in the ColorType's byte order. */
typedef struct jpgb_device_images {
    const void *data;       /* device address of image 0's first sample (plane 0 when planar) */
    uint64_t image_stride;  /* bytes between image i and image i + 1 (0: every image is the same pixels) */
    uint64_t row_stride;    /* bytes between row y and row y + 1 of an image (of a plane when planar) */
    uint64_t plane_stride;  /* 0: packed pixels, bpp bytes each in the ColorType's byte order;
                               > 0: channel-planar, channel c of the ColorType's byte order at data + c * plane_stride */
} jpgb_device_images;

/* jpgb_encode_batch_device for a jpgb_device_images layout: the same output (files back to back in context-owned
 * device memory, offsets[0..n]), and files byte-identical to those of the same pixels handed over packed. Per
 * ColorType the samples mean what they mean packed: Rgb, Bgr, Rgba, Bgra planes come in that channel order, and the
 * alpha plane of Rgba / Bgra is never read (it need not exist); Cmyk is inverted and CmykAsYcck converted; Ycbcr and
 * Ycck are taken verbatim; Luma planar is Luma packed.
 * Rejected before anything is enqueued (no launch), in this order, with JPGB_ERR_BAD_PARAMS unless noted:
 *   null arguments or n == 0;
 *   what jpgb_encode_batch_device rejects in `p` (same codes), except the BadImageData length check;
 *   row_stride < width*bpp (packed) or < width (planar); plane_stride > 0 but < width;
 *   an extent beyond 64-bit addresses;
 *   data that is not device or managed memory usable on the context's device;
 *   a last byte read outside the allocation that holds data: the byte at
 *     (n-1)*image_stride + (height-1)*row_stride + width*bpp - 1                        (packed)
 *     (n-1)*image_stride + c_max*plane_stride + (height-1)*row_stride + width - 1       (planar)
 *   where c_max is the highest plane read (2 for Rgb, Bgr, Ycbcr, Rgba, Bgra; 3 for Cmyk, CmykAsYcck, Ycck; 0 for Luma).
 * No kernel reads a byte outside the described samples. */
int jpgb_encode_batch_device_strided(jpgb_encoder *enc, const jpgb_params *p, const jpgb_device_images *images,
                                     uint32_t n, const void **d_files, uint64_t *offsets);

/* Order the context's stream after all work queued so far on `stream` (an event wait; the host does not block).
 * stream may be cudaStreamLegacy (1) or cudaStreamPerThread (2); the context's own stream is a no-op. Use it when
 * the pixels of the next encode are produced on a stream of the caller's. */
int jpgb_encoder_wait_stream(jpgb_encoder *enc, void *stream);

/* ---- one very large image split into strips of whole MCU rows (BASELINE config 5) ---------------
 * No reference equivalent: the crate encodes an image on one thread. A strip boundary must fall on
 * a restart boundary of *every* scan (src/encoder.rs:748-757, 833-839: the DC predictors reset and
 * the bit stream is byte aligned there), so strips need restart_interval > 0, first_row a multiple
 * of 8*Vmax, and in every scan (first unit of the strip) % restart_interval == 0.
 * Each strip is encoded on its own GPU; the final file is, scan by scan, the concatenation of the
 * strips' pieces: strip 0's piece of scan 0 starts with the file header (SOI .. first SOS), its
 * piece of scan k > 0 with that scan's SOS; every other piece starts with the RSTn marker that
 * precedes its first segment; the last strip's last piece ends with EOI. */
typedef struct jpgb_strip {
    uint32_t strip_index, n_strips;
    uint16_t first_row;   /* first pixel row of the strip in the whole image */
    uint16_t rows;        /* pixel rows in the strip */
    uint16_t full_height; /* height of the whole image (goes into SOF) */
} jpgb_strip;

/* number of scans the settings produce (1 interleaved, ncomp sequential, ncomp * scans progressive) */
int jpgb_scan_count(const jpgb_params *p, uint32_t *n_scans);

/* Largest number of equal-as-possible strips <= max_strips the image can be cut into, and their
 * (first_row, rows). Returns JPGB_ERR_BAD_PARAMS when the settings do not allow strips at all. */
int jpgb_plan_strips(const jpgb_params *p, uint32_t max_strips, jpgb_strip *strips, uint32_t *n_strips);

/* Encode one strip. `p->height` is the whole image's height; `d_pixels` (device) points at the
 * strip's first row. On return *d_bytes is device memory owned by the context holding the strip's
 * pieces back to back and piece_offsets[0..n_scans] (host) delimits piece k as
 * [piece_offsets[k], piece_offsets[k+1]). With optimized Huffman tables use the _optimized entry below. */
int jpgb_encode_strip_device(jpgb_encoder *enc, const jpgb_params *p, const jpgb_strip *strip, const void *d_pixels,
                             const void **d_bytes, uint64_t *piece_offsets);

/* Strips with optimized Huffman tables (src/encoder.rs:1086-1200 builds the tables from the symbol
 * histogram of the whole image, so the strips exchange theirs first):
 *  1. every strip: jpgb_strip_histogram_device -> hist[table 0|1][dc|ac][257] of the strip, its DC chain
 *     started at 0, and edge_dc[0..3] / edge_dc[4..7] = DC of the first / last block of each component;
 *  2. the caller sums the histograms over the strips (an all-reduce; jpeg_encoder_b200/sharding.py does it
 *     with NCCL) and gathers the edge_dc arrays in strip order (n_strips * 8 values);
 *  3. jpgb_merge_strip_histograms re-chains the first DC difference of every strip to the block in front
 *     of it (the reference's histogram never resets the DC predictor, Q17) -> hist_total;
 *  4. every strip: jpgb_encode_strip_device_optimized with hist_total. When it follows step 1 on the same context, strip and
 *     pixel pointer (the pixels untouched in between), the coefficients of step 1 are reused: the colour+DCT kernel runs once. */
#define JPGB_HIST_WORDS (2 * 2 * 257)
int jpgb_strip_histogram_device(jpgb_encoder *enc, const jpgb_params *p, const jpgb_strip *strip, const void *d_pixels,
                                uint32_t hist[JPGB_HIST_WORDS], int16_t edge_dc[8]);
int jpgb_merge_strip_histograms(const jpgb_params *p, uint32_t n_strips, const uint32_t hist_sum[JPGB_HIST_WORDS],
                                const int16_t *edge_dc /* n_strips * 8 */, uint32_t hist_total[JPGB_HIST_WORDS]);
int jpgb_encode_strip_device_optimized(jpgb_encoder *enc, const jpgb_params *p, const jpgb_strip *strip, const void *d_pixels,
                                       const uint32_t hist_total[JPGB_HIST_WORDS], const void **d_bytes, uint64_t *piece_offsets);

/* ---- gathering the strips' pieces on the root GPU, device to device (the "peer copy" of BASELINE config 5) ----
 * The assembled file is scan-major: for every scan, the pieces of strips 0..n-1 in order. Each GPU stores its own
 * pieces straight into the root's buffer:
 *   root:   jpgb_gather_target_create -> a device buffer + a 64-byte CUDA IPC handle that the other processes receive
 *           (jpeg_encoder_b200/sharding.py broadcasts it once over torch.distributed);
 *   others: jpgb_gather_target_open   -> the same memory as a peer pointer (NVLink);
 *   every step, every rank: piece offsets of the strip just encoded stay on the device (jpgb_last_piece_offsets_device),
 *           are all-gathered by the caller into one table of world * (n_scans + 1) u64 (one NCCL all-gather: the only
 *           collective of the path), then jpgb_gather_place_pieces launches one kernel that stores this rank's pieces
 *           at their final offsets. A barrier of the caller's choice tells the root when every rank is done.
 * All of it is asynchronous on the context's stream; nothing here synchronises with the host. */
int jpgb_gather_target_create(jpgb_encoder *enc, size_t capacity, void **d_target, uint8_t ipc_handle[64]);
int jpgb_gather_target_open(jpgb_encoder *enc, const uint8_t ipc_handle[64], void **d_target);
int jpgb_gather_target_close(jpgb_encoder *enc, void *d_target, int opened_from_handle);
int jpgb_last_piece_offsets_device(jpgb_encoder *enc, const uint64_t **d_offsets, uint32_t *n_scans);
/* d_table: world * (n_scans + 1) piece offsets in rank order (device memory). d_total (optional, device): receives the
 * size of the assembled file. Pieces are read from the output of the last jpgb_encode_strip_device* call. A piece that
 * would overrun target_capacity is not written; *d_total > target_capacity reports it. */
int jpgb_gather_place_pieces(jpgb_encoder *enc, void *d_target, size_t target_capacity, const uint64_t *d_table, uint32_t world,
                             uint32_t rank, uint64_t *d_total);

/* Copy `n` bytes of context-owned (or any) device memory to host memory; synchronous on the context's stream. */
int jpgb_download(jpgb_encoder *enc, const void *d_src, size_t n, void *host_dst);

/* ---- stage-level entry points (parity tests and roofline timing) ------------------------------ */

/* Layout of the coefficient buffer for `p` (64 i16 zig-zag coefficients per block; Q9). The buffer is ordered the
 * way the scans of the mode read it (Q14):
 *  - mcu_order = 1 (interleaved scan, src/encoder.rs:747-791): the blocks of the MCU-padded grids in coding order,
 *    block of (MCU m in raster order, slot s) = m * blocks_per_mcu + s, slot = slot_base[c] + v * comp_h[c] + h;
 *  - mcu_order = 0 (sequential / progressive, src/encoder.rs:1012-1031): per component the raster of its TRUE grid
 *    (true_w x true_h, the one encode_blocks walks), first block at block_offset[c]; blocks that exist only as MCU
 *    padding are never coded in these modes and are not stored. */
typedef struct jpgb_coef_layout {
    uint32_t n_components;
    uint32_t blocks_w[4], blocks_h[4]; /* padded grid = mcu_cols*H_c x mcu_rows*V_c */
    uint32_t true_w[4], true_h[4];     /* grid encode_blocks walks (src/encoder.rs:1012-1025) */
    uint64_t block_offset[4];          /* mcu_order = 0: first block of the component, in blocks */
    uint64_t blocks_per_image;
    uint32_t mcu_order, mcu_cols, mcu_rows, blocks_per_mcu;
    uint32_t slot_base[4], comp_h[4], comp_v[4];
} jpgb_coef_layout;
int jpgb_coef_layout_for(const jpgb_params *p, jpgb_coef_layout *layout);

/* Stage A only: colour conversion + decimation + level shift + fDCT + quantization
 * (image_buffer.rs, encoder.rs:1222-1272, fdct.rs, quantization.rs) on device memory.
 * d_coef must hold n * blocks_per_image * 64 int16. Asynchronous on the context's stream. */
int jpgb_stage_a_device(jpgb_encoder *enc, const jpgb_params *p, const void *d_pixels,
                        size_t image_stride, uint32_t n, void *d_coef);

/* Per-stage device time of the last jpgb_encode* call on this context, in milliseconds, measured
 * with CUDA events on the context's stream (enabled with jpgb_encoder_set_timing).
 * stage index: 0 = colour+DCT+quant kernel, 1 = histogram + table build (optimized only),
 * 2 = entropy coding into chunks + prefix sums, 3 = chunk placement (bit-granular copy into the stream),
 * 4 = byte stuffing + scatter, 5 = H2D, 6 = D2H. */
/* Per-stage timing covers the device-resident entry points (jpgb_encode_batch_device, the strip calls, jpgb_encode_planar):
 * with timing enabled they launch kernel by kernel between CUDA events instead of replaying their CUDA graph. The host
 * entry points (jpgb_encode, jpgb_encode_batch*) run several such passes overlapped with copies and report no stages. */
#define JPGB_N_STAGES 7
void jpgb_encoder_set_timing(jpgb_encoder *enc, int enabled);
int jpgb_encoder_last_timing(const jpgb_encoder *enc, float ms[JPGB_N_STAGES]);

/* number of kernel launches issued by the last jpgb_encode* / jpgb_stage_a_device call */
uint32_t jpgb_encoder_last_launch_count(const jpgb_encoder *enc);

/* ---- host-side planner, callable without a GPU (used by the CPU test-suite) ---------------------- */

/* The file header the encoder writes for `p` with the default (Annex K.3) Huffman tables: SOI, APP0,
 * [APP14], user APPn, SOF, DQT x2, DHT x2|4, [DRI], first SOS (src/encoder.rs:536-554, 633-667, 705).
 * Writes up to `cap` bytes to `buf`, the full length to *len. */
int jpgb_build_header(const jpgb_params *p, uint8_t *buf, size_t cap, size_t *len);

/* HuffmanTable::new_optimized (Annex K.2, src/huffman.rs:99-221) as the host planner runs it on the
 * device histogram: code-length counts, values in code order, number of values. */
int jpgb_optimized_huffman_table(const uint32_t freq[257], uint8_t length[16], uint8_t values[256], uint32_t *n_values);

/* The same on the device (csrc/tables.cu: what the optimized encode path runs, one warp per table): `n` histograms of
 * 257 counts each (host memory), every one built as an AC table (ac != 0) or a DC table. Per histogram: 16 length
 * counts, up to 256 values, the number of values, and 256 kernel-format code words (0 where a symbol has no code is
 * reported as its value size << 27). status[i] = JPGB_OK or JPGB_ERR_HUFFMAN. Test and diagnostics entry. */
int jpgb_optimized_huffman_tables_device(jpgb_encoder *enc, const uint32_t *freq /* n * 257 */, uint32_t n, int ac,
                                         uint8_t *lengths /* n * 16 */, uint8_t *values /* n * 256 */, uint32_t *n_values /* n */,
                                         uint32_t *words /* n * 256 */, int *status /* n */);

const char *jpgb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* JPEGENC_B200_H */
