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

/* ---- device images of wider samples: float32, float16, bfloat16 and uint16 (model outputs, raw and medical data) ----
 * Element types of jpgb_sample_format.type, all little-endian. (0 is uint8, which takes jpgb_encode_batch_device_strided.) */
enum { JPGB_SAMPLE_U16 = 1, JPGB_SAMPLE_F16 = 2, JPGB_SAMPLE_BF16 = 3, JPGB_SAMPLE_F32 = 4 };
typedef struct jpgb_sample_format {
    uint32_t type;        /* JPGB_SAMPLE_* */
    float scale, offset;  /* finite */
} jpgb_sample_format;

/* jpgb_encode_batch_device_strided for images whose samples are elements of fmt->type. The layout and the output mean
 * what they mean there; every stride stays in bytes, and sample ch of pixel (x, y) is one element of the type
 * (es = 2 or 4 bytes) at
 *   packed (plane_stride == 0): data + i*image_stride + y*row_stride + (x*bpp + ch)*es
 *   planar (plane_stride > 0):  data + i*image_stride + ch*plane_stride + y*row_stride + x*es
 * Each element x read becomes the 8-bit sample
 *   y = fadd_rn(fmul_rn(float(x), scale), offset)    two separately rounded fp32 operations, never a fused multiply-add
 *   sample = NaN(y) ? 0 : clamp(rint(y), 0, 255)     rint rounds half to even: 0.5 -> 0, 2.5 -> 2, 254.5 -> 254
 * (float(x) is exact for every type), and that sample takes the uint8 colour path unchanged: the files are byte-identical
 * to jpgb_encode_batch_device's for the converted image handed over packed. value_range (lo, hi) maps to
 * scale = float(255 / (hi - lo)), offset = float(-lo * 255 / (hi - lo)), each computed in double and rounded once.
 * Colour types: Luma, Rgb, Bgr, Rgba, Bgra. The alpha element is never converted, and never read when planar.
 * Rejected before anything is enqueued (no launch), in this order, with JPGB_ERR_BAD_PARAMS unless noted:
 *   null arguments (fmt included) or n == 0;
 *   what jpgb_encode_batch_device rejects in `p` (same codes), except the BadImageData length check;
 *   fmt->type 0 (uint8: use jpgb_encode_batch_device_strided) or not a JPGB_SAMPLE_* value;
 *   color_type Ycbcr, Cmyk, CmykAsYcck or Ycck;
 *   a scale or offset that is infinite or NaN;
 *   data, row_stride, plane_stride or image_stride not a multiple of es;
 *   then the layout checks of jpgb_encode_batch_device_strided in their order, counted in elements: a row is
 *   width*bpp*es bytes packed and width*es planar, and the last byte read is
 *     (n-1)*image_stride + (height-1)*row_stride + width*bpp*es - 1                       (packed)
 *     (n-1)*image_stride + c_max*plane_stride + (height-1)*row_stride + width*es - 1      (planar) */
int jpgb_encode_batch_device_samples(jpgb_encoder *enc, const jpgb_params *p, const jpgb_device_images *images,
                                     const jpgb_sample_format *fmt, uint32_t n, const void **d_files, uint64_t *offsets);

/* ---- YCbCr frames with subsampled chroma, as video decoders hand them out (I420, I422, I444, NV12, NV21, NV16) ----
 * A luma plane and two chroma planes, each read where it lies. With cw = ceil(width / c_h) and ch = ceil(height / c_v),
 * pixel (x, y) of image i is
 *   Y  = y [i*y_image_stride + y*y_row_stride + x]
 *   Cb = cb[i*c_image_stride + (y / c_v)*c_row_stride + (x / c_h)*c_sample_stride]
 *   Cr = cr[i*c_image_stride + (y / c_v)*c_row_stride + (x / c_h)*c_sample_stride]
 * that is, the full-resolution image whose chroma repeats every plane sample c_h x c_v times (nearest neighbour). The
 * file is byte-identical to jpgb_encode_batch_device's for that image handed over packed as JPGB_YCBCR. The JPEG
 * sampling factor is p->sampling, whatever the planes' subsampling: I420 at F_1_1 is upsampled, I444 at F_2_2 decimated,
 * both by point sampling as every path of the encoder does.
 * Samples are taken verbatim as full-range (JFIF) YCbCr: limited-range ("video range") samples are not expanded, and
 * BT.709 samples are not converted to the BT.601 matrix of JFIF. */
typedef struct jpgb_device_ycbcr {
    const void *y, *cb, *cr;   /* image 0's first sample of each plane (NV12: cr = cb + 1; NV21: cb = cr + 1) */
    uint64_t y_image_stride, y_row_stride;   /* bytes; an image stride of 0: every image is the same frame */
    uint64_t c_image_stride, c_row_stride;   /* bytes, shared by Cb and Cr */
    uint32_t c_sample_stride;  /* bytes between horizontally adjacent chroma samples: 1 planar, 2 interleaved */
    uint8_t c_h, c_v;          /* luma samples per chroma sample across / down: 1 or 2 (I420 / NV12: 2, 2; I422 / NV16: 2, 1) */
} jpgb_device_ycbcr;

/* Encode n frames laid out as `frames` describes. Output and lifetime as for jpgb_encode_batch_device_strided.
 * Rejected before anything is enqueued (no launch), in this order, with JPGB_ERR_BAD_PARAMS unless noted:
 *   null arguments (frames, y, cb or cr included) or n == 0;
 *   what jpgb_encode_batch_device rejects in `p` (same codes), except the BadImageData length check;
 *   color_type other than Ycbcr;
 *   c_h or c_v not 1 or 2; c_sample_stride not 1 or 2;
 *   y_row_stride < width; c_row_stride < (cw - 1)*c_sample_stride + 1;
 *   an extent beyond 64-bit addresses;
 *   then for y, cb and cr in turn: not device or managed memory usable on the context's device, or a last byte read
 *   outside the allocation that holds it. The last bytes read are
 *     y:      (n-1)*y_image_stride + (height-1)*y_row_stride + width - 1
 *     cb, cr: (n-1)*c_image_stride + (ch-1)*c_row_stride + (cw-1)*c_sample_stride
 * Interleaved chroma is read in whole byte pairs up to the channel's last sample, so the kernels may read the other
 * channel's bytes of a pair, never a byte past the last sample. A channel at an odd address is read from the byte in
 * front of it; that byte lies in the same allocation, because allocations start at aligned addresses. */
int jpgb_encode_batch_device_ycbcr(jpgb_encoder *enc, const jpgb_params *p, const jpgb_device_ycbcr *frames, uint32_t n,
                                   const void **d_files, uint64_t *offsets);

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

/* ---- one large image in strips without restart intervals ------------------------------------------
 * With restart_interval == 0 (Encoder::new's default, src/encoder.rs:239-275) a scan is one bit-contiguous stream: the
 * DC predictor never resets and nothing is byte aligned between the first and the last bit of a scan. Strips of whole
 * MCU rows are still coded on their own GPUs; the file bytes are the same as those of the whole image:
 *  1. every strip: jpgb_contiguous_strip_prepare_device runs stage A (and, with optimized tables, the strip histogram,
 *     as jpgb_strip_histogram_device does) and returns edge_dc[0..3] / edge_dc[4..7], the DC of the first / last block
 *     of each component in the order the scans code them (MCU order when interleaved, the raster of the component's
 *     true grid otherwise; jpgb_coef_layout_for);
 *  2. the caller all-gathers the edge_dc arrays in strip order (n_strips * 8 values); with optimized tables it also
 *     sums the histograms and merges them with jpgb_merge_strip_histograms -> hist_total;
 *  3. every strip: jpgb_encode_contiguous_strip_device codes its part of every scan, the first DC difference of each
 *     component taken against the last block of that component in the strip in front (strip 0: against 0). A piece is a
 *     bare bit string: no header, SOS, pad bits, 0xFF stuffing or EOI. The pieces lie in context memory (*d_bits),
 *     piece k at sum over j < k of its pieces' bytes rounded up to 16; jpgb_last_piece_bits_device gives their bit
 *     lengths (n_scans u64, device memory) for an all-gather into a world x n_scans table in rank order;
 *  4. every strip: jpgb_join_place_bits stores its pieces at their bit positions in a gather target (jpgb_gather_target_
 *     create / _open; rank 0's memory). The target holds a side table of 2 * world * n_scans 16-byte entries (rounded
 *     up to 128 bytes), then the joined stream: per scan its lead (the file header for scan 0, its SOS otherwise) and
 *     the pieces of strips 0..n-1 back to back at bit granularity. A rank stores the 32-bit words wholly inside its
 *     piece; the words it shares with a neighbour go to its own side-table entries. No atomics cross GPUs. Nothing is
 *     written when the stream would not fit in `capacity` bytes;
 *  5. rank 0, after a barrier that orders every rank's placement before it: jpgb_join_finish_device writes the header
 *     (its DHT segments from hist_total when optimized), the SOS leads, pad bits and EOI, ORs in the side table, and
 *     stuffs 0xFF: the file is in context memory, *d_file[0 .. *len).
 * `p` is the whole image's settings throughout (p->height = the whole image's height), and restart_interval must be 0.
 * The strip calls take the strip's pixels (packed rows back to back) at d_pixels. Steps 1 and 3 on the same context,
 * strip and pixel pointer (the pixels untouched in between) run the colour+DCT kernel once. */
int jpgb_plan_contiguous_strips(const jpgb_params *p, uint32_t max_strips, jpgb_strip *strips, uint32_t *n_strips); /* host only;
                               equal-as-possible strips of whole MCU rows, never more than MCU rows; BAD_PARAMS unless restart 0 */
int jpgb_contiguous_strip_prepare_device(jpgb_encoder *enc, const jpgb_params *p, const jpgb_strip *strip, const void *d_pixels,
                                         uint32_t *hist /* JPGB_HIST_WORDS; NULL unless optimize_huffman */, int16_t edge_dc[8]);
int jpgb_encode_contiguous_strip_device(jpgb_encoder *enc, const jpgb_params *p, const jpgb_strip *strip, const void *d_pixels,
                                        const int16_t *edge_dc_table /* n_strips * 8, strip order */,
                                        const uint32_t *hist_total /* NULL unless optimize_huffman */, const void **d_bits);
int jpgb_last_piece_bits_device(jpgb_encoder *enc, const uint64_t **d_bits_table, uint32_t *n_scans);
int jpgb_join_place_bits(jpgb_encoder *enc, void *d_target, size_t capacity, const uint64_t *d_bit_table /* world * n_scans */, uint32_t world,
                         uint32_t rank);
int jpgb_join_finish_device(jpgb_encoder *enc, const jpgb_params *p, void *d_target, size_t capacity, const uint64_t *d_bit_table, uint32_t world,
                            const uint32_t *hist_total /* NULL unless optimize_huffman */, const void **d_file, uint64_t *len);

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
