// Launchers of the CUDA kernels (sm_100a). All work is queued on `stream`; nothing here syncs.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <mutex>

#include "../../include/jpegenc_b200.h"
#include "device_types.h"

namespace jpgb {

// CTAs of a persistent `Kernel` that fit on the current device at once (SMs x resident CTAs per SM) at `threads`
// threads and `smem` bytes of dynamic shared memory, after opting the kernel in to that much shared memory. Each
// kernel launches with one block size and one shared-memory size, so the answer is computed once per device.
// Contexts on several host threads (and devices) launch concurrently: the table is guarded.
template <auto Kernel>
cudaError_t resident_ctas(int threads, size_t smem, unsigned long long &ctas) {
    constexpr int kMaxDevices = 64;
    static std::mutex mu;
    static struct {
        int dev = -1;
        unsigned long long ctas = 0;
    } cache[kMaxDevices];
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    auto &c = cache[dev < kMaxDevices ? dev : kMaxDevices - 1];
    if (c.dev != dev) {
        cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        int n_sms = 0, per_sm = 0;
        cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev);
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, Kernel, threads, smem);
        if (e != cudaSuccess) return e;
        c.ctas = (unsigned long long)n_sms * (per_sm < 1 ? 1 : per_sm);
        c.dev = dev;
    }
    ctas = c.ctas;
    return cudaSuccess;
}

// stage_a.cu -- colour + decimate + level shift + fDCT + quantize -> zig-zag i16 coefficients
cudaError_t launch_stage_a(const StageAParams &p, uint32_t n_images, cudaStream_t stream);

// Huffman code tables as the kernels see them: [image][table 0|1][class dc|ac][256] of (size<<16)|code
constexpr size_t kHuffWordsPerImage = 2 * 2 * 256;

// Buffers of one encode call (all device pointers). Sizes are in the comments; `n` = images. The plan itself
// (DevPlan, ~14 KB) travels to the kernels as a __grid_constant__ parameter: every field is a constant-bank operand.
struct EntropyBuffers {
    const int16_t *coef;           // n * blocks_per_image * 64
    const uint32_t *huff;          // n_huff * kHuffWordsPerImage; n_huff is 1 (shared) or n (optimized)
    int huff_per_image;            // 0: all images share tables[0]; 1: one set per image
    // coding: one chunk = the code bits of <= chunk_T consecutive visits of one restart segment of one scan
    uint32_t *scratch;             // per coding CTA: chunk_T visits x kSlotWords words (lives in L2)
    uint32_t *pool;                // chunk bit strings, MSB-first 32-bit words, each chunk 16-byte aligned, in completion order
    unsigned long long pool_cap;   // capacity of `pool` in 16-byte units
    uint32_t *chunk_bits;          // n * chunks_per_image: code bits of the chunk
    uint32_t *chunk_pool;          // n * chunks_per_image: where the chunk lies in `pool`, in 16-byte units
    unsigned long long *chunk_bitpos; // n * chunks_per_image + 1 (exclusive scan of chunk_bits)
    uint32_t *seglen;              // n * segs_per_image          (lead + data + tail bytes of a segment)
    unsigned long long *segpos;    // n * segs_per_image + 1      (exclusive scan of seglen)
    const uint32_t *hdr_len;       // n_huff entries: bytes of file header (SOI .. first SOS)
    const uint8_t *hdr;            // n_huff * hdr_stride bytes
    uint32_t hdr_stride;
    uint8_t *ustream;              // unstuffed stream incl. headers/markers, zero-initialised
    uint32_t *raw_mask;            // 1 bit per ustream byte: header/marker byte, exempt from stuffing
    uint32_t *ffcount;             // per chunk of kStuffChunk bytes
    unsigned long long *ffpos;     // exclusive scan of ffcount (+1)
    uint8_t *out;                  // final files back to back
    unsigned long long *file_off;  // n + 1 offsets into `out`
    void *scan_tmp;                // scratch for the scans
    // capacities (bytes) of ustream / out and the status block the kernels report into: the host sizes the
    // buffers from the previous call and checks `status` once at the end instead of syncing mid-pipeline
    unsigned long long ustream_cap, out_cap, n_segs_total;
    unsigned long long *status;    // kStatusWords entropy status words (kStat* below)
    size_t scan_tmp_bytes;
};

// The status block of one encode call, one device buffer: [n + 1 file offsets][kStatusWords entropy status words]
// [kStatusWords table-build status words][raw mask]. The first three parts are read back with one copy.
constexpr int kStatusWords = 8;
// Words of a status part: unstuffed bytes, 0xFF bytes of the coded data, flags, look-back scan error, work-item ticket
// of the coding kernel, pool cursor (16-byte units; it counts every request, also beyond the capacity).
constexpr int kStatUnstuffed = 0, kStatDataFF = 1, kStatFlags = 2, kStatScanError = 3, kStatTicket = 4, kStatPoolCursor = 5;
// Flag bits: overflow of the unstuffed stream, the output, the chunk pool; a scan segment over 4 GiB; an optimized
// Huffman code that does not fit (longer than 32 bits, or code plus value bits beyond 31; table-build part)
constexpr unsigned long long kFlagStream = 1, kFlagOut = 2, kFlagPool = 4, kFlagSegment4G = 8, kFlagHuffmanLong = 16;

struct StatusBlock {
    uint32_t n;        // images
    size_t mask_bytes; // raw mask: one bit per byte of the unstuffed stream
    size_t readback_bytes() const { return (size_t)(n + 1 + 2 * kStatusWords) * 8; }
    size_t bytes() const { return readback_bytes() + mask_bytes; }
    // the parts inside a block (device) or its read-back copy (host) at `base`
    unsigned long long *file_off(void *base) const { return static_cast<unsigned long long *>(base); }
    unsigned long long *status(void *base) const { return file_off(base) + n + 1; }
    unsigned long long *table_status(void *base) const { return status(base) + kStatusWords; }
    uint32_t *raw_mask(void *base) const { return reinterpret_cast<uint32_t *>(table_status(base) + kStatusWords); }
};
inline StatusBlock status_block(uint32_t n, unsigned long long ustream_cap) { return {n, (size_t)(ustream_cap / 32 + 2) * 4}; }

// A visit codes at most 1 + 63 symbols of <= 16 code + 11 value bits = 1728 bits = 54 words.
constexpr int kSlotWords = 56;
constexpr int kStuffChunk = 4096; // bytes of unstuffed stream per CTA in the stuffing kernels

// entropy.cu
cudaError_t launch_histogram(const DevPlan &hplan, const int16_t *coef, uint32_t n_images,
                             uint32_t *hist /* n * 2 tables * 2 classes * 257 */, cudaStream_t stream);
// persistent coding kernel: grid = what coder_grid() returns for this plan; `b.scratch` holds coder_scratch_bytes()
struct CoderLaunch {
    unsigned grid;
    size_t smem, scratch_bytes;
};
cudaError_t coder_launch_config(const DevPlan &hplan, uint32_t n_images, CoderLaunch &cfg);
cudaError_t launch_encode_chunks(const EntropyBuffers &b, const DevPlan &hplan, uint32_t n_images, const CoderLaunch &cfg, cudaStream_t stream);
cudaError_t launch_segment_lengths(const EntropyBuffers &b, const DevPlan &hplan, uint32_t n_images, cudaStream_t stream);
// small jobs: chunk positions (scan_chunks), segment lengths and segment positions in one single-CTA launch
cudaError_t launch_positions(const EntropyBuffers &b, const DevPlan &hplan, uint32_t n_images, bool scan_chunks, cudaStream_t stream);
cudaError_t launch_segment_leads(const EntropyBuffers &b, const DevPlan &hplan, uint32_t n_images, cudaStream_t stream);
cudaError_t launch_place_chunks(const EntropyBuffers &b, const DevPlan &hplan, uint32_t n_images, cudaStream_t stream);
cudaError_t launch_count_ff(const EntropyBuffers &b, cudaStream_t stream);   // grids sized by b.ustream_cap
// short streams: the scatter launch adds up the per-piece 0xFF counts itself and the prefix-sum launch is skipped
bool ff_scan_needed(const EntropyBuffers &b);
// pieces -> out, plus the file offsets (b.file_off) and, with piece_offs, the offset of every scan's first segment
cudaError_t launch_stuff_scatter(const EntropyBuffers &b, const DevPlan &hplan, uint32_t n_images, unsigned long long *piece_offs, cudaStream_t stream);

// tables.cu -- optimized Huffman tables (Annex K.2), kernel-format code words and the file header with its DHT
// segments, one CTA per image. hist: [image][table][dc|ac][257] (hist_per_image = 0: one histogram for all).
cudaError_t launch_build_tables(const uint32_t *hist, int hist_per_image, int n_tables, uint32_t n_images, uint32_t *huff, const uint8_t *head,
                                uint32_t head_len, const uint8_t *tail, uint32_t tail_len, uint8_t *hdr, uint32_t hdr_stride, uint32_t *hdr_len,
                                unsigned long long *status, cudaStream_t stream);

// one table per histogram, all of class `ac`: DHT segment bytes (5 + 16 + values, 277 apart), kernel words, error flags
cudaError_t launch_build_single_tables(const uint32_t *hist, uint32_t n, int ac, uint32_t *words, uint8_t *dht, uint32_t *dht_len, uint32_t *bad,
                                       cudaStream_t stream);

// gather.cu -- a rank's pieces stored at their place in the assembled file (possibly in a peer GPU's memory)
cudaError_t launch_place_pieces(const uint8_t *src, uint8_t *dst, unsigned long long dst_cap, const unsigned long long *table, unsigned world,
                                unsigned rank, unsigned n_scans, unsigned long long *total_out, cudaStream_t stream);

// scan.cu -- device-wide exclusive prefix sum of u32 into u64; out has n + 1 entries (out[n] = total)
size_t scan_tmp_bytes(uint64_t n);
cudaError_t launch_exclusive_scan(const uint32_t *in, unsigned long long *out, uint64_t n, void *tmp, cudaStream_t stream,
                                  uint32_t *launches, unsigned long long *err_flag = nullptr);

} // namespace jpgb
