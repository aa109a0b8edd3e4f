// C ABI (include/jpegenc_b200.h) and the per-call orchestration of the device pipeline.
// The product path has no CPU fallback: without a usable sm_100 device every entry point
// returns JPGB_ERR_CUDA.
#include <cuda.h>
#include <cuda_runtime.h>

#include <climits>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <string>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/jpegenc_b200.h"
#include "copy_pool.h"
#include "host.h"
#include "kernels.h"

using namespace jpgb;

namespace {

// test hook (JPGB_POISON_ALLOC=1): every buffer a context allocates starts out as all ones, so a read of memory that no
// call has written shows the same way every time instead of depending on what the allocator hands back. Read only when
// a buffer is (re)allocated: steady-state calls never get here.
bool poison_alloc() {
    const char *e = std::getenv("JPGB_POISON_ALLOC");
    return e && e[0] == '1';
}

// A device (cudaMalloc) or pinned host (cudaMallocHost) buffer, freed with its owner
template <bool kPinned>
struct Buf {
    void *p = nullptr;
    size_t cap = 0;
    Buf() = default;
    Buf(Buf &&o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    Buf &operator=(Buf o) noexcept { // the old buffer leaves with `o`
        std::swap(p, o.p);
        std::swap(cap, o.cap);
        return *this;
    }
    ~Buf() { if (p) kPinned ? cudaFreeHost(p) : cudaFree(p); }
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        *this = Buf();
        size_t want = bytes + bytes / 8 + 256; // grow-only with slack: steady-state calls never allocate
        if (!kPinned) want = (want + 255) & ~(size_t)255;
        cudaError_t e = kPinned ? cudaMallocHost(&p, want) : cudaMalloc(&p, want);
        if (e != cudaSuccess) return p = nullptr, e;
        cap = want;
        if (poison_alloc()) { // device memory is filled before the caller can enqueue work on another stream
            if (kPinned) std::memset(p, 0xFF, want);
            else if ((e = cudaMemset(p, 0xFF, want)) == cudaSuccess) e = cudaDeviceSynchronize();
        }
        return e;
    }
    template <typename T>
    T *as() const { return static_cast<T *>(p); }
};
using DevBuf = Buf<false>;
using PinnedBuf = Buf<true>;

// What the device plan is a function of: the caller's settings without the APPn payloads (they only change header
// bytes, which are uploaded, not baked into launches), the strip and the input kind.
struct PlanSig {
    jpgb_params p;
    jpgb_strip strip;
    uint32_t is_strip, planar;
};
inline PlanSig plan_sig(const Plan &plan) {
    PlanSig s;
    std::memset(&s, 0, sizeof(s)); // field by field: the caller's padding bytes must not take part in comparisons
    s.p.width = plan.p.width;
    s.p.height = plan.p.height;
    s.p.color_type = plan.p.color_type;
    s.p.quality = plan.p.quality;
    s.p.sampling = plan.p.sampling & 0x7F;
    for (int t = 0; t < 2; ++t) {
        s.p.qtable_kind[t] = plan.p.qtable_kind[t];
        if (plan.p.qtable_kind[t] == JPGB_QT_CUSTOM) std::memcpy(s.p.qtable_custom[t], plan.p.qtable_custom[t], sizeof(s.p.qtable_custom[t]));
    }
    s.p.progressive_scans = plan.p.progressive_scans;
    s.p.optimize_huffman = plan.p.optimize_huffman;
    s.p.restart_interval = plan.p.restart_interval;
    if (plan.is_strip) {
        s.strip.strip_index = plan.strip.strip_index;
        s.strip.n_strips = plan.strip.n_strips;
        s.strip.first_row = plan.strip.first_row;
        s.strip.rows = plan.strip.rows;
        s.strip.full_height = plan.strip.full_height;
    }
    s.is_strip = plan.is_strip;
    s.planar = plan.planar;
    return s;
}
struct CapKey {
    PlanSig sig;
    uint64_t raw_bytes;
    uint32_t n, pad;
};

// Capacities of one attempt: unstuffed stream and output in bytes, chunk pool in 16-byte units
struct Caps { uint64_t ustream, out, pool_units; };

// What a captured launch sequence bakes in (graph_key), word by word: no padding of the caller's structs takes part
struct GraphKey {
    PlanSig sig;
    uint64_t words[39];
};

// Replay of the launch sequence behind stage A as a CUDA graph (same settings, batch size and buffers)
struct GraphCache {
    struct Slot {
        cudaGraphExec_t exec = nullptr;
        GraphKey key{};
        uint32_t launches = 0;
        uint64_t used = 0;
    } slots[4]; // the pipelined host path alternates between two pixel / output buffers and ends on a shorter chunk
    uint64_t clock = 0;
    bool ok = true; // false once a capture failed (e.g. on the legacy default stream): launches go direct from then on
    ~GraphCache() {
        for (Slot &s : slots)
            if (s.exec) cudaGraphExecDestroy(s.exec);
    }
    // Launches the graph of `key`, first capturing it from `enqueue` (which counts its launches in `launches`) when no
    // slot holds it; the least recently used slot makes room. `replayed` stays false when capture failed: the caller
    // then enqueues directly.
    template <typename Enqueue>
    cudaError_t replay(const GraphKey &key, cudaStream_t st, uint32_t &launches, Enqueue &&enqueue, bool &replayed) {
        Slot *slot = nullptr, *victim = &slots[0];
        for (Slot &g : slots) {
            if (g.exec && std::memcmp(&g.key, &key, sizeof(key)) == 0) slot = &g;
            if (!g.exec || (victim->exec && g.used < victim->used)) victim = &g;
        }
        if (!slot) {
            if (victim->exec) cudaGraphExecDestroy(victim->exec), victim->exec = nullptr;
            const uint32_t launches_before = launches;
            cudaGraph_t graph = nullptr;
            const bool capturing = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
            const int rc = capturing ? enqueue() : JPGB_ERR_CUDA;
            if (capturing && cudaStreamEndCapture(st, &graph) == cudaSuccess && rc == JPGB_OK && graph &&
                cudaGraphInstantiate(&victim->exec, graph, 0) == cudaSuccess) {
                victim->key = key;
                victim->launches = launches - launches_before;
                slot = victim;
            } else {
                victim->exec = nullptr;
                ok = false;
            }
            if (graph) cudaGraphDestroy(graph);
            launches = launches_before;
            cudaGetLastError();
        }
        if (!slot) return cudaSuccess;
        slot->used = ++clock;
        const cudaError_t e = cudaGraphLaunch(slot->exec, st);
        if (e == cudaSuccess) launches += slot->launches, replayed = true;
        return e;
    }
};

} // namespace

struct jpgb_encoder {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    DevBuf pixels, coef, huff, hdr, hdr_len, scratch, pool, chunk_bits, chunk_pool, chunk_bitpos, seglen, segpos, ustream, ffcount, ffpos,
        out, scan_tmp, hist, piece_off, out2, pixels2, status, hdr_parts;
    std::vector<uint8_t> last_tables; // what the device currently holds
    double ucap_ratio = 0; // unstuffed-stream bytes to provision per raw pixel byte, learnt from earlier calls
    double pool_ratio = 0; // the same for the chunk pool (code bytes incl. per-chunk alignment)
    PinnedBuf h_small, h_hist, h_tables, h_pieces, h_out, h_stage[2];
    cudaEvent_t ev_stage[2] = {};
    bool stage_busy[2] = {};
    CopyPool copy_pool;
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    std::vector<cudaEvent_t> ev_slice;
    cudaEvent_t ev_in[2] = {}, ev_out[2] = {}, ev_enc[2] = {};
    cudaEvent_t ev_wait = nullptr; // jpgb_encoder_wait_stream
    bool timing = false;
    cudaEvent_t ev[JPGB_N_STAGES + 1][2] = {};
    bool ev_used[JPGB_N_STAGES] = {};
    float last_ms[JPGB_N_STAGES] = {};
    bool have_timing = false;
    uint32_t launches = 0;
    uint32_t last_piece_scans = 0; // scans of the last strip encode (its piece offsets are in piece_off)
    // whose coefficients `coef` holds (set by jpgb_strip_histogram_device, cleared by every other call that writes `coef`):
    // the optimized strip encode that follows on the same strip and pixels does not run the colour+DCT kernel again
    bool coef_tagged = false;
    PlanSig coef_sig{};
    const void *coef_pixels = nullptr;
    uint64_t coef_stride = 0;
    float coef_ms[2] = {0.f, 0.f}; // with timing on: what the colour+DCT kernel and the histogram of that call took (added to the reusing call's stages)
    GraphCache graphs;
    // Capacities are sticky per (settings, batch size): steady-state calls provision exactly what the last successful
    // call settled on, so the launch sequence has identical parameters call after call and is replayed as a CUDA graph.
    bool have_caps = false;
    CapKey cap_key{};
    Caps caps{};
};

namespace {

int fail(jpgb_encoder *e, int code, const std::string &msg) {
    if (e) e->err = msg;
    return code;
}
int fail_cuda(jpgb_encoder *e, cudaError_t ce, const char *what) {
    return fail(e, JPGB_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(ce));
}
#define CK(call, what)                                        \
    do {                                                      \
        cudaError_t ce__ = (call);                            \
        if (ce__ != cudaSuccess) return fail_cuda(enc, ce__, what); \
    } while (0)

struct StageTimer {
    jpgb_encoder *enc;
    int stage;
    StageTimer(jpgb_encoder *e, int s) : enc(e), stage(s) {
        if (enc->timing) {
            if (!enc->ev_used[stage]) cudaEventRecord(enc->ev[stage][0], enc->stream);
        }
    }
    ~StageTimer() {
        if (enc->timing) {
            cudaEventRecord(enc->ev[stage][1], enc->stream);
            enc->ev_used[stage] = true;
        }
    }
};

void timing_begin(jpgb_encoder *enc) {
    for (int i = 0; i < JPGB_N_STAGES; ++i) enc->ev_used[i] = false;
    enc->have_timing = false;
    enc->launches = 0;
}
void timing_end(jpgb_encoder *enc) {
    if (!enc->timing) return;
    cudaStreamSynchronize(enc->stream);
    for (int i = 0; i < JPGB_N_STAGES; ++i) {
        enc->last_ms[i] = 0.f;
        if (enc->ev_used[i]) cudaEventElapsedTime(&enc->last_ms[i], enc->ev[i][0], enc->ev[i][1]);
    }
    enc->have_timing = true;
}

int validate_and_plan(jpgb_encoder *enc, const jpgb_params *p, size_t len_each, Plan &plan) {
    if (!p) return fail(enc, JPGB_ERR_BAD_PARAMS, "null params");
    if (p->color_type > JPGB_YCCK) return fail(enc, JPGB_ERR_BAD_PARAMS, "bad color_type");
    const size_t required = (size_t)p->width * p->height * (size_t)bytes_per_pixel(p->color_type);
    if (len_each < required) { // BadImageData comes first, encoder.rs:447-454
        char m[128];
        snprintf(m, sizeof(m), "Image data too small for dimensions and color_type: %zu need at least %zu", len_each, required);
        return fail(enc, JPGB_ERR_BAD_IMAGE_DATA, m);
    }
    const int rc = plan.build(*p);
    if (rc != JPGB_OK) return fail(enc, rc, rc == JPGB_ERR_ZERO_DIMENSIONS ? "Image dimensions must be non zero" : "invalid parameters");
    return JPGB_OK;
}

typedef CUresult (*MemGetAddressRangeFn)(CUdeviceptr *, size_t *, CUdeviceptr);
MemGetAddressRangeFn mem_get_address_range_fn() {
    static MemGetAddressRangeFn fn = [] {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) f = nullptr;
        return reinterpret_cast<MemGetAddressRangeFn>(f);
    }();
    return fn;
}

// The checks of jpgb_encode_batch_device_strided on the layout, in the order the header lists them. Nothing is enqueued
// before they pass, so no kernel reads a byte outside the allocation that holds `data`.
int check_device_images(jpgb_encoder *enc, const Plan &plan, const jpgb_device_images &im, uint32_t n) {
    const uint64_t w = plan.p.width, h = plan.p.height;
    const bool planes = im.plane_stride != 0;
    const uint64_t row_bytes = planes ? w : w * (uint64_t)plan.bpp; // bytes of a row read (of one plane)
    char m[192];
    if (im.row_stride < row_bytes) {
        snprintf(m, sizeof(m), "row_stride %llu is shorter than a row (%llu bytes)", (unsigned long long)im.row_stride, (unsigned long long)row_bytes);
        return fail(enc, JPGB_ERR_BAD_PARAMS, m);
    }
    if (planes && im.plane_stride < w) {
        snprintf(m, sizeof(m), "plane_stride %llu is shorter than a row (%llu bytes)", (unsigned long long)im.plane_stride, (unsigned long long)w);
        return fail(enc, JPGB_ERR_BAD_PARAMS, m);
    }
    // the last byte read: (n-1)*image_stride + c_max*plane_stride + (h-1)*row_stride + row_bytes - 1 (alpha is not read)
    const uint8_t ct = plan.p.color_type;
    const uint64_t c_max = !planes ? 0 : (ct == JPGB_LUMA ? 0 : (plan.bpp == 3 || ct == JPGB_RGBA || ct == JPGB_BGRA) ? 2 : 3);
    uint64_t last = 0, t = 0;
    bool over = __builtin_mul_overflow((uint64_t)(n - 1), im.image_stride, &last);
    over |= __builtin_mul_overflow(c_max, im.plane_stride, &t) || __builtin_add_overflow(last, t, &last);
    over |= __builtin_mul_overflow(h - 1, im.row_stride, &t) || __builtin_add_overflow(last, t, &last);
    over |= __builtin_add_overflow(last, row_bytes - 1, &last);
    over |= __builtin_add_overflow((uint64_t)(uintptr_t)im.data, last, &t);
    if (over) return fail(enc, JPGB_ERR_BAD_PARAMS, "the described pixels extend beyond 64-bit addresses");
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    cudaPointerAttributes attr{};
    const bool known = cudaPointerGetAttributes(&attr, im.data) == cudaSuccess;
    cudaGetLastError();
    if (!known || !(attr.type == cudaMemoryTypeManaged || (attr.type == cudaMemoryTypeDevice && attr.device == enc->device)))
        return fail(enc, JPGB_ERR_BAD_PARAMS, "data is not device or managed memory of the context's device");
    MemGetAddressRangeFn range = mem_get_address_range_fn();
    CUdeviceptr base = 0;
    size_t size = 0;
    if (!range || range(&base, &size, (CUdeviceptr)(uintptr_t)im.data) != CUDA_SUCCESS)
        return fail(enc, JPGB_ERR_BAD_PARAMS, "no allocation is found at data");
    const uint64_t end = (uint64_t)(uintptr_t)im.data + last; // the last byte read
    if (end >= (uint64_t)base + size) {
        snprintf(m, sizeof(m), "the described pixels end %llu bytes past the end of the allocation that holds data",
                 (unsigned long long)(end + 1 - ((uint64_t)base + size)));
        return fail(enc, JPGB_ERR_BAD_PARAMS, m);
    }
    return JPGB_OK;
}

// Where the launches find the file headers in enc->hdr
struct HeaderLayout {
    size_t hdr_stride = 0;               // bytes between the headers of two images
    uint32_t head_len = 0, tail_len = 0; // optimized tables: header bytes in front of / behind the DHT segments
    int n_tables = 0;                    // optimized tables: tables per class and image (1 or 2)
};

// Huffman tables and the file header (SOI/APPn prefix, SOF/DQT/DHT/DRI, first SOS -- Q21).
// Default tables (Annex K.3): built on the host once per settings, shared by all images.
// Optimized tables: per image on the device, from its symbol histogram (tables.cu) -- no host round trip. Here only
// the header parts around the DHT segments, and for strips the whole image's histogram `given_hist`.
int setup_header(jpgb_encoder *enc, const Plan &plan, uint32_t n, const uint32_t *given_hist, HeaderLayout &hl) {
    cudaStream_t st = enc->stream;
    const bool optimized = plan.p.optimize_huffman != 0;
    const uint32_t n_huff = optimized ? n : 1;
    const size_t tab_bytes = kHuffWordsPerImage * 4;
    CK(enc->huff.reserve((size_t)n_huff * tab_bytes), "alloc huffman tables");
    CK(enc->hdr_len.reserve((size_t)n_huff * 4), "alloc header lengths");
    std::vector<uint8_t> fresh; // what the device is to hold
    if (!optimized) { // [kernel words of the four tables][header, padded to hdr_stride][header length]
        HuffTable tables[4];
        default_huffman_tables(reinterpret_cast<HuffTable(*)[2]>(tables));
        std::vector<uint8_t> h = plan.prefix;
        plan.frame_header(reinterpret_cast<const HuffTable(*)[2]>(tables), h);
        h.insert(h.end(), plan.scans[0].sos.begin(), plan.scans[0].sos.end());
        hl.hdr_stride = (h.size() + 15) & ~(size_t)15;
        fresh.assign(tab_bytes + hl.hdr_stride + 4, 0);
        CK(enc->h_tables.reserve(fresh.size()), "alloc tables (host)");
        for (int t = 0; t < 4; ++t) // [table][dc, ac]
            if (!tables[t].device_words(t & 1, reinterpret_cast<uint32_t *>(fresh.data() + (size_t)t * 1024)))
                return fail(enc, JPGB_ERR_HUFFMAN, "a Huffman code plus its value bits exceeds 31 bits");
        std::memcpy(fresh.data() + tab_bytes, h.data(), h.size());
        const uint32_t len = (uint32_t)h.size();
        std::memcpy(fresh.data() + tab_bytes + hl.hdr_stride, &len, 4);
    } else { // [head][tail][0xA5]: head = everything in front of the DHT segments, tail = what follows them (writer.rs:390-422, encoder.rs:633-667)
        std::vector<uint8_t> with;
        {
            HuffTable empty[2][2];
            const uint8_t none[16] = {0};
            for (auto &row : empty)
                for (HuffTable &e : row) e.set(none, nullptr, 0);
            with = plan.prefix;
            plan.frame_header(empty, with); // DHT segments with no values: 21 bytes each
        }
        hl.n_tables = plan.ncomp >= 3 ? 2 : 1; // encoder.rs:648-660, 1089
        size_t dht_at = plan.prefix.size(); // first DHT marker: behind SOF and the two DQT
        while (dht_at + 3 < with.size() && !(with[dht_at] == 0xFF && with[dht_at + 1] == 0xC4))
            dht_at += 2 + ((size_t)with[dht_at + 2] << 8 | with[dht_at + 3]);
        fresh.assign(with.begin(), with.begin() + dht_at);
        fresh.insert(fresh.end(), with.begin() + dht_at + (size_t)hl.n_tables * 2 * 21, with.end());
        fresh.insert(fresh.end(), plan.scans[0].sos.begin(), plan.scans[0].sos.end());
        hl.head_len = (uint32_t)dht_at;
        hl.tail_len = (uint32_t)(fresh.size() - dht_at);
        hl.hdr_stride = (fresh.size() + (size_t)hl.n_tables * 2 * (21 + 256) + 15) & ~(size_t)15;
        CK(enc->h_tables.reserve(fresh.size() + 16), "alloc header parts (host)");
        CK(enc->hdr_parts.reserve(fresh.size() + 16), "alloc header parts");
        fresh.push_back(0xA5); // never equal to the blob of the default-table path
        const size_t hist_words = (size_t)n * 2 * 2 * 257;
        CK(enc->hist.reserve(hist_words * 4), "alloc histogram");
        if (given_hist) { // strips: the whole image's histogram comes from the caller (n == 1)
            CK(enc->h_hist.reserve(hist_words * 4), "alloc histogram (host)");
            CK(cudaStreamSynchronize(st), "staging reuse sync");
            std::memcpy(enc->h_hist.p, given_hist, hist_words * 4);
            CK(cudaMemcpyAsync(enc->hist.p, enc->h_hist.p, hist_words * 4, cudaMemcpyHostToDevice, st), "upload histogram");
        }
    }
    CK(enc->hdr.reserve((size_t)n_huff * hl.hdr_stride), "alloc headers");
    if (enc->last_tables != fresh) { // repeated calls with the same settings skip the upload (the device copy is still valid)
        CK(cudaStreamSynchronize(st), "staging reuse sync"); // an earlier upload may still read h_tables
        enc->last_tables = fresh;
        const uint8_t *hb = enc->h_tables.as<uint8_t>();
        std::memcpy(enc->h_tables.p, fresh.data(), fresh.size());
        if (!optimized) {
            CK(cudaMemcpyAsync(enc->huff.p, hb, tab_bytes, cudaMemcpyHostToDevice, st), "upload huffman tables");
            CK(cudaMemcpyAsync(enc->hdr.p, hb + tab_bytes, hl.hdr_stride, cudaMemcpyHostToDevice, st), "upload headers");
            CK(cudaMemcpyAsync(enc->hdr_len.p, hb + tab_bytes + hl.hdr_stride, 4, cudaMemcpyHostToDevice, st), "upload header lengths");
        } else {
            CK(cudaMemcpyAsync(enc->hdr_parts.p, hb, hl.head_len + hl.tail_len, cudaMemcpyHostToDevice, st), "upload header parts");
        }
    }
    return JPGB_OK;
}

// ---- Capacities. No host round trip inside the pipeline: the pool, the unstuffed stream and the output are sized
// from what this context has seen before; the kernels read the real sizes on the device and raise a flag instead of
// overrunning, and the part of the pipeline that did not fit is repeated with room to spare.

// Attempt 0: what the last call with the same settings and batch size settled on, else the bytes per raw byte learnt
// from earlier calls (first call: a third of the raw size)
Caps first_caps(const jpgb_encoder *enc, const CapKey &ck, uint64_t n_chunks) {
    const uint64_t raw_bytes = ck.raw_bytes;
    Caps c;
    c.ustream = (enc->ucap_ratio > 0 ? (uint64_t)(raw_bytes * enc->ucap_ratio) : raw_bytes / 3) + (uint64_t)ck.n * 4096 + 65536;
    c.out = c.ustream + c.ustream / 32 + 4096;
    // every chunk is rounded up to 16 bytes in the pool
    c.pool_units = (enc->pool_ratio > 0 ? (uint64_t)(raw_bytes * enc->pool_ratio) : raw_bytes / 3) / 16 + n_chunks + 4096;
    if (enc->have_caps && std::memcmp(&enc->cap_key, &ck, sizeof(ck)) == 0) c = enc->caps;
    // test hook (JPGB_TIGHT_CAPS, a comma list of pool, stream, out): attempt 0 starts from the floor of each named
    // capacity, so the retry branch that capacity leads to (recode, tail with a larger stream, tail with a larger output)
    // runs on purpose
    if (const char *tight = std::getenv("JPGB_TIGHT_CAPS")) {
        const std::string t = std::string(",") + tight + ",";
        if (t.find(",pool,") != std::string::npos) c.pool_units = 1;
        if (t.find(",stream,") != std::string::npos) c.ustream = kStuffChunk;
        if (t.find(",out,") != std::string::npos) c.out = 4096;
    }
    return c;
}

// After an overflow, from the read-back entropy status of the attempt: room to spare for what did not fit.
// What survives a tail-only attempt is the device buffers the coder wrote (pool, chunk and segment positions), not
// the status block: it grows with the raw mask, so a larger stream reallocates it. Hence the pool cursor `pool_used`
// is read only from an attempt that ran the coder, and the table flag only from the attempt that built the tables.
void grow_caps(Caps &c, const unsigned long long *status, uint64_t pool_used) {
    const uint64_t ubytes = status[kStatUnstuffed];
    // the pool: code again (the cursor counted every request, so the exact need is known)
    if (status[kStatFlags] & kFlagPool) c.pool_units = pool_used + pool_used / 64 + 4096;
    if (status[kStatFlags] & kFlagStream) {
        c.ustream = ubytes + ubytes / 16 + 65536;
        c.out = c.ustream + c.ustream / 8 + 4096; // the 0xFF count is not known yet: generous
    } else if (status[kStatFlags] & kFlagOut) {
        c.out = ubytes + status[kStatDataFF] + 4096;
    }
}

// Next call with these settings: what this one needed plus 15 %, unless the present capacities are already within
// 5 .. 40 % of the need (then they stay, and with them the captured graph)
void settle_caps(jpgb_encoder *enc, const CapKey &ck, const Caps &c, uint64_t ubytes, uint64_t total, uint64_t pool_used, uint64_t n_chunks) {
    auto settle = [](uint64_t cap, uint64_t need, uint64_t slack) {
        const uint64_t lo = need + need / 20 + slack / 2, hi = need + need * 2 / 5 + 2 * slack;
        return (cap >= lo && cap <= hi) ? cap : need + need * 3 / 20 + slack;
    };
    enc->cap_key = ck;
    enc->caps.ustream = settle(c.ustream, ubytes, (uint64_t)ck.n * 4096 + 65536);
    enc->caps.out = std::max(settle(c.out, total, 4096), enc->caps.ustream + enc->caps.ustream / 64);
    enc->caps.pool_units = settle(c.pool_units, pool_used, 4096);
    enc->have_caps = true;
    const double raw = (double)std::max<uint64_t>(ck.raw_bytes, 1);
    enc->pool_ratio = std::max(enc->pool_ratio * 0.98, 1.1 * (double)((pool_used > n_chunks ? pool_used - n_chunks : 0) * 16) / raw);
    enc->ucap_ratio = std::max(enc->ucap_ratio * 0.98, 1.15 * (double)ubytes / raw);
}

// What one attempt's launch sequence runs: the optimized tables (first attempt only; with given_hist from the caller's
// histogram), the coder (else only the tail is repeated), the JPGB_POISON_STREAM hook, the read-back of strip pieces
struct SequenceFlags { bool tables, given_hist, coder, poison, pieces; };

// Everything behind stage A, for one attempt: tables, coding and positions, placement, stuffing, and the copy of the
// file offsets and status words to enc->h_small. Every launch counts itself in enc->launches.
int enqueue_sequence(jpgb_encoder *enc, const Plan &plan, const DevPlan &hp, const EntropyBuffers &b, uint32_t n, const CoderLaunch &coder,
                     const HeaderLayout &hl, const SequenceFlags &f) {
    cudaStream_t st = enc->stream;
    const uint64_t n_chunks = (uint64_t)plan.chunks_per_image * n, n_segs = b.n_segs_total, n_pieces = b.ustream_cap / kStuffChunk;
    const StatusBlock sb = status_block(n, b.ustream_cap);
    unsigned long long *scan_err = b.status + kStatScanError;
    // status words of the coder and of the table build (only the words the tail writes when only the tail is repeated)
    if (f.coder) {
        CK(cudaMemsetAsync(b.status, 0, 2 * kStatusWords * 8 + sb.mask_bytes, st), "clear status and raw mask");
    } else { // the pool cursor and the table status are not read again (grow_caps)
        CK(cudaMemsetAsync(b.status, 0, (kStatScanError + 1) * 8, st), "clear status");
        CK(cudaMemsetAsync(b.raw_mask, 0, sb.mask_bytes, st), "clear raw mask");
    }
    if (f.tables) { // histogram + Annex K.2 on the device
        StageTimer t(enc, 1);
        if (!f.given_hist) {
            CK(cudaMemsetAsync(enc->hist.p, 0, (size_t)n * 2 * 2 * 257 * 4, st), "clear histogram");
            CK(launch_histogram(hp, b.coef, n, enc->hist.as<uint32_t>(), st), "histogram launch");
            enc->launches += 1;
        }
        CK(launch_build_tables(enc->hist.as<uint32_t>(), 1, hl.n_tables, n, enc->huff.as<uint32_t>(), enc->hdr_parts.as<uint8_t>(), hl.head_len,
                               enc->hdr_parts.as<uint8_t>() + hl.head_len, hl.tail_len, enc->hdr.as<uint8_t>(), (uint32_t)hl.hdr_stride,
                               enc->hdr_len.as<uint32_t>(), sb.table_status(b.file_off), st),
           "table build launch");
        enc->launches += 1;
    }
    if (f.coder) {
        StageTimer t(enc, 2);
        CK(launch_encode_chunks(b, hp, n, coder, st), "coding launch");
        enc->launches += 1;
        const bool few_chunks = n_chunks <= 4096, few_segs = n_segs <= 4096;
        if (!few_chunks) CK(launch_exclusive_scan(b.chunk_bits, b.chunk_bitpos, n_chunks, b.scan_tmp, st, &enc->launches, scan_err), "chunk position scan");
        if (few_segs) { // chunk positions (when few), segment lengths and positions in one single-CTA launch
            CK(launch_positions(b, hp, n, few_chunks, st), "positions launch");
            enc->launches += 1;
        } else {
            if (few_chunks) CK(launch_exclusive_scan(b.chunk_bits, b.chunk_bitpos, n_chunks, b.scan_tmp, st, &enc->launches, scan_err), "chunk position scan");
            CK(launch_segment_lengths(b, hp, n, st), "segment length launch");
            CK(launch_exclusive_scan(b.seglen, b.segpos, n_segs, b.scan_tmp, st, &enc->launches, scan_err), "segment position scan");
            enc->launches += 1;
        }
    }
    {
        StageTimer t(enc, 3);
        // test hook: the stream starts out as all ones, so a byte that the kernels neither store nor zero shows in the output
        if (f.poison) CK(cudaMemsetAsync(b.ustream, 0xFF, b.ustream_cap + 64, st), "poison stream");
        CK(launch_segment_leads(b, hp, n, st), "segment lead launch");
        CK(launch_place_chunks(b, hp, n, st), "placement launch");
        enc->launches += 2;
    }
    {
        StageTimer t(enc, 4);
        CK(launch_count_ff(b, st), "count ff launch");
        if (ff_scan_needed(b)) CK(launch_exclusive_scan(b.ffcount, b.ffpos, n_pieces, b.scan_tmp, st, &enc->launches, scan_err), "ff scan");
        // ... and the file offsets (for a strip also where each scan's bytes start) by extra CTAs of the same launch
        CK(launch_stuff_scatter(b, hp, n, f.pieces ? enc->piece_off.as<unsigned long long>() : nullptr, st), "scatter launch");
        enc->launches += 2;
        if (f.pieces)
            CK(cudaMemcpyAsync(enc->h_pieces.p, enc->piece_off.p, (plan.scans.size() + 1) * 8, cudaMemcpyDeviceToHost, st), "read piece offsets");
        CK(cudaMemcpyAsync(enc->h_small.p, b.file_off, sb.readback_bytes(), cudaMemcpyDeviceToHost, st), "read file offsets and status");
    }
    return JPGB_OK;
}

// Every value enqueue_sequence bakes into the launches, with the plan through its signature
GraphKey graph_key(const jpgb_encoder *enc, const PlanSig &sig, const EntropyBuffers &b, uint32_t n, const CoderLaunch &coder,
                   const HeaderLayout &hl, const SequenceFlags &f) {
    static_assert(sizeof(EntropyBuffers) == 26 * 8, "every field of EntropyBuffers takes part in the graph key");
    GraphKey k{{}, {
        (uint64_t)b.coef, (uint64_t)b.huff, (uint64_t)b.huff_per_image, (uint64_t)b.scratch, (uint64_t)b.pool, b.pool_cap,
        (uint64_t)b.chunk_bits, (uint64_t)b.chunk_pool, (uint64_t)b.chunk_bitpos, (uint64_t)b.seglen, (uint64_t)b.segpos,
        (uint64_t)b.hdr_len, (uint64_t)b.hdr, b.hdr_stride, (uint64_t)b.ustream, (uint64_t)b.raw_mask, (uint64_t)b.ffcount,
        (uint64_t)b.ffpos, (uint64_t)b.out, (uint64_t)b.file_off, (uint64_t)b.scan_tmp, b.ustream_cap, b.out_cap, b.n_segs_total,
        (uint64_t)b.status, b.scan_tmp_bytes,
        coder.grid, coder.smem, coder.scratch_bytes, n,
        (uint64_t)f.tables | (uint64_t)f.given_hist << 1 | (uint64_t)f.coder << 2 | (uint64_t)f.poison << 3 | (uint64_t)f.pieces << 4,
        hl.head_len, hl.tail_len, (uint64_t)hl.n_tables,
        (uint64_t)enc->hist.p, (uint64_t)enc->hdr_parts.p, (uint64_t)enc->piece_off.p, (uint64_t)enc->h_small.p, (uint64_t)enc->h_pieces.p}};
    std::memcpy(&k.sig, &sig, sizeof(sig));
    return k;
}

// Packed pixels, rows back to back, images `image_stride` apart; the ImageBuffer planes of a planar plan (one byte per
// sample) back to back
jpgb_device_images contiguous_images(const Plan &plan, const void *d_pixels, uint64_t image_stride) {
    const uint64_t row = (uint64_t)plan.p.width * (plan.planar ? 1 : plan.bpp);
    return {d_pixels, image_stride, row, plan.planar ? row * plan.p.height : 0};
}

// Where stage A finds the pixels (jpgb_device_images, include/jpegenc_b200.h). Channel-planar pixels of a packed
// ColorType are staged by the kernels with byte k of a pixel taken from plane plane_of[k]: Bgr, Rgba and Bgra are the
// Rgb kernels with their R, G, B planes in that order (the alpha plane is not read).
void set_pixel_layout(StageAParams &ap, const Plan &plan, const jpgb_device_images &im) {
    ap.pixels = static_cast<const uint8_t *>(im.data);
    ap.image_stride = im.image_stride;
    ap.row_stride = im.row_stride;
    if (plan.planar) {
        ap.plane_stride = im.plane_stride;
    } else if (im.plane_stride && plan.ncomp > 1) {
        const uint8_t ct = plan.p.color_type;
        const bool bgr = ct == JPGB_BGR || ct == JPGB_BGRA;
        ap.channel_planar = 1;
        ap.plane_stride = im.plane_stride;
        for (int k = 0; k < 4; ++k) ap.plane_of[k] = (bgr && k < 3) ? 2 - k : k;
        if (ct == JPGB_BGR || ct == JPGB_RGBA || ct == JPGB_BGRA) {
            ap.color_type = JPGB_RGB;
            ap.bpp = 3;
        }
    }
}

// The whole device pipeline for `n` device-resident images. On success the files lie back to back
// in `out` and `offsets` (host, n + 1) delimits them.
// `given_hist` (strips with optimized tables): the symbol histogram of the *whole* image, [table][dc|ac][257],
// used instead of the one of these pixels.
int encode_device(jpgb_encoder *enc, const Plan &plan, const jpgb_device_images &images, uint32_t n, DevBuf &out,
                  std::vector<uint64_t> &offsets, std::vector<uint64_t> *piece_offsets = nullptr, const uint32_t *given_hist = nullptr,
                  bool coef_ready = false) {
    cudaStream_t st = enc->stream;
    DevPlan hp;
    plan.fill_device_plan(hp);

    const uint64_t n_segs = (uint64_t)plan.segs_per_image * n;
    const uint64_t n_chunks = (uint64_t)plan.chunks_per_image * n;

    CK(enc->coef.reserve(plan.blocks_per_image * n * 128), "alloc coefficients");
    // ---- stage A (unless the caller has already run it slice by slice behind the upload) ----
    if (!coef_ready) {
        enc->coef_tagged = false;
        StageAParams ap;
        plan.fill_stage_a(ap);
        set_pixel_layout(ap, plan, images);
        ap.coef = enc->coef.as<int16_t>();
        StageTimer t(enc, 0);
        CK(launch_stage_a(ap, n, st), "stage A launch");
        enc->launches += 1;
    }

    HeaderLayout hl;
    int rc = setup_header(enc, plan, n, given_hist, hl);
    if (rc != JPGB_OK) return rc;

    // ---- entropy coding: chunks -> pool, two small prefix sums, placement, stuffing ----
    CK(enc->chunk_bits.reserve(n_chunks * 4), "alloc chunk sizes");
    CK(enc->chunk_pool.reserve(n_chunks * 4), "alloc chunk places");
    CK(enc->chunk_bitpos.reserve((n_chunks + 1) * 8), "alloc chunk positions");
    CK(enc->seglen.reserve(n_segs * 4), "alloc seglen");
    CK(enc->segpos.reserve((n_segs + 1) * 8), "alloc segpos");
    CoderLaunch coder{};
    CK(coder_launch_config(hp, n, coder), "coder configuration");
    CK(enc->scratch.reserve(coder.scratch_bytes), "alloc coder scratch");
    CK(enc->h_small.reserve(status_block(n, 0).readback_bytes()), "alloc readback");
    if (piece_offsets) {
        CK(enc->piece_off.reserve((plan.scans.size() + 1) * 8), "alloc piece offsets");
        CK(enc->h_pieces.reserve((plan.scans.size() + 1) * 8), "alloc piece offsets (host)");
    }

    EntropyBuffers b{};
    b.coef = enc->coef.as<int16_t>();
    b.huff = enc->huff.as<uint32_t>();
    b.huff_per_image = plan.p.optimize_huffman != 0 ? 1 : 0;
    b.scratch = enc->scratch.as<uint32_t>();
    b.chunk_bits = enc->chunk_bits.as<uint32_t>();
    b.chunk_pool = enc->chunk_pool.as<uint32_t>();
    b.chunk_bitpos = enc->chunk_bitpos.as<unsigned long long>();
    b.seglen = enc->seglen.as<uint32_t>();
    b.segpos = enc->segpos.as<unsigned long long>();
    b.hdr_len = enc->hdr_len.as<uint32_t>();
    b.hdr = enc->hdr.as<uint8_t>();
    b.hdr_stride = (uint32_t)hl.hdr_stride;
    b.n_segs_total = n_segs;

    CapKey ck;
    std::memset(&ck, 0, sizeof(ck));
    ck.sig = plan_sig(plan);
    ck.raw_bytes = (uint64_t)plan.p.width * plan.p.height * plan.bpp * n;
    ck.n = n;
    Caps caps = first_caps(enc, ck, n_chunks);
    const char *poison_env = std::getenv("JPGB_POISON_STREAM");
    uint64_t ubytes = 0, total = 0, pool_used = 0;
    bool coded = false;
    for (int attempt = 0;; ++attempt) {
        caps.ustream = (caps.ustream + kStuffChunk - 1) / kStuffChunk * kStuffChunk;
        const uint64_t n_pieces = caps.ustream / kStuffChunk;
        const StatusBlock sb = status_block(n, caps.ustream);
        CK(enc->ustream.reserve(caps.ustream + 64), "alloc unstuffed stream");
        CK(enc->status.reserve(sb.bytes()), "alloc status and raw mask");
        CK(enc->ffcount.reserve((n_pieces + 1) * 4), "alloc ff counts");
        CK(enc->ffpos.reserve((n_pieces + 2) * 8), "alloc ff positions");
        CK(enc->scan_tmp.reserve(scan_tmp_bytes(std::max<uint64_t>(n_pieces, std::max(n_chunks, n_segs)))), "alloc scan scratch");
        CK(enc->pool.reserve(caps.pool_units * 16), "alloc chunk pool");
        CK(out.reserve(caps.out + 64), "alloc output");
        b.pool = enc->pool.as<uint32_t>();
        b.pool_cap = caps.pool_units;
        b.ustream = enc->ustream.as<uint8_t>();
        b.file_off = sb.file_off(enc->status.p);
        b.status = sb.status(enc->status.p);
        b.raw_mask = sb.raw_mask(enc->status.p);
        b.ffcount = enc->ffcount.as<uint32_t>();
        b.ffpos = enc->ffpos.as<unsigned long long>();
        b.scan_tmp = enc->scan_tmp.p;
        b.out = out.as<uint8_t>();
        b.ustream_cap = caps.ustream;
        b.out_cap = caps.out;
        const SequenceFlags f{plan.p.optimize_huffman != 0 && attempt == 0, given_hist != nullptr, !coded, poison_env && poison_env[0] == '1',
                              piece_offsets != nullptr};
        auto enqueue = [&] { return enqueue_sequence(enc, plan, hp, b, n, coder, hl, f); };
        // Everything behind stage A is one fixed launch sequence per (settings, batch size, buffers): captured once,
        // replayed afterwards (a dozen launches cost ~10 us each from the host; a 1080p frame needs 70 us of kernels).
        bool replayed = false;
        if (attempt == 0 && enc->graphs.ok && !enc->timing)
            CK(enc->graphs.replay(graph_key(enc, ck.sig, b, n, coder, hl, f), st, enc->launches, enqueue, replayed), "graph launch");
        if (!replayed) {
            rc = enqueue();
            if (rc != JPGB_OK) return rc;
        }
        CK(cudaStreamSynchronize(st), "final sync");
        const unsigned long long *status = sb.status(enc->h_small.p);
        if (status[kStatScanError]) return fail(enc, JPGB_ERR_CUDA, "internal: prefix-sum look-back timed out");
        if (status[kStatFlags] & kFlagSegment4G) return fail(enc, JPGB_ERR_BAD_PARAMS, "a scan segment exceeds 4 GiB (use a restart interval)");
        if (f.tables && (sb.table_status(enc->h_small.p)[kStatFlags] & kFlagHuffmanLong))
            return fail(enc, JPGB_ERR_HUFFMAN, "an optimized Huffman code does not fit (longer than 32 bits, or code plus value bits beyond 31)");
        ubytes = status[kStatUnstuffed];
        if (f.coder) pool_used = status[kStatPoolCursor];
        if (status[kStatFlags] == 0) {
            total = ubytes + status[kStatDataFF];
            break;
        }
        if (attempt >= 3) return fail(enc, JPGB_ERR_CUDA, "internal: buffer capacity retry did not converge");
        // overflow: the sizing results are still on the device; a pool overflow codes again, the rest repeats the tail
        coded = !(status[kStatFlags] & kFlagPool);
        grow_caps(caps, status, pool_used);
    }
    settle_caps(enc, ck, caps, ubytes, total, pool_used, n_chunks);
    if (piece_offsets) {
        piece_offsets->assign(enc->h_pieces.as<uint64_t>(), enc->h_pieces.as<uint64_t>() + plan.scans.size() + 1);
        enc->last_piece_scans = (uint32_t)plan.scans.size();
    }
    offsets.assign(enc->h_small.as<uint64_t>(), enc->h_small.as<uint64_t>() + n + 1);
    if (offsets[n] != total) return fail(enc, JPGB_ERR_CUDA, "internal: file offsets disagree with stream size");
    return JPGB_OK;
}

// Host -> device copy of caller memory. Pinned (or registered) memory goes straight to the copy engine. Pageable
// memory -- what `Encoder::encode(&[u8])` hands over -- is staged through two pinned buffers owned by the context:
// while the copy engine drains one, the host fills the other, so the DMA never waits for a page-locked bounce
// inside the driver and the copy stays asynchronous.
constexpr size_t kStageBytes = 16u << 20;
cudaError_t upload_host(jpgb_encoder *enc, void *d_dst, const uint8_t *src, size_t bytes, cudaStream_t s) {
    cudaPointerAttributes attr{};
    const bool pinned = cudaPointerGetAttributes(&attr, src) == cudaSuccess && (attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged);
    cudaGetLastError(); // an unregistered pointer may leave a sticky-free error code behind on older runtimes
    if (pinned || bytes <= 65536) return cudaMemcpyAsync(d_dst, src, bytes, cudaMemcpyHostToDevice, s);
    // pieces of 16 MB; an input of 16 .. 32 MB goes in two pieces (of whole MB) so that the DMA of the first one runs
    // behind the copy of the second. Smaller inputs go in one piece: measured on a 1080p frame, two pieces and helper
    // threads cost more in wake-ups (0.95 ms per call) than they save (0.84 ms with the caller copying alone).
    size_t piece = kStageBytes;
    if (bytes >= kStageBytes && bytes < 2 * kStageBytes) piece = ((bytes / 2 + (1u << 20) - 1) >> 20) << 20;
    unsigned hw = std::thread::hardware_concurrency();
    if (const char *e = std::getenv("JPGB_COPY_THREADS")) hw = (unsigned)std::max(1, std::atoi(e)); // test hook: 1 = the caller alone
    for (size_t off = 0, k = 0; off < bytes; off += piece, ++k) {
        const int b = (int)(k & 1);
        const size_t n = std::min(piece, bytes - off);
        cudaError_t e = enc->h_stage[b].reserve(kStageBytes);
        if (e != cudaSuccess) return e;
        if (enc->stage_busy[b]) { // the DMA that last read this buffer must be done before the host overwrites it
            e = cudaEventSynchronize(enc->ev_stage[b]);
            if (e != cudaSuccess) return e;
        }
        unsigned threads = (unsigned)std::min<size_t>(4, n >> 22); // at least 4 MB per thread
        if (hw && threads > hw) threads = hw;
        enc->copy_pool.copy(enc->h_stage[b].p, src + off, n, threads);
        e = cudaMemcpyAsync(static_cast<uint8_t *>(d_dst) + off, enc->h_stage[b].p, n, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) return e;
        e = cudaEventRecord(enc->ev_stage[b], s);
        if (e != cudaSuccess) return e;
        enc->stage_busy[b] = true;
    }
    return cudaSuccess;
}

// Host pixels -> host files for n images, pipelined in chunks over three streams: while chunk c is
// encoded on the context's stream, chunk c+1 is uploaded (s_h2d) and the files of chunk c-1 are
// downloaded (s_d2h) into one pinned buffer owned by the context. PCIe moves 3 B/pixel in and the
// files out; the device pipeline itself is ~10x faster, so the copies set the pace.
// On success file i is h_out[offsets[i] .. offsets[i+1]).
int encode_host_pipelined(jpgb_encoder *enc, const Plan &plan, const uint8_t *const *pixels, uint32_t n,
                          std::vector<uint64_t> &offsets) {
    const size_t img_bytes = (size_t)plan.p.width * plan.p.height * plan.bpp;
    const size_t stride = (img_bytes + 255) & ~(size_t)255;
    uint32_t chunk = (uint32_t)std::max<size_t>(1, (96u << 20) / stride); // ~96 MB of pixels per chunk
    chunk = std::min(chunk, n);
    const uint32_t n_chunks = (n + chunk - 1) / chunk;
    CK(enc->pixels.reserve(stride * chunk), "alloc pixels");
    if (n_chunks > 1) CK(enc->pixels2.reserve(stride * chunk), "alloc pixels");
    CK(enc->h_out.reserve(std::max<size_t>(img_bytes * n / 3, 1 << 20)), "alloc pinned output");
    offsets.assign(1, 0);
    cudaStream_t st = enc->stream;

    // One large image: the upload dominates (3 B/pixel over PCIe against ~1 ms of device work), so the image is cut into
    // slices of whole MCU rows and the colour+DCT kernel runs on slice k while slice k + 1 is still on the link.
    if (n == 1 && !plan.planar && img_bytes >= (48u << 20)) {
        const size_t row_bytes = (size_t)plan.p.width * plan.bpp;
        const uint32_t mcu_px = 8 * plan.vmax;
        uint32_t rows_per_slice = (uint32_t)std::max<size_t>(1, (32u << 20) / (row_bytes * mcu_px)); // in MCU rows, ~32 MB
        rows_per_slice = (rows_per_slice + 3) & ~3u; // whole warp tiles (up to four MCU rows each)
        const uint32_t n_slices = (plan.mcu_rows + rows_per_slice - 1) / rows_per_slice;
        CK(enc->pixels.reserve(stride), "alloc pixels");
        CK(enc->coef.reserve(plan.blocks_per_image * 128), "alloc coefficients");
        enc->coef_tagged = false;
        while (enc->ev_slice.size() < n_slices) {
            cudaEvent_t e;
            CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "create event");
            enc->ev_slice.push_back(e);
        }
        StageAParams ap;
        plan.fill_stage_a(ap);
        for (uint32_t k = 0; k < n_slices; ++k) { // all uploads are queued first: the link never idles
            const size_t r0 = (size_t)k * rows_per_slice * mcu_px, r1 = std::min<size_t>(plan.p.height, r0 + (size_t)rows_per_slice * mcu_px);
            CK(upload_host(enc, enc->pixels.as<uint8_t>() + r0 * row_bytes, pixels[0] + r0 * row_bytes, (r1 - r0) * row_bytes, enc->s_h2d), "upload slice");
            CK(cudaEventRecord(enc->ev_slice[k], enc->s_h2d), "record slice");
        }
        for (uint32_t k = 0; k < n_slices; ++k) {
            const size_t r0 = (size_t)k * rows_per_slice * mcu_px, r1 = std::min<size_t>(plan.p.height, r0 + (size_t)rows_per_slice * mcu_px);
            StageAParams sp = ap;
            sp.pixels = enc->pixels.as<uint8_t>() + r0 * row_bytes;
            sp.coef = enc->coef.as<int16_t>();
            sp.image_stride = stride;
            sp.height = (int)(r1 - r0);
            sp.mcu_row0 = (int)(k * rows_per_slice);
            sp.mcu_rows = (int)std::min<uint32_t>(rows_per_slice, plan.mcu_rows - k * rows_per_slice);
            CK(cudaStreamWaitEvent(st, enc->ev_slice[k], 0), "wait slice");
            CK(launch_stage_a(sp, 1, st), "stage A launch");
            enc->launches += 1;
        }
        std::vector<uint64_t> off;
        const int rc = encode_device(enc, plan, contiguous_images(plan, enc->pixels.p, stride), 1, enc->out, off, nullptr, nullptr, true);
        if (rc != JPGB_OK) return rc;
        CK(enc->h_out.reserve(std::max<size_t>(off[1], 1 << 20)), "alloc pinned output");
        CK(cudaMemcpyAsync(enc->h_out.p, enc->out.p, off[1], cudaMemcpyDeviceToHost, st), "download file");
        CK(cudaStreamSynchronize(st), "download sync");
        offsets.push_back(off[1]);
        return JPGB_OK;
    }

    auto upload = [&](uint32_t c) -> cudaError_t {
        DevBuf &px = (c & 1) ? enc->pixels2 : enc->pixels;
        const uint32_t lo = c * chunk, hi = std::min(n, lo + chunk);
        if (c >= 2) { // the buffer was last read by the encode of chunk c-2
            cudaError_t e = cudaStreamWaitEvent(enc->s_h2d, enc->ev_enc[c & 1], 0);
            if (e != cudaSuccess) return e;
        }
        for (uint32_t i = lo; i < hi; ++i) {
            cudaError_t e = upload_host(enc, px.as<uint8_t>() + stride * (i - lo), pixels[i], img_bytes, enc->s_h2d);
            if (e != cudaSuccess) return e;
        }
        return cudaEventRecord(enc->ev_in[c & 1], enc->s_h2d);
    };

    {
        StageTimer t(enc, 5);
        CK(upload(0), "upload pixels");
    }
    uint64_t total = 0;
    for (uint32_t c = 0; c < n_chunks; ++c) {
        const uint32_t lo = c * chunk, hi = std::min(n, lo + chunk), cn = hi - lo;
        if (c + 1 < n_chunks) CK(upload(c + 1), "upload pixels");
        DevBuf &px = (c & 1) ? enc->pixels2 : enc->pixels;
        DevBuf &ob = (c & 1) ? enc->out2 : enc->out;
        CK(cudaStreamWaitEvent(st, enc->ev_in[c & 1], 0), "wait upload");
        if (c >= 2) CK(cudaStreamWaitEvent(st, enc->ev_out[c & 1], 0), "wait download"); // out slot reused
        std::vector<uint64_t> off;
        const int rc = encode_device(enc, plan, contiguous_images(plan, px.p, stride), cn, ob, off);
        if (rc != JPGB_OK) return rc;
        CK(cudaEventRecord(enc->ev_enc[c & 1], st), "record encode");
        const uint64_t bytes = off[cn];
        if (total + bytes > enc->h_out.cap) { // grow the pinned buffer, keeping what is already there
            CK(cudaStreamSynchronize(enc->s_d2h), "download sync");
            PinnedBuf bigger;
            CK(bigger.reserve((total + bytes) * 2), "grow pinned output");
            std::memcpy(bigger.p, enc->h_out.p, total);
            std::swap(enc->h_out, bigger);
        }
        // encode_device has synchronised the context's stream: the files are complete in `ob`
        CK(cudaMemcpyAsync(enc->h_out.as<uint8_t>() + total, ob.p, bytes, cudaMemcpyDeviceToHost, enc->s_d2h), "download files");
        CK(cudaEventRecord(enc->ev_out[c & 1], enc->s_d2h), "record download");
        for (uint32_t i = 0; i < cn; ++i) offsets.push_back(total + off[i + 1]);
        total += bytes;
    }
    {
        StageTimer t(enc, 6);
        CK(cudaStreamSynchronize(enc->s_d2h), "download sync");
    }
    return JPGB_OK;
}

int encode_host_batch(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *const *pixels, size_t len_each, uint32_t n,
                      uint8_t **outs, size_t *out_lens, const uint8_t **pinned_base, uint64_t *pinned_offsets) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    const bool pinned_api = pinned_base != nullptr;
    if (!pixels || n == 0 || (pinned_api ? !pinned_offsets : (!outs || !out_lens))) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    if (!pinned_api)
        for (uint32_t i = 0; i < n; ++i) outs[i] = nullptr, out_lens[i] = 0;
    Plan plan;
    int rc = validate_and_plan(enc, p, len_each, plan);
    if (rc != JPGB_OK) return rc;
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    const bool was_timing = enc->timing;
    enc->timing = false; // per-stage events are per encode_device call; the pipelined path runs several
    timing_begin(enc);
    std::vector<uint64_t> off;
    rc = encode_host_pipelined(enc, plan, pixels, n, off);
    enc->timing = was_timing;
    if (rc != JPGB_OK) return rc;
    if (pinned_api) {
        *pinned_base = enc->h_out.as<uint8_t>();
        std::memcpy(pinned_offsets, off.data(), (size_t)(n + 1) * 8);
        return JPGB_OK;
    }
    for (uint32_t i = 0; i < n; ++i) {
        const size_t sz = (size_t)(off[i + 1] - off[i]);
        outs[i] = static_cast<uint8_t *>(std::malloc(sz ? sz : 1));
        if (!outs[i]) {
            for (uint32_t k = 0; k < i; ++k) std::free(outs[k]), outs[k] = nullptr;
            return fail(enc, JPGB_ERR_NOMEM, "out of host memory");
        }
        out_lens[i] = sz;
        std::memcpy(outs[i], enc->h_out.as<uint8_t>() + off[i], sz);
    }
    return JPGB_OK;
}

} // namespace

extern "C" {

void jpgb_params_default(jpgb_params *p, uint8_t quality) {
    std::memset(p, 0, sizeof(*p));
    p->quality = quality;
    p->sampling = quality < 90 ? 0x22 : 0x11; // encoder.rs:256-260
    p->density_unit = 0;                       // PixelDensity::default, writer.rs:37-45
    p->density_x = p->density_y = 1;
}

int jpgb_encoder_create(int device, void *cuda_stream, jpgb_encoder **out) {
    if (!out) return JPGB_ERR_BAD_PARAMS;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return JPGB_ERR_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return JPGB_ERR_CUDA;
    if (prop.major != 10) return JPGB_ERR_CUDA; // kernels are built for sm_100a only; there is no fallback
    if (cudaSetDevice(device) != cudaSuccess) return JPGB_ERR_CUDA;
    jpgb_encoder *e = new (std::nothrow) jpgb_encoder();
    if (!e) return JPGB_ERR_NOMEM;
    e->device = device;
    if (cuda_stream) {
        e->stream = static_cast<cudaStream_t>(cuda_stream);
    } else {
        if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete e;
            return JPGB_ERR_CUDA;
        }
        e->own_stream = true;
    }
    for (int i = 0; i < JPGB_N_STAGES; ++i)
        for (int k = 0; k < 2; ++k) cudaEventCreate(&e->ev[i][k]);
    cudaStreamCreateWithFlags(&e->s_h2d, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&e->s_d2h, cudaStreamNonBlocking);
    for (int i = 0; i < 2; ++i) {
        cudaEventCreateWithFlags(&e->ev_in[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&e->ev_out[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&e->ev_enc[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&e->ev_stage[i], cudaEventDisableTiming);
    }
    cudaEventCreateWithFlags(&e->ev_wait, cudaEventDisableTiming);
    *out = e;
    return JPGB_OK;
}

void jpgb_encoder_destroy(jpgb_encoder *e) {
    if (!e) return;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    if (e->s_h2d) cudaStreamDestroy(e->s_h2d);
    if (e->s_d2h) cudaStreamDestroy(e->s_d2h);
    for (cudaEvent_t ev : e->ev_slice) cudaEventDestroy(ev);
    for (int i = 0; i < 2; ++i) {
        if (e->ev_in[i]) cudaEventDestroy(e->ev_in[i]);
        if (e->ev_out[i]) cudaEventDestroy(e->ev_out[i]);
        if (e->ev_enc[i]) cudaEventDestroy(e->ev_enc[i]);
        if (e->ev_stage[i]) cudaEventDestroy(e->ev_stage[i]);
    }
    if (e->ev_wait) cudaEventDestroy(e->ev_wait);
    for (int i = 0; i < JPGB_N_STAGES; ++i)
        for (int k = 0; k < 2; ++k)
            if (e->ev[i][k]) cudaEventDestroy(e->ev[i][k]);
    if (e->own_stream) cudaStreamDestroy(e->stream);
    delete e; // frees the buffers and graphs
}

const char *jpgb_last_error(const jpgb_encoder *e) { return e ? e->err.c_str() : "no encoder"; }

int jpgb_encode(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *pixels, size_t len, uint8_t **out, size_t *out_len) {
    if (!out || !out_len) return JPGB_ERR_BAD_PARAMS;
    *out = nullptr;
    *out_len = 0;
    const uint8_t *px[1] = {pixels};
    return encode_host_batch(enc, p, px, len, 1, out, out_len, nullptr, nullptr);
}

void jpgb_free(void *buf) { std::free(buf); }

// Encoder::encode_image's planes -> the file in the context's pinned output buffer (enc->h_out)
static int encode_planar_pinned(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *const planes[4], size_t plane_len, size_t *out_len) {
    if (!p || !planes) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    const uint8_t ct = p->color_type;
    if (ct != JPGB_LUMA && ct != JPGB_YCBCR && ct != JPGB_CMYK && ct != JPGB_YCCK)
        return fail(enc, JPGB_ERR_BAD_PARAMS, "planar input takes a JPEG colour type: Luma, Ycbcr, Cmyk or Ycck");
    const size_t plane_bytes = (size_t)p->width * p->height;
    if (plane_len < plane_bytes) return fail(enc, JPGB_ERR_BAD_IMAGE_DATA, "plane shorter than width*height");
    Plan plan;
    plan.planar = true;
    const int rc = plan.build(*p);
    if (rc != JPGB_OK) return fail(enc, rc, rc == JPGB_ERR_ZERO_DIMENSIONS ? "Image dimensions must be non zero" : "invalid parameters");
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    timing_begin(enc);
    const size_t stride = (plane_bytes * plan.ncomp + 255) & ~(size_t)255;
    CK(enc->pixels.reserve(stride), "alloc planes");
    for (int c = 0; c < plan.ncomp; ++c) {
        if (!planes[c]) return fail(enc, JPGB_ERR_BAD_PARAMS, "null plane");
        CK(upload_host(enc, enc->pixels.as<uint8_t>() + plane_bytes * c, planes[c], plane_bytes, enc->stream), "upload plane");
    }
    std::vector<uint64_t> off;
    const int rc2 = encode_device(enc, plan, contiguous_images(plan, enc->pixels.p, stride), 1, enc->out, off);
    if (rc2 != JPGB_OK) return rc2;
    const size_t sz = (size_t)off[1];
    CK(enc->h_out.reserve(sz ? sz : 1), "alloc pinned output");
    CK(cudaMemcpyAsync(enc->h_out.p, enc->out.p, sz, cudaMemcpyDeviceToHost, enc->stream), "download file");
    CK(cudaStreamSynchronize(enc->stream), "download sync");
    *out_len = sz;
    timing_end(enc);
    return JPGB_OK;
}

int jpgb_encode_planar(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *const planes[4], size_t plane_len, uint8_t **out,
                       size_t *out_len) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!out || !out_len) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    *out = nullptr;
    *out_len = 0;
    size_t sz = 0;
    const int rc = encode_planar_pinned(enc, p, planes, plane_len, &sz);
    if (rc != JPGB_OK) return rc;
    *out = static_cast<uint8_t *>(std::malloc(sz ? sz : 1));
    if (!*out) return fail(enc, JPGB_ERR_NOMEM, "out of host memory");
    std::memcpy(*out, enc->h_out.p, sz);
    *out_len = sz;
    return JPGB_OK;
}

int jpgb_encode_planar_to_sink(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *const planes[4], size_t plane_len,
                               jpgb_write_all_fn write_all, void *user) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!write_all) return fail(enc, JPGB_ERR_BAD_PARAMS, "null sink");
    size_t sz = 0;
    const int rc = encode_planar_pinned(enc, p, planes, plane_len, &sz);
    if (rc != JPGB_OK) return rc;
    if (write_all(user, enc->h_out.as<uint8_t>(), sz) != 0) return fail(enc, JPGB_ERR_SINK, "sink write_all failed");
    return JPGB_OK;
}

// The sink receives the file straight from the context's pinned download buffer: one write_all call, no
// intermediate copy (the reference makes many small write_all calls, src/writer.rs:123-202; only the number of
// calls differs, the bytes and the error propagation do not).
int jpgb_encode_to_sink(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *pixels, size_t len, jpgb_write_all_fn write_all,
                        void *user) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!write_all) return fail(enc, JPGB_ERR_BAD_PARAMS, "null sink");
    const uint8_t *px[1] = {pixels};
    const uint8_t *files = nullptr;
    uint64_t offs[2] = {0, 0};
    const int rc = encode_host_batch(enc, p, px, len, 1, nullptr, nullptr, &files, offs);
    if (rc != JPGB_OK) return rc;
    if (write_all(user, files + offs[0], (size_t)(offs[1] - offs[0])) != 0) return fail(enc, JPGB_ERR_SINK, "sink write_all failed");
    return JPGB_OK;
}

int jpgb_encode_batch(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *const *pixels, size_t len_each, uint32_t n,
                      uint8_t **outs, size_t *out_lens) {
    return encode_host_batch(enc, p, pixels, len_each, n, outs, out_lens, nullptr, nullptr);
}

int jpgb_encode_batch_pinned(jpgb_encoder *enc, const jpgb_params *p, const uint8_t *const *pixels, size_t len_each, uint32_t n,
                             const uint8_t **files, uint64_t *offsets) {
    if (!files) return JPGB_ERR_BAD_PARAMS;
    return encode_host_batch(enc, p, pixels, len_each, n, nullptr, nullptr, files, offsets);
}

int jpgb_encode_batch_device(jpgb_encoder *enc, const jpgb_params *p, const void *d_pixels, size_t image_stride, uint32_t n,
                             const void **d_files, uint64_t *offsets) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!d_pixels || !d_files || !offsets || n == 0) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    Plan plan;
    int rc = validate_and_plan(enc, p, image_stride, plan);
    if (rc != JPGB_OK) return rc;
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    timing_begin(enc);
    std::vector<uint64_t> off;
    rc = encode_device(enc, plan, contiguous_images(plan, d_pixels, image_stride), n, enc->out, off);
    if (rc != JPGB_OK) return rc;
    timing_end(enc);
    std::memcpy(offsets, off.data(), (size_t)(n + 1) * 8);
    *d_files = enc->out.p;
    return JPGB_OK;
}

int jpgb_encode_batch_device_strided(jpgb_encoder *enc, const jpgb_params *p, const jpgb_device_images *images, uint32_t n,
                                     const void **d_files, uint64_t *offsets) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    enc->launches = 0; // a rejected call reports no launches
    if (!images || !images->data || !d_files || !offsets || n == 0) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    Plan plan;
    int rc = validate_and_plan(enc, p, SIZE_MAX, plan); // a strided layout has no length to check
    if (rc != JPGB_OK) return rc;
    rc = check_device_images(enc, plan, *images, n);
    if (rc != JPGB_OK) return rc;
    // Ycbcr and Ycck planes are the ImageBuffer planes: samples taken verbatim, one plane per component
    plan.planar = images->plane_stride != 0 && (p->color_type == JPGB_YCBCR || p->color_type == JPGB_YCCK);
    timing_begin(enc);
    std::vector<uint64_t> off;
    rc = encode_device(enc, plan, *images, n, enc->out, off);
    if (rc != JPGB_OK) return rc;
    timing_end(enc);
    std::memcpy(offsets, off.data(), (size_t)(n + 1) * 8);
    *d_files = enc->out.p;
    return JPGB_OK;
}

int jpgb_encoder_wait_stream(jpgb_encoder *enc, void *stream) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (s == enc->stream) return JPGB_OK;
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    CK(cudaEventRecord(enc->ev_wait, s), "record the caller's stream");
    CK(cudaStreamWaitEvent(enc->stream, enc->ev_wait, 0), "wait for the caller's stream");
    return JPGB_OK;
}

int jpgb_scan_count(const jpgb_params *p, uint32_t *n_scans) {
    if (!p || !n_scans) return JPGB_ERR_BAD_PARAMS;
    Plan plan;
    const int rc = plan.build(*p);
    if (rc != JPGB_OK) return rc;
    *n_scans = (uint32_t)plan.scans.size();
    return JPGB_OK;
}

int jpgb_plan_strips(const jpgb_params *p, uint32_t max_strips, jpgb_strip *strips, uint32_t *n_strips) {
    if (!p || !strips || !n_strips || max_strips == 0) return JPGB_ERR_BAD_PARAMS;
    Plan plan;
    const int rc = plan.build(*p);
    if (rc != JPGB_OK) return rc;
    const uint32_t R = p->restart_interval;
    if (R == 0) return JPGB_ERR_BAD_PARAMS;
    auto gcd = [](uint64_t a, uint64_t b) { while (b) { const uint64_t t = a % b; a = b; b = t; } return a; };
    // a strip may start at MCU row r only if r * (units per MCU row) is a multiple of R in every scan
    uint64_t step = 1;
    for (const Scan &s : plan.scans) {
        const uint64_t upr = s.comp < 0 ? plan.mcu_cols : (uint64_t)plan.comps[s.comp].v * plan.true_w[s.comp];
        const uint64_t need = R / gcd(R, upr);
        step = step / gcd(step, need) * need;
    }
    const uint64_t groups = (plan.mcu_rows + step - 1) / step; // groups of `step` MCU rows (the last may be short)
    uint32_t n = (uint32_t)std::min<uint64_t>(max_strips, groups);
    if (n == 0) n = 1;
    const uint32_t rows_per_mcu = 8 * plan.vmax;
    uint64_t g0 = 0;
    for (uint32_t i = 0; i < n; ++i) {
        const uint64_t g1 = groups * (i + 1) / n;
        const uint64_t r0 = g0 * step * rows_per_mcu, r1 = std::min<uint64_t>(g1 * step * rows_per_mcu, p->height);
        strips[i].strip_index = i;
        strips[i].n_strips = n;
        strips[i].first_row = (uint16_t)r0;
        strips[i].rows = (uint16_t)(r1 - r0);
        strips[i].full_height = p->height;
        g0 = g1;
    }
    *n_strips = n;
    return JPGB_OK;
}

static int encode_strip(jpgb_encoder *enc, const jpgb_params *p, const jpgb_strip *strip, const void *d_pixels, const uint32_t *hist_total,
                        const void **d_bytes, uint64_t *piece_offsets) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!p || !strip || !d_pixels || !d_bytes || !piece_offsets) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    if (p->color_type > JPGB_YCCK) return fail(enc, JPGB_ERR_BAD_PARAMS, "bad color_type");
    if ((p->optimize_huffman != 0) != (hist_total != nullptr))
        return fail(enc, JPGB_ERR_BAD_PARAMS, "optimized tables with strips take the whole image's histogram (jpgb_encode_strip_device_optimized); other settings take none");
    Plan plan;
    const int rc = plan.build(*p, strip);
    if (rc != JPGB_OK) return fail(enc, rc, "settings or strip geometry do not allow strip encoding (needs restart intervals aligned in every scan)");
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    timing_begin(enc);
    std::vector<uint64_t> off, pieces;
    const size_t stride = (size_t)p->width * strip->rows * bytes_per_pixel(p->color_type);
    bool reuse = false;
    if (hist_total && enc->coef_tagged && enc->coef_pixels == d_pixels && enc->coef_stride == uint64_t(stride)) {
        const PlanSig sig = plan_sig(plan);
        reuse = std::memcmp(&sig, &enc->coef_sig, sizeof(sig)) == 0;
    }
    const int rc2 = encode_device(enc, plan, contiguous_images(plan, d_pixels, stride), 1, enc->out, off, &pieces, hist_total, reuse);
    enc->coef_tagged = false;
    if (rc2 != JPGB_OK) return rc2;
    timing_end(enc);
    if (reuse && enc->timing) { // the stages that ran in the histogram call belong to this strip's encode
        enc->last_ms[0] += enc->coef_ms[0];
        enc->last_ms[1] += enc->coef_ms[1];
    }
    std::memcpy(piece_offsets, pieces.data(), pieces.size() * 8);
    *d_bytes = enc->out.p;
    return JPGB_OK;
}

int jpgb_encode_strip_device(jpgb_encoder *enc, const jpgb_params *p, const jpgb_strip *strip, const void *d_pixels,
                             const void **d_bytes, uint64_t *piece_offsets) {
    return encode_strip(enc, p, strip, d_pixels, nullptr, d_bytes, piece_offsets);
}

int jpgb_encode_strip_device_optimized(jpgb_encoder *enc, const jpgb_params *p, const jpgb_strip *strip, const void *d_pixels,
                                       const uint32_t hist_total[JPGB_HIST_WORDS], const void **d_bytes, uint64_t *piece_offsets) {
    if (enc && !hist_total) return fail(enc, JPGB_ERR_BAD_PARAMS, "null histogram");
    return encode_strip(enc, p, strip, d_pixels, hist_total, d_bytes, piece_offsets);
}

int jpgb_strip_histogram_device(jpgb_encoder *enc, const jpgb_params *p, const jpgb_strip *strip, const void *d_pixels,
                                uint32_t hist[JPGB_HIST_WORDS], int16_t edge_dc[8]) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!p || !strip || !d_pixels || !hist || !edge_dc) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    if (p->color_type > JPGB_YCCK || !p->optimize_huffman) return fail(enc, JPGB_ERR_BAD_PARAMS, "strip histograms belong to optimized Huffman tables");
    Plan plan;
    const int rc = plan.build(*p, strip);
    if (rc != JPGB_OK) return fail(enc, rc, "settings or strip geometry do not allow strip encoding (needs restart intervals aligned in every scan)");
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    cudaStream_t st = enc->stream;
    DevPlan hp;
    plan.fill_device_plan(hp);
    StageAParams ap;
    plan.fill_stage_a(ap);
    CK(enc->coef.reserve(plan.blocks_per_image * 128), "alloc coefficients");
    ap.pixels = static_cast<const uint8_t *>(d_pixels);
    ap.coef = enc->coef.as<int16_t>();
    ap.image_stride = (size_t)p->width * strip->rows * bytes_per_pixel(p->color_type);
    timing_begin(enc);
    {
        StageTimer t(enc, 0);
        CK(launch_stage_a(ap, 1, st), "stage A launch");
    }
    const size_t hist_bytes = JPGB_HIST_WORDS * 4;
    CK(enc->hist.reserve(hist_bytes), "alloc histogram");
    CK(enc->h_hist.reserve(hist_bytes + 16), "alloc histogram (host)");
    {
        StageTimer t(enc, 1);
        CK(cudaMemsetAsync(enc->hist.p, 0, hist_bytes, st), "clear histogram");
        CK(launch_histogram(hp, enc->coef.as<int16_t>(), 1, enc->hist.as<uint32_t>(), st), "histogram launch");
    }
    enc->launches = 2;
    CK(cudaMemcpyAsync(enc->h_hist.p, enc->hist.p, hist_bytes, cudaMemcpyDeviceToHost, st), "download histogram");
    // DC of the first and of the last block of every component's true grid (the histogram chains DC differences
    // across the whole image without restart resets, encoder.rs:1086-1200: the neighbours need them)
    int16_t *edge = reinterpret_cast<int16_t *>(enc->h_hist.as<uint8_t>() + hist_bytes);
    std::memset(edge, 0, 16);
    for (int c = 0; c < plan.ncomp; ++c) {
        const uint64_t first = plan.block_off[c], last = plan.block_off[c] + (uint64_t)plan.true_w[c] * plan.true_h[c] - 1; // raster of the true grid
        CK(cudaMemcpyAsync(edge + c, enc->coef.as<int16_t>() + first * 64, 2, cudaMemcpyDeviceToHost, st), "read edge DC");
        CK(cudaMemcpyAsync(edge + 4 + c, enc->coef.as<int16_t>() + last * 64, 2, cudaMemcpyDeviceToHost, st), "read edge DC");
    }
    CK(cudaStreamSynchronize(st), "histogram sync");
    std::memcpy(hist, enc->h_hist.p, hist_bytes);
    std::memcpy(edge_dc, edge, 16);
    enc->coef_sig = plan_sig(plan);
    enc->coef_pixels = d_pixels;
    enc->coef_stride = uint64_t(ap.image_stride);
    enc->coef_tagged = true;
    timing_end(enc);
    enc->coef_ms[0] = enc->timing ? enc->last_ms[0] : 0.f;
    enc->coef_ms[1] = enc->timing ? enc->last_ms[1] : 0.f;
    return JPGB_OK;
}

int jpgb_merge_strip_histograms(const jpgb_params *p, uint32_t n_strips, const uint32_t hist_sum[JPGB_HIST_WORDS], const int16_t *edge_dc,
                                uint32_t hist_total[JPGB_HIST_WORDS]) {
    if (!p || !hist_sum || !edge_dc || !hist_total || n_strips == 0) return JPGB_ERR_BAD_PARAMS;
    Plan plan;
    const int rc = plan.build(*p);
    if (rc != JPGB_OK) return rc;
    std::memcpy(hist_total, hist_sum, JPGB_HIST_WORDS * 4);
    auto category = [](int diff) { // get_num_bits of the i16 difference, encoder.rs:1244-1257
        int a = (int16_t)diff;
        a = a < 0 ? -a : a;
        int n = 0;
        while (a) ++n, a >>= 1;
        return n;
    };
    for (uint32_t s = 1; s < n_strips; ++s)
        for (int c = 0; c < plan.ncomp; ++c) {
            uint32_t *dc = hist_total + (size_t)plan.comps[c].dc_table * 2 * 257;
            const int first = edge_dc[s * 8 + c], prev_last = edge_dc[(s - 1) * 8 + 4 + c];
            dc[category(first)] -= 1;             // the strip counted its first block against a predictor of 0
            dc[category(first - prev_last)] += 1; // the whole image chains it to the block before
        }
    return JPGB_OK;
}

int jpgb_gather_target_create(jpgb_encoder *enc, size_t capacity, void **d_target, uint8_t ipc_handle[64]) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!d_target || !ipc_handle || capacity == 0) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the C ABI carries the IPC handle as 64 bytes");
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    void *p = nullptr;
    CK(cudaMalloc(&p, capacity + 64), "alloc gather target");
    cudaIpcMemHandle_t h;
    const cudaError_t ce = cudaIpcGetMemHandle(&h, p);
    if (ce != cudaSuccess) {
        cudaFree(p);
        return fail_cuda(enc, ce, "cudaIpcGetMemHandle");
    }
    std::memcpy(ipc_handle, &h, 64);
    *d_target = p;
    return JPGB_OK;
}

int jpgb_gather_target_open(jpgb_encoder *enc, const uint8_t ipc_handle[64], void **d_target) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!d_target || !ipc_handle) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    cudaIpcMemHandle_t h;
    std::memcpy(&h, ipc_handle, 64);
    void *p = nullptr;
    CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle (peer access over NVLink)");
    *d_target = p;
    return JPGB_OK;
}

int jpgb_gather_target_close(jpgb_encoder *enc, void *d_target, int opened_from_handle) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!d_target) return JPGB_OK;
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    CK(cudaStreamSynchronize(enc->stream), "sync before releasing the gather target");
    if (opened_from_handle) CK(cudaIpcCloseMemHandle(d_target), "cudaIpcCloseMemHandle");
    else CK(cudaFree(d_target), "free gather target");
    return JPGB_OK;
}

int jpgb_last_piece_offsets_device(jpgb_encoder *enc, const uint64_t **d_offsets, uint32_t *n_scans) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!d_offsets || !n_scans || !enc->piece_off.p || enc->last_piece_scans == 0) return fail(enc, JPGB_ERR_BAD_PARAMS, "no strip has been encoded on this context");
    *d_offsets = enc->piece_off.as<uint64_t>();
    *n_scans = enc->last_piece_scans;
    return JPGB_OK;
}

int jpgb_gather_place_pieces(jpgb_encoder *enc, void *d_target, size_t target_capacity, const uint64_t *d_table, uint32_t world, uint32_t rank,
                             uint64_t *d_total) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!d_target || !d_table || world == 0 || rank >= world || enc->last_piece_scans == 0) return fail(enc, JPGB_ERR_BAD_PARAMS, "bad gather arguments");
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    CK(launch_place_pieces(enc->out.as<uint8_t>(), static_cast<uint8_t *>(d_target), target_capacity, reinterpret_cast<const unsigned long long *>(d_table),
                           world, rank, enc->last_piece_scans, reinterpret_cast<unsigned long long *>(d_total), enc->stream),
       "piece placement launch");
    return JPGB_OK;
}

int jpgb_download(jpgb_encoder *enc, const void *d_src, size_t n, void *host_dst) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (n == 0) return JPGB_OK;
    if (!d_src || !host_dst) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    CK(cudaMemcpyAsync(host_dst, d_src, n, cudaMemcpyDeviceToHost, enc->stream), "download");
    CK(cudaStreamSynchronize(enc->stream), "download sync");
    return JPGB_OK;
}

int jpgb_coef_layout_for(const jpgb_params *p, jpgb_coef_layout *l) {
    if (!p || !l) return JPGB_ERR_BAD_PARAMS;
    Plan plan;
    const int rc = plan.build(*p);
    if (rc != JPGB_OK) return rc;
    std::memset(l, 0, sizeof(*l));
    l->n_components = (uint32_t)plan.ncomp;
    for (int c = 0; c < plan.ncomp; ++c) {
        l->blocks_w[c] = plan.pad_w[c];
        l->blocks_h[c] = plan.pad_h[c];
        l->true_w[c] = plan.true_w[c];
        l->true_h[c] = plan.true_h[c];
        l->block_offset[c] = plan.block_off[c];
        l->slot_base[c] = plan.slot_base[c];
        l->comp_h[c] = plan.comps[c].h;
        l->comp_v[c] = plan.comps[c].v;
    }
    l->blocks_per_image = plan.blocks_per_image;
    l->mcu_order = plan.mode == Mode::Interleaved;
    l->mcu_cols = plan.mcu_cols;
    l->mcu_rows = plan.mcu_rows;
    l->blocks_per_mcu = plan.bpu_interleaved;
    return JPGB_OK;
}

int jpgb_stage_a_device(jpgb_encoder *enc, const jpgb_params *p, const void *d_pixels, size_t image_stride, uint32_t n, void *d_coef) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!d_pixels || !d_coef || n == 0) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    Plan plan;
    const int rc = validate_and_plan(enc, p, image_stride, plan);
    if (rc != JPGB_OK) return rc;
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    StageAParams ap;
    plan.fill_stage_a(ap);
    ap.pixels = static_cast<const uint8_t *>(d_pixels);
    ap.coef = static_cast<int16_t *>(d_coef);
    ap.image_stride = image_stride;
    enc->launches = 0;
    CK(launch_stage_a(ap, n, enc->stream), "stage A launch");
    enc->launches = 1;
    return JPGB_OK;
}

void jpgb_encoder_set_timing(jpgb_encoder *enc, int enabled) {
    if (enc) enc->timing = enabled != 0;
}
int jpgb_encoder_last_timing(const jpgb_encoder *enc, float ms[JPGB_N_STAGES]) {
    if (!enc || !enc->have_timing) return JPGB_ERR_BAD_PARAMS;
    std::memcpy(ms, enc->last_ms, sizeof(enc->last_ms));
    return JPGB_OK;
}
uint32_t jpgb_encoder_last_launch_count(const jpgb_encoder *enc) { return enc ? enc->launches : 0; }

int jpgb_build_header(const jpgb_params *p, uint8_t *buf, size_t cap, size_t *len) {
    if (!p || !len) return JPGB_ERR_BAD_PARAMS;
    Plan plan;
    const int rc = plan.build(*p);
    if (rc != JPGB_OK) return rc;
    HuffTable huff[2][2];
    default_huffman_tables(huff);
    std::vector<uint8_t> h = plan.prefix;
    plan.frame_header(huff, h);
    h.insert(h.end(), plan.scans[0].sos.begin(), plan.scans[0].sos.end());
    *len = h.size();
    if (buf) std::memcpy(buf, h.data(), std::min(cap, h.size()));
    return JPGB_OK;
}

int jpgb_optimized_huffman_table(const uint32_t freq[257], uint8_t length[16], uint8_t values[256], uint32_t *n_values) {
    if (!freq || !length || !values || !n_values) return JPGB_ERR_BAD_PARAMS;
    HuffTable t;
    if (!t.set_optimized(freq)) return JPGB_ERR_HUFFMAN;
    std::memcpy(length, t.length, 16);
    std::memcpy(values, t.values.data(), t.values.size());
    *n_values = (uint32_t)t.values.size();
    return JPGB_OK;
}

int jpgb_optimized_huffman_tables_device(jpgb_encoder *enc, const uint32_t *freq, uint32_t n, int ac, uint8_t *lengths, uint8_t *values,
                                         uint32_t *n_values, uint32_t *words, int *status) {
    if (!enc) return JPGB_ERR_BAD_PARAMS;
    if (!freq || !lengths || !values || !n_values || !words || !status || n == 0) return fail(enc, JPGB_ERR_BAD_PARAMS, "null argument");
    CK(cudaSetDevice(enc->device), "cudaSetDevice");
    cudaStream_t st = enc->stream;
    DevBuf d_hist, d_words, d_dht, d_len, d_bad;
    std::vector<uint8_t> dht((size_t)n * 277);
    std::vector<uint32_t> len(n), bad(n);
    cudaError_t e = d_hist.reserve((size_t)n * 257 * 4);
    if (e == cudaSuccess) e = d_words.reserve((size_t)n * 1024);
    if (e == cudaSuccess) e = d_dht.reserve((size_t)n * 277);
    if (e == cudaSuccess) e = d_len.reserve((size_t)n * 4);
    if (e == cudaSuccess) e = d_bad.reserve((size_t)n * 4);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_hist.p, freq, (size_t)n * 257 * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = launch_build_single_tables(d_hist.as<uint32_t>(), n, ac, d_words.as<uint32_t>(), d_dht.as<uint8_t>(), d_len.as<uint32_t>(), d_bad.as<uint32_t>(), st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(words, d_words.p, (size_t)n * 1024, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dht.data(), d_dht.p, dht.size(), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(len.data(), d_len.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(bad.data(), d_bad.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail_cuda(enc, e, "device table build");
    for (uint32_t i = 0; i < n; ++i) {
        status[i] = bad[i] ? JPGB_ERR_HUFFMAN : JPGB_OK;
        n_values[i] = bad[i] ? 0 : len[i] - 21;
        std::memcpy(lengths + (size_t)i * 16, dht.data() + (size_t)i * 277 + 5, 16);
        std::memcpy(values + (size_t)i * 256, dht.data() + (size_t)i * 277 + 21, 256);
    }
    return JPGB_OK;
}

const char *jpgb_version(void) { return "jpeg-encoder_b200 0.1 (sm_100a; parity target: jpeg-encoder 0.7.0)"; }

} // extern "C"
