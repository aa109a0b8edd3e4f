// Optimized Huffman tables on the device: HuffmanTable::new_optimized (Annex K.2, /root/reference/src/huffman.rs:99-221),
// create_lookup_table (:240-288) and the DHT segments of the frame header (src/writer.rs:253-269), for every image of
// a batch at once. The reference builds them on one thread from the symbol histogram of optimize_huffman_table
// (src/encoder.rs:1086-1200); here one CTA per image does it, one warp per table, straight from the histogram the
// histogram kernel left in HBM -- no host round trip in the middle of the pipeline.
//
// The result must be the reference's table bit for bit (the DHT bytes are part of the file), so the selection rule of
// Figure K.1 is kept exactly: the least frequency wins, ties go to the LARGEST symbol index (the reference scans upward
// with `<=`), v2 is chosen the same way among the rest, the merged frequency lives on at v1. What the reference keeps
// as linked lists (`others`) is kept here as tree membership: every symbol knows the root of its tree, and a merge
// adds one to the code size of every member of both trees -- the same increments the list walk makes.
#include "kernels.h"

namespace jpgb {
namespace {

constexpr int kSym = 257;      // 256 symbols + the reserved code point (src/encoder.rs:1092-1095)
constexpr int kPerLane = 9;    // ceil(257 / 32): entry i of the packed symbol list belongs to lane i % 32
constexpr unsigned kNone = 0xFFFFFFFFu;

struct TableSmem {
    uint32_t freq[kSym + 31];
    uint16_t root[kSym + 31], sym[kSym + 31]; // K.1 runs on the symbols that occur, packed to the front
    uint8_t csz[kSym + 31];                   // code size of packed entry i
    uint16_t parent[2 * (kSym + 31)];         // merge tree: leaves 0..n-1 (the packed entries), inner nodes from n; 0xFFFF = no parent
    uint8_t codesize[kSym + 31];              // ... and of symbol s
    uint8_t values[256];
    uint8_t len[16];      // BITS after Figure K.3
    uint32_t n_values;
    uint32_t start[34];   // first position (in `values`) of code size s
    uint32_t counter[34];
    uint32_t first_code[17], first_pos[17];
};

// One warp builds one table. `freq_in` = 257 counts (entry 256 is forced to 1). Writes the kernel-format words
// ((code length + value size) << 27 | code << size) and the DHT segment; returns false if a code does not fit.
__device__ bool build_one(TableSmem &S, const uint32_t *freq_in, bool ac, int table_id, uint32_t *words, uint8_t *dht, uint32_t &dht_len) {
    const int lane = threadIdx.x & 31;
    // Only symbols that occur take part in Figure K.1 (a zero frequency is never selected): they are packed to the
    // front in symbol order, so "the largest index among equal frequencies" is still the largest symbol.
    unsigned n = 0;
    for (int base = 0; base < kSym + 31; base += 32) {
        const int sym = base + lane;
        const uint32_t f = sym < 256 ? freq_in[sym] : (sym == 256 ? 1u : 0u);
        const unsigned have = __ballot_sync(0xffffffffu, f != 0);
        if (f) {
            const unsigned at = n + __popc(have & ((1u << lane) - 1u));
            S.freq[at] = f;
            S.sym[at] = (uint16_t)sym;
            S.root[at] = (uint16_t)at;
        }
        if (sym < kSym + 31) S.codesize[sym] = 0;
        n += __popc(have);
    }
    for (int i = lane; i < 2 * (kSym + 31); i += 32) S.parent[i] = 0xFFFF;
    __syncwarp();
    // every lane keeps the frequencies of its (at most nine) entries in registers: entry i belongs to lane i % 32
    uint32_t f[kPerLane];
#pragma unroll
    for (int j = 0; j < kPerLane; ++j) f[j] = (unsigned)(lane + 32 * j) < n ? S.freq[lane + 32 * j] : 0u;
    // least non-zero frequency among the lane's entries, ties to the largest index; `skip` is left out
    auto lane_least = [&](unsigned skip, uint32_t &fo, unsigned &io) {
        fo = kNone;
        io = kNone;
#pragma unroll
        for (int j = 0; j < kPerLane; ++j) {
            const unsigned i = lane + 32 * j;
            if (f[j] != 0 && i != skip && f[j] <= fo) {
                fo = f[j];
                io = i;
            }
        }
    };
    uint32_t lf;
    unsigned li;
    lane_least(kNone, lf, li);
    bool ok = true;
    // Figure K.1. What the reference keeps as linked lists (`others`, every member's code size bumped at each merge) is
    // kept here as the merge tree itself: entry i currently stands for tree node root[i]; a merge hangs the two nodes
    // under a new one. A symbol's code size is the depth of its leaf, read off the parent links afterwards.
    unsigned next_node = n;
    for (;;) {
        const uint32_t m1 = __reduce_min_sync(0xffffffffu, lf);
        if (m1 == kNone) break;
        const unsigned v1 = __reduce_max_sync(0xffffffffu, lf == m1 ? li : 0u); // indices of equal frequency: the largest
        // v2: the same rule over everything but v1; only v1's lane has to look again
        uint32_t lf2 = lf;
        unsigned li2 = li;
        if ((v1 & 31) == (unsigned)lane) lane_least(v1, lf2, li2);
        const uint32_t m2 = __reduce_min_sync(0xffffffffu, lf2);
        if (m2 == kNone) break;
        const unsigned v2 = __reduce_max_sync(0xffffffffu, lf2 == m2 ? li2 : 0u);
        if (lane == 0) {
            S.parent[S.root[v1]] = (uint16_t)next_node;
            S.parent[S.root[v2]] = (uint16_t)next_node;
            S.root[v1] = (uint16_t)next_node; // v1 now stands for the merged tree
        }
        ++next_node;
        // the merged frequency lives on at v1, v2 leaves the game: their owners update their registers and look again
        const bool own1 = (v1 & 31) == (unsigned)lane, own2 = (v2 & 31) == (unsigned)lane;
        if (own1 || own2) {
#pragma unroll
            for (int j = 0; j < kPerLane; ++j) {
                if (own1 && (int)(v1 >> 5) == j) f[j] = m1 + m2;
                if (own2 && (int)(v2 >> 5) == j) f[j] = 0;
            }
            lane_least(kNone, lf, li);
        }
    }
    __syncwarp();
    for (unsigned i = lane; i < n; i += 32) { // depth of leaf i
        unsigned d = 0, node = i;
        while (S.parent[node] != 0xFFFF && d < 40) node = S.parent[node], ++d;
        if (d > 32) ok = false; // the reference panics on its fixed arrays
        S.csz[i] = (uint8_t)d;
    }
    __syncwarp();
    for (unsigned i = lane; i < n; i += 32) S.codesize[S.sym[i]] = S.csz[i]; // back to symbol order
    __syncwarp();
    if (n < 2) return false; // nothing but the reserved code point: no code at all (the reference indexes out of bounds and panics)
    ok = __all_sync(0xffffffffu, ok);
    if (!ok) return false;

    // Figure K.2: number of codes of each size; K.3: no code longer than 16 bits; drop the reserved code point
    if (lane == 0) {
        uint8_t bits[33];
        for (int i = 0; i <= 32; ++i) bits[i] = 0;
        for (int i = 0; i < kSym; ++i)
            if (S.codesize[i]) ++bits[S.codesize[i]];
        uint32_t pos = 0;
        for (int s = 0; s <= 33; ++s) { // positions by ORIGINAL code size (Figure K.4 sorts by it)
            S.start[s] = pos;
            S.counter[s] = 0;
            if (s >= 1 && s <= 32) pos += bits[s];
        }
        int i = 32;
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
        --bits[i];
        uint32_t code = 0, k = 0;
        for (int l = 1; l <= 16; ++l) { // Figures C.1 - C.3: first code and first position of every length
            S.len[l - 1] = bits[l];
            S.first_code[l] = code;
            S.first_pos[l] = k;
            code = (code + bits[l]) << 1;
            k += bits[l];
        }
        S.n_values = k;
    }
    __syncwarp();
    // Figure K.4: symbols 0..255 by code size, then by value. Rank inside a size class = symbols of that size with a
    // smaller value: counted 32 symbols at a time (match_any groups the lanes of equal size).
    for (int base = 0; base < 256; base += 32) {
        const int sym = base + lane;
        const unsigned cs = S.codesize[sym];
        const unsigned peers = __match_any_sync(0xffffffffu, cs);
        const unsigned before = __popc(peers & ((1u << lane) - 1u));
        if (cs) {
            const unsigned pos = S.start[cs] + S.counter[cs] + before;
            if (pos < 256) S.values[pos] = (uint8_t)sym;
        }
        __syncwarp();
        if (cs && before + 1 == (unsigned)__popc(peers)) S.counter[cs] += __popc(peers); // the group's last lane
        __syncwarp();
    }
    // lookup: symbol values[k] gets the k-th code in order of length
    for (int i = lane; i < 256; i += 32) words[i] = 0; // a symbol without a code: only its value bits are written (Q18)
    __syncwarp();
    const uint32_t nv = S.n_values;
    for (uint32_t k = lane; k < nv; k += 32) {
        int l = 1;
        while (l < 16 && k >= S.first_pos[l] + S.len[l - 1]) ++l;
        const uint32_t code = S.first_code[l] + (k - S.first_pos[l]);
        const unsigned sym = S.values[k];
        if (!ac && sym > 15) continue; // DC categories are 0..15
        const unsigned z = ac ? (sym & 15u) : sym;
        if ((unsigned)l + z > 31 || (((unsigned long long)code << z) >> 27)) ok = false;
        words[sym] = ((uint32_t)(l + z) << 27) | (code << z);
    }
    // symbols without a code still carry their value size in the length field
    __syncwarp();
    for (int i = lane; i < 256; i += 32) {
        if (!ac && i > 15) continue;
        if (words[i] == 0) {
            const unsigned z = ac ? (i & 15u) : (unsigned)i;
            words[i] = z << 27;
        }
    }
    // DHT segment (writer.rs:253-269)
    if (lane == 0) {
        dht[0] = 0xFF;
        dht[1] = 0xC4;
        const uint32_t seg = 2 + 1 + 16 + nv;
        dht[2] = (uint8_t)(seg >> 8);
        dht[3] = (uint8_t)seg;
        dht[4] = (uint8_t)(((ac ? 1 : 0) << 4) | table_id);
        dht_len = 5 + 16 + nv;
    }
    for (int i = lane; i < 16; i += 32) dht[5 + i] = S.len[i];
    for (uint32_t i = lane; i < nv; i += 32) dht[21 + i] = S.values[i];
    __syncwarp();
    return __all_sync(0xffffffffu, ok);
}

// grid = images; block = 128 threads = one warp per (table, class). hist: [image][table][dc|ac][257].
// huff: [image][table][dc|ac][256] words, preset with the default tables (tables that are not optimized keep them).
// Header of image i = head (SOI .. DQT) + the DHT segments + tail (DRI, first SOS), at hdr + i * hdr_stride.
__global__ void __launch_bounds__(128) build_tables_kernel(const uint32_t *__restrict__ hist, int hist_per_image, int n_tables, uint32_t *huff,
                                                           const uint8_t *__restrict__ head, uint32_t head_len, const uint8_t *__restrict__ tail,
                                                           uint32_t tail_len, uint8_t *hdr, uint32_t hdr_stride, uint32_t *hdr_len,
                                                           unsigned long long *status) {
    __shared__ TableSmem S[4];
    __shared__ uint8_t dht[4][5 + 16 + 256];
    __shared__ uint32_t dht_len[4];
    __shared__ uint32_t words[4][256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned long long img = blockIdx.x;
    const int t = warp >> 1, cls = warp & 1;
    if (lane == 0) dht_len[warp] = 0;
    if (t < n_tables) {
        const uint32_t *f = hist + (hist_per_image ? img : 0) * (2 * 2 * 257) + (size_t)(t * 2 + cls) * 257;
        const bool ok = build_one(S[warp], f, cls == 1, t, words[warp], dht[warp], dht_len[warp]);
        if (!ok && lane == 0) atomicOr(status + kStatFlags, kFlagHuffmanLong);
        uint32_t *dst = huff + img * kHuffWordsPerImage + (size_t)(t * 2 + cls) * 256;
        for (int i = lane; i < 256; i += 32) dst[i] = words[warp][i];
    }
    __syncthreads();
    uint8_t *out = hdr + img * hdr_stride;
    uint32_t pos = head_len;
    for (uint32_t i = threadIdx.x; i < head_len; i += blockDim.x) out[i] = head[i];
    for (int w = 0; w < 4; ++w) {
        const uint32_t n = dht_len[w];
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) out[pos + i] = dht[w][i];
        pos += n;
    }
    for (uint32_t i = threadIdx.x; i < tail_len; i += blockDim.x) out[pos + i] = tail[i];
    if (threadIdx.x == 0) hdr_len[img] = pos + tail_len;
}

// test / diagnostics: one warp per histogram, every histogram on its own
__global__ void __launch_bounds__(128) build_single_tables_kernel(const uint32_t *__restrict__ hist, unsigned n, int ac, uint32_t *words_out,
                                                                  uint8_t *dht_out, uint32_t *dht_len_out, uint32_t *bad) {
    __shared__ TableSmem S[4];
    __shared__ uint8_t dht[4][5 + 16 + 256];
    __shared__ uint32_t dht_len[4];
    __shared__ uint32_t words[4][256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned i = blockIdx.x * 4 + warp;
    if (i >= n) return;
    if (lane == 0) dht_len[warp] = 0;
    __syncwarp();
    const bool ok = build_one(S[warp], hist + (size_t)i * 257, ac != 0, 0, words[warp], dht[warp], dht_len[warp]);
    __syncwarp();
    if (lane == 0) {
        bad[i] = ok ? 0u : 1u;
        dht_len_out[i] = ok ? dht_len[warp] : 0u;
    }
    for (int k = lane; k < 256; k += 32) words_out[(size_t)i * 256 + k] = ok ? words[warp][k] : 0u;
    for (unsigned k = lane; k < 5 + 16 + 256; k += 32) dht_out[(size_t)i * 277 + k] = ok && k < dht_len[warp] ? dht[warp][k] : 0;
}

} // namespace

cudaError_t launch_build_single_tables(const uint32_t *hist, uint32_t n, int ac, uint32_t *words, uint8_t *dht, uint32_t *dht_len, uint32_t *bad,
                                       cudaStream_t stream) {
    build_single_tables_kernel<<<(n + 3) / 4, 128, 0, stream>>>(hist, n, ac, words, dht, dht_len, bad);
    return cudaGetLastError();
}

cudaError_t launch_build_tables(const uint32_t *hist, int hist_per_image, int n_tables, uint32_t n_images, uint32_t *huff, const uint8_t *head,
                                uint32_t head_len, const uint8_t *tail, uint32_t tail_len, uint8_t *hdr, uint32_t hdr_stride, uint32_t *hdr_len,
                                unsigned long long *status, cudaStream_t stream) {
    build_tables_kernel<<<n_images, 128, 0, stream>>>(hist, hist_per_image, n_tables, huff, head, head_len, tail, tail_len, hdr, hdr_stride, hdr_len,
                                                     status);
    return cudaGetLastError();
}

} // namespace jpgb
