// Stage B: quantized coefficients -> JFIF bytes, entirely on the device.
//
// Replaces the reference's serial entropy coder and bit writer
//   write_dc / write_ac_block / write_block / get_code      src/writer.rs:331-388, 455-470
//   write_bits / flush / finalize_bit_buffer (0xFF stuffing) src/writer.rs:138-202
//   the MCU / block walks with restart bookkeeping           src/encoder.rs:727-804, 823-861, 885-972
//   optimize_huffman_table's symbol histogram                src/encoder.rs:1086-1200
//
// Vocabulary. A *visit* is one block coded in one scan. A *segment* is the run of visits between two restart
// points of one scan (one segment per scan when restarts are off); its bits start byte-aligned and end padded
// with 1-bits. A *chunk* is the code of <= chunk_T consecutive visits of one segment: one bit string. A *group*
// is the set of scans that walk the same blocks (a component's DC scan and AC bands in progressive mode).
// The *unstuffed stream* is the complete file before 0xFF stuffing: per image the header, then per segment its
// lead (RSTn marker or the next scan's SOS) and its data bytes, then EOI. `raw_mask` flags header/marker bytes
// so that the stuffing pass leaves their 0xFF alone.
//
//   encode_chunks_kernel persistent; a CTA takes a chunk, stages its blocks once (the coefficient buffer is laid
//                        out in scan order, so they are one contiguous run), codes every visit for every scan of
//                        the group, prefix-sums the bit counts inside the CTA and writes each scan's chunk as one
//                        contiguous bit string into `pool` (+ its bit count)
//   [exclusive scan]     bit position of every chunk (one element per chunk, not per block)
//   segment_len_kernel   segment -> lead + ceil(bits/8) + tail bytes
//   [exclusive scan]     byte position of every segment in the unstuffed stream
//   positions_kernel     small jobs: the three steps above (or the last two) in one single-CTA launch
//   segment_lead_kernel  writes headers / RSTn / SOS / EOI, sets raw_mask; zeroes the stream words that two chunks
//                        share (the stream is never cleared as a whole)
//   place_chunks_kernel  streams every chunk from `pool` to its bit position (funnel shift): stores the words a chunk
//                        owns, ORs into the shared ones; pad bits at segment end
//   count_ff_kernel      4 KB piece of the stream -> number of data 0xFF bytes
//   [exclusive scan]     skipped for short streams (the scatter CTAs add the counts up themselves)
//   stuff_scatter_kernel copies every byte to its final place, inserting 0x00 after data 0xFF; extra CTAs work out
//                        the file offsets and a strip's piece offsets
//   histogram_kernel     optimized tables: symbol statistics of every image (same walk as the coder)

#include "kernels.h"

namespace jpgb {
namespace {

__device__ __forceinline__ int find_scan_by_seg(const DevPlan &P, unsigned s) {
    int lo = 0, hi = P.n_scans - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (P.scans[mid].seg_base <= s) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}
__device__ __forceinline__ int find_scan_by_chunk(const DevPlan &P, unsigned c) {
    int lo = 0, hi = P.n_scans - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (P.scans[mid].chunk_base <= c) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// get_code, writer.rs:455-470: size = bit length of |v|, bits = low `size` bits of (v - (v<0))
__device__ __forceinline__ void value_code(int v, int &size, uint32_t &bits) {
    const int a = v < 0 ? -v : v;
    int top; // index of the highest set bit, -1 for 0
    asm("bfind.u32 %0, %1;" : "=r"(top) : "r"(a));
    size = top + 1;
    uint32_t mask;
    asm("bmsk.clamp.b32 %0, 0, %1;" : "=r"(mask) : "r"(size));
    bits = (uint32_t)(v + (v >> 31)) & mask;
}

__device__ __forceinline__ unsigned nonzero16x2(unsigned x) {
    unsigned r;
    asm("min.u16x2 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(0x00010001u));
    return r;
}

// Bit sink of one visit. Codes are packed MSB-first into 32-bit words; word j of the visit with index i inside
// its chunk goes to scratch[j * T + i] (the lanes of a warp write one contiguous line per word). The scratch of a
// coding CTA is T x kSlotWords words that it overwrites chunk after chunk, so it stays in L2. Where the bits
// belong in the chunk is decided after all visits of the chunk are coded, from the prefix sum of their lengths.
template <int T>
struct BitSink {
    unsigned long long acc = 0;
    int n = 0;
    unsigned off = 0; // bytes written so far, scaled by the tile stride
    uint32_t *slot0;

    __device__ __forceinline__ BitSink(uint32_t *scratch, int visit) : slot0(scratch + visit) {}
    __device__ __forceinline__ void put(uint32_t code, int len) { // len <= 31, n < 32 on entry
        acc = (acc << len) | code;
        n += len;
        if (n >= 32) {
            n -= 32;
            *reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(slot0) + off) = (uint32_t)(acc >> n);
            off += T * 4;
        }
    }
    __device__ __forceinline__ unsigned finish() {
        if (n > 0) *reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(slot0) + off) = (uint32_t)(acc << (32 - n)); // left-aligned tail
        return off / (T * 4) * 32 + n;
    }
};

// Table words as the host uploads them (api.cu): for the symbol (run << 4 | size), or the DC category
// `size`, (code_length + size) << 27 | code << size: OR-ing the value bits in gives the whole
// write_bits argument of huffman_encode_value (writer.rs:320-329). A symbol without a code is
// size << 27: only the value bits are written (release-build behaviour of the reference, SURVEY.md Q18).
constexpr uint32_t kCodeBits = 0x07FFFFFFu;

constexpr int kStageStride = 72;    // int16 per staged block: 128 B of coefficients + 16 B pad (128-bit rows stay conflict-free)
constexpr int kAsmWordsProg = 3072; // progressive: words of the chunk assembly buffer (the staged blocks stay live across the group's scans)

// Zero runs longer than 15 in front of a non-zero coefficient take one ZRL symbol per 16 zeros (writer.rs:369-373).
// `m` has bit k set for every non-zero coefficient k of the band [first_ac, se]. Returns the positions of the
// zeros that end such a group of 16: start of the run + 15, + 31, + 47.
__device__ __forceinline__ unsigned long long zrl_markers(unsigned long long m, int first_ac) {
    const unsigned long long z = m | (1ull << (first_ac - 1)); // the position in front of the band ends "run 0"
    // s16 / s32 / s48: bit p is set when z has a set bit among the 16 / 32 / 48 positions p, p - 1, ...
    unsigned long long s = z;
    s |= s << 1;
    s |= s << 2;
    s |= s << 4;
    const unsigned long long s16 = s | (s << 8);
    const unsigned long long s32 = s16 | (s16 << 16);
    const unsigned long long s48 = s32 | (s16 << 32);
    // a zero exactly 16 / 32 / 48 positions behind the nearest set bit below it
    unsigned long long marks = ((z << 16) & ~s16) | ((z << 32) & ~s32) | ((z << 48) & ~s48);
    // ... and only in front of a non-zero coefficient (zeros at the end of the band become EOB, writer.rs:383-385)
    const int top = 63 - __clzll((long long)m); // -1 when the band is empty: the shift below then clears everything
    marks &= top > 0 ? (~0ull >> (64 - top)) : 0ull;
    return marks;
}

// write_ac_block restricted to the band (writer.rs:354-388) for one visit. The positions to code come as two
// bit-reversed masks: coefficient k of the half [BASE, BASE + 32) is bit 31 - (k - BASE), so the next one in
// zig-zag order is the highest set bit (one FLO, no bit reversal). One iteration per set bit: a non-zero
// coefficient, or a ZRL marker (zrl_markers): a zero 15 positions after the start of its run, for which the same
// arithmetic yields the symbol 0xF0 with no value bits (writer.rs:369-373), so the loop has no ZRL branch.
template <int BASE, int T>
__device__ __forceinline__ void code_half(unsigned m, int &next, unsigned c_shared, const uint32_t *__restrict__ tab, BitSink<T> &sink) {
#pragma unroll 1
    while (m) {
        int p;
        asm("bfind.u32 %0, %1;" : "=r"(p) : "r"(m));
        unsigned bit;
        asm("bmsk.clamp.b32 %0, %1, 1;" : "=r"(bit) : "r"(p));
        m ^= bit;
        const int k = BASE + 31 - p;
        int v;
        asm("ld.shared.s16 %0, [%1];" : "=r"(v) : "r"(c_shared + 2 * k));
        const int run = k - next; // next = first position of the current zero run; <= 15 thanks to the ZRL markers
        next = k + 1;
        int size;
        uint32_t bits;
        value_code(v, size, bits);
        const uint32_t e = (tab + run * 16)[size]; // (code length + size) << 27 | code << size
        sink.put((e & kCodeBits) | bits, (int)(e >> 27));
    }
}
template <int T>
__device__ __forceinline__ void code_nonzeros(unsigned lo_rev, unsigned hi_rev, int first_ac, int se, const int16_t *__restrict__ c,
                                              const uint32_t *__restrict__ tab, BitSink<T> &sink) {
    int next = first_ac;
    const unsigned c_shared = (unsigned)__cvta_generic_to_shared(c);
    code_half<0, T>(lo_rev, next, c_shared, tab, sink);
    code_half<32, T>(hi_rev, next, c_shared, tab, sink);
    if (next <= se) { // the band ends in zeros: EOB (writer.rs:383-385)
        const uint32_t e = tab[0];
        sink.put(e & kCodeBits, (int)(e >> 27));
    }
}

// what thread 0 works out for the CTA's next chunk
struct __align__(16) ItemInfo {
    unsigned long long img, blk0, chunk_index0; // first block of the chunk (global); img * chunks_per_image + seg * cps + chunk
    unsigned v_in_seg0, n_valid, group;
    int done;
};

// shared-memory carve-up of the coding CTA
template <int T, bool FULL>
struct CoderSmem {
    static constexpr int kCoefBytes = T * kStageStride * 2;
    static constexpr int kAsmWords = FULL ? kCoefBytes / 4 : kAsmWordsProg; // FULL: the staged blocks are dead once coded -> reuse
    static constexpr int oAsm = FULL ? 0 : kCoefBytes;
    // per visit: band mask (8 B), DC code word (4 B), table | valid (4 B) live in the 16 pad bytes behind its staged block
    static constexpr int oAc = kCoefBytes + (FULL ? 0 : kAsmWordsProg * 4);
    static constexpr int oDc = oAc + 2048;  // AC tables: 2 x 256 packed words
    static constexpr int oSlot = oDc + 256; // DC tables: 2 x 16 x {code << size, length}
    static constexpr int oBin = oSlot + 128; // per MCU slot: table | distance to the DC predecessor << 8 | first of its component << 16 | component << 24;
                                             // words kMaxSlots .. + 3: each component's DC predictor at the start of a segment (kStatDcPred)
    static_assert(kMaxSlots + 4 <= 32, "the DC predictors follow the slot words");
    static constexpr int oNb = oBin + 256;
    static constexpr int oOrder = oNb + T * 4;
    static constexpr int oWsum = oOrder + T * 2;
    static constexpr int oItem = oWsum + 64;
    static constexpr int kBytes = oItem + 2 * 64; // two ItemInfo: the chunk being coded and the next one
};

// write_dc + write_ac_block for one chunk after the other (persistent CTAs, a ticket per chunk):
//  1. the chunk's blocks -- one contiguous run of the scan-ordered coefficient buffer -- are copied into shared
//     memory with coalesced 16-byte cp.async; every thread then owns visit `tid`: the 64-bit mask of its non-zero
//     coefficients and its DC difference (the predecessor is a fixed distance back in the same run);
//  then for every scan of the group (one, except in progressive mode: DC scan and AC bands share the staging):
//  2. band mask + ZRL markers; the CTA sorts its visits by their number of symbols (counting sort);
//  3. thread t codes the visit of rank t -- the lanes of a warp then run nearly the same number of iterations of
//     the per-coefficient loop, which is where the time goes -- into the CTA's L2-resident scratch;
//  4. prefix sum of the visits' bit counts, then every thread shifts its visit's words to their place in the
//     chunk's bit string, assembled in shared memory and written to `pool` with coalesced 128-bit stores.
// Resident CTAs per SM the register allocation aims at. The sequential coder needs 51 registers, which the allocation
// granularity turns into 9 CTAs of 128 threads; capped at 48 (no spills) it is 10, as many as the shared memory allows:
// 2.91 -> 2.80 ms on C3. The progressive variant (62 registers, 8 CTAs) spills when pushed to 10 (C5: 0.75 -> 0.78 ms) and
// gains nothing at 9 (56 registers, no spill: 0.76 ms): it is left alone.
__host__ __device__ constexpr int coder_min_ctas(int T, bool full) { return full && T >= 128 ? 1280 / T : 1024 / T; } // 48 / 64 registers

// FULL: every scan of the plan covers the whole block (baseline and sequential modes).
template <int T, bool FULL>
__global__ void __launch_bounds__(T, coder_min_ctas(T, FULL)) encode_chunks_kernel(const __grid_constant__ EntropyBuffers b, const __grid_constant__ DevPlan P,
                                                          unsigned long long n_items) {
    using L = CoderSmem<T, FULL>;
    extern __shared__ __align__(16) unsigned char smem[];
    int16_t *coef = reinterpret_cast<int16_t *>(smem);
    uint32_t *asmbuf = reinterpret_cast<uint32_t *>(smem + L::oAsm);
    uint32_t *ac_tab = reinterpret_cast<uint32_t *>(smem + L::oAc);
    uint2 *dc_tab = reinterpret_cast<uint2 *>(smem + L::oDc);
    uint32_t *slot_tab = reinterpret_cast<uint32_t *>(smem + L::oSlot);
    uint32_t *bin = reinterpret_cast<uint32_t *>(smem + L::oBin);
    uint32_t *nbv = reinterpret_cast<uint32_t *>(smem + L::oNb);
    // the 16 bytes behind the 128 coefficient bytes of visit v: {band mask lo, band mask hi, DC code word, table | valid << 8}
    auto visit_meta = [&](int v) { return reinterpret_cast<uint4 *>(smem + v * (kStageStride * 2) + 128); };
    uint16_t *order = reinterpret_cast<uint16_t *>(smem + L::oOrder);
    uint32_t *wsum = reinterpret_cast<uint32_t *>(smem + L::oWsum); // [0..7] warp sums, [8] pool offset of the chunk
    ItemInfo *items = reinterpret_cast<ItemInfo *>(smem + L::oItem);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *scratch = b.scratch + (size_t)blockIdx.x * (T * kSlotWords);
    long long tab_img = -1; // whose Huffman tables the shared copy holds
    for (int i = tid; i < 64; i += T) bin[i] = 0;
    if (tid < kMaxSlots)
        slot_tab[tid] = (unsigned)P.comp_tbl[P.slot_comp[tid]] | (unsigned)P.slot_back[tid] << 8 | (unsigned)P.slot_first[tid] << 16 |
                        (unsigned)(uint8_t)P.slot_comp[tid] << 24;
    else if (tid < kMaxSlots + 4) slot_tab[tid] = (unsigned)(int)(int16_t)(b.status[kStatDcPred] >> (16 * (tid - kMaxSlots)));
    // Work items are handed out by a ticket counter. Thread 0 runs one chunk ahead: while the CTA codes chunk i it
    // requests the ticket of chunk i + 2 and works out where chunk i + 1 lies, so neither the round trip of the
    // atomic nor the arithmetic is ever waited for.
    auto decode = [&](unsigned long long ticket, ItemInfo &it) {
        it.done = ticket >= n_items;
        if (it.done) return;
        unsigned long long img;
        unsigned r;
        if ((ticket >> 32) == 0) {
            unsigned q;
            divmod((unsigned)ticket, P.div_items, q, r);
            img = q;
        } else {
            img = ticket / P.items_per_image;
            r = (unsigned)(ticket - img * P.items_per_image);
        }
        int g = 0;
        while (g + 1 < P.n_groups && r >= P.groups[g + 1].item_base) ++g;
        const DevGroup &G = P.groups[g];
        unsigned seg, chunk;
        divmod(r - G.item_base, G.div_cps, seg, chunk);
        const unsigned long long seg_start = (unsigned long long)seg * G.seg_visits;
        const unsigned long long v0 = seg_start + (unsigned long long)chunk * T;
        unsigned long long seg_end = seg_start + G.seg_visits;
        if (seg_end > G.n_visits) seg_end = G.n_visits;
        it.img = img;
        it.group = (unsigned)g;
        it.v_in_seg0 = chunk * T;
        it.n_valid = v0 < seg_end ? (unsigned)(seg_end - v0 < (unsigned long long)T ? seg_end - v0 : T) : 0u;
        it.blk0 = img * P.blocks_per_image + G.block_base + v0;
        it.chunk_index0 = img * P.chunks_per_image + (r - G.item_base);
    };
    unsigned long long next_ticket = 0;
    if (tid == 0) {
        decode(atomicAdd(b.status + kStatTicket, 1ull), items[0]);
        next_ticket = atomicAdd(b.status + kStatTicket, 1ull);
    }

    for (unsigned round = 0;; ++round) {
        __syncthreads(); // the previous chunk is completely written out; items[round & 1] is ready
        const ItemInfo it = items[round & 1];
        if (it.done) break;
        if (tid == 0) {
            decode(next_ticket, items[(round & 1) ^ 1]);
            next_ticket = atomicAdd(b.status + kStatTicket, 1ull);
        }
        if (it.n_valid == 0) { // a chunk slot past the end of a short last segment: it exists only as an (empty) descriptor
            for (int j = tid; j < P.spg; j += T) {
                const unsigned long long ci = it.chunk_index0 + P.scans[it.group + j * P.n_groups].chunk_base;
                b.chunk_bits[ci] = 0;
                b.chunk_pool[ci] = 0;
            }
            continue;
        }
        const DevGroup &G = P.groups[it.group];
        const bool valid = (unsigned)tid < it.n_valid;

        // Huffman tables of this image (or the shared default ones) -> shared memory, when they change
        const long long want_tab = b.huff_per_image ? (long long)it.img : 0;
        if (want_tab != tab_img) {
            const uint32_t *set = b.huff + (size_t)want_tab * kHuffWordsPerImage;
            for (int i = tid; i < 512; i += T) { // table 0 / 1, AC
                ac_tab[i] = __ldg(set + (i >> 8) * 512 + 256 + (i & 255));
            }
            if (tid < 32) { // DC categories 0..15
                const uint32_t e = __ldg(set + (tid >> 4) * 512 + (tid & 15));
                dc_tab[tid] = make_uint2(e & kCodeBits, e >> 27);
            }
            tab_img = want_tab;
        }

        // ---- 1. stage the chunk's blocks: n_valid * 128 contiguous bytes ----
        const int16_t *src_blocks = b.coef + it.blk0 * 64;
        {
            const unsigned pieces = it.n_valid * 8;
            const char *g = reinterpret_cast<const char *>(src_blocks) + (size_t)tid * 16;
            const unsigned d = (unsigned)__cvta_generic_to_shared(coef) + (tid >> 3) * (kStageStride * 2) + (tid & 7) * 16;
            if (it.n_valid == T) { // a full chunk: no bounds to test
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + k * (T / 8) * (kStageStride * 2)), "l"(g + k * T * 16) : "memory");
            } else {
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if ((unsigned)(tid + k * T) < pieces)
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + k * (T / 8) * (kStageStride * 2)), "l"(g + k * T * 16) : "memory");
            }
            asm volatile("cp.async.wait_all;" ::: "memory");
        }
        __syncthreads();

        // mask of all non-zero coefficients of this thread's block, its DC difference, its table
        unsigned long long m_all = 0;
        int dcdiff = 0, tbl = 0;
        if (valid) {
            const uint4 *mine = reinterpret_cast<const uint4 *>(coef + tid * kStageStride);
            unsigned m_lo = 0, m_hi = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                const uint4 q = mine[w];
                // per 16-bit half min(x, 1) = (x != 0); dp2a weighs the two halves 1 and 2 and accumulates
                unsigned byte = __dp2a_lo(nonzero16x2(q.x), 0x0201u, 0u);
                byte = __dp2a_lo(nonzero16x2(q.y), 0x0804u, byte);
                byte = __dp2a_lo(nonzero16x2(q.z), 0x2010u, byte);
                byte = __dp2a_lo(nonzero16x2(q.w), 0x8040u, byte);
                if (w < 4) m_lo |= byte << (8 * w);
                else m_hi |= byte << (8 * (w - 4));
            }
            m_all = (((unsigned long long)m_hi << 32) | m_lo) & ~1ull;
            // DC predictor (encoder.rs:753-756, 838, 900): the previous block of the component in scan order, 0 at a restart
            const unsigned v_in_seg = it.v_in_seg0 + tid;
            unsigned unit = v_in_seg, slot = 0;
            if (G.bpu > 1) divmod(v_in_seg, G.div_bpu, unit, slot);
            const unsigned sinfo = G.comp < 0 ? slot_tab[slot] : ((unsigned)P.comp_tbl[G.comp] | 0x10100u | (unsigned)G.comp << 24);
            tbl = sinfo & 0xFF;
            const int back = (sinfo >> 8) & 0xFF;
            const bool first_of_comp = (sinfo >> 16) & 1;
            int prev;
            if (!(unit == 0 && first_of_comp)) prev = tid >= back ? (int)coef[(tid - back) * kStageStride] : (int)__ldg(src_blocks + ((long long)tid - back) * 64);
            else prev = (int)slot_tab[kMaxSlots + (sinfo >> 24)]; // 0, or the strip in front's last DC

            dcdiff = (int)(int16_t)(coef[tid * kStageStride] - prev);
        }

        for (int j = 0; j < (FULL ? 1 : P.spg); ++j) {
            const DevScan &S = P.scans[it.group + j * P.n_groups];
            const int ss = FULL ? 0 : S.ss, se = FULL ? 63 : S.se;
            const int first_ac = ss == 0 ? 1 : ss;
            // ---- 2. band mask with ZRL markers, DC code, sort key ----
            unsigned m_lo = 0, m_hi = 0;
            uint32_t first = 0;
            if (valid) {
                if (se > 0) {
                    unsigned long long m = FULL ? m_all : m_all & (~0ull << first_ac) & (~0ull >> (63 - se));
                    m |= zrl_markers(m, first_ac);
                    m_lo = __brev((unsigned)m); // coded from the highest bit down
                    m_hi = __brev((unsigned)(m >> 32));
                }
                if (ss == 0) { // write_dc, writer.rs:342-352
                    int size;
                    uint32_t bits;
                    value_code(dcdiff, size, bits);
                    const uint2 e = dc_tab[tbl * 16 + size];
                    first = e.x | bits | e.y << 27;
                }
            }
            *visit_meta(tid) = make_uint4(m_lo, m_hi, first, (unsigned)tbl | (valid ? 0x100u : 0u));
            if (se > 0) {
                const int nnz = __popc(m_lo) + __popc(m_hi); // <= 63
                const unsigned rank = atomicAdd(&bin[nnz], 1u);
                __syncthreads();
                { // exclusive prefix over the 64 bins, two per lane; every warp computes it for itself
                    const unsigned a = bin[2 * lane], c = bin[2 * lane + 1];
                    unsigned inc = a + c;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        const unsigned o = __shfl_up_sync(0xffffffffu, inc, d);
                        if (lane >= d) inc += o;
                    }
                    const unsigned even = inc - a - c, odd = inc - c; // first rank of bins 2*lane and 2*lane + 1
                    const unsigned e = __shfl_sync(0xffffffffu, even, nnz >> 1), o = __shfl_sync(0xffffffffu, odd, nnz >> 1);
                    order[((nnz & 1) ? o : e) + rank] = (uint16_t)tid;
                }
                __syncthreads();
                for (int i = tid; i < 64; i += T) bin[i] = 0; // for the next sort (several barriers away)
            } else {
                order[tid] = (uint16_t)tid; // one code per visit at most: nothing to balance
                __syncthreads();
            }

            if (j == 0) { // the next chunk's blocks on their way into L2 while this one is coded (thread 0 has already decoded it)
                const ItemInfo &nx = items[(round & 1) ^ 1];
                if (!nx.done && (unsigned)tid < nx.n_valid)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(b.coef + (nx.blk0 + tid) * 64));
            }
            // ---- 3. code the visit of rank tid ----
            {
                const int src = order[tid];
                const uint4 meta = *visit_meta(src);
                const unsigned inf = meta.w;
                unsigned nb = 0;
                if (inf & 0x100u) {
                    const uint32_t dc_code = meta.z;
                    BitSink<T> sink(scratch, src);
                    sink.put(dc_code & kCodeBits, (int)(dc_code >> 27));
                    if (se > 0) code_nonzeros<T>(meta.x, meta.y, first_ac, se, coef + src * kStageStride, ac_tab + (inf & 0xFF) * 256, sink);
                    nb = sink.finish();
                }
                nbv[src] = nb;
            }
            __syncthreads(); // all code words are in the scratch (visible to the CTA), all reads of the staged blocks are done

            // ---- 4. bit offsets of the visits inside the chunk, assembly, write-out ----
            const unsigned myb = nbv[tid];
            const unsigned nw = (myb + 31) >> 5;
            const uint32_t *mine = scratch + tid;
            uint32_t pre[4]; // nearly every visit has at most four words: request them before the prefix sum
#pragma unroll
            for (int q = 0; q < 4; ++q) pre[q] = __ldcg(mine + q * T);
            unsigned inc = myb;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned o = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane >= d) inc += o;
            }
            // sums of the other warps' visits: every warp adds them up itself (one REDUX each) instead of meeting at a barrier
            unsigned off = inc - myb, total = 0;
#pragma unroll
            for (int w = 0; w < T / 32; ++w) {
                const unsigned sw = __reduce_add_sync(0xffffffffu, nbv[w * 32 + lane]);
                if (w < warp) off += sw;
                total += sw;
            }
            const unsigned total_words = (total + 31) >> 5;
            const unsigned long long ci = it.chunk_index0 + S.chunk_base;
            // room in the pool: requested now, looked at only when the chunk is written out (the atomic's round trip
            // overlaps the assembly)
            const unsigned pool_units = (total_words + 3) >> 2; // 16-byte units
            unsigned long long pool_at = 0;
            if (tid == 0) {
                if (pool_units) pool_at = atomicAdd(b.status + kStatPoolCursor, (unsigned long long)pool_units);
                b.chunk_bits[ci] = total;
            }
            for (unsigned wb = 0; wb < total_words; wb += L::kAsmWords) { // one pass unless the chunk is larger than the buffer
                const unsigned nwin = total_words - wb < (unsigned)L::kAsmWords ? total_words - wb : (unsigned)L::kAsmWords;
                for (unsigned i = tid * 4; i < nwin; i += T * 4) *reinterpret_cast<uint4 *>(asmbuf + i) = make_uint4(0, 0, 0, 0);
                __syncthreads();
                if (myb) { // shift this visit's words to bit offset `off` of the chunk; only its first and last word are shared with the neighbours
                    const unsigned d0 = off >> 5, dl = (off + myb - 1) >> 5, sft = off & 31;
                    auto word = [&](unsigned q) -> uint32_t {
                        if (q >= nw) return 0u;
                        if (q < 4) return q == 0 ? pre[0] : (q == 1 ? pre[1] : (q == 2 ? pre[2] : pre[3]));
                        return __ldcg(mine + q * T);
                    };
                    if (wb == 0 && dl < nwin) { // the usual case: the whole visit lies in this window
                        uint32_t prev = pre[0];
                        atomicOr(asmbuf + d0, prev >> sft);
                        unsigned jw = 1;
                        for (unsigned d = d0 + 1; d < dl; ++d, ++jw) {
                            const uint32_t cur = word(jw);
                            asmbuf[d] = __funnelshift_r(cur, prev, sft);
                            prev = cur;
                        }
                        if (dl > d0) atomicOr(asmbuf + dl, __funnelshift_r(word(jw), prev, sft));
                    } else {
                        const unsigned lo = d0 > wb ? d0 : wb, hi = dl < wb + nwin - 1 ? dl : wb + nwin - 1;
                        if (lo <= hi) {
                            unsigned jw = lo - d0; // source word that starts in destination word `lo`
                            uint32_t prev = jw > 0 ? word(jw - 1) : 0u;
                            for (unsigned d = lo; d <= hi; ++d, ++jw) {
                                const uint32_t cur = word(jw);
                                atomicOr(asmbuf + (d - wb), __funnelshift_r(cur, prev, sft));
                                prev = cur;
                            }
                        }
                    }
                }
                if (tid == 0 && wb == 0) {
                    if (pool_at + pool_units > b.pool_cap) {
                        atomicOr(b.status + kStatFlags, kFlagPool);
                        pool_at = ~0ull;
                    }
                    wsum[8] = (uint32_t)pool_at;
                    wsum[9] = (uint32_t)(pool_at >> 32);
                    b.chunk_pool[ci] = (uint32_t)pool_at;
                }
                __syncthreads();
                const unsigned long long at = ((unsigned long long)wsum[9] << 32) | wsum[8];
                if (at != ~0ull) {
                    uint4 *dst = reinterpret_cast<uint4 *>(b.pool) + at + (wb >> 2);
                    for (unsigned i = tid; i * 4 < nwin; i += T) dst[i] = reinterpret_cast<const uint4 *>(asmbuf)[i];
                }
                if (wb + L::kAsmWords < total_words || !FULL) __syncthreads(); // the buffer is reused
            }
        }
    }
}

// lead of local segment `s`: what the reference writes between the previous segment's last byte
// and this segment's first: the file header (first segment of the image), the SOS of a later scan
// (writer.rs:424-452) or RSTn (encoder.rs:748-752: marker index = restarts % 8).
__device__ __forceinline__ unsigned lead_len(const EntropyBuffers &b, const DevPlan &P, unsigned long long img, int k,
                                             unsigned seg_in_scan) {
    if (P.bare) return 0;
    if (P.scans[k].rst_base + seg_in_scan > 0) return 2; // RSTn (for a strip: also before its first segment)
    if (k > 0) return P.scans[k].sos_len;
    return b.hdr_len[b.huff_per_image ? img : 0];
}

// bytes of local segment g (lead + data + EOI); the caller raises kFlagSegment4G beyond 4 GiB
__device__ __forceinline__ unsigned long long segment_bytes(const EntropyBuffers &b, const DevPlan &P, unsigned long long g) {
    const unsigned long long img = g / P.segs_per_image;
    const unsigned s = (unsigned)(g - img * P.segs_per_image);
    const int k = find_scan_by_seg(P, s);
    const DevScan &S = P.scans[k];
    const unsigned i = s - S.seg_base;
    const unsigned cps = P.groups[k % P.n_groups].cps;
    // the segment's chunks are consecutive; the chunk after its last one starts the next segment (or scan, or image)
    const unsigned long long c0 = img * P.chunks_per_image + S.chunk_base + (unsigned long long)i * cps;
    const unsigned long long bits = b.chunk_bitpos[c0 + cps] - b.chunk_bitpos[c0];
    if (P.bare) return (bits + 127) >> 7 << 4;
    const unsigned tail = (s == P.segs_per_image - 1 && P.has_eoi) ? 2u : 0u; // EOI, encoder.rs:564
    return lead_len(b, P, img, k, i) + ((bits + 7) >> 3) + tail;
}

__global__ void __launch_bounds__(256) segment_len_kernel(const __grid_constant__ EntropyBuffers b, const __grid_constant__ DevPlan P, unsigned long long n_segs) {
    const unsigned long long g = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_segs) return;
    const unsigned long long bytes = segment_bytes(b, P, g);
    if (bytes > 0xFFFFFFFFull) atomicOr(b.status + kStatFlags, kFlagSegment4G); // seglen is 32-bit: reported, never wrapped silently
    b.seglen[g] = (unsigned)bytes;
}

// exclusive prefix over the 1024 threads of a CTA (sm: 33 words); `total` = the CTA's sum
__device__ __forceinline__ unsigned long long cta1024_exclusive(unsigned long long v, unsigned long long *sm, unsigned long long &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) sm[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const unsigned long long w = sm[lane];
        unsigned long long winc = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long o = __shfl_up_sync(0xffffffffu, winc, d);
            if (lane >= d) winc += o;
        }
        sm[lane] = winc - w;
        if (lane == 31) sm[32] = winc;
    }
    __syncthreads();
    const unsigned long long ex = sm[warp] + inc - v;
    total = sm[32];
    __syncthreads(); // sm is reused by the caller's next round
    return ex;
}

// Small jobs (a few thousand chunks and segments: one image, or a short batch): the prefix sum of the chunk sizes, the
// segment lengths and their prefix sum in ONE single-CTA kernel instead of four launches. With scan_chunks == 0 the
// chunk positions come from the look-back scan (many chunks, few segments).
__global__ void __launch_bounds__(1024) positions_kernel(const __grid_constant__ EntropyBuffers b, const __grid_constant__ DevPlan P, unsigned long long n_chunks,
                                                         unsigned long long n_segs, int scan_chunks) {
    __shared__ unsigned long long sm[33];
    unsigned long long carry = 0, total;
    if (scan_chunks) {
        for (unsigned long long base = 0; base < n_chunks; base += 1024) {
            const unsigned long long i = base + threadIdx.x;
            const unsigned long long ex = cta1024_exclusive(i < n_chunks ? b.chunk_bits[i] : 0ull, sm, total);
            if (i < n_chunks) b.chunk_bitpos[i] = carry + ex;
            carry += total;
        }
        if (threadIdx.x == 0) b.chunk_bitpos[n_chunks] = carry;
        __syncthreads(); // the positions are read back below by other threads of this CTA
    }
    carry = 0;
    for (unsigned long long base = 0; base < n_segs; base += 1024) {
        const unsigned long long g = base + threadIdx.x;
        unsigned long long bytes = 0;
        if (g < n_segs) {
            bytes = segment_bytes(b, P, g);
            if (bytes > 0xFFFFFFFFull) atomicOr(b.status + kStatFlags, kFlagSegment4G);
        }
        const unsigned long long ex = cta1024_exclusive(bytes, sm, total);
        if (g < n_segs) b.segpos[g] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) b.segpos[n_segs] = carry;
}

// Unstuffed stream size as computed on the device; kernels that write the stream bail out (and the
// first one raises the overflow flag) when it exceeds the capacity the host provided.
__device__ __forceinline__ unsigned long long stream_bytes(const EntropyBuffers &b) { return b.segpos[b.n_segs_total]; }
__device__ __forceinline__ bool stream_fits(const EntropyBuffers &b) { return stream_bytes(b) <= b.ustream_cap; }

__device__ __forceinline__ void put_raw(const EntropyBuffers &b, unsigned long long pos, uint8_t byte) {
    b.ustream[pos] = byte;
    atomicOr(b.raw_mask + (pos >> 5), 1u << (pos & 31));
}

__global__ void __launch_bounds__(128) segment_lead_kernel(const __grid_constant__ EntropyBuffers b, const __grid_constant__ DevPlan P, unsigned long long n_segs,
                                                           const unsigned wps) {
    // `wps` warps per segment: each takes a slice of the segment's chunk boundaries; the first one also writes the lead
    // (lanes stride over its bytes: headers can be long -- ICC, EXIF) and the EOI
    const unsigned long long gw = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned long long g = gw / wps;
    const unsigned slice = (unsigned)(gw - g * wps);
    const int lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0) { // size of the unstuffed stream for the host; too large for the buffer: nothing is written
        const unsigned long long bytes = stream_bytes(b);
        b.status[kStatUnstuffed] = bytes;
        if (bytes > b.ustream_cap) atomicOr(b.status + kStatFlags, kFlagStream);
    }
    if (g >= n_segs || !stream_fits(b)) return;
    const unsigned long long img = g / P.segs_per_image;
    const unsigned s = (unsigned)(g - img * P.segs_per_image);
    const int k = find_scan_by_seg(P, s);
    const DevScan &S = P.scans[k];
    const unsigned i = s - S.seg_base;
    const unsigned long long pos = b.segpos[g];
    {   // The stream is not cleared as a whole. The placement kernel stores the words a chunk owns and ORs its bits into
        // the words it shares: the word in which a chunk ends and the next one begins (every chunk boundary that is not
        // word aligned, the segment's first and last data bit included). Those words are zeroed here -- only their bytes
        // that hold this segment's entropy-coded data: lead, EOI and the neighbouring segments' bytes in the same word
        // are stored byte-wise by whoever owns them, in any order.
        const bool eoi = s == P.segs_per_image - 1 && P.has_eoi;
        const unsigned cps = P.groups[k % P.n_groups].cps;
        const unsigned long long c0 = img * P.chunks_per_image + S.chunk_base + (unsigned long long)i * cps;
        const unsigned long long bit0 = b.chunk_bitpos[c0];
        const unsigned long long data0 = pos + lead_len(b, P, img, k, i), data1 = b.segpos[g + 1] - (eoi ? 2u : 0u);
        const unsigned per = (cps + wps) / wps; // cps + 1 boundaries over wps warps
        const unsigned q1 = (slice + 1) * per < cps + 1 ? (slice + 1) * per : cps + 1;
        for (unsigned q = slice * per + lane; q < q1; q += 32) {
            const unsigned long long pbit = data0 * 8 + (b.chunk_bitpos[c0 + q] - bit0);
            if ((pbit & 31) == 0) continue;
            const unsigned long long w = pbit >> 5;
            const unsigned long long lo = w * 4 > data0 ? w * 4 : data0, hi = w * 4 + 4 < data1 ? w * 4 + 4 : data1;
            if (lo + 4 == hi) reinterpret_cast<uint32_t *>(b.ustream)[w] = 0u;
            else
                for (unsigned long long x = lo; x < hi; ++x) b.ustream[x] = 0;
        }
    }
    if (slice != 0 || P.bare) return;
    if (S.rst_base + i > 0) {
        if (lane == 0) {
            put_raw(b, pos, 0xFF);
            put_raw(b, pos + 1, (uint8_t)(0xD0 + ((S.rst_base + i - 1) & 7)));
        }
    } else if (k > 0) {
        for (unsigned j = lane; j < S.sos_len; j += 32) put_raw(b, pos + j, P.blob[S.sos_off + j]);
    } else {
        const unsigned long long h = b.huff_per_image ? img : 0;
        const unsigned n = b.hdr_len[h];
        const uint8_t *src = b.hdr + h * b.hdr_stride;
        // the bytes (independent loads, several in flight), then the raw flags one 32-bit mask word at a time
#pragma unroll 4
        for (unsigned j = lane; j < n; j += 32) b.ustream[pos + j] = src[j];
        const unsigned long long w0 = pos >> 5, w1 = (pos + n - 1) >> 5;
        for (unsigned long long w = w0 + lane; w <= w1 && n; w += 32) {
            const unsigned long long lo = w * 32 > pos ? w * 32 : pos, hi = (w + 1) * 32 < pos + n ? (w + 1) * 32 : pos + n; // [lo, hi) of this word
            const unsigned bits = (unsigned)(hi - lo);
            atomicOr(b.raw_mask + w, (bits == 32 ? 0xFFFFFFFFu : ((1u << bits) - 1u)) << (unsigned)(lo & 31));
        }
    }
    if (s == P.segs_per_image - 1 && P.has_eoi && lane == 0) {
        const unsigned long long end = b.segpos[g + 1];
        put_raw(b, end - 2, 0xFF);
        put_raw(b, end - 1, 0xD9);
    }
}

// finalize_bit_buffer (writer.rs:138-145): ones behind the segment's last bit up to the byte boundary
__device__ __forceinline__ void put_pad(uint32_t *stream, unsigned long long data_byte, unsigned long long seg_bits) {
    const unsigned pad = (unsigned)(-(long long)seg_bits) & 7u;
    if (pad) {
        const unsigned long long pbit = data_byte * 8 + seg_bits;
        const unsigned s2 = (unsigned)(pbit & 31); // pad never crosses a byte, hence never a word
        atomicOr(stream + (pbit >> 5), __byte_perm(((1u << pad) - 1u) << (32 - s2 - pad), 0, 0x0123));
    }
}

// Streams chunk c from `pool` to its place in the unstuffed stream: a bit-granular copy (funnel shift by the
// start position modulo 32), one warp per chunk, 128 bytes per step, reads and writes coalesced. The first and the
// last stream word of a chunk are shared with its neighbours and are merged with atomicOr (the stream is
// zero-initialised); words in between are owned and stored. The warp of a segment's first chunk also writes the
// pad bits of finalize_bit_buffer behind the segment's last bit (writer.rs:138-145: ones up to the byte boundary).
__global__ void __launch_bounds__(256) place_chunks_kernel(const __grid_constant__ EntropyBuffers b, const __grid_constant__ DevPlan P, unsigned long long n_chunks,
                                                           const unsigned per_warp) {
    if (!stream_fits(b) || (b.status[kStatFlags] & kFlagPool)) return;
    const int lane = threadIdx.x & 31;
    const unsigned long long warps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    uint32_t *stream = reinterpret_cast<uint32_t *>(b.ustream);
    // A warp takes `per_warp` (1..32) consecutive chunks. First every lane works out where ONE of them goes (a chain of
    // dependent loads: sizes, positions, segment start -- up to 32 chains in flight instead of one), then the warp
    // copies them one after the other with all lanes. Small jobs take one chunk per warp: they need the warps.
    for (unsigned long long c0 = (((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * per_warp; c0 < n_chunks; c0 += warps * per_warp) {
        const unsigned long long c = c0 + lane;
        unsigned my_bits = 0, my_pool = 0;
        unsigned long long my_bitpos = 0;
        if ((unsigned)lane < per_warp && c < n_chunks) {
            const unsigned long long img = c / P.chunks_per_image;
            const unsigned r = (unsigned)(c - img * P.chunks_per_image);
            const int k = find_scan_by_chunk(P, r);
            const DevScan &S = P.scans[k];
            const DevGroup &G = P.groups[k % P.n_groups];
            unsigned seg, q;
            divmod(r - S.chunk_base, G.div_cps, seg, q);
            my_bits = b.chunk_bits[c];
            if (my_bits != 0 || q == 0) {
                const unsigned long long seg_first = b.chunk_bitpos[c - q];
                const unsigned long long data_byte = b.segpos[img * P.segs_per_image + S.seg_base + seg] + lead_len(b, P, img, k, seg);
                my_bitpos = data_byte * 8 + (b.chunk_bitpos[c] - seg_first);
                if (my_bits) my_pool = b.chunk_pool[c];
                if (q == 0 && !P.bare) put_pad(stream, data_byte, b.chunk_bitpos[c + G.cps] - seg_first);
            }
        }
        unsigned todo = __ballot_sync(0xffffffffu, my_bits != 0);
        while (todo) {
            const int who = __ffs(todo) - 1;
            todo &= todo - 1;
            const unsigned bits = __shfl_sync(0xffffffffu, my_bits, who);
            const unsigned long long bitpos = __shfl_sync(0xffffffffu, my_bitpos, who);
            const uint32_t *src = b.pool + (size_t)__shfl_sync(0xffffffffu, my_pool, who) * 4;
            const unsigned sft = (unsigned)(bitpos & 31);
            uint32_t *dst = stream + (bitpos >> 5);
            const unsigned nw = (bits + 31) >> 5, ndw = (sft + bits + 31) >> 5;
            const bool first_owned = sft == 0, last_owned = ((sft + bits) & 31) == 0;
            uint32_t carry = 0; // source word in front of this step's first one
            // 128 words per step: four independent, coalesced loads per lane are in flight together
            for (unsigned base = 0; base < ndw; base += 128) {
                uint32_t cur[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const unsigned d = base + 32 * u + lane;
                    cur[u] = d < nw ? __ldg(src + d) : 0u;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const unsigned d = base + 32 * u + lane;
                    uint32_t prev = __shfl_up_sync(0xffffffffu, cur[u], 1);
                    if (lane == 0) prev = carry;
                    carry = __shfl_sync(0xffffffffu, cur[u], 31);
                    if (d < ndw) {
                        const uint32_t val = sft ? __funnelshift_r(cur[u], prev, sft) : cur[u];
                        const uint32_t be = __byte_perm(val, 0, 0x0123);
                        const bool owned = (d > 0 || first_owned) && (d + 1 < ndw || last_owned);
                        if (owned) dst[d] = be;
                        else atomicOr(dst + d, be);
                    }
                }
            }
        }
    }
}

// ---- strips without restart intervals -----------------------------------------------------------
// A bare strip (one image, one segment per scan): the bits of its piece of every scan
__global__ void __launch_bounds__(256) piece_bits_kernel(const __grid_constant__ EntropyBuffers b, const __grid_constant__ DevPlan P,
                                                         unsigned long long *bits) {
    for (int k = threadIdx.x; k < P.n_scans; k += blockDim.x) {
        const unsigned c1 = k + 1 < P.n_scans ? P.scans[k + 1].chunk_base : P.chunks_per_image;
        bits[k] = b.chunk_bitpos[c1] - b.chunk_bitpos[P.scans[k].chunk_base];
    }
}

// The root of a join: chunk k * world + r of its plan is rank r's piece of scan k (table: world x n_scans, rank order)
__global__ void __launch_bounds__(256) join_chunks_kernel(const EntropyBuffers b, const unsigned long long *__restrict__ table, unsigned world,
                                                          unsigned n_scans) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= world * n_scans) return;
    const unsigned k = i / world, r = i - k * world;
    const unsigned long long bits = table[(unsigned long long)r * n_scans + k];
    if (bits > 0xFFFFFFFFull) atomicOr(b.status + kStatFlags, kFlagSegment4G); // chunk sizes are 32-bit
    b.chunk_bits[i] = (uint32_t)bits;
}

// The root of a join, once every rank's stores have landed and segment_lead_kernel has written the leads and zeroed the
// shared words: the pad bits behind every scan and the ranks' side words
__global__ void __launch_bounds__(256) join_merge_kernel(const __grid_constant__ EntropyBuffers b, const __grid_constant__ DevPlan P,
                                                         const JoinSideWord *__restrict__ side, unsigned world) {
    if (!stream_fits(b)) return;
    uint32_t *stream = reinterpret_cast<uint32_t *>(b.ustream);
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (unsigned)P.n_scans) {
        const unsigned long long c0 = P.scans[i].chunk_base;
        put_pad(stream, b.segpos[i] + lead_len(b, P, 0, (int)i, 0), b.chunk_bitpos[c0 + world] - b.chunk_bitpos[c0]);
    }
    if (i < 2 * world * (unsigned)P.n_scans) {
        const JoinSideWord sw = side[i];
        if (sw.word < b.ustream_cap / 4) atomicOr(stream + sw.word, sw.value);
    }
}

// ---- 0xFF stuffing (writer.rs:156-167) as count / scan / scatter ---------------------------------
// A thread owns 16 consecutive bytes of the unstuffed stream and the 16 raw_mask bits beside them.
// 0x80 in every byte of w that equals 0xFF, exact (no carries cross bytes): a byte of ~w is zero iff neither its
// low seven bits (sum with 0x7F stays below 0x80) nor its top bit are set.
__device__ __forceinline__ uint32_t ff_flags(uint32_t w) {
    const uint32_t x = ~w;
    const uint32_t t = ((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x;
    return ~t & 0x80808080u;
}
// flags at bits 7, 15, 23, 31 -> bits 0..3 (the four products land on distinct bits 21..24)
__device__ __forceinline__ unsigned flags_to_nibble(uint32_t z) { return (((z >> 7) * 0x00204081u) >> 21) & 0xFu; }

__device__ __forceinline__ unsigned ff_bits16(const uint4 d, unsigned raw16, unsigned valid) {
    unsigned m = flags_to_nibble(ff_flags(d.x)) | flags_to_nibble(ff_flags(d.y)) << 4 | flags_to_nibble(ff_flags(d.z)) << 8 |
                 flags_to_nibble(ff_flags(d.w)) << 12;
    m &= ~raw16;
    if (valid < 16) m &= (1u << valid) - 1u;
    return m;
}
// number of data 0xFF bytes among the 16 (same as popc(ff_bits16), cheaper when nothing is raw)
__device__ __forceinline__ unsigned ff_count16(const uint4 d, unsigned raw16, unsigned valid) {
    if (raw16 == 0 && valid >= 16) return __popc(ff_flags(d.x)) + __popc(ff_flags(d.y)) + __popc(ff_flags(d.z)) + __popc(ff_flags(d.w));
    return __popc(ff_bits16(d, raw16, valid));
}

__global__ void __launch_bounds__(256) count_ff_kernel(const EntropyBuffers b) {
    __shared__ unsigned warp_sums[8];
    const unsigned long long bytes = stream_fits(b) ? stream_bytes(b) : 0ull;
    const unsigned long long base = (unsigned long long)blockIdx.x * kStuffChunk + (unsigned long long)threadIdx.x * 16;
    unsigned cnt = 0;
    if (base < bytes) {
        const uint4 d = *reinterpret_cast<const uint4 *>(b.ustream + base);
        const unsigned raw = (b.raw_mask[base >> 5] >> (base & 31)) & 0xFFFFu;
        const unsigned valid = bytes - base < 16 ? (unsigned)(bytes - base) : 16u;
        cnt = ff_count16(d, raw, valid);
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned t = 0;
        for (int i = 0; i < 8; ++i) t += warp_sums[i];
        b.ffcount[blockIdx.x] = t;
    }
}

// Short streams (up to kDirectPieces pieces): no prefix-sum launch over the per-piece 0xFF counts; whoever needs
// "0xFF bytes in front of piece i" adds the counts up itself.
constexpr unsigned kDirectPieces = 2048;

// sum of ffcount[0, idx) and of all n_pieces counts, by one warp
__device__ __forceinline__ void ff_sums_warp(const uint32_t *ffcount, unsigned n_pieces, unsigned idx, int lane, unsigned long long &before, unsigned long long &total) {
    unsigned a = 0, t = 0;
    for (unsigned j = lane; j < n_pieces; j += 32) {
        const unsigned v = ffcount[j];
        t += v;
        if (j < idx) a += v;
    }
    before = __reduce_add_sync(0xffffffffu, a);
    total = __reduce_add_sync(0xffffffffu, t);
}

// data 0xFF bytes in [chunk start, pos) of the unstuffed stream, counted by one warp with 128-bit loads
__device__ __forceinline__ unsigned ff_before_in_chunk(const EntropyBuffers &b, unsigned long long pos, int lane) {
    const unsigned long long start = pos / kStuffChunk * kStuffChunk;
    unsigned ff = 0;
    for (unsigned long long i = start + (unsigned long long)lane * 16; i < pos; i += 32 * 16) {
        const uint4 d = *reinterpret_cast<const uint4 *>(b.ustream + i);
        const unsigned raw = (b.raw_mask[i >> 5] >> (i & 31)) & 0xFFFFu;
        const unsigned valid = pos - i < 16 ? (unsigned)(pos - i) : 16u;
        ff += ff_count16(d, raw, valid);
    }
    return __reduce_add_sync(0xffffffffu, ff);
}

// CTAs [0, n_pieces): piece blockIdx.x of the unstuffed stream -> its place in `out`, 0x00 inserted behind data 0xFF.
// CTAs behind them, one warp per position: the byte offset in `out` of every file (position of the image's first
// segment plus the data 0xFF bytes in front of it) and, for a strip, of every scan's first segment (the pieces).
__global__ void __launch_bounds__(256) stuff_scatter_kernel(const __grid_constant__ EntropyBuffers b, const __grid_constant__ DevPlan P, unsigned n_pieces,
                                                            unsigned n_images, unsigned long long *piece_offs) {
    if (!stream_fits(b)) return;
    const unsigned long long bytes = stream_bytes(b);
    const bool direct = n_pieces <= kDirectPieces;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (blockIdx.x >= n_pieces) { // ---- offsets ----
        const unsigned k = (blockIdx.x - n_pieces) * 8 + warp;
        const unsigned n_pos = n_images + 1 + (piece_offs ? (unsigned)P.n_scans + 1 : 0u);
        if (k >= n_pos) return;
        unsigned long long pos;
        unsigned long long *dst;
        if (k <= n_images) {
            pos = k == n_images ? bytes : b.segpos[(unsigned long long)k * P.segs_per_image];
            dst = b.file_off + k;
        } else {
            const unsigned sc = k - (n_images + 1);
            pos = sc == (unsigned)P.n_scans ? bytes : b.segpos[P.scans[sc].seg_base];
            dst = piece_offs + sc;
        }
        const unsigned long long piece = pos / kStuffChunk;
        unsigned long long before, total;
        if (direct) ff_sums_warp(b.ffcount, n_pieces, (unsigned)piece, lane, before, total);
        else before = b.ffpos[piece];
        const unsigned ff = ff_before_in_chunk(b, pos, lane);
        if (lane == 0) *dst = pos + before + ff;
        return;
    }
    __shared__ unsigned warp_excl[9];
    __shared__ unsigned long long ff_sm[2];
    __shared__ __align__(16) uint8_t stage[2 * kStuffChunk + 32];
    unsigned long long ff_before, ff_total;
    if (direct) { // every CTA adds up the counts in front of its piece (and all of them) itself
        if (warp == 0) {
            unsigned long long a, t;
            ff_sums_warp(b.ffcount, n_pieces, blockIdx.x, lane, a, t);
            if (lane == 0) ff_sm[0] = a, ff_sm[1] = t;
        }
        __syncthreads();
        ff_before = ff_sm[0];
        ff_total = ff_sm[1];
    } else {
        ff_before = b.ffpos[blockIdx.x];
        ff_total = b.ffpos[n_pieces];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        b.status[kStatDataFF] = ff_total;
        if (bytes + ff_total > b.out_cap) atomicOr(b.status + kStatFlags, kFlagOut);
    }
    if (bytes + ff_total > b.out_cap) return;
    if ((unsigned long long)blockIdx.x * kStuffChunk >= bytes) return;
    // The chunk's output is first laid out in shared memory at the same offset modulo 16 as its place
    // in `out`, then copied with aligned 128-bit stores (single bytes only at the two ends).
    const unsigned long long base = (unsigned long long)blockIdx.x * kStuffChunk + (unsigned long long)threadIdx.x * 16;
    uint4 d = make_uint4(0, 0, 0, 0);
    unsigned m = 0, valid = 0;
    if (base < bytes) {
        d = *reinterpret_cast<const uint4 *>(b.ustream + base);
        const unsigned raw = (b.raw_mask[base >> 5] >> (base & 31)) & 0xFFFFu;
        valid = bytes - base < 16 ? (unsigned)(bytes - base) : 16u;
        m = ff_bits16(d, raw, valid);
    }
    const unsigned cnt = __popc(m);
    unsigned inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) warp_excl[warp + 1] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
        warp_excl[0] = 0;
        for (int i = 1; i <= 8; ++i) warp_excl[i] += warp_excl[i - 1];
    }
    __syncthreads();
    const unsigned long long chunk_base = (unsigned long long)blockIdx.x * kStuffChunk;
    const unsigned long long out0 = chunk_base + ff_before; // first output byte of this chunk
    const unsigned pad = (unsigned)(out0 & 15);
    const unsigned chunk_in = bytes - chunk_base < kStuffChunk ? (unsigned)(bytes - chunk_base) : (unsigned)kStuffChunk;
    const unsigned total = chunk_in + warp_excl[8];
    if (valid) {
        unsigned o = pad + threadIdx.x * 16 + warp_excl[warp] + (inc - cnt);
        const uint32_t w[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            if ((unsigned)i < valid) {
                stage[o++] = (uint8_t)(w[i >> 2] >> ((i & 3) * 8));
                if (m & (1u << i)) stage[o++] = 0x00;
            }
        }
    }
    __syncthreads();
    uint8_t *dst = b.out + (out0 - pad); // 16-byte aligned (b.out comes from cudaMalloc)
    const unsigned end = pad + total;
    for (unsigned o = threadIdx.x * 16; o < end; o += 256 * 16) {
        if (o >= pad && o + 16 <= end) {
            *reinterpret_cast<uint4 *>(dst + o) = *reinterpret_cast<const uint4 *>(stage + o);
        } else {
            for (unsigned k = (o < pad ? pad : o); k < o + 16 && k < end; ++k) dst[k] = stage[k];
        }
    }
}

// ---- optimized-table histogram (encoder.rs:1086-1200) --------------------------------------------
// One CTA per 256 consecutive blocks of one image, staged like a coding chunk (the coefficient buffer holds every
// component's true grid in raster order -- optimized tables always code non-interleaved -- so the blocks are one
// contiguous run and the block in front is the DC predecessor). Every thread walks the set bits of its block's
// non-zero mask, band by band: AC run/size symbols (runs restart per band), ZRL through the marker trick of the coder,
// EOB when a band ends in zeros; DC category of the chained difference with NO restart resets (Q17).
// Bins: [image][table][dc|ac][257], collected per CTA in shared memory. One launch for the whole batch.
template <int BASE>
__device__ __forceinline__ void count_half(unsigned m, int &next, unsigned c_shared, unsigned *ha) {
#pragma unroll 1
    while (m) { // same walk as code_half: the highest set bit of the reversed mask is the next position in zig-zag order
        int p;
        asm("bfind.u32 %0, %1;" : "=r"(p) : "r"(m));
        unsigned bit;
        asm("bmsk.clamp.b32 %0, %1, 1;" : "=r"(bit) : "r"(p));
        m ^= bit;
        const int k = BASE + 31 - p;
        int v;
        asm("ld.shared.s16 %0, [%1];" : "=r"(v) : "r"(c_shared + 2 * k));
        const int run = k - next; // <= 15 thanks to the markers; a marker is a zero: size 0 -> symbol 0xF0
        next = k + 1;
        const int a = v < 0 ? -v : v;
        int top;
        asm("bfind.u32 %0, %1;" : "=r"(top) : "r"(a));
        atomicAdd(ha + ((run << 4) | (top + 1)), 1u);
    }
}

__global__ void __launch_bounds__(256) histogram_kernel(const __grid_constant__ DevPlan P, const int16_t *coef, unsigned n_images, uint32_t *hist,
                                                        int bands, int per_band) {
    __shared__ unsigned sh[2 * 2 * 257];
    __shared__ __align__(16) int16_t blk[256 * kStageStride];
    const int tid = threadIdx.x;
    const unsigned long long g0 = (unsigned long long)blockIdx.x * 256; // first block of this CTA inside the image
    const unsigned n_here = P.blocks_per_image - g0 < 256 ? (unsigned)(P.blocks_per_image - g0) : 256u;
    for (unsigned img = blockIdx.y; img < n_images; img += gridDim.y) {
        for (int i = tid; i < 2 * 2 * 257; i += 256) sh[i] = 0;
        const int16_t *src = coef + ((unsigned long long)img * P.blocks_per_image + g0) * 64;
        {
            const unsigned pieces = n_here * 8;
            const char *g = reinterpret_cast<const char *>(src) + (size_t)tid * 16;
            const unsigned d = (unsigned)__cvta_generic_to_shared(blk) + (tid >> 3) * (kStageStride * 2) + (tid & 7) * 16;
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if ((unsigned)(tid + k * 256) < pieces)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + k * 32 * (kStageStride * 2)), "l"(g + k * 256 * 16) : "memory");
            asm volatile("cp.async.wait_all;" ::: "memory");
        }
        __syncthreads();
        if ((unsigned)tid < n_here) {
            const unsigned long long g = g0 + tid;
            int comp = 0;
            while (comp + 1 < P.n_groups && g >= P.groups[comp + 1].block_base) ++comp;
            const int16_t *mine = blk + tid * kStageStride;
            const uint4 *m4 = reinterpret_cast<const uint4 *>(mine);
            unsigned m_lo = 0, m_hi = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                const uint4 q = m4[w];
                unsigned byte = __dp2a_lo(nonzero16x2(q.x), 0x0201u, 0u);
                byte = __dp2a_lo(nonzero16x2(q.y), 0x0804u, byte);
                byte = __dp2a_lo(nonzero16x2(q.z), 0x2010u, byte);
                byte = __dp2a_lo(nonzero16x2(q.w), 0x8040u, byte);
                if (w < 4) m_lo |= byte << (8 * w);
                else m_hi |= byte << (8 * (w - 4));
            }
            const unsigned long long m_all = (((unsigned long long)m_hi << 32) | m_lo) & ~1ull;
            const int prev = g > P.groups[comp].block_base ? (tid > 0 ? (int)mine[-kStageStride] : (int)__ldg(src - 64)) : 0;
            unsigned *h = sh + P.comp_tbl[comp] * 2 * 257;
            const int diff = (int)(int16_t)(mine[0] - prev);
            atomicAdd(h + (32 - __clz(diff < 0 ? -diff : diff)), 1u);
            unsigned *ha = h + 257;
            const unsigned c_shared = (unsigned)__cvta_generic_to_shared(mine);
            for (int b = 0; b < bands; ++b) { // band b covers [max(b * per, 1), (b + 1) * per), the last one to 63
                const int first_ac = b == 0 ? 1 : b * per_band, se = b == bands - 1 ? 63 : (b + 1) * per_band - 1;
                if (se < first_ac) continue; // the empty first band of 34..64 scans
                unsigned long long m = m_all & (~0ull << first_ac) & (~0ull >> (63 - se));
                m |= zrl_markers(m, first_ac);
                int next = first_ac;
                count_half<0>(__brev((unsigned)m), next, c_shared, ha);
                count_half<32>(__brev((unsigned)(m >> 32)), next, c_shared, ha);
                if (next <= se) atomicAdd(ha, 1u); // the band ends in zeros: EOB
            }
        }
        __syncthreads();
        uint32_t *dst = hist + (size_t)img * (2 * 2 * 257);
        for (int i = tid; i < 2 * 2 * 257; i += 256)
            if (sh[i]) atomicAdd(dst + i, sh[i]);
        __syncthreads();
    }
}

} // namespace

static inline unsigned grid_for(unsigned long long n, unsigned block) { return (unsigned)((n + block - 1) / block); }

cudaError_t launch_histogram(const DevPlan &hp, const int16_t *coef, uint32_t n_images, uint32_t *hist,
                             cudaStream_t stream) {
    // sequential / progressive plans only (optimized tables never code interleaved)
    const int bands = hp.spg > 1 ? hp.spg - 1 : 1;
    const int per_band = bands > 1 ? 64 / bands : 64;
    dim3 grid(grid_for(hp.blocks_per_image, 256), n_images < 32768 ? n_images : 32768);
    histogram_kernel<<<grid, 256, 0, stream>>>(hp, coef, n_images, hist, bands, per_band);
    return cudaGetLastError();
}

namespace {
template <int T, bool FULL>
cudaError_t coder_config(unsigned long long n_items, CoderLaunch &cfg) {
    unsigned long long grid = 0;
    cudaError_t e = resident_ctas<encode_chunks_kernel<T, FULL>>(T, CoderSmem<T, FULL>::kBytes, grid);
    if (e != cudaSuccess) return e;
    if (grid > n_items) grid = n_items;
    if (grid < 1) grid = 1;
    cfg.grid = (unsigned)grid;
    cfg.smem = CoderSmem<T, FULL>::kBytes;
    cfg.scratch_bytes = (size_t)grid * T * kSlotWords * 4;
    return cudaSuccess;
}
// progressive plans end with an AC band; in every other mode all scans cover the whole block
inline bool plan_is_full(const DevPlan &hp) { return hp.scans[hp.n_scans - 1].ss == 0 && hp.scans[hp.n_scans - 1].se == 63; }
} // namespace

#define JPGB_CODER_DISPATCH(CALL)                              \
    do {                                                       \
        const bool full = plan_is_full(hp);                    \
        switch (hp.chunk_T) {                                  \
        case 32: if (full) { CALL(32, true); } else { CALL(32, false); } break;    \
        case 64: if (full) { CALL(64, true); } else { CALL(64, false); } break;    \
        case 128: if (full) { CALL(128, true); } else { CALL(128, false); } break; \
        default: if (full) { CALL(256, true); } else { CALL(256, false); } break;  \
        }                                                      \
    } while (0)

cudaError_t coder_launch_config(const DevPlan &hp, uint32_t n, CoderLaunch &cfg) {
    const unsigned long long n_items = (unsigned long long)hp.items_per_image * n;
#define JPGB_CFG(T, F) return coder_config<T, F>(n_items, cfg)
    JPGB_CODER_DISPATCH(JPGB_CFG);
#undef JPGB_CFG
    return cudaErrorInvalidValue;
}
cudaError_t launch_encode_chunks(const EntropyBuffers &b, const DevPlan &hp, uint32_t n, const CoderLaunch &cfg, cudaStream_t s) {
    const unsigned long long n_items = (unsigned long long)hp.items_per_image * n;
#define JPGB_RUN(T, F) encode_chunks_kernel<T, F><<<cfg.grid, T, cfg.smem, s>>>(b, hp, n_items)
    JPGB_CODER_DISPATCH(JPGB_RUN);
#undef JPGB_RUN
    return cudaGetLastError();
}
cudaError_t launch_segment_lengths(const EntropyBuffers &b, const DevPlan &hp, uint32_t n, cudaStream_t s) {
    const unsigned long long ns = (unsigned long long)hp.segs_per_image * n;
    segment_len_kernel<<<grid_for(ns, 256), 256, 0, s>>>(b, hp, ns);
    return cudaGetLastError();
}
cudaError_t launch_positions(const EntropyBuffers &b, const DevPlan &hp, uint32_t n, bool scan_chunks, cudaStream_t s) {
    positions_kernel<<<1, 1024, 0, s>>>(b, hp, (unsigned long long)hp.chunks_per_image * n, (unsigned long long)hp.segs_per_image * n, scan_chunks ? 1 : 0);
    return cudaGetLastError();
}
cudaError_t launch_segment_leads(const EntropyBuffers &b, const DevPlan &hp, uint32_t n, cudaStream_t s) {
    const unsigned long long ns = (unsigned long long)hp.segs_per_image * n;
    unsigned cps = 1;
    for (int g = 0; g < hp.n_groups; ++g) cps = hp.groups[g].cps > cps ? hp.groups[g].cps : cps;
    unsigned wps = (cps + 1 + 127) / 128; // a warp looks at up to 128 chunk boundaries (four dependent loads per lane)
    wps = wps > 1024 ? 1024 : wps;
    segment_lead_kernel<<<grid_for(ns * wps * 32, 128), 128, 0, s>>>(b, hp, ns, wps);
    return cudaGetLastError();
}
cudaError_t launch_place_chunks(const EntropyBuffers &b, const DevPlan &hp, uint32_t n, cudaStream_t s) {
    const unsigned long long nc = (unsigned long long)hp.chunks_per_image * n;
    unsigned per_warp = 1; // chunks per warp: as many as leaves ~16 K warps of work
    while (per_warp < 32 && nc / (per_warp * 2) >= 16384) per_warp *= 2;
    const unsigned long long ctas = (nc + 8ull * per_warp - 1) / (8ull * per_warp); // grid-stride beyond 64 K CTAs
    place_chunks_kernel<<<(unsigned)(ctas < 65536 ? (ctas ? ctas : 1) : 65536), 256, 0, s>>>(b, hp, nc, per_warp);
    return cudaGetLastError();
}
cudaError_t launch_piece_bits(const EntropyBuffers &b, const DevPlan &hp, unsigned long long *bits, cudaStream_t s) {
    piece_bits_kernel<<<1, 256, 0, s>>>(b, hp, bits);
    return cudaGetLastError();
}
cudaError_t launch_join_chunks(const EntropyBuffers &b, const unsigned long long *table, unsigned world, unsigned n_scans, cudaStream_t s) {
    join_chunks_kernel<<<grid_for((unsigned long long)world * n_scans, 256), 256, 0, s>>>(b, table, world, n_scans);
    return cudaGetLastError();
}
cudaError_t launch_join_merge(const EntropyBuffers &b, const DevPlan &hp, const JoinSideWord *side, unsigned world, cudaStream_t s) {
    join_merge_kernel<<<grid_for(2ull * world * hp.n_scans, 256), 256, 0, s>>>(b, hp, side, world);
    return cudaGetLastError();
}
cudaError_t launch_count_ff(const EntropyBuffers &b, cudaStream_t s) {
    count_ff_kernel<<<grid_for(b.ustream_cap, kStuffChunk), 256, 0, s>>>(b);
    return cudaGetLastError();
}
bool ff_scan_needed(const EntropyBuffers &b) { return grid_for(b.ustream_cap, kStuffChunk) > kDirectPieces; }
cudaError_t launch_stuff_scatter(const EntropyBuffers &b, const DevPlan &hp, uint32_t n, unsigned long long *piece_offs, cudaStream_t s) {
    const unsigned n_pieces = grid_for(b.ustream_cap, kStuffChunk);
    const unsigned n_pos = n + 1 + (piece_offs ? (unsigned)hp.n_scans + 1 : 0u);
    stuff_scatter_kernel<<<n_pieces + (n_pos + 7) / 8, 256, 0, s>>>(b, hp, n_pieces, n, piece_offs);
    return cudaGetLastError();
}

} // namespace jpgb
