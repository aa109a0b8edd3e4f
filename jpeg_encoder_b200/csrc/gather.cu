// Strips of one very large image live on different GPUs (SURVEY.md section 8e, BASELINE config 5). The file is the
// scan-major concatenation of the strips' pieces, assembled on the root GPU. Every GPU places its own pieces: one
// kernel per rank reads the table of all ranks' piece offsets (device memory, e.g. the result of an NCCL all-gather
// -- the only collective of the path), works out where each of its pieces belongs in the file and stores the bytes
// straight into the root's buffer through a peer pointer (CUDA IPC mapping over NVLink). No host round trip, no
// staging copy on the root.
#include "kernels.h"

namespace jpgb {
namespace {

// 16 bytes from an arbitrarily aligned address: five aligned words, shifted
__device__ __forceinline__ uint4 load16_unaligned(const uint8_t *p) {
    const unsigned mis = (unsigned)(reinterpret_cast<uintptr_t>(p) & 3);
    const uint32_t *w = reinterpret_cast<const uint32_t *>(p - mis);
    const uint32_t a = w[0], b = w[1], c = w[2], d = w[3];
    if (mis == 0) return make_uint4(a, b, c, d);
    const uint32_t e = w[4];
    const unsigned sh = mis * 8;
    return make_uint4(__funnelshift_r(a, b, sh), __funnelshift_r(b, c, sh), __funnelshift_r(c, d, sh), __funnelshift_r(d, e, sh));
}

// table[r * (n_scans + 1) + k] = byte offset of rank r's piece k inside its own output (entry n_scans = its end).
// Piece k of rank r goes behind all pieces of scans < k and behind the pieces of scan k of the ranks < r.
__global__ void __launch_bounds__(256) place_pieces_kernel(const uint8_t *__restrict__ src, uint8_t *dst, unsigned long long dst_cap,
                                                           const unsigned long long *__restrict__ table, unsigned world, unsigned rank,
                                                           unsigned n_scans, unsigned long long *total_out) {
    const unsigned np = n_scans + 1;
    for (unsigned k = blockIdx.y; k < n_scans; k += gridDim.y) {
        unsigned long long at = 0;
        for (unsigned kk = 0; kk <= k; ++kk)
            for (unsigned r = 0; r < world; ++r)
                if (kk < k || r < rank) at += table[r * np + kk + 1] - table[r * np + kk];
        const unsigned long long s0 = table[rank * np + k], len = table[rank * np + k + 1] - s0;
        if (at + len > dst_cap) continue; // not written; the caller sees *total_out > dst_cap
        const uint8_t *s = src + s0;
        uint8_t *d = dst + at;
        // head: up to the first 16-byte boundary of the destination; body: aligned 128-bit peer stores; tail: the rest
        const unsigned long long head = len < 16 ? len : ((16 - (reinterpret_cast<uintptr_t>(d) & 15)) & 15);
        const unsigned long long body = (len - head) / 16;
        const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (unsigned long long)gridDim.x * blockDim.x;
        if (tid < head) d[tid] = s[tid];
        for (unsigned long long i = tid; i < body; i += stride)
            *reinterpret_cast<uint4 *>(d + head + i * 16) = load16_unaligned(s + head + i * 16);
        const unsigned long long done = head + body * 16;
        if (tid < len - done) d[done + tid] = s[done + tid];
    }
    if (total_out && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
        unsigned long long t = 0;
        for (unsigned r = 0; r < world; ++r) t += table[r * np + n_scans] - table[r * np];
        *total_out = t;
    }
}

__device__ __forceinline__ unsigned long long warp_sum64(unsigned long long v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}

// Strips without restart intervals. table[r * n + k] = bits of rank r's piece of scan k. The target holds the side table
// (join_side_bytes) and then the root's unstuffed stream: per scan its lead, the pieces of ranks 0..world-1 back to back
// at bit granularity, pad bits up to the byte; EOI at the end. Piece k of this rank lies in `src` at the sum of its
// earlier pieces rounded up to 16 bytes each. Every rank derives the same positions from the same table.
__global__ void __launch_bounds__(256) join_place_kernel(const uint8_t *__restrict__ src, uint8_t *target, unsigned long long target_cap,
                                                         const unsigned long long *__restrict__ table, unsigned world, unsigned rank,
                                                         const __grid_constant__ JoinLeads L) {
    __shared__ unsigned long long at_sh[4];
    const unsigned n = L.n_scans;
    const unsigned long long side_bytes = join_side_bytes(world, n);
    uint32_t *stream = reinterpret_cast<uint32_t *>(target + side_bytes);
    JoinSideWord *side = reinterpret_cast<JoinSideWord *>(target);
    const int lane = threadIdx.x & 31;
    for (unsigned k = blockIdx.y; k < n; k += gridDim.y) {
        if (threadIdx.x < 32) { // where the piece comes from and goes to, and whether the stream fits
            unsigned long long s0 = 0, before = 0, all = 0, in_front = 0;
            for (unsigned j = lane; j < n; j += 32) {
                unsigned long long t = 0;
                for (unsigned r = 0; r < world; ++r) {
                    const unsigned long long v = table[(unsigned long long)r * n + j];
                    t += v;
                    if (j == k && r < rank) before += v;
                }
                const unsigned long long bytes = L.lead[j] + ((t + 7) >> 3);
                all += bytes;
                if (j < k) in_front += bytes, s0 += (table[(unsigned long long)rank * n + j] + 127) >> 7 << 4;
            }
            s0 = warp_sum64(s0), before = warp_sum64(before), all = warp_sum64(all), in_front = warp_sum64(in_front);
            if (lane == 0) {
                at_sh[0] = s0;
                at_sh[1] = (in_front + L.lead[k]) * 8 + before;
                at_sh[2] = side_bytes + all + 2 <= target_cap; // + EOI
            }
        }
        __syncthreads();
        const unsigned long long s0 = at_sh[0], B = at_sh[1], bits = table[(unsigned long long)rank * n + k];
        const bool fits = at_sh[2] != 0;
        __syncthreads(); // at_sh is rewritten for the next scan
        const uint32_t *sw = reinterpret_cast<const uint32_t *>(src + s0);
        const unsigned long long nw = (bits + 31) >> 5;
        const unsigned sft = (unsigned)(B & 31), tail_bits = (unsigned)(bits & 31);
        // source word i as a big-endian number, zero outside the piece
        auto word = [&](long long i) -> uint32_t {
            if (i < 0 || (unsigned long long)i >= nw) return 0u;
            uint32_t v = __byte_perm(__ldg(sw + i), 0, 0x0123);
            if ((unsigned long long)i == nw - 1 && tail_bits) v &= ~0u << (32 - tail_bits);
            return v;
        };
        const unsigned long long dw0 = B >> 5;
        // destination word d in memory byte order
        auto dst_word = [&](unsigned long long d) -> uint32_t {
            const long long i = (long long)(d - dw0);
            const uint32_t v = sft ? __funnelshift_r(word(i), word(i - 1), sft) : word(i);
            return __byte_perm(v, 0, 0x0123);
        };
        const unsigned long long o0 = (B + 31) >> 5, o1 = (B + bits) >> 5; // words wholly inside the piece: [o0, o1)
        if (fits && o0 < o1) {
            const unsigned long long a0 = (o0 + 3) & ~3ull, a1 = o1 & ~3ull;
            const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (unsigned long long)gridDim.x * blockDim.x;
            if (a0 < a1) { // aligned 128-bit peer stores for the body, single words at the two ends
                for (unsigned long long q = a0 + tid * 4; q < a1; q += stride * 4)
                    *reinterpret_cast<uint4 *>(stream + q) = make_uint4(dst_word(q), dst_word(q + 1), dst_word(q + 2), dst_word(q + 3));
                if (tid < a0 - o0) stream[o0 + tid] = dst_word(o0 + tid);
                if (tid < o1 - a1) stream[a1 + tid] = dst_word(a1 + tid);
            } else if (tid < o1 - o0) {
                stream[o0 + tid] = dst_word(o0 + tid);
            }
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) { // the shared words: the one holding the first bit and the one holding the last
            const unsigned long long head = (fits && bits && sft) ? dw0 : ~0ull;
            unsigned long long tail = (fits && bits && ((B + bits) & 31)) ? (B + bits - 1) >> 5 : ~0ull;
            if (tail == head) tail = ~0ull;
            JoinSideWord *slot = side + ((unsigned long long)k * world + rank) * 2;
            slot[0] = {head, head != ~0ull ? dst_word(head) : 0u, 0u};
            slot[1] = {tail, tail != ~0ull ? dst_word(tail) : 0u, 0u};
        }
    }
}

} // namespace

cudaError_t launch_join_place(const uint8_t *src, uint8_t *target, unsigned long long target_cap, const unsigned long long *table, unsigned world,
                              unsigned rank, const JoinLeads &leads, cudaStream_t stream) {
    dim3 grid(148, leads.n_scans < 64 ? leads.n_scans : 64);
    join_place_kernel<<<grid, 256, 0, stream>>>(src, target, target_cap, table, world, rank, leads);
    return cudaGetLastError();
}

cudaError_t launch_place_pieces(const uint8_t *src, uint8_t *dst, unsigned long long dst_cap, const unsigned long long *table, unsigned world,
                                unsigned rank, unsigned n_scans, unsigned long long *total_out, cudaStream_t stream) {
    dim3 grid(148, n_scans < 64 ? n_scans : 64);
    place_pieces_kernel<<<grid, 256, 0, stream>>>(src, dst, dst_cap, table, world, rank, n_scans, total_out);
    return cudaGetLastError();
}

} // namespace jpgb
