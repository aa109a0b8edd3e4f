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

} // namespace

cudaError_t launch_place_pieces(const uint8_t *src, uint8_t *dst, unsigned long long dst_cap, const unsigned long long *table, unsigned world,
                                unsigned rank, unsigned n_scans, unsigned long long *total_out, cudaStream_t stream) {
    dim3 grid(148, n_scans < 64 ? n_scans : 64);
    place_pieces_kernel<<<grid, 256, 0, stream>>>(src, dst, dst_cap, table, world, rank, n_scans, total_out);
    return cudaGetLastError();
}

} // namespace jpgb
