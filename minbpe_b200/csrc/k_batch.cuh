// k_batch.cuh — batched encode: [tok.encode(t) for t in docs] in one device call (bpe_encode_batch_gpt4).
//
// The documents are joined by single 0xFF bytes (BATCH_SEP, a byte UTF-8 never contains, so it can neither collide
// with text nor with a special token).  Every separator is handled like a one-byte special-token occurrence of the
// splitter's front end (k_special.cuh): its meta byte gets the boundary class SC_B, so the WITH_B rule code of
// split_logic.h splits the text on either side on its own, and it becomes a chunk of its own with a chunk start right
// behind it.  Here:
//   k_batch_sep_meta    meta[i] = SC_B | SM_START at every separator (after k_split_classify)
//   k_batch_sep_flags   flag[i] = flag[i + 1] = 1 at every separator (after k_split_apply<WITH_B>)
// The memoised encode kernels (k_encode2.cuh, BATCH = true) then skip every chunk that starts with a separator — it is
// never memoised and produces no ids — and k_enc_write<true> stores, for every separator, the output position where
// the next document starts.
#pragma once
#include "common.cuh"
#include "split_logic.h"
#include "k_encode2.cuh"

// nonzero iff one of the four bytes of x is 0xFF (a zero byte of ~x)
__device__ __forceinline__ u32 has_ff(u32 x) { const u32 v = ~x; return (v - 0x01010101u) & ~v & 0x80808080u; }

// 16 bytes per thread and step; n is the length of the piece (its buffers are 256-byte aligned, the tail is bytewise)
__global__ void __launch_bounds__(256) k_batch_sep_meta(const unsigned char *__restrict__ b, u64 n, unsigned char *__restrict__ meta) {
    const u64 nv = n / 16;
    for (u64 v = (u64)blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += (u64)gridDim.x * blockDim.x) {
        const uint4 w = reinterpret_cast<const uint4 *>(b)[v];
        if (!(has_ff(w.x) | has_ff(w.y) | has_ff(w.z) | has_ff(w.w))) continue;
        for (u32 k = 0; k < 16; ++k)
            if (b[16 * v + k] == BATCH_SEP) meta[16 * v + k] = (unsigned char)(SC_B | SM_START);
    }
    for (u64 i = nv * 16 + (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (b[i] == BATCH_SEP) meta[i] = (unsigned char)(SC_B | SM_START);
}

// the separator is a chunk of its own and the next document starts a chunk (the WITH_B rule answers false for SC_B bytes)
__global__ void __launch_bounds__(256) k_batch_sep_flags(const unsigned char *__restrict__ b, u64 n, unsigned char *__restrict__ flag) {
    const u64 nv = n / 16;
    for (u64 v = (u64)blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += (u64)gridDim.x * blockDim.x) {
        const uint4 w = reinterpret_cast<const uint4 *>(b)[v];
        if (!(has_ff(w.x) | has_ff(w.y) | has_ff(w.z) | has_ff(w.w))) continue;
        for (u32 k = 0; k < 16; ++k) {
            const u64 i = 16 * v + k;
            if (b[i] == BATCH_SEP) { flag[i] = 1; if (i + 1 < n) flag[i + 1] = 1; }
        }
    }
    for (u64 i = nv * 16 + (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (b[i] == BATCH_SEP) { flag[i] = 1; if (i + 1 < n) flag[i + 1] = 1; }
}
