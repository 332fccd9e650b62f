// common.cuh -- device helpers shared by the codec kernels (sm_100a).
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "snappy_b200.h"

namespace sb200 {

constexpr uint32_t kBlock = SNAPPY_B200_BLOCK_SIZE;
constexpr uint32_t kSlot = SNAPPY_B200_SLOT_STRIDE;
constexpr unsigned kFull = 0xffffffffu;
constexpr uint32_t kHashMul = 0x1e35a7bdu;  // reference: src/snappy_compression.c:82
constexpr uint32_t kAbortMark = 0xffffffffu; // sizes[] entry of a block a table tier gave up on

// ---- framed streams (csrc/frame.cu): one data chunk, as the host walk of the chunk headers describes it
constexpr uint32_t kChunkCompressed = 0x00, kChunkUncompressed = 0x01;
struct FrameChunk {
    uint64_t in_off;   // stream offset of the chunk's body: the elements (after the varint), or the raw bytes
    uint64_t out_off;  // output offset of its first byte
    uint32_t in_len;   // body bytes
    uint32_t out_len;  // uncompressed bytes, <= 65536
    uint32_t type;     // kChunkCompressed / kChunkUncompressed
    uint32_t crc;      // the stored (masked) CRC-32C
};

// ---- read-only input access -------------------------------------------------------------
// `base` is 4-byte aligned.  Word `last_word` is the last one that holds a valid byte, so the
// second load is clamped instead of running past the buffer when pos is word aligned.
__device__ __forceinline__ uint32_t ld_le32(const uint8_t *__restrict__ base, uint32_t pos, uint32_t last_word)
{
    const uint32_t *w = reinterpret_cast<const uint32_t *>(base);
    const uint32_t i = pos >> 2;
    const uint32_t lo = __ldg(w + i);
    const uint32_t hi = __ldg(w + min(i + 1, last_word));
    return __funnelshift_r(lo, hi, (pos & 3u) * 8u);
}

__device__ __forceinline__ uint32_t bswap32(uint32_t x) { return __byte_perm(x, 0, 0x0123); }

// Big-endian 4-byte load: reference get_next_u32, src/snappy_compression.c:239-241.
__device__ __forceinline__ uint32_t ld_be32(const uint8_t *__restrict__ base, uint32_t pos, uint32_t last_word)
{
    return bswap32(ld_le32(base, pos, last_word));
}

// Little-endian 32 bits at an arbitrarily aligned address; the aligned words touched are
// clamped to `last_word`, the last aligned word that still holds a byte of the stream.
__device__ __forceinline__ uint32_t ld_le32_any(const uint8_t *__restrict__ p, const uint32_t *__restrict__ last_word)
{
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t *w0 = reinterpret_cast<const uint32_t *>(a & ~uintptr_t(3));
    const uint32_t *w1 = w0 + 1;
    w0 = w0 > last_word ? last_word : w0;
    w1 = w1 > last_word ? last_word : w1;
    return __funnelshift_r(__ldg(w0), __ldg(w1), (uint32_t)(a & 3u) * 8u);
}


// ---- cooperative byte copy, global -> global, any alignment -------------------------------
cudaError_t peek_u32(uint32_t *h_pinned_dst, const void *d_src, uint32_t n_u32, cudaStream_t st); // abi.cu
uint32_t *thread_pinned_scratch();                                                                // abi.cu

// Ask for a line to be brought into L2.  The parse and decode chains are latency-bound, and the
// first touch of every input line is otherwise a full DRAM round trip on the critical path.
__device__ __forceinline__ void prefetch_l2(const void *p)
{
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

// `nt` threads (ids 0..nt-1) copy len bytes.  src is read through the read-only path, so it
// must not alias anything written by this kernel.  Large copies go in 16-byte destination
// chunks; the source words are funnel-shifted to the destination alignment.
__device__ __forceinline__ void coop_copy_ro(uint8_t *__restrict__ dst, const uint8_t *__restrict__ src, uint32_t len,
                                             uint32_t tid, uint32_t nt)
{
    if (len < 64) {
        for (uint32_t i = tid; i < len; i += nt)
            dst[i] = __ldg(src + i);
        return;
    }
    const uint32_t head = (16u - (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u;
    for (uint32_t i = tid; i < head; i += nt)
        dst[i] = __ldg(src + i);
    const uint32_t nchunk = (len - head) >> 4;
    const uint8_t *s0 = src + head;
    const uint32_t sa = (uint32_t)(reinterpret_cast<uintptr_t>(s0) & 3u);
    const uint32_t *sw = reinterpret_cast<const uint32_t *>(s0 - sa);
    uint4 *d4 = reinterpret_cast<uint4 *>(dst + head);
    const uint32_t sh = sa * 8u;
    const uint32_t w4i = sa ? 4u : 3u; // the fifth word is only touched when it holds wanted bytes
    for (uint32_t c = tid; c < nchunk; c += nt) {
        const uint32_t *p = sw + 4u * c;
        const uint32_t w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2), w3 = __ldg(p + 3), w4 = __ldg(p + w4i);
        uint4 v;
        v.x = __funnelshift_r(w0, w1, sh);
        v.y = __funnelshift_r(w1, w2, sh);
        v.z = __funnelshift_r(w2, w3, sh);
        v.w = __funnelshift_r(w3, w4, sh);
        d4[c] = v;
    }
    for (uint32_t i = head + (nchunk << 4) + tid; i < len; i += nt)
        dst[i] = __ldg(src + i);
}

} // namespace sb200
