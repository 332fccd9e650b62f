// frame.cu -- the Snappy framing format (google/snappy framing_format.txt): the stream identifier, then one chunk
// per 64 KiB block, each with a 4-byte header (type, 24-bit length) and the masked CRC-32C of its uncompressed bytes.
//
//   k_crc32c_chunks : CRC-32C of up to 65536 bytes per CTA -- the input blocks (compress: masked values for the
//                     gather) or the decoded chunks (decompress: compared with the stored value, ST_CHECKSUM)
//   k_frame_sizes   : per block, compressed (0x00) or uncompressed (0x01) chunk, and its size
//   k_frame_gather  : one CTA per block: header, masked CRC, then varint(n) + the block's slot or the raw input
// The placement between the two is k_scan_sizes (compact.cu) with base 10 (the identifier) and no varint.  The
// chunk decoder, k_frame_decode, shares the block routines of csrc/decode.cu and lives there.
#include "common.cuh"

namespace sb200 {

cudaError_t launch_scan_sizes(const uint32_t *, uint64_t, uint64_t, uint64_t, int, uint8_t *, uint64_t, uint64_t *,
                              uint64_t *, uint32_t *, cudaStream_t, uint64_t *); // compact.cu

namespace {

constexpr uint32_t kCrcPoly = 0x82F63B78u; // CRC-32C (Castagnoli), reflected
constexpr uint32_t kCrcThreads = 256;
constexpr uint32_t kCrcSeg = kBlock / kCrcThreads; // 256 contiguous bytes per thread
constexpr uint32_t kCrcMaskDelta = 0xa282ead8u;

// Column i of kShift.m[j] is what the zero-init CRC register holding bit i becomes after 2^j zero bytes: the
// operator that shifts a partial CRC past 2^j further bytes (crc(A || B) = shift(crc(A), |B|) ^ crc(B)).
struct ShiftOps {
    uint32_t m[17][32];
};

constexpr uint32_t gf2_apply(const uint32_t *M, uint32_t v)
{
    uint32_t r = 0;
    for (int i = 0; i < 32; ++i)
        if ((v >> i) & 1u)
            r ^= M[i];
    return r;
}

constexpr ShiftOps make_shift_ops()
{
    ShiftOps s{};
    for (int i = 0; i < 32; ++i) {
        uint32_t c = 1u << i;
        for (int k = 0; k < 8; ++k)
            c = (c & 1u) ? (c >> 1) ^ kCrcPoly : c >> 1;
        s.m[0][i] = c;
    }
    for (int j = 1; j < 17; ++j)
        for (int i = 0; i < 32; ++i)
            s.m[j][i] = gf2_apply(s.m[j - 1], s.m[j - 1][i]);
    return s;
}

__constant__ ShiftOps kShift = make_shift_ops();

// Every thread of the warp passes the same j: the constant reads are broadcasts.
__device__ __forceinline__ uint32_t crc_shift_pow2(uint32_t v, int j)
{
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < 32; ++i)
        r ^= ((v >> i) & 1u) ? kShift.m[j][i] : 0u;
    return r;
}

__device__ __forceinline__ uint32_t sel4(uint32_t o, uint32_t a, uint32_t b, uint32_t c, uint32_t d)
{
    return o == 0 ? a : (o == 1 ? b : (o == 2 ? c : d));
}

// The chunk [p0, p0 + len), len <= 65536, is placed right-aligned in a virtual 65536-byte buffer: the zero-init
// CRC does not change under leading zero bytes, so every chunk length runs the same tree.  Thread t takes virtual
// bytes [256 t, 256 t + 256) -- 16-byte loads, realigned with funnel shifts, slicing-by-4 out of shared-memory
// tables -- and shifts its partial CRC past the 256 (255 - t) bytes behind it; the partials are XOR-reduced.  The
// register init 0xffffffff is one more shifted term (past all len bytes), the final xor is applied once.
__device__ __forceinline__ uint32_t crc32c_chunk(const uint8_t *p0, uint32_t len, const uint32_t (*T)[256],
                                                 uint32_t *part, uint32_t tid)
{
    const int64_t vs = (int64_t)len - (int64_t)kBlock + (int64_t)(kCrcSeg * tid); // my first byte, p0-relative
    uint32_t crc = 0;
    if (vs + (int64_t)kCrcSeg > 0) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(p0) + (intptr_t)vs;
        const uintptr_t a0 = a & ~uintptr_t(15);
        const uintptr_t lo = reinterpret_cast<uintptr_t>(p0) & ~uintptr_t(15);
        const uintptr_t hi = (reinterpret_cast<uintptr_t>(p0) + len - 1) & ~uintptr_t(15);
        const uint32_t o = (uint32_t)(a & 15u) >> 2, sh = (uint32_t)(a & 3u) * 8u;
        uint32_t W[4 * (kCrcSeg / 16 + 1)];
#pragma unroll
        for (uint32_t q = 0; q <= kCrcSeg / 16; ++q) {
            // a line that holds none of the chunk's bytes is clamped into it (its bytes are masked or shifted out)
            uintptr_t qa = a0 + 16u * q;
            qa = qa < lo ? lo : (qa > hi ? hi : qa);
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(qa));
            W[4 * q] = v.x, W[4 * q + 1] = v.y, W[4 * q + 2] = v.z, W[4 * q + 3] = v.w;
        }
#pragma unroll
        for (uint32_t i = 0; i < kCrcSeg / 4; ++i) {
            uint32_t m = __funnelshift_r(sel4(o, W[i], W[i + 1], W[i + 2], W[i + 3]),
                                         sel4(o, W[i + 1], W[i + 2], W[i + 3], W[i + 4]), sh);
            const int64_t at = vs + 4 * (int64_t)i; // bytes before p0 count as the leading zeros
            if (at < 0)
                m = at <= -4 ? 0u : m & (0xffffffffu << (uint32_t)(-at * 8));
            crc ^= m;
            crc = T[3][crc & 0xffu] ^ T[2][(crc >> 8) & 0xffu] ^ T[1][(crc >> 16) & 0xffu] ^ T[0][crc >> 24];
        }
    }
    const uint32_t behind = kCrcThreads - 1u - tid; // 256-byte segments after mine
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint32_t s = crc_shift_pow2(crc, 8 + j);
        crc = ((behind >> j) & 1u) ? s : crc;
    }
    crc = __reduce_xor_sync(kFull, crc);
    if ((tid & 31u) == 0)
        part[tid >> 5] = crc;
    __syncthreads();
    uint32_t all = 0;
    if (tid == 0) {
        uint32_t init = 0xffffffffu;
        for (int j = 0; j < 17; ++j)
            if ((len >> j) & 1u)
                init = crc_shift_pow2(init, j);
        all = init;
        for (uint32_t w = 0; w < kCrcThreads / 32; ++w)
            all ^= part[w];
        all = ~all;
        all = ((all >> 15) | (all << 17)) + kCrcMaskDelta;
    }
    return all; // thread 0 only
}

// chunks == nullptr: compress mode, CTA b takes input block b of n_bytes and writes the masked CRC to masked[b].
// Otherwise CTA c takes the output bytes of chunks[c] at base and sets ST_CHECKSUM if they do not match its CRC.
__global__ void __launch_bounds__(kCrcThreads) k_crc32c_chunks(const uint8_t *__restrict__ base, uint64_t n_bytes,
                                                               const FrameChunk *__restrict__ chunks,
                                                               uint32_t *__restrict__ masked,
                                                               uint32_t *__restrict__ status)
{
    __shared__ uint32_t T[4][256];
    __shared__ uint32_t part[kCrcThreads / 32];
    const uint32_t tid = threadIdx.x;
    {
        uint32_t c = tid;
#pragma unroll
        for (int k = 0; k < 8; ++k)
            c = (c & 1u) ? (c >> 1) ^ kCrcPoly : c >> 1;
        T[0][tid] = c;
    }
    __syncthreads();
#pragma unroll
    for (int k = 1; k < 4; ++k) {
        const uint32_t prev = T[k - 1][tid];
        T[k][tid] = (prev >> 8) ^ T[0][prev & 0xffu];
        __syncthreads();
    }
    const uint64_t c = blockIdx.x;
    if (chunks) {
        const FrameChunk ch = chunks[c];
        const uint32_t got = crc32c_chunk(base + ch.out_off, ch.out_len, T, part, tid);
        if (tid == 0 && got != ch.crc)
            atomicOr(status, SNAPPY_B200_ST_CHECKSUM);
    } else {
        const uint64_t left = n_bytes - c * kBlock;
        const uint32_t got = crc32c_chunk(base + c * kBlock, left < kBlock ? (uint32_t)left : kBlock, T, part, tid);
        if (tid == 0)
            masked[c] = got;
    }
}

__device__ __forceinline__ uint32_t block_len(uint64_t n_bytes, uint64_t b)
{
    const uint64_t left = n_bytes - b * kBlock;
    return left < kBlock ? (uint32_t)left : kBlock;
}

__device__ __forceinline__ uint32_t varint_len_block(uint32_t n) { return n < (1u << 7) ? 1u : (n < (1u << 14) ? 2u : 3u); }

// The writer rule of golang/snappy: a compressed chunk only when it saves at least 1/8 of the block.
__global__ void k_frame_sizes(const uint32_t *__restrict__ sizes, uint64_t n_bytes, uint64_t n_blocks,
                              uint32_t *__restrict__ fsizes)
{
    const uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (b >= n_blocks)
        return;
    const uint32_t n = block_len(n_bytes, b);
    const uint32_t r = varint_len_block(n) + sizes[b];
    fsizes[b] = 8u + (r < n - n / 8 ? r : n);
}

__global__ void __launch_bounds__(128) k_frame_gather(const uint8_t *__restrict__ in, uint64_t n_bytes,
                                                      uint64_t n_blocks, const uint8_t *__restrict__ scratch,
                                                      const uint32_t *__restrict__ sizes,
                                                      const uint32_t *__restrict__ fsizes,
                                                      const uint32_t *__restrict__ crcs,
                                                      const uint64_t *__restrict__ offsets, int identifier,
                                                      uint8_t *__restrict__ out, uint64_t out_capacity)
{
    const uint64_t blk = blockIdx.x;
    const uint32_t tid = threadIdx.x;
    if (identifier && blk == 0 && tid < 10 && out_capacity >= 10) // ff 06 00 00 "sNaPpY"
        out[tid] = tid < 8 ? (uint8_t)(0x50614e73000006ffull >> (8 * tid)) : (tid == 8 ? 'p' : 'Y');
    if (blk >= n_blocks)
        return;
    const uint32_t fs = fsizes[blk];
    const uint64_t off = offsets[blk];
    if (off + fs > out_capacity)
        return; // k_scan_sizes has already flagged SNAPPY_B200_ST_CAPACITY
    const uint32_t n = block_len(n_bytes, blk);
    const bool comp = fs - 8u < n; // an uncompressed chunk carries exactly n bytes
    const uint32_t vl = comp ? varint_len_block(n) : 0u;
    if (tid == 0) {
        uint8_t *h = out + off;
        const uint32_t L = fs - 4u, crc = crcs[blk];
        h[0] = comp ? kChunkCompressed : kChunkUncompressed;
        h[1] = (uint8_t)L, h[2] = (uint8_t)(L >> 8), h[3] = (uint8_t)(L >> 16);
        h[4] = (uint8_t)crc, h[5] = (uint8_t)(crc >> 8), h[6] = (uint8_t)(crc >> 16), h[7] = (uint8_t)(crc >> 24);
        if (comp) {
            uint32_t v = n, k = 8;
            while (v >= 0x80u) {
                h[k++] = (uint8_t)(v | 0x80u);
                v >>= 7;
            }
            h[k] = (uint8_t)v;
        }
    }
    if (comp)
        coop_copy_ro(out + off + 8 + vl, scratch + blk * (uint64_t)kSlot, sizes[blk], tid, blockDim.x);
    else
        coop_copy_ro(out + off + 8, in + blk * (uint64_t)kBlock, n, tid, blockDim.x);
}

} // namespace

// After launch_compress: the chunks of n_bytes of input at d_in into d_out, the identifier in front when
// `identifier` is set.  crcs / fsizes: n_blocks words each; offsets: n_blocks + 1 entries.
cudaError_t launch_frame_compact(const uint8_t *d_in, uint64_t n_bytes, const uint8_t *d_scratch,
                                 const uint32_t *d_sizes, uint32_t *d_crcs, uint32_t *d_fsizes, int identifier,
                                 uint8_t *d_out, uint64_t out_capacity, uint64_t *d_offsets, uint64_t *d_out_bytes,
                                 uint32_t *d_status, cudaStream_t st, uint64_t *launches)
{
    const uint64_t nb = (n_bytes + kBlock - 1) / kBlock;
    if (nb > 0x7fffffffull)
        return cudaErrorInvalidValue;
    if (nb > 0) {
        k_crc32c_chunks<<<(unsigned)nb, kCrcThreads, 0, st>>>(d_in, n_bytes, nullptr, d_crcs, d_status);
        k_frame_sizes<<<(unsigned)((nb + 255) / 256), 256, 0, st>>>(d_sizes, n_bytes, nb, d_fsizes);
        *launches += 2;
    }
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess)
        e = launch_scan_sizes(d_fsizes, nb, n_bytes, identifier ? 10 : 0, 0, d_out, out_capacity, d_offsets,
                              d_out_bytes, d_status, st, launches);
    if (e != cudaSuccess)
        return e;
    if (nb > 0 || identifier) {
        k_frame_gather<<<(unsigned)(nb ? nb : 1), 128, 0, st>>>(d_in, n_bytes, nb, d_scratch, d_sizes, d_fsizes, d_crcs,
                                                               d_offsets, identifier, d_out, out_capacity);
        *launches += 1;
    }
    return cudaGetLastError();
}

// Checks the CRC of every data chunk of a framed stream against the decoded output at d_out.
cudaError_t launch_frame_check(const uint8_t *d_out, const FrameChunk *d_chunks, uint64_t n_chunks, uint32_t *d_status,
                               cudaStream_t st, uint64_t *launches)
{
    if (n_chunks == 0)
        return cudaSuccess;
    if (n_chunks > 0x7fffffffull)
        return cudaErrorInvalidValue;
    k_crc32c_chunks<<<(unsigned)n_chunks, kCrcThreads, 0, st>>>(d_out, 0, d_chunks, nullptr, d_status);
    *launches += 1;
    return cudaGetLastError();
}

} // namespace sb200
