// compact.cu -- K3: turn the per-block scratch slots into one contiguous reference-format
// stream: varint(total) || block_0 || block_1 ...   (reference: write_dim_varint
// src/snappy_compression.c:171-174 + write_block_compressed :334-336, i.e. fwrite in order).
//
//   k_scan_sizes : exclusive prefix sum of the per-block compressed sizes (one CTA, the
//                  array is tiny: 16 Ki entries per GiB), writes the varint and the total
//   k_gather     : one CTA per block, 16-byte stores, source funnel-shifted to the
//                  destination alignment (block offsets in the stream are arbitrary)
#include "common.cuh"

namespace sb200 {

constexpr int kScanThreads = 1024;
constexpr int kScanItems = 8;

// Plain LEB128, reference parse_to_varint src/varint.c:12-20.
__device__ __forceinline__ uint32_t dev_put_varint(uint64_t v, uint8_t *dst)
{
    uint32_t k = 0;
    while (v >= 0x80u) {
        dst[k++] = (uint8_t)(v | 0x80u);
        v >>= 7;
    }
    dst[k++] = (uint8_t)v;
    return k;
}

__host__ __device__ inline uint32_t varint_len(uint64_t v)
{
    uint32_t k = 1;
    while (v >= 0x80u) {
        v >>= 7;
        ++k;
    }
    return k;
}

__global__ void __launch_bounds__(kScanThreads) k_scan_sizes(const uint32_t *__restrict__ sizes, uint64_t n_blocks,
                                                             uint64_t n_bytes, uint64_t base, int write_varint,
                                                             uint8_t *__restrict__ out, uint64_t out_capacity,
                                                             uint64_t *__restrict__ offsets,
                                                             uint64_t *__restrict__ out_bytes,
                                                             uint32_t *__restrict__ status)
{
    __shared__ uint64_t warp_sum[kScanThreads / 32];
    __shared__ uint64_t carry_s;
    const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0)
        carry_s = base;
    __syncthreads();
    for (uint64_t start = 0; start < n_blocks; start += (uint64_t)kScanThreads * kScanItems) {
        uint64_t v[kScanItems];
        uint64_t sum = 0;
        const uint64_t i0 = start + (uint64_t)tid * kScanItems;
#pragma unroll
        for (int k = 0; k < kScanItems; ++k) {
            v[k] = (i0 + k < n_blocks) ? sizes[i0 + k] : 0;
            sum += v[k];
        }
        uint64_t incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint64_t t = __shfl_up_sync(kFull, incl, d);
            if ((int)lane >= d)
                incl += t;
        }
        if (lane == 31)
            warp_sum[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            uint64_t w = warp_sum[lane];
            uint64_t wi = w;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint64_t t = __shfl_up_sync(kFull, wi, d);
                if ((int)lane >= d)
                    wi += t;
            }
            warp_sum[lane] = wi - w; // exclusive
        }
        __syncthreads();
        const uint64_t carry = carry_s;
        uint64_t run = carry + warp_sum[wid] + (incl - sum);
#pragma unroll
        for (int k = 0; k < kScanItems; ++k) {
            if (i0 + k < n_blocks)
                offsets[i0 + k] = run;
            run += v[k];
        }
        __syncthreads();
        if (tid == kScanThreads - 1)
            carry_s = run;
        __syncthreads();
    }
    if (tid == 0) {
        const uint64_t total = carry_s;
        offsets[n_blocks] = total;
        *out_bytes = total;
        if (total > out_capacity)
            atomicOr(status, SNAPPY_B200_ST_CAPACITY);
        else if (write_varint && n_blocks > 0)
            dev_put_varint(n_bytes, out);
    }
}

__global__ void __launch_bounds__(128) k_gather(const uint8_t *__restrict__ scratch, const uint32_t *__restrict__ sizes,
                                                const uint64_t *__restrict__ offsets, uint8_t *__restrict__ out,
                                                uint64_t out_capacity)
{
    const uint64_t blk = blockIdx.x;
    const uint32_t len = sizes[blk];
    const uint64_t off = offsets[blk];
    if (off + len > out_capacity)
        return; // k_scan_sizes has already flagged SNAPPY_B200_ST_CAPACITY
    coop_copy_ro(out + off, scratch + blk * (uint64_t)kSlot, len, threadIdx.x, blockDim.x);
}

cudaError_t launch_compact(const uint8_t *d_scratch, const uint32_t *d_sizes, uint64_t n_blocks, uint64_t n_bytes,
                           uint64_t base, int write_varint, uint8_t *d_out, uint64_t out_capacity, uint64_t *d_offsets,
                           uint64_t *d_out_bytes, uint32_t *d_status, cudaStream_t st, uint64_t *launches)
{
    k_scan_sizes<<<1, kScanThreads, 0, st>>>(d_sizes, n_blocks, n_bytes, base, write_varint, d_out, out_capacity,
                                             d_offsets, d_out_bytes, d_status);
    *launches += 1;
    if (n_blocks > 0) {
        k_gather<<<(unsigned)n_blocks, 128, 0, st>>>(d_scratch, d_sizes, d_offsets, d_out, out_capacity);
        *launches += 1;
    }
    return cudaGetLastError();
}

cudaError_t launch_scan_sizes(const uint32_t *d_sizes, uint64_t n_blocks, uint64_t n_bytes, uint64_t base,
                              int write_varint, uint8_t *d_out, uint64_t out_capacity, uint64_t *d_offsets,
                              uint64_t *d_out_bytes, uint32_t *d_status, cudaStream_t st, uint64_t *launches)
{
    k_scan_sizes<<<1, kScanThreads, 0, st>>>(d_sizes, n_blocks, n_bytes, base, write_varint, d_out, out_capacity,
                                             d_offsets, d_out_bytes, d_status);
    *launches += 1;
    return cudaGetLastError();
}

uint32_t host_varint_len(uint64_t v) { return varint_len(v); }

} // namespace sb200
