// decode_tile.cu -- K4/K5: decompression of an index-less stream, one CTA per 64 KiB output block,
// the whole output block resident in shared memory.
//
// reference: decompressor src/snappy_decompression.c:290-333 (tag dispatch), do_literal :193-224,
// write_literal :232-239, do_copy :253-265, write_copy :273-280.
//
// The reference walks the elements one after another and moves every byte with a scalar loop.
// Here K0 (index.cu) has already left, for every 128-byte segment of the stream, the exact bit map
// of the element starts in it and the output offset of its first element, so the elements of
// different segments can be decoded independently:
//
//   staging   the compressed bytes of the block come into shared memory in 4 KiB chunks (32
//             segments) with bulk asynchronous copies (cp.async.bulk + mbarrier, double buffered:
//             chunk j+1 is in flight while chunk j is decoded).
//   phase A   a warp takes one segment: lane l owns the (at most two) elements that start in
//             stream bytes 4l..4l+3, decodes their headers through a tag table, and one warp
//             prefix sum gives every element its place in the output block.
//   phase B   every lane moves its own literals from the staged stream into the 64 KiB output
//             tile (no dependencies: all literals of all segments go in parallel).
//   phase C   copies.  A copy may read what an earlier copy wrote, so the warp works in rounds
//             (multi-round resolution): a copy is executed by its lane as soon as its whole source
//             range lies below the high-water mark = the output position below which every element
//             is final.  Inside a segment the mark is the first pending copy of the warp; across
//             segments every warp publishes its mark in shared memory (release/acquire) and a warp
//             looks at the first unfinished segment before its own.  Sources are read from the tile
//             (shared memory), 16 bytes per lane per step with word loads/stores; copies that
//             overlap themselves (offset < length, write_copy :273-280) are pattern fills.
//   store     the finished tile goes to HBM once, with a bulk shared->global copy.
// A block that is a single literal (incompressible data) is moved global->global with 16-byte stores
// and never touches the tile.  Unlike the reference, malformed input is detected and reported in
// *status instead of being undefined behaviour (SURVEY.md Q7).
#include <mutex>

#include "common.cuh"
#include "lanecopy.cuh"
#include "tags.cuh"

namespace sb200 {

namespace {

constexpr uint32_t kSegB = 128;                        // K0 segment size (csrc/index.cu)
constexpr uint32_t kChunkSegs = 32;                    // segments staged together
constexpr uint32_t kChunkBytes = kChunkSegs * kSegB;   // 4 KiB
constexpr uint32_t kHalo = 96;                         // 15 (alignment) + 2 (header) + 64 (payload) + word slack
constexpr uint32_t kStageBytes = kChunkBytes + kHalo;  // multiple of 16
constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr uint32_t kShortLit = 64;                     // literals up to this long are moved by their lane

struct TileSmem {
    alignas(128) uint8_t tile[kBlock];
    alignas(16) uint8_t stage[2][kStageBytes];
    uint32_t seg_start[kChunkSegs + 1]; // output offset (block relative) at which segment s of the chunk starts
    uint32_t seg_hwm[kChunkSegs];       // everything of segment s below this output offset is final
    uint16_t lut[256];
    alignas(8) unsigned long long mbar[2];
    uint32_t produced; // output bytes of the block's own elements
};

// ---- PTX: bulk asynchronous copies and their barriers ------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long *b, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *b, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *b, uint32_t parity)
{
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok)
                     : "r"(smem_u32(b)), "r"(parity)
                     : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *b)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(b))
                 : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *dst, const void *src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit_wait_read()
{
    asm volatile("cp.async.bulk.commit_group;\n\tcp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void st_release(uint32_t *p, uint32_t v)
{
    asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
    return v;
}

// len bytes src -> dst where the ranges are at least min(len, 16) bytes apart (or do not alias at all).
__device__ __forceinline__ void copy_fwd(uint8_t *dst, const uint8_t *src, uint32_t len)
{
    for (uint32_t k = 0; k < len; k += 16) {
        const uint32_t n = min(16u, len - k);
        store16(dst + k, load16(src + k, n), n);
    }
}

// dest[m + i] = dest[m - offset + i], i ascending (write_copy :273-280); off >= 1, d - off inside the tile.
__device__ __forceinline__ void do_copy(uint8_t *d, uint32_t off, uint32_t len)
{
    const uint8_t *s = d - off;
    if (off >= 16 || off >= len) {
        copy_fwd(d, s, len);
    } else if (off == 1 || off == 2 || off == 4) {
        // the pattern fits a word and keeps its phase from one 16-byte step to the next
        const uint32_t p = load16(s, off).a;
        const uint32_t w = off == 1 ? (p & 0xffu) * 0x01010101u : (off == 2 ? (p & 0xffffu) * 0x00010001u : p);
        V4 v;
        v.a = v.b = v.c = v.d = w;
        for (uint32_t k = 0; k < len; k += 16)
            store16(d + k, v, min(16u, len - k));
    } else {
        // the periodic region doubles with every pass: each pass is a plain copy over a distance
        // (a multiple of the offset) that is at least its length
        uint32_t done = 0, dist = off;
        while (done < len) {
            const uint32_t n = min(dist, len - done);
            copy_fwd(d + done, d + done - dist, n);
            done += n;
            dist <<= 1;
        }
    }
}

__device__ __forceinline__ uint32_t lds_le32_any(const uint8_t *p)
{
    const uint32_t a = (uint32_t)reinterpret_cast<uintptr_t>(p) & 3u;
    const uint32_t *w = reinterpret_cast<const uint32_t *>(p - a);
    return __funnelshift_r(w[0], w[1], a * 8u);
}

__global__ void __launch_bounds__(kThreads, 3)
    k_decode_tile(const uint8_t *__restrict__ stream, uint64_t body_offset, const uint64_t *__restrict__ offsets,
                  const uint4 *__restrict__ starts, const uint64_t *__restrict__ outoff, uint64_t total_out,
                  uint8_t *out_base, uint32_t *__restrict__ status, uint64_t n_blocks, uint64_t blk_base)
{
    extern __shared__ __align__(128) uint8_t smem_raw[];
    TileSmem &sm = *reinterpret_cast<TileSmem *>(smem_raw);
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint64_t blk = blockIdx.x;
    if (*reinterpret_cast<volatile uint32_t *>(status) != 0)
        return; // K0 rejected the stream: its maps are not trustworthy
    const uint64_t c0 = offsets[blk], c1 = offsets[blk + 1];
    const uint64_t stream_bytes = offsets[n_blocks];
    if (c1 <= c0 || c0 < body_offset || c1 > stream_bytes || c1 - c0 > 2u * kBlock) {
        // a range that does not fit the stream is an error; a block of more than 2 * 65536 stream bytes is valid
        // raw Snappy (non-minimal encodings) that only the general decoder takes
        if (tid == 0)
            atomicOr(status, c1 > c0 && c0 >= body_offset && c1 <= stream_bytes ? SNAPPY_B200_ST_FRAMING
                                                                                 : SNAPPY_B200_ST_CORRUPT);
        return;
    }
    uint8_t *out = out_base + blk * (uint64_t)kBlock;
    const uint64_t oleft = total_out - blk * (uint64_t)kBlock;
    const uint32_t olen = oleft < kBlock ? (uint32_t)oleft : kBlock;

    // ---- a block that is one literal (incompressible data): straight global -> global
    {
        const uint8_t *p = stream + c0;
        const uint32_t tag = __ldg(p);
        const uint32_t k = (tag >> 2) - 59u; // length bytes when this is a long-form literal
        if ((tag & 3u) == 0 && (tag >> 2) >= 60u && c1 - c0 > 1 + k) {
            uint32_t raw = 0;
            for (uint32_t i = 0; i < k; ++i)
                raw |= (uint32_t)__ldg(p + 1 + i) << (8u * i);
            if ((uint64_t)raw + 1 == olen && c1 - c0 == 1ull + k + olen) {
                coop_copy_ro(out, p + 1 + k, olen, tid, kThreads);
                return;
            }
        }
    }

    // ---- stream geometry.  Positions P below are relative to the first segment the block touches.
    const uint64_t b0 = c0 - body_offset, b1 = c1 - body_offset;
    const uint64_t t0 = b0 / kSegB, t1 = (b1 - 1) / kSegB;
    const uint8_t *__restrict__ in = stream + body_offset + t0 * kSegB;
    const uint32_t first = (uint32_t)(b0 - t0 * kSegB); // where the block starts
    const uint32_t lim = (uint32_t)(b1 - t0 * kSegB);   // where it ends
    const uint32_t mis = (uint32_t)reinterpret_cast<uintptr_t>(in) & 15u;
    const uint8_t *gsrc0 = in - mis; // 16-byte aligned
    const uint8_t *gend = reinterpret_cast<const uint8_t *>(
        (reinterpret_cast<uintptr_t>(stream + stream_bytes) + 15u) & ~uintptr_t(15)); // same 16-byte granule as the last byte
    const uint32_t nchunk = ((uint32_t)(t1 - t0) + kChunkSegs) / kChunkSegs;
    const int64_t obase = (int64_t)(blk * (uint64_t)kBlock);

    for (uint32_t i = tid; i < 256; i += kThreads)
        sm.lut[i] = (uint16_t)tag_facts(i);
    if (tid == 0) {
        mbar_init(&sm.mbar[0], 1);
        mbar_init(&sm.mbar[1], 1);
        sm.produced = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
    }
    __syncthreads();
    auto issue = [&](uint32_t j) {
        const uint8_t *g = gsrc0 + (size_t)j * kChunkBytes;
        const uint64_t avail = (uint64_t)(gend - g);
        const uint32_t bytes = avail < kStageBytes ? (uint32_t)avail : kStageBytes;
        mbar_expect_tx(&sm.mbar[j & 1u], bytes);
        bulk_g2s(sm.stage[j & 1u], g, bytes, &sm.mbar[j & 1u]);
    };
    if (tid == 0)
        issue(0);

    uint32_t err = 0;
    for (uint32_t j = 0; j < nchunk; ++j) {
        const uint32_t buf = j & 1u;
        if (tid == 0 && j + 1 < nchunk)
            issue(j + 1); // the other buffer: its last readers passed the barrier that ended chunk j-1
        if (tid <= kChunkSegs) {
            const uint64_t t = t0 + (uint64_t)j * kChunkSegs + tid;
            int64_t s = t > t1 ? (int64_t)olen : (int64_t)__ldg(outoff + t) - obase;
            s = s < 0 ? 0 : (s > (int64_t)olen ? (int64_t)olen : s);
            sm.seg_start[tid] = (uint32_t)s;
            if (tid < kChunkSegs)
                sm.seg_hwm[tid] = (uint32_t)s;
        }
        mbar_wait(&sm.mbar[buf], (j >> 1) & 1u);
        __syncthreads();

        // stg[P] = stream byte at position P, for the positions of this chunk (+ halo)
        const uint8_t *stg = sm.stage[buf] + mis - (size_t)j * kChunkBytes;
        uint32_t fr = 0; // first segment of the chunk not known to be finished
        for (uint32_t s = warp; s < kChunkSegs; s += kWarps) {
            const uint64_t t = t0 + (uint64_t)j * kChunkSegs + s;
            if (t > t1)
                break;
            const uint4 sv = __ldg(starts + t);
            const uint32_t R[4] = {sv.x, sv.y, sv.z, sv.w};
            const uint32_t seg_lo = (j * kChunkSegs + s) * kSegB;
            const uint32_t w = lane >> 3, sh = (lane & 7u) * 4u; // my nibble of the 128-bit start map
            const uint32_t Rw = w == 0 ? R[0] : (w == 1 ? R[1] : (w == 2 ? R[2] : R[3]));
            const uint32_t nib = (Rw >> sh) & 15u;
            const uint32_t cnt = __popc(nib);
            const bool has0 = cnt >= 1, has1 = cnt >= 2;
            const uint32_t pos0 = seg_lo + 4 * lane + (uint32_t)(__ffs((int)nib) - 1);
            const uint32_t pos1 = seg_lo + 4 * lane + (uint32_t)(31 - __clz((int)nib));
            // ---- phase A: headers
            const uint32_t v0 = lds_le32_any(stg + (has0 ? pos0 : seg_lo));
            const uint32_t v1 = lds_le32_any(stg + (has1 ? pos1 : seg_lo));
            const Header h0 = decode_header_lut(sm.lut, v0, pos0), h1 = decode_header_lut(sm.lut, v1, pos1);
            uint32_t len0 = has0 ? h0.len : 0u, len1 = has1 ? h1.len : 0u;
            uint32_t info0 = h0.info, info1 = h1.info;
            if (has0 && h0.slow) { // the fifth header byte: top of a 4-byte literal length / of a copy-4 offset
                const uint32_t top = (uint32_t)stg[pos0 + 4] << 24;
                if (h0.is_lit)
                    len0 = ((v0 >> 8) | top) + 1u;
                else
                    info0 = (v0 >> 8) | top;
            }
            if (has1 && h1.slow) {
                const uint32_t top = (uint32_t)stg[pos1 + 4] << 24;
                if (h1.is_lit)
                    len1 = ((v1 >> 8) | top) + 1u;
                else
                    info1 = (v1 >> 8) | top;
            }
            // output offsets (lengths clamped so that an absurd literal length cannot wrap the sum)
            const uint32_t lc0 = min(len0, kBlock + 1u), lc1 = min(len1, kBlock + 1u);
            uint32_t end = lc0 + lc1;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t u = __shfl_up_sync(kFull, end, d);
                if ((int)lane >= d)
                    end += u;
            }
            const int64_t segbase = (int64_t)__ldg(outoff + t) - obase; // negative: the previous block's elements
            const int64_t d0 = segbase + (int64_t)(end - lc0 - lc1), d1 = d0 + lc0;
            // own elements: those of this block (only the first / last segment can hold others)
            bool ok0 = has0 && pos0 >= first && pos0 < lim, ok1 = has1 && pos1 >= first && pos1 < lim;
            uint32_t e = cnt > 2 ? SNAPPY_B200_ST_CORRUPT : 0u;
            if (ok0) {
                if (pos0 + h0.hdr > lim || (h0.is_lit && (uint64_t)pos0 + h0.hdr + len0 > lim) ||
                    (!h0.is_lit && info0 == 0))
                    e |= SNAPPY_B200_ST_CORRUPT, ok0 = false;
                else if (d0 < 0 || d0 + len0 > olen)
                    e |= SNAPPY_B200_ST_FRAMING, ok0 = false;
                else if (!h0.is_lit && (int64_t)info0 > d0) // reaches back into an earlier block
                    e |= (uint64_t)info0 > (blk_base + blk) * (uint64_t)kBlock + (uint64_t)d0 ? SNAPPY_B200_ST_CORRUPT
                                                                                              : SNAPPY_B200_ST_FRAMING,
                        ok0 = false;
            }
            if (ok1) {
                if (pos1 + h1.hdr > lim || (h1.is_lit && (uint64_t)pos1 + h1.hdr + len1 > lim) ||
                    (!h1.is_lit && info1 == 0))
                    e |= SNAPPY_B200_ST_CORRUPT, ok1 = false;
                else if (d1 < 0 || d1 + len1 > olen)
                    e |= SNAPPY_B200_ST_FRAMING, ok1 = false;
                else if (!h1.is_lit && (int64_t)info1 > d1)
                    e |= (uint64_t)info1 > (blk_base + blk) * (uint64_t)kBlock + (uint64_t)d1 ? SNAPPY_B200_ST_CORRUPT
                                                                                              : SNAPPY_B200_ST_FRAMING,
                        ok1 = false;
            }
            err |= e;
            const uint32_t mylen = (ok0 ? len0 : 0u) + (ok1 ? len1 : 0u);
            const uint32_t seglen = __reduce_add_sync(kFull, mylen);
            if (lane == 0 && seglen)
                atomicAdd(&sm.produced, seglen);
            const uint32_t dst0 = (uint32_t)d0, dst1 = (uint32_t)d1;

            // ---- phase B: literals
            const bool lit0 = ok0 && h0.is_lit, lit1 = ok1 && h1.is_lit;
            if (lit0 && len0 <= kShortLit)
                copy_fwd(sm.tile + dst0, stg + info0, len0);
            if (lit1 && len1 <= kShortLit)
                copy_fwd(sm.tile + dst1, stg + info1, len1);
            unsigned L = __ballot_sync(kFull, lit0 && len0 > kShortLit);
            while (L) { // long literals: the whole warp, straight from the stream in global memory
                const int src = __ffs((int)L) - 1;
                L &= L - 1;
                const uint32_t dd = __shfl_sync(kFull, dst0, src), ll = __shfl_sync(kFull, len0, src),
                               ii = __shfl_sync(kFull, info0, src);
                coop_copy_ro(sm.tile + dd, in + ii, ll, lane, 32);
            }
            L = __ballot_sync(kFull, lit1 && len1 > kShortLit);
            while (L) {
                const int src = __ffs((int)L) - 1;
                L &= L - 1;
                const uint32_t dd = __shfl_sync(kFull, dst1, src), ll = __shfl_sync(kFull, len1, src),
                               ii = __shfl_sync(kFull, info1, src);
                coop_copy_ro(sm.tile + dd, in + ii, ll, lane, 32);
            }

            // ---- phase C: copies, in rounds under the high-water mark
            bool pend0 = ok0 && !h0.is_lit, pend1 = ok1 && !h1.is_lit;
            // a copy is ready when everything below `need` is final (a self-overlapping copy: below its own start)
            const uint32_t need0 = info0 >= len0 ? dst0 - info0 + len0 : dst0;
            const uint32_t need1 = info1 >= len1 ? dst1 - info1 + len1 : dst1;
            const uint32_t seg_end = sm.seg_start[s + 1];
            uint32_t published = sm.seg_start[s];
            uint32_t hlast = 0;
            for (;;) {
                const uint32_t mine = pend0 ? dst0 : (pend1 ? dst1 : 0xffffffffu);
                const uint32_t lh = __reduce_min_sync(kFull, mine);
                const uint32_t cur = lh == 0xffffffffu ? seg_end : lh; // this segment is final below cur
                if (cur != published) {
                    __syncwarp();
                    if (lane == 0)
                        st_release(&sm.seg_hwm[s], cur);
                    published = cur;
                }
                if (lh == 0xffffffffu)
                    break;
                while (fr < s) {
                    hlast = ld_acquire(&sm.seg_hwm[fr]);
                    if (hlast != sm.seg_start[fr + 1])
                        break;
                    ++fr;
                }
                const uint32_t G = fr == s ? lh : hlast;
                bool did = false;
                if (pend0 && need0 <= G) {
                    do_copy(sm.tile + dst0, info0, len0);
                    pend0 = false;
                    did = true;
                }
                if (pend1 && need1 <= G) {
                    do_copy(sm.tile + dst1, info1, len1);
                    pend1 = false;
                    did = true;
                }
                if (!__any_sync(kFull, did))
                    __nanosleep(64); // waiting for an earlier segment: leave the issue slots to its warp
            }
        }
        __syncthreads();
    }
    // a refused element has produced nothing: the byte count is only a finding when every element was taken
    // (a valid unframed stream must report ST_FRAMING alone, so that the general decoder takes it)
    const int refused = __syncthreads_or(err != 0);
    if (tid == 0 && !refused && sm.produced != olen)
        err |= SNAPPY_B200_ST_CORRUPT;
    if (err)
        atomicOr(status, err);

    // ---- the finished tile goes out once
    fence_proxy_async();
    __syncthreads();
    if ((reinterpret_cast<uintptr_t>(out) & 15u) == 0) {
        const uint32_t bulk = olen & ~15u;
        if (tid == 0 && bulk) {
            for (uint32_t o = 0; o < bulk; o += 16384u)
                bulk_s2g(out + o, sm.tile + o, min(16384u, bulk - o));
            bulk_commit_wait_read();
        }
        if (tid < (olen & 15u))
            out[bulk + tid] = sm.tile[bulk + tid];
    } else {
        for (uint32_t i = tid; i < olen; i += kThreads)
            out[i] = sm.tile[i];
    }
}

std::once_flag g_attr_once[64];

} // namespace

cudaError_t launch_decode_tile(const uint8_t *d_stream, uint64_t body_offset, const uint64_t *d_offsets,
                               const uint4 *d_starts, const uint64_t *d_outoff, uint64_t n_blocks, uint64_t total_out,
                               uint8_t *d_out, uint32_t *d_status, uint64_t blk_base, cudaStream_t st,
                               uint64_t *launches)
{
    if (n_blocks == 0)
        return cudaSuccess;
    if (n_blocks > 0x7fffffffull)
        return cudaErrorInvalidValue;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess)
        return e;
    // the opt-in to > 48 KiB of dynamic shared memory is per device
    cudaError_t attr = cudaSuccess;
    std::call_once(g_attr_once[dev & 63], [&] {
        attr = cudaFuncSetAttribute(k_decode_tile, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TileSmem));
    });
    if (attr != cudaSuccess)
        return attr;
    k_decode_tile<<<(unsigned)n_blocks, kThreads, sizeof(TileSmem), st>>>(d_stream, body_offset, d_offsets, d_starts,
                                                                         d_outoff, total_out, d_out, d_status, n_blocks,
                                                                         blk_base);
    *launches += 1;
    return cudaGetLastError();
}

} // namespace sb200
