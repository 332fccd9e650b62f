// lanecopy.cuh -- byte moves done by ONE lane, any alignment, 16 bytes per step with word accesses.
//
// The tile decoder (decode_tile.cu) gives every element (literal or copy, src/snappy_decompression.c:232-239,
// :273-280) to one lane; the destination is always shared memory, the source shared or global memory (generic
// pointers).
#pragma once

#include "common.cuh"

namespace sb200 {

struct V4 {
    uint32_t a, b, c, d;
};

// Bytes [src, src + n), n <= 16, as four little-endian words (bytes past n are don't-care).  Only the
// aligned words that hold a requested byte are read.
__device__ __forceinline__ V4 load16(const uint8_t *src, uint32_t n)
{
    const uint32_t sa = (uint32_t)reinterpret_cast<uintptr_t>(src) & 3u;
    const uint32_t *w = reinterpret_cast<const uint32_t *>(src - sa);
    const uint32_t need = sa + n; // bytes of the aligned words that are touched
    const uint32_t w0 = w[0];
    const uint32_t w1 = need > 4 ? w[1] : 0u;
    const uint32_t w2 = need > 8 ? w[2] : 0u;
    const uint32_t w3 = need > 12 ? w[3] : 0u;
    const uint32_t w4 = need > 16 ? w[4] : 0u;
    const uint32_t sh = sa * 8u;
    V4 v;
    v.a = __funnelshift_r(w0, w1, sh);
    v.b = __funnelshift_r(w1, w2, sh);
    v.c = __funnelshift_r(w2, w3, sh);
    v.d = __funnelshift_r(w3, w4, sh);
    return v;
}

// The first n bytes of v to [dst, dst + n): bytes up to the next word boundary, whole words, tail bytes.
__device__ __forceinline__ void store16(uint8_t *dst, const V4 &v, uint32_t n)
{
    const uint32_t da = (uint32_t)reinterpret_cast<uintptr_t>(dst) & 3u;
    const uint32_t h = min(n, (4u - da) & 3u);
    if (h > 0)
        dst[0] = (uint8_t)v.a;
    if (h > 1)
        dst[1] = (uint8_t)(v.a >> 8);
    if (h > 2)
        dst[2] = (uint8_t)(v.a >> 16);
    const uint32_t sh = h * 8u;
    const uint32_t u0 = __funnelshift_r(v.a, v.b, sh), u1 = __funnelshift_r(v.b, v.c, sh),
                   u2 = __funnelshift_r(v.c, v.d, sh), u3 = v.d >> sh;
    uint32_t *dw = reinterpret_cast<uint32_t *>(dst + h);
    const uint32_t r = n - h, nf = r >> 2;
    if (nf > 0)
        dw[0] = u0;
    if (nf > 1)
        dw[1] = u1;
    if (nf > 2)
        dw[2] = u2;
    if (nf > 3)
        dw[3] = u3;
    const uint32_t t = r & 3u;
    if (t) {
        const uint32_t tv = nf == 0 ? u0 : (nf == 1 ? u1 : (nf == 2 ? u2 : u3));
        uint8_t *dt = dst + h + 4u * nf;
        dt[0] = (uint8_t)tv;
        if (t > 1)
            dt[1] = (uint8_t)(tv >> 8);
        if (t > 2)
            dt[2] = (uint8_t)(tv >> 16);
    }
}

} // namespace sb200
