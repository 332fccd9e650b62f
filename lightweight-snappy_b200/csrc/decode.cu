// decode.cu -- K4/K5: decompression, one warp per 64 KiB output block.
//
// reference: decompressor src/snappy_decompression.c:290-333 (tag dispatch), do_literal
// :193-224, write_literal :232-239, do_copy :253-265, write_copy :273-280.
//
// The reference walks one element at a time.  Both kernels here decode many elements per step
// and then produce the output bytes of all of them 32 at a time:
//   * a warp prefix sum of the output lengths gives every element its output offset;
//   * the elements go into a small shared-memory table; in every round the lane that produces
//     output byte k finds its element from a bit map of the element starts inside the round
//     (rank = #elements before the round + popc(map up to k) - 1), then reads either the
//     stream (literal) or the output written earlier (copy; offset < length repeats the
//     pattern, write_copy :273-280).  A source byte produced by the very same round is
//     resolved inside the round: k_decode_seg sends every lane to the root of its chain (a
//     literal or a byte written earlier) by pointer doubling over shuffles, k_decode_warp follows
//     the chain back through the round's elements.
// Literals of 64 bytes or more are moved by the 16-byte copy loop, and the rare element kinds
// whose header does not fit the 4 bytes a lane holds (copy-4, 4-byte literal length) take a
// one-element path.  Copies read the output through global memory; __syncwarp() orders the
// read-after-write.  Unlike the reference, malformed input is detected and reported in
// *status instead of being undefined behaviour (SURVEY.md Q7).
//
// What differs is how a step finds its elements:
//   k_decode_seg   (index-less streams, after K0) takes them from the exact element-start bit
//                  maps K0 leaves per 128-byte stream segment.  A step is one segment: lane l
//                  owns the (at most two) elements that start in stream bytes 4l..4l+3, their
//                  rank is a popcount of the map below, headers come from a tag table.
//   k_decode_warp  (caller supplied block index, no K0) looks at a 32-byte window: every lane
//                  decodes the byte at its offset as if an element started there, and the
//                  real starts are the orbit of lane 0 under "next = lane + element size",
//                  found with pointer doubling over shuffles and five warp-wide OR reductions.
#include <cstdlib>

#include "common.cuh"
#include "tags.cuh"

namespace sb200 {

constexpr uint32_t kLongLiteral = 64;
constexpr uint32_t kSegBytes = 128; // K0 segment size (csrc/index.cu)

// One element, handled by the whole warp (warp-uniform arguments): long literals, copy-4,
// literals with a 4-byte length.  `in` + ip is the tag, lim the end of the compressed block.
// Returns an error status or 0; advances ip / op.
__device__ __forceinline__ uint32_t single_element(const uint8_t *__restrict__ in, uint32_t lim, uint32_t t0,
                                                   uint8_t *out, uint32_t olen, uint64_t blk, uint32_t &ip, uint32_t &op,
                                                   uint32_t lane)
{
    const uint32_t tg = t0 & 0xffu;
    const uint32_t ty = tg & 3u;
    const uint32_t b4 = (ip + 4 < lim) ? (uint32_t)__ldg(in + ip + 4) : 0u;
    uint32_t h, l;
    if (ty == 0) {
        const uint32_t m = tg >> 2;
        const uint32_t k = m >= 60 ? m - 59 : 0;
        h = 1 + k;
        const uint32_t raw = (t0 >> 8) | (b4 << 24);
        l = k == 0 ? m : (k == 4 ? raw : raw & ((1u << (8 * k)) - 1u));
        if (ip + h > lim || l >= olen - op || (uint64_t)ip + h + l + 1 > lim)
            return (ip + h <= lim && (uint64_t)ip + h + l + 1 <= lim) ? SNAPPY_B200_ST_FRAMING
                                                                      : SNAPPY_B200_ST_CORRUPT;
        l += 1;
        coop_copy_ro(out + op, in + ip + h, l, lane, 32);
        ip += h + l;
    } else {
        uint32_t off;
        if (ty == 1) {
            h = 2, l = ((tg >> 2) & 7u) + 4, off = ((tg >> 5) << 8) | ((t0 >> 8) & 0xffu);
        } else if (ty == 2) {
            h = 3, l = (tg >> 2) + 1, off = (t0 >> 8) & 0xffffu;
        } else { // copy-4 (src/snappy_decompression.c:323-327)
            h = 5, l = (tg >> 2) + 1, off = (t0 >> 8) | (b4 << 24);
        }
        if (ip + h > lim || off == 0)
            return SNAPPY_B200_ST_CORRUPT;
        if (off > op || l > olen - op)
            return ((uint64_t)off > blk * (uint64_t)kBlock + op) ? SNAPPY_B200_ST_CORRUPT : SNAPPY_B200_ST_FRAMING;
        __syncwarp();
        for (uint32_t i = lane; i < l; i += 32)
            out[op + i] = out[op - off + (off >= l ? i : i % off)];
        ip += h;
    }
    op += l;
    __syncwarp();
    return 0;
}

// Produces T output bytes at out[op ..) from the ne elements in `elems`:
//   x = window-relative start, y = offset (0: literal) | (floor(2^15/offset)+1) << 16 when the copy
//   overlaps itself, (z,w) = pointer p such that byte k of the window is p[k] -- the stream for a
//   literal, out + op - offset for a copy.
// In every round the lane that produces output byte k finds its element from a bit map of the
// element starts inside the round (rank = #elements before the round + popc(map up to k) - 1).
// A copy whose source byte is produced by the very same round is followed back through the
// round's elements until it leaves the round or lands in a literal.
__device__ __forceinline__ void produce(uint8_t *out, uint32_t op, uint32_t T, const uint4 *elems, uint32_t ne,
                                        uint32_t lane)
{
    const uint32_t my_start = lane < ne ? elems[lane].x : 0xffffffffu;
    for (uint32_t c = 0; c < T; c += 32) {
        const uint32_t before = __popc(__ballot_sync(kFull, my_start < c));
        const uint32_t rel = my_start - c;
        const unsigned B = __reduce_or_sync(kFull, rel < 32u ? 1u << rel : 0u);
        uint32_t k = c + lane; // window-relative output byte
        bool pending = k < T;
        uint32_t val = 0;
        do {
            if (pending) {
                const uint32_t r = before + __popc(B & (0xffffffffu >> (31u - (k - c)))) - 1u;
                const uint4 e = elems[r];
                const uint32_t off = e.y & 0xffffu, inv = e.y >> 16;
                uint32_t kk = k;
                if (inv) { // write_copy :273-280: byte i comes from i mod offset when the copy overlaps itself
                    const uint32_t i = k - e.x;
                    kk = e.x + i - off * ((i * inv) >> 15);
                }
                if (off == 0 || kk < c + off) {
                    // a literal, or a copy whose source was written by an earlier step / round
                    const uint8_t *p = reinterpret_cast<const uint8_t *>(((uint64_t)e.w << 32) | e.z);
                    val = p[kk];
                    pending = false;
                } else {
                    k = kk - off; // produced by this very round: follow it back
                }
            }
        } while (__any_sync(kFull, pending));
        if (c + lane < T)
            out[op + c + lane] = (uint8_t)val;
        __syncwarp(); // the next round may read what this one wrote
    }
}

// Shared tail of a step: prefix sum, validation, table, production.  `mine` lanes hold an
// element (h, at stream position pos relative to `in`, lim = end of the compressed block);
// rank = number of element lanes below, ne = their total.  Returns an error status or 0; adds
// the produced bytes to op.
__device__ __forceinline__ uint32_t run_step(const uint8_t *__restrict__ in, uint32_t lim, uint8_t *out, uint32_t olen,
                                             uint32_t &op, bool mine, uint32_t rank, uint32_t ne, const Header &h,
                                             uint32_t pos, uint4 *elems, uint32_t lane)
{
    const uint32_t mylen = mine ? h.len : 0u;
    uint32_t end = mylen;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(kFull, end, d);
        if ((int)lane >= d)
            end += t;
    }
    const uint32_t T = __shfl_sync(kFull, end, 31);
    const uint32_t start = end - mylen; // window-relative output offset of my element
    const bool bad_corrupt = mine && (pos + h.hdr > lim || (h.is_lit && pos + h.hdr + h.len > lim) ||
                                      (!h.is_lit && h.info == 0));
    bool bad_framing = mine && !h.is_lit && h.info > op + start;
    if (T > olen - op)
        bad_framing = true;
    const unsigned BC = __ballot_sync(kFull, bad_corrupt), BF = __ballot_sync(kFull, bad_framing);
    if (BC | BF)
        return BC ? SNAPPY_B200_ST_CORRUPT : SNAPPY_B200_ST_FRAMING;
    if (mine) {
        uint32_t y = 0;
        const uint8_t *p;
        if (h.is_lit) {
            p = in + h.info - start; // byte k of the window = stream byte info + (k - start)
        } else {
            const uint32_t off = h.info; // <= 65535 here (copy-4 takes the one-element path)
            y = off | (off < h.len ? (32768u / off + 1u) << 16 : 0u);
            p = out + op - off; // byte k of the window = output byte op + k - off
        }
        const uint64_t pa = reinterpret_cast<uint64_t>(p);
        elems[rank] = make_uint4(start, y, (uint32_t)pa, (uint32_t)(pa >> 32));
    }
    __syncwarp(); // also: stores of earlier steps are visible to every lane from here
    produce(out, op, T, elems, ne, lane);
    op += T;
    return 0;
}

// ------------------------------------------------------------------ segment-driven decoder
// One step = one 128-byte stream segment.  Lane l looks at the four start bits of stream bytes
// 4l..4l+3: an element is at least two bytes long, so at most two elements start there, and
// the rank of the first one is a popcount of the map below.  All elements of the segment
// (<= 64) go into the shared-memory table at once; their output offsets come from one warp
// prefix sum over the per-lane sums.
constexpr uint32_t kSegElems = 64;
constexpr uint32_t kRunBytes = kSegElems * 64; // output bytes of a run of ordinary elements (each <= 64)

struct SegSmem {
    uint16_t lut[256];
    uint4 elems[kSegElems];
    uint32_t bm[kRunBytes / 32 + 4]; // element starts inside the current run, one bit per output byte
};

// Bit 31 of a source position: the byte is in the stream (relative to `in`), not in the output (relative
// to the block's `out`, always below 65536).  A literal's stream position is below 2 * 65536 + 256.
constexpr uint32_t kFromStream = 0x80000000u;

// Table entry of an element that starts at window-relative output byte `start` (after it: `len` bytes,
// offset `info` for a copy, stream position `info` of the first literal byte):
//   x = start, y = offset (0: literal) | (floor(2^15/offset)+1) << 16 when the copy overlaps itself,
//   z = source position of window byte 0, so that window byte k comes from position z + k (32-bit wrap-around),
//   kFromStream set for a literal; w is unused.
// A special element (one-element path) has y = 0xffffffff and z = the stream position `pos` of its tag.
__device__ __forceinline__ uint4 seg_entry(uint32_t op, uint32_t start, const Header &h, uint32_t len, uint32_t pos,
                                           bool special)
{
    if (special)
        return make_uint4(start, 0xffffffffu, pos, 0u);
    const uint32_t off = h.is_lit ? 0u : h.info; // <= 65535 (copy-4 is special)
    const uint32_t y = off | (off != 0 && off < len ? (32768u / off + 1u) << 16 : 0u);
    return make_uint4(start, y, h.is_lit ? h.info - start + kFromStream : op - off, 0u);
}

// Produces the output bytes [k_lo, k_hi) (window-relative) of the elements e_lo.. of the table;
// `bm` holds their starts relative to k_lo.  Same per-byte rule as produce() above, but a source byte produced
// by the same round is resolved by pointer doubling instead of following the chain back.
//
// The lane of byte k = c + lane looks its element up once.  A literal, or a copy whose source byte
// s = kk - offset lies before the round (s < c), is a root and knows the position it reads; any other lane
// copies lane s - c < lane, its parent.  Five pointer-doubling shuffles take every lane to its root (a chain
// inside a round has fewer than 32 links), one more fetches the root's position, and every lane does exactly
// one load.  Rounds in which no lane has a parent skip the shuffles.  (Measured, B200, 1 GiB per class: a
// doubling loop that ends on a ballot once every parent is a root lost on low-entropy data, 3.83 against
// 3.64 ms; five shuffles in every round lost on text, 6.10 against 5.88 ms; following each chain back through
// the table, as produce() does, lost too, DESIGN.md §6.)
__device__ __forceinline__ void produce_run(const uint8_t *__restrict__ in, uint8_t *out, uint32_t op, uint32_t k_lo,
                                            uint32_t k_hi, uint32_t e_lo, const SegSmem &sm, uint32_t lane)
{
    const unsigned le_mask = 0xffffffffu >> (31u - lane);
    uint32_t before = e_lo; // table index of the first element that starts in this round, if any does
    uint8_t *o = out + op + k_lo + lane;
    for (uint32_t c = k_lo; c < k_hi; c += 32, o += 32) {
        const unsigned B = sm.bm[(c - k_lo) >> 5];
        // every lane's look-up is a valid table entry (the element at or before it), also past k_hi
        const uint4 e = sm.elems[before + __popc(B & le_mask) - 1u];
        const uint32_t off = e.y & 0xffffu, inv = e.y >> 16;
        uint32_t kk = c + lane;
        if (inv) { // write_copy :273-280: byte i comes from i mod offset when the copy overlaps itself
            const uint32_t i = kk - e.x;
            kk = e.x + i - off * ((i * inv) >> 15);
        }
        uint32_t src = e.z + kk;
        // produced by this very round: the parent is a lower lane (a lane past k_hi has no children)
        uint32_t parent = off != 0 && kk >= c + off ? kk - off - c : lane;
        if (__any_sync(kFull, parent != lane)) {
#pragma unroll
            for (int d = 0; d < 5; ++d)
                parent = __shfl_sync(kFull, parent, parent);
            src = __shfl_sync(kFull, src, parent);
        }
        if (c + lane < k_hi) {
            const uint8_t *base = (src & kFromStream) ? in : out;
            *o = base[src & ~kFromStream];
        }
        before += __popc(B);
        __syncwarp(); // the next round may read what this one wrote
    }
}

__global__ void __launch_bounds__(64, 20) k_decode_seg(const uint8_t *__restrict__ stream, uint64_t body_offset,
                                                         const uint64_t *__restrict__ offsets,
                                                         const uint4 *__restrict__ starts, uint64_t total_out,
                                                         uint8_t *out_base, uint32_t *__restrict__ status,
                                                         uint64_t n_blocks, uint64_t blk_base,
                                                         const uint32_t *__restrict__ order)
{
    __shared__ SegSmem sm2[2];
    SegSmem &sm = sm2[threadIdx.x >> 5];
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t slot = blockIdx.x * 2ull + (threadIdx.x >> 5);
    if (slot >= n_blocks)
        return;
    if (*reinterpret_cast<volatile uint32_t *>(status) != 0)
        return; // K0 rejected the stream: its maps are not trustworthy
    const uint64_t blk = order ? order[slot] : slot; // longest blocks first (k_block_order)
    const uint64_t c0 = offsets[blk], c1 = offsets[blk + 1];
    const uint64_t stream_bytes = offsets[n_blocks];
    if (c1 <= c0 || c0 < body_offset || c1 > stream_bytes || c1 - c0 > 2u * kBlock) {
        // a range that does not fit the stream is an error; a block of more than 2 * 65536 stream bytes is valid
        // raw Snappy (non-minimal encodings) that only the general decoder takes
        if (lane == 0)
            atomicOr(status, c1 > c0 && c0 >= body_offset && c1 <= stream_bytes ? SNAPPY_B200_ST_FRAMING
                                                                                 : SNAPPY_B200_ST_CORRUPT);
        return;
    }
    {
        const uint64_t oleft0 = total_out - blk * (uint64_t)kBlock;
        if (one_literal_block(stream, c0, c1, oleft0 < kBlock ? (uint32_t)oleft0 : kBlock))
            return; // k_copy_literal_blocks has moved it
    }
    const uint32_t *last_word = reinterpret_cast<const uint32_t *>(
        reinterpret_cast<uintptr_t>(stream + stream_bytes - 1) & ~uintptr_t(3));
    // stream positions below are relative to the first segment the block touches
    const uint64_t b0 = c0 - body_offset, b1 = c1 - body_offset; // body-relative
    const uint64_t t0 = b0 / kSegBytes, t1 = (b1 - 1) / kSegBytes;
    const uint8_t *__restrict__ in = stream + body_offset + t0 * kSegBytes;
    const uint32_t first = (uint32_t)(b0 - t0 * kSegBytes); // where the block starts
    const uint32_t lim = (uint32_t)(b1 - t0 * kSegBytes);   // where it ends
    uint8_t *out = out_base + blk * (uint64_t)kBlock;
    const uint64_t oleft = total_out - blk * (uint64_t)kBlock;
    const uint32_t olen = oleft < kBlock ? (uint32_t)oleft : kBlock;
    const uint4 *__restrict__ seg_starts = starts + t0;
    const uint32_t ns = (uint32_t)(t1 - t0); // segments t0..t1 are s = 0..ns
    const uint32_t w = lane >> 3, sh = (lane & 7u) * 4u; // my nibble of the 128-bit start map
    for (uint32_t i = lane; i < 256; i += 32)
        sm.lut[i] = (uint16_t)tag_facts(i);
    __syncwarp();

    uint32_t op = 0, err = 0;
    for (uint32_t s = 0; s <= ns && !err; ++s) {
        const uint4 sv = __ldg(seg_starts + s);
        uint32_t R[4] = {sv.x, sv.y, sv.z, sv.w};
        const uint32_t seg_lo = s * kSegBytes;
        // the block is one serial chain: have the stream (and its maps) on their way before they are needed
        // (every 8 segments: the 8 stream lines 16..23 segments ahead, one lane each, and the line of their maps)
        if ((s & 7u) == 0 && lane <= 8 && s + 16 + lane <= ns) {
            if (lane < 8)
                prefetch_l2(in + seg_lo + (16 + lane) * kSegBytes);
            else
                prefetch_l2(seg_starts + s + 16);
        }
        // keep only the starts that belong to this block (only the first / last segment can hold others)
        if (s == 0 || s == ns)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t lo = seg_lo + 32 * q; // stream position of bit 0 of this word
                if (lo + 32 <= first || lo >= lim) {
                    R[q] = 0;
                } else {
                    if (lo < first)
                        R[q] &= ~((1u << (first - lo)) - 1u);
                    if (lo + 32 > lim)
                        R[q] &= (1u << (lim - lo)) - 1u;
                }
            }
        const uint32_t n0 = __popc(R[0]), n1 = n0 + __popc(R[1]), n2 = n1 + __popc(R[2]), ne = n2 + __popc(R[3]);
        if (ne == 0)
            continue;
        const uint32_t Rw = w == 0 ? R[0] : (w == 1 ? R[1] : (w == 2 ? R[2] : R[3]));
        const uint32_t nib = (Rw >> sh) & 15u;
        const uint32_t rank = (w == 0 ? 0u : (w == 1 ? n0 : (w == 2 ? n1 : n2))) + __popc(Rw & ((1u << sh) - 1u));
        const uint32_t cnt = __popc(nib);
        const bool has0 = cnt >= 1, has1 = cnt >= 2;
        // my (up to) two elements
        const uint32_t pos0 = seg_lo + 4 * lane + (uint32_t)(__ffs((int)nib) - 1);
        const uint32_t pos1 = seg_lo + 4 * lane + (uint32_t)(31 - __clz((int)nib));
        const uint32_t v0 = ld_le32_any(in + (has0 ? pos0 : seg_lo), last_word);
        const uint32_t v1 = ld_le32_any(in + (has1 ? pos1 : seg_lo), last_word);
        const Header h0 = decode_header_lut(sm.lut, v0, pos0), h1 = decode_header_lut(sm.lut, v1, pos1);
        const bool sp0 = has0 && (h0.slow || (h0.is_lit && h0.len >= kLongLiteral));
        const bool sp1 = has1 && (h1.slow || (h1.is_lit && h1.len >= kLongLiteral));
        // a 4-byte literal length does not fit v: take its top byte from the stream
        uint32_t len0 = has0 ? h0.len : 0u, len1 = has1 ? h1.len : 0u;
        if (has0 && h0.is_lit && h0.hdr == 5)
            len0 = (((v0 >> 8) | ((pos0 + 4 < lim ? (uint32_t)__ldg(in + pos0 + 4) : 0u) << 24))) + 1u;
        if (has1 && h1.is_lit && h1.hdr == 5)
            len1 = (((v1 >> 8) | ((pos1 + 4 < lim ? (uint32_t)__ldg(in + pos1 + 4) : 0u) << 24))) + 1u;
        // output offsets.  Lengths are clamped to one more than a block can hold before they are
        // summed (an absurd literal length cannot wrap the sum, and still trips the T > room test)
        const uint32_t lc0 = min(len0, kBlock + 1u), lc1 = min(len1, kBlock + 1u);
        uint32_t end = lc0 + lc1;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t u = __shfl_up_sync(kFull, end, d);
            if ((int)lane >= d)
                end += u;
        }
        const uint32_t T64 = __shfl_sync(kFull, end, 31);
        const uint32_t start0 = end - lc0 - lc1, start1 = start0 + lc0;
        const bool corrupt0 = has0 && (pos0 + h0.hdr > lim || (h0.is_lit && (uint64_t)pos0 + h0.hdr + len0 > lim) ||
                                       (!h0.is_lit && !h0.slow && h0.info == 0));
        const bool corrupt1 = has1 && (pos1 + h1.hdr > lim || (h1.is_lit && (uint64_t)pos1 + h1.hdr + len1 > lim) ||
                                       (!h1.is_lit && !h1.slow && h1.info == 0));
        bool framing = (has0 && !h0.is_lit && !h0.slow && h0.info > op + start0) ||
                       (has1 && !h1.is_lit && !h1.slow && h1.info > op + start1);
        if (T64 > olen - op)
            framing = true;
        const unsigned BC = __ballot_sync(kFull, corrupt0 || corrupt1 || cnt > 2), BF = __ballot_sync(kFull, framing);
        if (BC | BF) {
            err = BC ? SNAPPY_B200_ST_CORRUPT : SNAPPY_B200_ST_FRAMING;
            break;
        }
        const uint32_t T = T64;
        const unsigned S = __ballot_sync(kFull, sp0 || sp1);
        // ---- the table
        if (has0)
            sm.elems[rank] = seg_entry(op, start0, h0, len0, pos0, sp0);
        if (has1)
            sm.elems[rank + 1] = seg_entry(op, start1, h1, len1, pos1, sp1);
        if (S == 0) {
            // ---- the ordinary segment: one run
            const uint32_t words = (T + 31) >> 5;
            for (uint32_t i = lane; i < words; i += 32)
                sm.bm[i] = 0;
            __syncwarp();
            if (has0)
                atomicOr(&sm.bm[start0 >> 5], 1u << (start0 & 31u));
            if (has1)
                atomicOr(&sm.bm[start1 >> 5], 1u << (start1 & 31u));
            __syncwarp(); // also: stores of earlier steps are visible to every lane from here
            produce_run(in, out, op, 0, T, 0, sm, lane);
        } else {
            // ---- runs of ordinary elements between the special ones (long literals, copy-4, ...)
            __syncwarp();
            uint32_t e_lo = 0;
            while (e_lo < ne && !err) {
                // first special element at or after e_lo
                uint32_t mine = 0xffffffffu;
                if (sp0 && rank >= e_lo)
                    mine = rank;
                else if (sp1 && rank + 1 >= e_lo)
                    mine = rank + 1;
                const uint32_t e_sp = __reduce_min_sync(kFull, mine); // 0xffffffff: none
                const uint32_t e_hi = min(e_sp, ne);
                const uint32_t k_lo = sm.elems[e_lo].x;
                const uint32_t k_hi = e_hi < ne ? sm.elems[e_hi].x : T;
                if (e_hi > e_lo) {
                    const uint32_t words = (k_hi - k_lo + 31) >> 5;
                    for (uint32_t i = lane; i < words; i += 32)
                        sm.bm[i] = 0;
                    __syncwarp();
                    if (has0 && rank >= e_lo && rank < e_hi)
                        atomicOr(&sm.bm[(start0 - k_lo) >> 5], 1u << ((start0 - k_lo) & 31u));
                    if (has1 && rank + 1 >= e_lo && rank + 1 < e_hi)
                        atomicOr(&sm.bm[(start1 - k_lo) >> 5], 1u << ((start1 - k_lo) & 31u));
                    __syncwarp();
                    produce_run(in, out, op, k_lo, k_hi, e_lo, sm, lane);
                }
                if (e_hi < ne) {
                    uint32_t ip = sm.elems[e_hi].z, o2 = op + k_hi;
                    const uint32_t tv = ld_le32_any(in + ip, last_word);
                    err = single_element(in, lim, tv, out, olen, blk_base + blk, ip, o2, lane);
                }
                e_lo = e_hi + 1;
            }
        }
        op += T;
    }
    if (!err && op != olen)
        err = SNAPPY_B200_ST_CORRUPT;
    if (err && lane == 0)
        atomicOr(status, err);
}

// ------------------------------------------------------------------ window decoder (block index only)
// One compressed block of clen stream bytes at `in` into olen output bytes at `out`, by one warp.  `elems` is the
// warp's 32-entry shared table; `last_word` clamps the loads to the stream.  Returns an error status or 0.
// `blk` only tells ST_CORRUPT from ST_FRAMING for a copy that reaches before the block.
__device__ __forceinline__ uint32_t decode_block_warp(const uint8_t *__restrict__ in, uint32_t clen,
                                                      const uint32_t *__restrict__ last_word, uint8_t *out, uint32_t olen,
                                                      uint64_t blk, uint4 *elems, uint32_t lane)
{
    uint32_t ip = 0, op = 0;
    uint32_t err = 0;
    while (op < olen && !err) {
        if (ip >= clen) {
            err = SNAPPY_B200_ST_CORRUPT;
            break;
        }
        // ---- speculative decode of the element that would start at ip + lane
        const uint32_t pos = ip + lane;
        const bool inside = pos < clen;
        const uint32_t v = ld_le32_any(in + (inside ? pos : clen - 1), last_word);
        const Header h = decode_header(v, pos);
        const uint32_t size = h.hdr + (h.is_lit ? h.len : 0u); // stream bytes of the element

        // ---- which lanes are element starts: orbit of lane 0 under lane -> lane + size
        // (an element that ends at or past the end of the compressed block leaves the window)
        uint32_t j0 = (inside && pos + size < clen) ? min(lane + size, 32u) : 32u;
        uint32_t j1 = __shfl_sync(kFull, j0, j0 & 31);
        j1 = j0 < 32 ? j1 : 32u;
        uint32_t j2 = __shfl_sync(kFull, j1, j1 & 31);
        j2 = j1 < 32 ? j2 : 32u;
        uint32_t j3 = __shfl_sync(kFull, j2, j2 & 31);
        j3 = j2 < 32 ? j3 : 32u;
        uint32_t j4 = __shfl_sync(kFull, j3, j3 & 31);
        j4 = j3 < 32 ? j4 : 32u;
        unsigned M = 1u;
        M |= __reduce_or_sync(kFull, ((M >> lane) & 1u) && j4 < 32 ? 1u << j4 : 0u);
        M |= __reduce_or_sync(kFull, ((M >> lane) & 1u) && j3 < 32 ? 1u << j3 : 0u);
        M |= __reduce_or_sync(kFull, ((M >> lane) & 1u) && j2 < 32 ? 1u << j2 : 0u);
        M |= __reduce_or_sync(kFull, ((M >> lane) & 1u) && j1 < 32 ? 1u << j1 : 0u);
        M |= __reduce_or_sync(kFull, ((M >> lane) & 1u) && j0 < 32 ? 1u << j0 : 0u);

        // cut the step before the first element that needs special handling
        const bool special = h.slow || (h.is_lit && h.len >= kLongLiteral);
        const unsigned S = __ballot_sync(kFull, ((M >> lane) & 1u) && special);
        if (S & 1u) {
            const uint32_t v0 = __shfl_sync(kFull, v, 0);
            err = single_element(in, clen, v0, out, olen, blk, ip, op, lane);
            continue;
        }
        if (S)
            M &= (1u << (__ffs((int)S) - 1)) - 1u;
        const bool mine = (M >> lane) & 1u;
        const int last = 31 - __clz((int)M);
        const uint32_t consumed = __shfl_sync(kFull, lane + size, last);
        if (__ballot_sync(kFull, mine && !inside)) {
            err = SNAPPY_B200_ST_CORRUPT;
            break;
        }
        err = run_step(in, clen, out, olen, op, mine, __popc(M & ((1u << lane) - 1u)), __popc(M), h, pos, elems, lane);
        ip += consumed;
    }
    if (!err && ip != clen)
        err = SNAPPY_B200_ST_CORRUPT; // the index said this block ends at c1
    return err;
}

__global__ void __launch_bounds__(32) k_decode_warp(const uint8_t *__restrict__ stream,
                                                    const uint64_t *__restrict__ offsets, uint64_t total_out,
                                                    uint8_t *out_base, uint32_t *__restrict__ status)
{
    __shared__ uint4 elems[32];
    const uint32_t lane = threadIdx.x;
    const uint64_t blk = blockIdx.x;
    if (*reinterpret_cast<volatile uint32_t *>(status) != 0)
        return; // an earlier stage rejected the stream: the offsets are not trustworthy
    const uint64_t c0 = offsets[blk], c1 = offsets[blk + 1];
    const uint64_t stream_bytes = offsets[gridDim.x]; // entry n_blocks of the index = end of the stream
    const uint64_t clen64 = c1 - c0;
    if (c1 < c0 || c1 > stream_bytes || clen64 > 2u * kBlock) { // a compressor's block never needs more than 65536+1010
        // a longer block is valid raw Snappy (non-minimal encodings) that only the general decoder takes
        if (lane == 0)
            atomicOr(status, c1 < c0 || c1 > stream_bytes ? SNAPPY_B200_ST_CORRUPT : SNAPPY_B200_ST_FRAMING);
        return;
    }
    const uint8_t *__restrict__ in = stream + c0;
    const uint32_t *last_word = reinterpret_cast<const uint32_t *>(
        reinterpret_cast<uintptr_t>(stream + stream_bytes - 1) & ~uintptr_t(3));
    uint8_t *out = out_base + blk * (uint64_t)kBlock;
    const uint64_t oleft = total_out - blk * (uint64_t)kBlock;
    const uint32_t olen = oleft < kBlock ? (uint32_t)oleft : kBlock;
    const uint32_t err = decode_block_warp(in, (uint32_t)clen64, last_word, out, olen, blk, elems, lane);
    if (err && lane == 0)
        atomicOr(status, err);
}

// ------------------------------------------------------------------ general decoder (no framing assumed)
// Raw Snappy allows what no block-framed compressor emits: elements that straddle a 64 KiB output block
// and copies that reach back into earlier blocks (the reference decoder resolves any offset into its
// whole-file buffer, src/snappy_decompression.c:349, :253-280, copy-4 :323-327).  The block-parallel
// decoders report such streams as ST_FRAMING; this kernel then decodes them the way the reference does, one
// element after the other over the whole output, with one warp moving the bytes of each element.  It is a
// correctness fallback for rare foreign streams (about an element per microsecond), not a fast path.
// The element loop over stream bytes [ip, stream_bytes) into total_out bytes at `out`, one warp; copies reach at
// most back to out[0].  Returns an error status or 0.
__device__ __forceinline__ uint32_t decode_sequential_warp(const uint8_t *__restrict__ stream, uint64_t ip,
                                                           uint64_t stream_bytes, uint8_t *out, uint64_t total_out,
                                                           uint32_t lane)
{
    uint64_t op = 0;
    uint32_t err = 0;
    while (op < total_out) {
        if (ip >= stream_bytes) {
            err = SNAPPY_B200_ST_CORRUPT;
            break;
        }
        uint32_t b[5];
#pragma unroll
        for (int k = 0; k < 5; ++k)
            b[k] = ip + k < stream_bytes ? (uint32_t)__ldg(stream + ip + k) : 0u;
        const uint32_t tag = b[0], type = tag & 3u;
        uint64_t hdr, len, off = 0;
        if (type == 0) {
            const uint32_t m = tag >> 2;
            const uint32_t k = m >= 60 ? m - 59 : 0;
            const uint64_t raw = (uint64_t)b[1] | ((uint64_t)b[2] << 8) | ((uint64_t)b[3] << 16) | ((uint64_t)b[4] << 24);
            hdr = 1 + k;
            len = (k == 0 ? m : (raw & (k == 4 ? 0xffffffffull : ((1ull << (8 * k)) - 1)))) + 1;
            if (ip + hdr + len > stream_bytes || len > total_out - op) {
                err = SNAPPY_B200_ST_CORRUPT;
                break;
            }
            coop_copy_ro(out + op, stream + ip + hdr, (uint32_t)len, lane, 32);
            ip += hdr + len;
        } else {
            if (type == 1)
                hdr = 2, len = ((tag >> 2) & 7u) + 4, off = ((uint64_t)(tag >> 5) << 8) | b[1];
            else if (type == 2)
                hdr = 3, len = (tag >> 2) + 1, off = (uint64_t)b[1] | ((uint64_t)b[2] << 8);
            else
                hdr = 5, len = (tag >> 2) + 1,
                off = (uint64_t)b[1] | ((uint64_t)b[2] << 8) | ((uint64_t)b[3] << 16) | ((uint64_t)b[4] << 24);
            if (ip + hdr > stream_bytes || off == 0 || off > op || len > total_out - op) {
                err = SNAPPY_B200_ST_CORRUPT;
                break;
            }
            __syncwarp(); // the bytes earlier elements wrote are visible to every lane
            for (uint64_t i = lane; i < len; i += 32) // write_copy :273-280: ascending, so an overlap repeats the pattern
                out[op + i] = out[op - off + (off >= len ? i : i % off)];
            ip += hdr;
        }
        op += len;
        __syncwarp();
    }
    if (!err && ip != stream_bytes)
        err = SNAPPY_B200_ST_CORRUPT; // trailing bytes after the declared length
    return err;
}

__global__ void __launch_bounds__(32) k_decode_sequential(const uint8_t *__restrict__ stream, uint64_t stream_bytes,
                                                          uint64_t body_offset, uint64_t total_out, uint8_t *out,
                                                          uint32_t *__restrict__ status)
{
    const uint32_t lane = threadIdx.x;
    const uint32_t err = decode_sequential_warp(stream, body_offset, stream_bytes, out, total_out, lane);
    if (err && lane == 0)
        atomicOr(status, err);
}

cudaError_t launch_decode_sequential(const uint8_t *d_stream, uint64_t stream_bytes, uint64_t body_offset,
                                     uint64_t total_out, uint8_t *d_out, uint32_t *d_status, cudaStream_t st,
                                     uint64_t *launches)
{
    if (total_out == 0)
        return cudaSuccess;
    k_decode_sequential<<<1, 32, 0, st>>>(d_stream, stream_bytes, body_offset, total_out, d_out, d_status);
    *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_decode(const uint8_t *d_stream, const uint64_t *d_offsets, uint64_t n_blocks, uint64_t total_out,
                          uint8_t *d_out, uint32_t *d_status, cudaStream_t st, uint64_t *launches)
{
    if (n_blocks == 0)
        return cudaSuccess;
    if (n_blocks > 0x7fffffffull)
        return cudaErrorInvalidValue;
    k_decode_warp<<<(unsigned)n_blocks, 32, 0, st>>>(d_stream, d_offsets, total_out, d_out, d_status);
    *launches += 1;
    return cudaGetLastError();
}

// ------------------------------------------------------------------ framed streams (csrc/frame.cu)
// One warp per data chunk of a framed stream.  A chunk is self-contained, so any error -- also what the block
// routine calls ST_FRAMING (a copy before the chunk, output past its length) -- is ST_CORRUPT here.  A compressed
// body longer than the window decoder takes (non-minimal encodings: up to 6 stream bytes per output byte) goes
// through the element loop of the general decoder, so a valid framed stream never needs a host fallback.
__global__ void __launch_bounds__(32) k_frame_decode(const uint8_t *__restrict__ stream, uint64_t stream_bytes,
                                                     const FrameChunk *__restrict__ chunks, uint8_t *out_base,
                                                     uint32_t *__restrict__ status)
{
    __shared__ uint4 elems[32];
    const uint32_t lane = threadIdx.x;
    const FrameChunk c = chunks[blockIdx.x];
    uint8_t *out = out_base + c.out_off;
    const uint8_t *__restrict__ in = stream + c.in_off;
    uint32_t err = 0;
    if (c.type == kChunkUncompressed) {
        coop_copy_ro(out, in, c.out_len, lane, 32);
    } else if (c.in_len <= 2u * kBlock) {
        const uint32_t *last_word = reinterpret_cast<const uint32_t *>(
            reinterpret_cast<uintptr_t>(stream + stream_bytes - 1) & ~uintptr_t(3));
        err = decode_block_warp(in, c.in_len, last_word, out, c.out_len, 0, elems, lane);
    } else {
        err = decode_sequential_warp(in, 0, c.in_len, out, c.out_len, lane);
    }
    if (err && lane == 0)
        atomicOr(status, SNAPPY_B200_ST_CORRUPT);
}

cudaError_t launch_frame_decode(const uint8_t *d_stream, uint64_t stream_bytes, const FrameChunk *d_chunks,
                                uint64_t n_chunks, uint8_t *d_out, uint32_t *d_status, cudaStream_t st, uint64_t *launches)
{
    if (n_chunks == 0)
        return cudaSuccess;
    if (n_chunks > 0x7fffffffull)
        return cudaErrorInvalidValue;
    k_frame_decode<<<(unsigned)n_chunks, 32, 0, st>>>(d_stream, stream_bytes, d_chunks, d_out, d_status);
    *launches += 1;
    return cudaGetLastError();
}

namespace {

// Runs in front of k_decode_seg: a block that is one literal (incompressible data) is moved stream -> output by the
// whole CTA with 16-byte vector copies, and k_decode_seg skips it.
__global__ void __launch_bounds__(256) k_copy_literal_blocks(const uint8_t *__restrict__ stream, uint64_t body_offset,
                                                             const uint64_t *__restrict__ offsets, uint64_t total_out,
                                                             uint8_t *out_base, const uint32_t *__restrict__ status,
                                                             uint64_t n_blocks)
{
    const uint64_t blk = blockIdx.x;
    if (*reinterpret_cast<const volatile uint32_t *>(status) != 0)
        return;
    const uint64_t c0 = offsets[blk], c1 = offsets[blk + 1];
    if (c1 <= c0 || c0 < body_offset || c1 > offsets[n_blocks] || c1 - c0 > 2u * kBlock)
        return; // k_decode_seg reports it (a bad range as ST_CORRUPT, an oversized block as ST_FRAMING)
    const uint64_t oleft = total_out - blk * (uint64_t)kBlock;
    const uint32_t olen = oleft < kBlock ? (uint32_t)oleft : kBlock;
    if (!one_literal_block(stream, c0, c1, olen))
        return;
    const uint32_t hdr = ((uint32_t)__ldg(stream + c0) >> 2) - 58u; // tag + length bytes
    coop_copy_ro(out_base + blk * (uint64_t)kBlock, stream + c0 + hdr, olen, threadIdx.x, 256);
}

} // namespace

// A block is one serial chain (about 2 ms for a text block, 1.5 ms for a low-entropy one, nothing for a block
// that k_copy_literal_blocks has moved), and 1 GiB is fewer than two waves of them: started in stream order the
// last wave ends with a few long blocks on an otherwise idle GPU.  The blocks are therefore handed out longest
// first, by compressed size (counting sort into 1 KiB classes, one CTA).
__global__ void __launch_bounds__(1024) k_block_order(const uint64_t *__restrict__ offsets, uint64_t n_blocks,
                                                      const uint32_t *__restrict__ status, uint32_t *__restrict__ order)
{
    __shared__ uint32_t cnt[64], base[64];
    if (*reinterpret_cast<const volatile uint32_t *>(status) != 0)
        return; // (k_decode_seg returns before it reads `order`)
    if (threadIdx.x < 64)
        cnt[threadIdx.x] = 0;
    __syncthreads();
    for (uint64_t b = threadIdx.x; b < n_blocks; b += blockDim.x)
        atomicAdd(&cnt[min((uint64_t)63, (offsets[b + 1] - offsets[b]) >> 10)], 1u);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t pos = 0;
        for (int k = 63; k >= 0; --k) {
            base[k] = pos;
            pos += cnt[k];
        }
    }
    __syncthreads();
    for (uint64_t b = threadIdx.x; b < n_blocks; b += blockDim.x)
        order[atomicAdd(&base[min((uint64_t)63, (offsets[b + 1] - offsets[b]) >> 10)], 1u)] = (uint32_t)b;
}

cudaError_t launch_decode_tile(const uint8_t *, uint64_t, const uint64_t *, const uint4 *, const uint64_t *, uint64_t,
                               uint64_t, uint8_t *, uint32_t *, uint64_t, cudaStream_t, uint64_t *); // decode_tile.cu

// Decoder for the maps K0 leaves behind.  Inputs of at most 32 blocks go to the tile decoder (k_decode_tile), whose
// eight warps per block give the lower latency; larger ones to the warp-per-block, segment-driven decoder above
// (k_decode_seg), preceded by k_copy_literal_blocks, which moves the blocks that are a single literal.
// SNAPPY_B200_DECODER=seg|tile (read once per process) forces one of the two on any input, so that both can be tested
// on either side of the threshold; unset or =auto picks by size.  The other block decoders that were built and
// measured, and why they lost, are in DESIGN.md §4.
cudaError_t launch_decode_seg(const uint8_t *d_stream, uint64_t body_offset, const uint64_t *d_offsets,
                              const uint4 *d_starts, const uint64_t *d_outoff, uint64_t n_blocks, uint64_t total_out,
                              uint8_t *d_out, uint32_t *d_status, uint64_t blk_base, cudaStream_t st,
                              uint64_t *launches)
{
    if (n_blocks == 0)
        return cudaSuccess;
    if (n_blocks > 0x7fffffffull)
        return cudaErrorInvalidValue;
    static const char which_env = [] {
        const char *v = getenv("SNAPPY_B200_DECODER");
        return v ? v[0] : 'a';
    }();
    // 'a' (default): the tile decoder for small inputs, the segment decoder otherwise.  A block is one serial
    // chain for k_decode_seg's single warp (about 0.8 ms on an idle GPU); k_decode_tile puts eight warps on the
    // block, which is the better trade when there are too few blocks to fill the machine anyway (measured, host
    // API, 64 KiB: 1.18 -> 0.72 ms; 1 MiB: 1.40 -> 0.88 ms; 16 MiB: 2.78 vs 3.70 ms the other way round).
    constexpr uint64_t kTileMaxBlocks = 32;
    const char which = which_env != 'a' ? which_env : (n_blocks <= kTileMaxBlocks && d_outoff ? 't' : 's');
    if (which == 't')
        return launch_decode_tile(d_stream, body_offset, d_offsets, d_starts, d_outoff, n_blocks, total_out, d_out,
                                  d_status, blk_base, st, launches);

    k_copy_literal_blocks<<<(unsigned)n_blocks, 256, 0, st>>>(d_stream, body_offset, d_offsets, total_out, d_out, d_status,
                                                             n_blocks);
    *launches += 1;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
        return e;
    // The order array lives in the memory of K0's per-segment output offsets, which this decoder does not need
    // (8 bytes per 128 stream bytes; a 64 KiB block is at least 2 KiB of stream, so it always fits).
    uint32_t *d_order = nullptr;
    if (d_outoff && n_blocks > 1) {
        d_order = reinterpret_cast<uint32_t *>(const_cast<uint64_t *>(d_outoff));
        k_block_order<<<1, 1024, 0, st>>>(d_offsets, n_blocks, d_status, d_order);
        *launches += 1;
    }
    // two blocks (warps) per CTA and a 48-register cap: 40 warps per SM instead of the 32 that one-warp
    // CTAs allow (measured: 64 registers / 32 warps 6.92, 48 / 40 6.72, 40 / 48 6.84 ms per GiB, K0 included)
    k_decode_seg<<<(unsigned)((n_blocks + 1) / 2), 64, 0, st>>>(d_stream, body_offset, d_offsets, d_starts, total_out,
                                                                d_out, d_status, n_blocks, blk_base, d_order);
    *launches += 1;
    return cudaGetLastError();
}

} // namespace sb200
