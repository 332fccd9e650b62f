// compress_parallel.cu -- the parse of SNAPPY_B200_MODE_PARALLEL: a valid Snappy stream in the reference's
// format, deterministic, not byte-identical to the reference.  csrc/parallel_parse.h defines the parse;
// tests/parallel_parse.c is the CPU model these kernels are held to byte for byte.
//
// k_par_cand -- one CTA of SB200_PAR_STEP threads per block, one position per thread and step.  The block is
// staged into shared memory first (64 KiB) next to the hash table (2^14 32-bit slots, 64 KiB): one CTA per SM.
// A slot holds position + 1 in its high half and a 16-bit fingerprint of that position's key in its low half.
// Each step reads its snapshot of the table, finds the in-group predecessor with __match_any_sync, and after a
// barrier the last position of each warp's same-hash group enters itself with atomicMax, whose result does not
// depend on the order the warps arrive in (the position is the high half, so the max is the latest position).
// The candidates are then checked against the staged block -- the table's one only when the fingerprints agree,
// the in-group one through the shuffled key of its lane -- and the match of the chosen one is measured up to 16
// bytes.  Out go a u16 offset per position and a length byte per position (0 = no candidate, len - 3 for a
// match shorter than 16 bytes, 255 for one of 16 or more); the length bytes live in the block's output slot
// until k_emit.  The offsets (128 KiB) do not fit into shared memory beside the block and the table.
//
// k_par_walk -- one warp per block, one lane per 2 KiB slice: the greedy walk over the length bytes (a word of
// them at a time) and the offsets; only matches of 16 bytes or more are extended from the input.  A block whose
// copies cover fewer than SB200_PAR_MIN_COVER bytes gets no records at all.  Otherwise a lane writes its
// records into its own 512-record stretch of the block's record array, then the warp scans the counts, sets
// the literal run of each slice's first record from the last copy of the slices before it, and compacts the
// records to the front (a record only ever moves down, and each 32-record window is read whole before it is
// written).  The records are the ones k_parse* writes: k_emit, k_scan_sizes and k_gather follow unchanged.
#include <mutex>

#include "common.cuh"
#include "parallel_parse.h"

namespace sb200 {

constexpr uint32_t kMaxRecords = 16384; // compress.cu
constexpr uint32_t kParSlots = 1u << SB200_PAR_TABLE_LOG;
constexpr uint32_t kParSliceRecs = SB200_PAR_SLICE / 4; // a copy covers >= 4 bytes
constexpr int kParWalkWarps = 4;
static_assert(SB200_PAR_GROUP == 32, "the in-group search is one warp's __match_any_sync");
static_assert(SB200_PAR_STEP % 32 == 0 && SB200_PAR_STEP <= 1024, "a step is whole warps of one CTA");
static_assert(SB200_PAR_SLICE * 32 == SNAPPY_B200_BLOCK_SIZE, "one lane per slice");
static_assert(kParSliceRecs * 32 == kMaxRecords, "every slice's records fit its stretch of the record array");
static_assert(SB200_PAR_CMP_WORDS == 1, "k_par_cand compares one word after the key");

__device__ __forceinline__ uint32_t par_hash(uint32_t key) { return (key * kHashMul) >> (32 - SB200_PAR_TABLE_LOG); }

// equal leading bytes of two little-endian words whose xor is x, counting at most `valid`
__device__ __forceinline__ uint32_t eq_bytes(uint32_t x, uint32_t valid)
{
    return min(x ? (uint32_t)(__ffs((int)x) - 1) >> 3 : 4u, valid);
}

// shared memory of k_par_cand: the block (+ 16 zero bytes, so that a word pair at any position is inside), the table
constexpr uint32_t kParStage = SNAPPY_B200_BLOCK_SIZE + 16;
constexpr uint32_t kParCandSmem = kParStage + kParSlots * 4;

__device__ __forceinline__ uint32_t par_fingerprint(uint32_t key) { return (key * 0x9e3779b1u) >> 16; }

// little-endian 32 bits at any position of the staged block
__device__ __forceinline__ uint32_t sld32(const uint32_t *w, uint32_t pos)
{
    return __funnelshift_r(w[pos >> 2], w[(pos >> 2) + 1], (pos & 3u) * 8u);
}

__global__ void __launch_bounds__(SB200_PAR_STEP, 1) k_par_cand(const uint8_t *__restrict__ in, uint64_t n_bytes,
                                                                uint16_t *__restrict__ cand, uint8_t *__restrict__ scratch,
                                                                uint32_t *__restrict__ nrec)
{
    extern __shared__ __align__(16) uint8_t par_smem[];
    const uint32_t *w = reinterpret_cast<const uint32_t *>(par_smem);
    uint32_t *T = reinterpret_cast<uint32_t *>(par_smem + kParStage); // (position + 1) << 16 | fingerprint; 0 = empty
    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    const uint64_t blk = blockIdx.x;
    const uint8_t *__restrict__ b = in + blk * (uint64_t)kBlock; // 16-byte aligned
    const uint64_t left = n_bytes - blk * (uint64_t)kBlock;
    const uint32_t n = left < kBlock ? (uint32_t)left : kBlock;
    uint16_t *__restrict__ off_out = cand + blk * (uint64_t)kBlock;
    uint8_t *__restrict__ len_out = scratch + blk * (uint64_t)kSlot;
    const uint32_t n16 = n / 16;
    for (uint32_t i = tid; i < n16; i += SB200_PAR_STEP)
        reinterpret_cast<uint4 *>(par_smem)[i] = __ldg(reinterpret_cast<const uint4 *>(b) + i);
    for (uint32_t i = 16 * n16 + tid; i < min(16 * n16 + 32, kParStage); i += SB200_PAR_STEP)
        par_smem[i] = i < n ? __ldg(b + i) : 0;
    for (uint32_t i = tid; i < kParSlots / 4; i += SB200_PAR_STEP)
        reinterpret_cast<uint4 *>(T)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();

    const uint32_t np = n >= 4 ? n - 3 : 0; // positions with a key
    // (CTA-uniform) steps in a row without a candidate, steps to skip, candidates so far
    uint32_t misses = 0, skip = 0, found = 0;
    bool pending = false; // the last step looked up is not counted yet: its candidates are in `code`
    uint32_t code = 0;
    for (uint32_t g0 = 0; g0 < np; g0 += SB200_PAR_STEP) {
        const uint32_t p = g0 + tid;
        const bool valid = p < np;
        if (skip) { // passed over: no lookups, nothing entered, no candidates
            --skip;
            if (valid)
                len_out[p] = 0;
            continue;
        }
        const uint32_t key = valid ? sld32(w, p) : 0u;
        const uint32_t kn = valid ? sld32(w, p + 4) : 0u; // the next word, to choose between two candidates
        const uint32_t h = par_hash(key);
        const uint32_t t = valid ? T[h] : 0u;
        const unsigned grp = __match_any_sync(kFull, valid ? h : 0xffffffffu);
        const unsigned earlier = grp & ((1u << lane) - 1u);
        const uint32_t src = earlier ? (uint32_t)(31 - __clz((int)earlier)) : lane;
        const uint32_t key2 = __shfl_sync(kFull, key, src), kn2 = __shfl_sync(kFull, kn, src);
        const uint32_t fp = par_fingerprint(key);
        // every snapshot read is done; count the previous step looked up (the skip starts after this step)
        const int prev_hits = __syncthreads_count(code != 0);
        if (pending) {
            found += (uint32_t)prev_hits;
            if (prev_hits) {
                misses = 0;
            } else {
                ++misses;
                skip = min(1u << min(misses - 1, 30u), (uint32_t)SB200_PAR_SKIP_MAX);
            }
        }
        pending = true;
        if (valid && (grp >> lane) == 1u)
            atomicMax(&T[h], (p + 1) << 16 | fp);
        __syncthreads();
        code = 0;
        if (valid) {
            const uint32_t nx = min(4u, n - (p + 4)); // (p + 4 <= n)
            bool v1 = false;
            uint32_t c1 = 0, e1 = 0;
            if (t && (t & 0xffffu) == fp) {
                c1 = (t >> 16) - 1;
                v1 = sld32(w, c1) == key;
                e1 = eq_bytes(sld32(w, c1 + 4) ^ kn, nx);
            }
            const bool v2 = earlier && key2 == key;
            const uint32_t e2 = eq_bytes(kn2 ^ kn, nx);
            uint32_t off = 0;
            if (v1 || v2) {
                const bool two = v2 && (!v1 || e2 >= e1);
                const uint32_t c = two ? p - lane + src : c1;
                uint32_t len = 4 + (two ? e2 : e1);
                if (len == 8) { // (then p + 8 <= n)
                    for (uint32_t k = 8; k < 16; k += 4) {
                        const uint32_t lim = p + k < n ? min(4u, n - (p + k)) : 0u;
                        const uint32_t ek = lim ? eq_bytes(sld32(w, c + k) ^ sld32(w, p + k), lim) : 0u;
                        len += ek;
                        if (ek < 4)
                            break;
                    }
                }
                off = p - c;
                code = len < 16 ? len - 3 : 255u;
            }
            off_out[p] = (uint16_t)off;
            len_out[p] = (uint8_t)code;
        }
    }
    found += (uint32_t)__syncthreads_count(code != 0); // the last step looked up
    if (tid == 0)
        nrec[blk] = found ? 1u : 0u; // k_par_walk leaves a block without any candidate at 0 records
}

// equal bytes of b[c..] and b[q..], at most max_len (q + max_len <= n, c < q)
__device__ __forceinline__ uint32_t match_len(const uint8_t *__restrict__ b, uint32_t c, uint32_t q, uint32_t max_len,
                                              uint32_t last_word)
{
    uint32_t k = 0;
    while (k < max_len) {
        const uint32_t valid = min(4u, max_len - k);
        const uint32_t e = eq_bytes(ld_le32(b, c + k, last_word) ^ ld_le32(b, q + k, last_word), valid);
        k += e;
        if (e < valid)
            break;
    }
    return k;
}

__global__ void __launch_bounds__(32 * kParWalkWarps) k_par_walk(const uint8_t *__restrict__ in, uint64_t n_bytes,
                                                                 uint64_t n_blocks, const uint16_t *__restrict__ cand,
                                                                 const uint8_t *__restrict__ scratch,
                                                                 uint2 *__restrict__ recs, uint32_t *__restrict__ nrec)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t blk = (uint64_t)blockIdx.x * kParWalkWarps + (threadIdx.x >> 5);
    if (blk >= n_blocks)
        return; // (warp-uniform)
    if (__ldcg(nrec + blk) == 0)
        return; // no candidate anywhere in the block: one literal
    const uint8_t *__restrict__ b = in + blk * (uint64_t)kBlock;
    const uint64_t left = n_bytes - blk * (uint64_t)kBlock;
    const uint32_t n = left < kBlock ? (uint32_t)left : kBlock;
    const uint32_t last_word = (n - 1) >> 2;
    const uint16_t *__restrict__ off = cand + blk * (uint64_t)kBlock;
    const uint32_t *__restrict__ codes = reinterpret_cast<const uint32_t *>(scratch + blk * (uint64_t)kSlot);
    uint2 *__restrict__ my_recs = recs + blk * (uint64_t)kMaxRecords;
    uint2 *__restrict__ mine = my_recs + lane * kParSliceRecs;

    const uint32_t s0 = lane * SB200_PAR_SLICE, s1 = min(s0 + SB200_PAR_SLICE, n);
    uint32_t cnt = 0, p = s0, prev = s0, covered = 0;
    uint2 first = make_uint2(0, 0);
    uint32_t cw = 0, cw_at = 0xffffffffu; // the word of length bytes that holds position p
    while (p + 4 <= s1) {
        if (p >> 2 != cw_at) {
            cw_at = p >> 2;
            cw = __ldg(codes + cw_at);
        }
        const uint32_t rest = cw >> (8 * (p & 3u));
        if (!(rest & 0xffu)) { // no candidate: on to the next position that has one (bytes past n - 4 end the loop)
            p = rest ? p + ((uint32_t)(__ffs((int)rest) - 1) >> 3) : (p | 3u) + 1;
            continue;
        }
        const uint32_t code = rest & 0xffu, room = s1 - p;
        const uint32_t o = __ldg(off + p);
        const uint32_t len = code != 255u ? min(code + 3, room)
                             : room <= 16 ? room
                                          : 16 + match_len(b, p - o + 16, p + 16, room - 16, last_word);
        const uint2 rec = make_uint2(p | (o << 16), len | ((p - prev) << 16));
        if (cnt == 0)
            first = rec;
        else
            mine[cnt] = rec;
        ++cnt;
        covered += len;
        p += len;
        prev = p;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1)
        covered += __shfl_xor_sync(kFull, covered, d);
    if (covered < SB200_PAR_MIN_COVER) { // (warp-uniform) no records: the block is one literal
        if (lane == 0)
            nrec[blk] = 0;
        return;
    }

    // counts -> slots; the literal before a slice's first copy starts at the last copy end of the slices before it
    uint32_t incl = cnt, last_end = cnt ? prev : 0u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t a = __shfl_up_sync(kFull, incl, d);
        const uint32_t e = __shfl_up_sync(kFull, last_end, d);
        if ((int)lane >= d) {
            incl += a;
            last_end = max(last_end, e);
        }
    }
    const uint32_t excl = incl - cnt, total = __shfl_sync(kFull, incl, 31);
    uint32_t prev_end = __shfl_up_sync(kFull, last_end, 1);
    if (lane == 0)
        prev_end = 0;
    if (cnt) {
        const uint32_t p0 = first.x & 0xffffu;
        first.y = (first.y & 0xffffu) | ((p0 - prev_end) << 16);
        mine[0] = first;
    }
    __syncwarp();
    for (uint32_t d0 = 0; d0 < total; d0 += 32) {
        const uint32_t d = d0 + lane;
        uint32_t k = 0; // the last slice whose first slot is <= d
#pragma unroll
        for (uint32_t s = 16; s; s >>= 1)
            if (__shfl_sync(kFull, excl, k + s) <= d)
                k += s;
        const uint32_t ek = __shfl_sync(kFull, excl, k);
        uint2 r = make_uint2(0, 0);
        if (d < total)
            r = my_recs[k * kParSliceRecs + (d - ek)];
        __syncwarp();
        if (d < total)
            my_recs[d] = r;
        __syncwarp();
    }
    if (lane == 0)
        nrec[blk] = total;
}

// d_scratch: the blocks' output slots, which hold the length bytes until k_emit overwrites them
cudaError_t launch_parallel_parse(const uint8_t *d_in, uint64_t n_bytes, uint64_t n_blocks, uint16_t *d_cand,
                                  uint8_t *d_scratch, uint2 *d_recs, uint32_t *d_nrec, cudaStream_t st,
                                  uint64_t *launches)
{
    if (!d_cand)
        return cudaErrorInvalidValue;
    // (the opt-in to > 48 KiB of dynamic shared memory is per device: once per device, thread-safe)
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess)
        return e;
    static std::once_flag attr_once[64];
    std::call_once(attr_once[dev & 63], [&] {
        e = cudaFuncSetAttribute(k_par_cand, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kParCandSmem);
    });
    if (e != cudaSuccess)
        return e;
    k_par_cand<<<(unsigned)n_blocks, SB200_PAR_STEP, kParCandSmem, st>>>(d_in, n_bytes, d_cand, d_scratch, d_nrec);
    k_par_walk<<<(unsigned)((n_blocks + kParWalkWarps - 1) / kParWalkWarps), 32 * kParWalkWarps, 0, st>>>(
        d_in, n_bytes, n_blocks, d_cand, d_scratch, d_recs, d_nrec);
    *launches += 2;
    return cudaGetLastError();
}

size_t parallel_cand_bytes(uint64_t n_blocks) { return n_blocks * (size_t)kBlock * sizeof(uint16_t); }

} // namespace sb200
