// compress.cu -- K1 (hash-table parse), K2 (exact-key parse) and K1e (element emission).
//
// What is computed is exactly the greedy parse of the reference
//   hash mode : src/snappy_compression.c:384-403 (compress_next_block)
//   exact mode: src/snappy_compression_tree.c:269-288 with the dictionary of src/BST.c
// and the element encodings of src/snappy_compression.c:95-165.  How it is computed is not.
//
// k_parse -- one warp per 64 KiB block; the serial part, kept as lean as possible.
// The parse is serial in the table state, so the warp speculates.  Each step lays the next 16
// probe positions out as 32 "events" (lane 2j = the p-1 insertion that probe j would make on
// a miss, lane 2j+1 = probe j itself), under the assumption that every earlier probe of the
// step misses.  Lanes look their key up in the shared-memory table AND in the earlier lanes
// of the same step (__match_any_sync), which reproduces what the table would hold after
// those misses.  The first probe that hits (or reaches the end-of-block test) cuts the step:
// the misses before it are committed to the table in one go and the hit is extended with a
// warp-wide 4-byte-per-lane compare.  Everything the speculation assumed about lanes after
// the cut is discarded, so the result is the reference's parse, bit for bit.  The warp does
// not write compressed bytes: it leaves one 8-byte record per copy {position, offset,
// length, literal run before it}.
//
// Hash-mode table: u16 position + u8 key fingerprint per slot, in two arrays (8 KiB in global
// memory, 4 KiB in shared memory, see k_parse_hash_global).  The fingerprint is bits 19..12 of
// key*0x1e35a7bd -- together with the 12-bit slot index it pins 20 of the 32 bits of an
// injective function of the key, so the "does the candidate's 4 bytes equal mine" test of the
// reference (found_match, :259-265) is almost always answered from shared memory; lanes whose
// fingerprint matches confirm against the candidate bytes, all at once, and compare the next
// four bytes in the same fetch (most matches end there, which saves the separate extension
// round trip).  The reference's zero-filled table ("candidate = position 0") becomes
// (position 0, fingerprint of the block's first 4 bytes).
//
// Exact mode keeps an open-addressing table of u16 positions keyed by the exact 4 bytes
// (0xffff = empty, which no insertable position can be: positions >= n-15 are never probed).
// Keys are compared through the block itself.  Tables come in three sizes; a block whose
// dictionary outgrows the small table is marked and redone by the next tier.
//
// k_emit -- one CTA per block, one thread per record: literal header + bytes and the copy
// tags (write_literal :95-120, write_copy :153-165, write_single_copy :131-145) are sized,
// prefix-summed and written in parallel into the block's scratch slot; long literals are
// copied by the whole CTA with 16-byte stores.
#include <algorithm>

#include <mutex>
#include <type_traits>

#include "common.cuh"

namespace sb200 {

constexpr uint32_t kMaxRecords = 16384; // a copy covers >= 4 bytes

// reference: find_copy_length :61-72 (+4 for the bytes the probe already matched).
// Lane l compares bytes [base+4l, base+4l+4) of the two strings; the first lane that sees a
// difference (or the end of the block) decides.
__device__ __forceinline__ uint32_t match_extend(const uint8_t *__restrict__ b, uint32_t p, uint32_t c, uint32_t n,
                                                 uint32_t last_word, uint32_t lane, uint32_t base = 4)
{
    uint32_t width = 8; // most matches are short: first look at 32 bytes, then 128 at a time
    for (;;) {
        uint32_t t = 4; // number of equal bytes in this lane's word; 4 = keep going
        const uint32_t pp = p + base + 4 * lane;
        if (lane < width) {
            if (pp >= n) {
                t = 0;
            } else {
                const uint32_t nvalid = min(4u, n - pp);
                uint32_t x = ld_le32(b, pp, last_word) ^ ld_le32(b, c + base + 4 * lane, last_word);
                if (nvalid < 4)
                    x = (x & ((1u << (8 * nvalid)) - 1u)) | (1u << (8 * nvalid));
                if (x)
                    t = (uint32_t)(__ffs((int)x) - 1) >> 3;
            }
        }
        const unsigned stop = __ballot_sync(kFull, t < 4);
        if (stop) {
            const int l = __ffs((int)stop) - 1;
            return base + 4 * (uint32_t)l + __shfl_sync(kFull, t, l);
        }
        base += 4 * width;
        width = 32;
    }
}

// ------------------------------------------------------------------------------- exact table
// GLOBAL: the table lives in global memory (the big tier, see launch_compress).  It is private to
// one warp, but lanes insert with atomics, which are performed in L2: the reads then go to L2 as
// well (__ldcg) instead of trusting a line in L1.
// In the global tiers an entry is 32 bits: the position and a 16-bit fingerprint of the key (the low half
// of key * golden; the high bits give the home slot).  A probe that walks over other keys' entries then
// costs one L2 access per entry instead of two dependent ones (entry, then the key bytes through the
// block): the key bytes are only fetched when the fingerprint matches, i.e. practically only on a hit.
template <int LOG_SLOTS, bool GLOBAL = false> struct ExactTable {
    static constexpr uint32_t kSlots = 1u << LOG_SLOTS;
    using Entry = typename std::conditional<GLOBAL, uint32_t, uint16_t>::type;
    static constexpr uint32_t kEmpty = GLOBAL ? 0xffffffffu : 0xffffu;
    static constexpr uint32_t kBytes = kSlots * sizeof(Entry);
    Entry *tab;

    __device__ __forceinline__ uint32_t home(uint32_t key) const { return (key * 0x9e3779b1u) >> (32 - LOG_SLOTS); }
    __device__ __forceinline__ uint32_t entry(uint32_t key, uint32_t pos) const
    {
        return GLOBAL ? pos | ((key * 0x9e3779b1u) << 16) : pos;
    }

    // Returns the slot holding `key`, or the first empty slot of its probe sequence.
    __device__ __forceinline__ uint32_t find(const uint8_t *__restrict__ b, uint32_t last_word, uint32_t key,
                                             bool &found, uint32_t &pos) const
    {
        uint32_t s = home(key);
        const uint32_t fp = (key * 0x9e3779b1u) & 0xffffu;
        for (;;) {
            const uint32_t v = GLOBAL ? (uint32_t)__ldcg(tab + s) : (uint32_t)tab[s];
            if (v == kEmpty) {
                found = false;
                pos = 0;
                return s;
            }
            if ((!GLOBAL || (v >> 16) == fp) && ld_be32(b, v & 0xffffu, last_word) == key) {
                found = true;
                pos = v & 0xffffu;
                return s;
            }
            s = (s + 1) & (kSlots - 1);
        }
    }

    // Inserts a key known to be absent (several lanes may insert different keys at once).
    __device__ __forceinline__ void insert_absent(uint32_t key, uint32_t pos)
    {
        uint32_t s = home(key);
        for (;;) {
            if (GLOBAL) {
                if (atomicCAS(reinterpret_cast<unsigned int *>(tab + s), kEmpty, entry(key, pos)) == kEmpty)
                    return;
            } else {
                const unsigned short old = atomicCAS(reinterpret_cast<unsigned short *>(tab + s),
                                                     (unsigned short)kEmpty, (unsigned short)pos);
                if (old == kEmpty)
                    return;
            }
            s = (s + 1) & (kSlots - 1);
        }
    }
    __device__ __forceinline__ void set(uint32_t slot, uint32_t key, uint32_t pos) { tab[slot] = (Entry)entry(key, pos); }
};

// ------------------------------------------------------------------------------- the parse
// MODE 0 = hash table (LOG_SLOTS ignored: up to 4096 u16 positions at smem_raw, one u8 fingerprint per
//          slot at fp_mem)
// MODE 1 = exact dictionary with 2^LOG_SLOTS u16 slots; a block whose dictionary would grow
//          past 3/4 of the table gives up (nrec[blk] = kAbortMark) unless FINAL.
// smem_raw: the table memory (shared, or global when GLOBAL).
template <int MODE, int LOG_SLOTS, bool FINAL, bool GLOBAL = false>
__device__ __forceinline__ void parse_block(const uint8_t *__restrict__ in, uint64_t n_bytes, uint2 *__restrict__ recs,
                                            uint32_t *__restrict__ nrec, uint64_t blk, uint8_t *smem_raw,
                                            uint8_t *fp_mem = nullptr)
{
    const uint32_t lane = threadIdx.x & 31u;

    const uint8_t *__restrict__ b = in + blk * (uint64_t)kBlock;
    const uint64_t left = n_bytes - blk * (uint64_t)kBlock;
    const uint32_t n = left < kBlock ? (uint32_t)left : kBlock;
    const uint32_t last_word = (n - 1) >> 2;
    uint2 *__restrict__ my_recs = recs + blk * (uint64_t)kMaxRecords;

    // per-miss skip bookkeeping: hash mode skip += 1 per miss and the step uses the value the
    // end test saw (:229-232, :283-287); BST mode post-increments inside the end test as well
    // (tree.c:154-157), so skip += 2 per miss and the step sees skip+1.
    constexpr uint32_t C = MODE == 0 ? 1 : 2;
    constexpr uint32_t D = MODE == 0 ? 0 : 1;

    uint16_t *hpos = reinterpret_cast<uint16_t *>(smem_raw); // hash mode: candidate position per slot
    uint8_t *hfp = fp_mem;                                    // hash mode: key fingerprint per slot
    ExactTable<LOG_SLOTS, GLOBAL> et{reinterpret_cast<typename ExactTable<LOG_SLOTS, GLOBAL>::Entry *>(smem_raw)};
    uint32_t shift = 20;
    uint32_t n_keys = 0; // exact mode: dictionary population (warp-uniform)

    if (MODE == 0) {
        // set_htable_size, :198-204
        uint32_t lg = 8;
        while ((1u << lg) < SNAPPY_B200_HTABLE_SIZE && (1u << lg) < n)
            ++lg;
        shift = 32 - lg;
        const uint32_t f0 = n >= 4 ? ((ld_be32(b, 0, last_word) * kHashMul) >> 12) & 0xffu : 0;
        const uint32_t f4 = f0 * 0x01010101u;
        uint4 *p4 = reinterpret_cast<uint4 *>(hpos);
        uint4 *q4 = reinterpret_cast<uint4 *>(hfp);
        for (uint32_t i = lane; i < (1u << lg) / 8; i += 32)
            p4[i] = make_uint4(0, 0, 0, 0);
        for (uint32_t i = lane; i < (1u << lg) / 16; i += 32)
            q4[i] = make_uint4(f4, f4, f4, f4);
    } else {
        uint4 *t4 = reinterpret_cast<uint4 *>(smem_raw);
        const uint4 init = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
        for (uint32_t i = lane; i < ExactTable<LOG_SLOTS, GLOBAL>::kBytes / 16; i += 32)
            t4[i] = init;
    }
    __syncwarp();

    uint32_t pos = 1, skip = 33, prev_end = 0; // :386-387: the first byte is a literal
    uint32_t nh = 0;                           // records so far
    uint2 rec = make_uint2(0, 0);              // lane (nh & 31) holds record nh until 32 are full

    const uint32_t j = lane >> 1;
    const uint32_t odd = lane & 1u; // odd lanes are the probes
    const unsigned vis_mask = lane >= 1 ? (1u << (lane - 1)) - 1u : 0u; // events a probe may see

    const uint32_t hl = (lane + 1) >> 1; // stride-1 layout: event position = pos - 1 + hl
    bool narrow = false;                 // the last probe hit at once: try the first probe alone

    uint32_t pf = 0; // input prefetched into L2 up to here (4 KiB at a time, 4..8 KiB ahead)

    for (;;) {
        if (pos + 4096u > pf) {
            if (pf + 128u * lane < n)
                prefetch_l2(b + pf + 128u * lane);
            pf += 4096u;
        }
        // ---- fast path of the hash parse: all 16 probes one byte apart (skip + 15 < 64) and none
        // of them near the end of the block.  Same events, same rules as the general step below,
        // with the positions, the end test and a few shuffles folded away.
        if (MODE == 0 && skip <= 48u && pos + 34u <= n) {
            if (narrow) {
                // First probe after a copy.  Runs and repeated phrases hit again at once (every
                // time on low-entropy data, one time in four on text), so try that probe alone
                // with warp-uniform work -- no event layout, no match, no ballot.  On a miss
                // nothing has been changed and the full step below takes over.
                const uint32_t *wp = reinterpret_cast<const uint32_t *>(b) + (pos >> 2);
                const uint32_t psh = (pos & 3u) * 8u;
                const uint32_t k0 = __ldg(wp), k1 = __ldg(wp + 1), k2 = __ldg(wp + 2), k3 = __ldg(wp + 3),
                               k4 = __ldg(wp + 4); // pos + 19 < n
                const uint32_t key = bswap32(__funnelshift_r(k0, k1, psh));
                const uint32_t prod = key * kHashMul;
                const uint32_t idx = prod >> shift;
                const uint32_t ph = (prod >> 12) & 0xffu;
                uint32_t cand = 0;
                bool hit = false;
                uint32_t ext = 0;
                if (hfp[idx] == ph) {
                    cand = hpos[idx];
                    const uint32_t *cw = reinterpret_cast<const uint32_t *>(b) + (cand >> 2);
                    const uint32_t sh = (cand & 3u) * 8u;
                    const uint32_t w0 = __ldg(cw), w1 = __ldg(cw + 1), w2 = __ldg(cw + 2),
                                   w3 = __ldg(cw + 3), w4 = __ldg(cw + 4);
                    hit = __funnelshift_r(w0, w1, sh) == __funnelshift_r(k0, k1, psh);
                    const uint32_t x1 = __funnelshift_r(w1, w2, sh) ^ __funnelshift_r(k1, k2, psh);
                    const uint32_t x2 = __funnelshift_r(w2, w3, sh) ^ __funnelshift_r(k2, k3, psh);
                    const uint32_t x3 = __funnelshift_r(w3, w4, sh) ^ __funnelshift_r(k3, k4, psh);
                    // little-endian words: trailing equal bytes
                    ext = x1   ? (uint32_t)(__ffs((int)x1) - 1) >> 3
                          : x2 ? 4 + ((uint32_t)(__ffs((int)x2) - 1) >> 3)
                          : x3 ? 8 + ((uint32_t)(__ffs((int)x3) - 1) >> 3)
                               : 0x10c;
                }
                if (hit) {
                    __syncwarp();
                    if (lane == 0) { // emit_copy :327
                        hpos[idx] = (uint16_t)pos;
                        hfp[idx] = (uint8_t)ph;
                    }
                    const uint32_t p = pos;
                    const uint32_t len =
                        ext < 0x100 ? 4 + ext : match_extend(b, p, cand, n, last_word, lane, 4 + (ext & 0xffu));
                    if (lane == (nh & 31u))
                        rec = make_uint2(p | ((p - cand) << 16), len | ((p - prev_end) << 16));
                    ++nh;
                    if ((nh & 31u) == 0)
                        my_recs[nh - 32 + lane] = rec;
                    pos = p + len;
                    prev_end = pos;
                    skip = 32;
                    __syncwarp();
                    continue;
                }
                narrow = false;
            }
            const uint32_t ev = pos - 1u + hl;
            const uint32_t *wp = reinterpret_cast<const uint32_t *>(b) + (ev >> 2);
            const uint32_t key = __byte_perm(__ldg(wp), __ldg(wp + 1), 0x0123u + 0x1111u * (ev & 3u)); // big-endian
            const uint32_t prod = key * kHashMul; // hash_bytes :81-84
            const uint32_t idx = prod >> shift;
            const uint32_t ph = (prod >> 12) & 0xffu;
            // my next 12 bytes are the keys of the lanes 8, 16 and 24 up (two lanes per byte step)
            const uint32_t nk1 = __shfl_down_sync(kFull, key, 8);
            const uint32_t nk2 = __shfl_down_sync(kFull, key, 16);
            const uint32_t nk3 = __shfl_down_sync(kFull, key, 24);
            const uint32_t tfp = hfp[idx];
            // found_match :259-265 and a head start on find_copy_length :61-72: probes whose
            // fingerprint agrees fetch the candidate's bytes now, so that the round trip overlaps
            // the in-step forwarding below (tpos + 19 < pos + 19 < n: all five words are inside).
            // Only they read the position (the fingerprints are the array that is kept closest).
            const bool want = odd && tfp == ph;
            const uint32_t tpos = want ? hpos[idx] : 0u;
            const uint32_t *cw = reinterpret_cast<const uint32_t *>(b) + (tpos >> 2);
            uint32_t w0 = 0, w1 = 0, w2 = 0, w3 = 0, w4 = 0;
            if (want) {
                w0 = __ldg(cw);
                w1 = __ldg(cw + 1);
                w2 = __ldg(cw + 2);
                w3 = __ldg(cw + 3);
                w4 = __ldg(cw + 4);
            }
            const unsigned grp = __match_any_sync(kFull, idx);
            const unsigned vis = odd ? grp & vis_mask : 0u;
            bool hit = false;
            uint32_t cand = tpos;
            uint32_t ext = 0x100; // bit 8: the match may go on past the bytes compared here (low bits: how many)
            if (__any_sync(kFull, vis != 0u)) {
                // rare: a probe's slot is written by an earlier event of this same step
                const int src = 31 - __clz((int)vis); // latest earlier writer of the slot (-1: none)
                const uint32_t skey = __shfl_sync(kFull, key, src);
                if (vis) {
                    hit = skey == key;
                    cand = pos - 1u + ((uint32_t)(src + 1) >> 1);
                }
            }
            if (vis) {
            } else if (want) {
                const uint32_t sh = (tpos & 3u) * 8u;
                hit = bswap32(__funnelshift_r(w0, w1, sh)) == key;
                const uint32_t x1 = bswap32(__funnelshift_r(w1, w2, sh)) ^ nk1;
                const uint32_t x2 = bswap32(__funnelshift_r(w2, w3, sh)) ^ nk2;
                const uint32_t x3 = bswap32(__funnelshift_r(w3, w4, sh)) ^ nk3;
                // big-endian words: leading equal bytes.  Lanes too high to have neighbours
                // 8 / 16 / 24 up stop at what they can see and leave the rest to match_extend.
                if (lane >= 24)
                    ext = 0x100;
                else if (x1)
                    ext = (uint32_t)__clz((int)x1) >> 3;
                else if (lane >= 16)
                    ext = 0x104;
                else if (x2)
                    ext = 4 + ((uint32_t)__clz((int)x2) >> 3);
                else if (lane >= 8)
                    ext = 0x108;
                else if (x3)
                    ext = 8 + ((uint32_t)__clz((int)x3) >> 3);
                else
                    ext = 0x10c;
            }
            const unsigned H = __ballot_sync(kFull, odd && hit);
            if (H == 0) { // 16 misses: update_hash_table :303-307, the last writer of a slot wins
                if ((grp >> lane) == 1u) {
                    hpos[idx] = (uint16_t)ev;
                    hfp[idx] = (uint8_t)ph;
                }
                pos += 16;
                skip += 16;
                continue;
            }
            const int f = __ffs((int)H) - 1;
            if (((grp & ((1u << (f - 1)) - 1u)) >> lane) == 1u) { // the misses before the cut
                hpos[idx] = (uint16_t)ev;
                hfp[idx] = (uint8_t)ph;
            }
            __syncwarp();
            const uint32_t p = pos + ((uint32_t)f >> 1);
            const uint32_t c = __shfl_sync(kFull, cand, f);
            const uint32_t ex = __shfl_sync(kFull, ext, f);
            if ((int)lane == f) { // emit_copy :327
                hpos[idx] = (uint16_t)ev;
                hfp[idx] = (uint8_t)ph;
            }
            const uint32_t len = ex < 0x100 ? 4 + ex : match_extend(b, p, c, n, last_word, lane, 4 + (ex & 0xffu));
            if (lane == (nh & 31u))
                rec = make_uint2(p | ((p - c) << 16), len | ((p - prev_end) << 16));
            ++nh;
            if ((nh & 31u) == 0)
                my_recs[nh - 32 + lane] = rec;
            pos = p + len;
            prev_end = pos;
            skip = 32; // start_new_literal :271-274
            narrow = true; // (trying the first probe alone costs little even when it then misses)
            __syncwarp();
            continue;
        }

        // ---- exact mode, first probe after a copy, tried alone with warp-uniform work (see the
        // hash-mode single-probe step above; a key that is in the dictionary always hits)
        if (MODE == 1 && narrow && skip == 32u && pos + 34u <= n) {
            const uint32_t key = ld_be32(b, pos, last_word);
            bool found;
            uint32_t tpos;
            const uint32_t slot = et.find(b, last_word, key, found, tpos); // found_match_tree tree.c:174-180
            if (found) {
                et.set(slot, key, pos); // tree.c:221 (every lane stores the same value)
                const uint32_t len = match_extend(b, pos, tpos, n, last_word, lane);
                if (lane == (nh & 31u))
                    rec = make_uint2(pos | ((pos - tpos) << 16), len | ((pos - prev_end) << 16));
                ++nh;
                if ((nh & 31u) == 0)
                    my_recs[nh - 32 + lane] = rec;
                pos += len;
                prev_end = pos;
                __syncwarp();
                continue; // skip stays 32: start_new_literal tree.c:182-186
            }
            narrow = false;
        }

        // ---- lay out 16 probes under the all-miss assumption
        const uint32_t a = skip + D;
        const uint32_t q = a >> 5, r = a & 31u;
        const uint32_t k1 = (32u - r + C - 1u) / C; // first probe index whose step is q+1
        const uint32_t pj = pos + j * q + (j > k1 ? j - k1 : 0u);
        const bool end_j = pj + ((skip + C * j) >> 5) + 15u > n; // is_block_end
        const uint32_t ev_pos = pj - 1 + odd;
        const uint32_t key = ld_be32(b, end_j ? 0u : ev_pos, last_word);
        const bool probe = odd && !end_j;

        bool hit;       // this lane's probe hits
        uint32_t cand;  // ... this candidate position
        uint32_t idx = 0, ph = 0;
        unsigned grp;
        bool in_table = false;

        uint32_t ext4 = 4; // equal bytes among the four that follow the key (4 = unknown / all)
        if (MODE == 0) {
            const uint32_t prod = key * kHashMul; // hash_bytes :81-84
            idx = prod >> shift;
            ph = (prod >> 12) & 0xffu;
            grp = __match_any_sync(kFull, idx);
            const unsigned vis = grp & vis_mask;
            const int src = 31 - __clz((int)vis); // latest earlier writer of the slot (-1: none)
            const uint32_t skey = __shfl_sync(kFull, key, src);
            const uint32_t spos = __shfl_sync(kFull, ev_pos, src);
            // my next four bytes are the key of the lane 8 up (steps of one byte, two lanes each)
            const uint32_t nkey = __shfl_down_sync(kFull, key, 8);
            const bool nend = __shfl_down_sync(kFull, (int)end_j, 8);
            const bool nkey_ok = lane < 24 && !nend && skip + D + C * 15 < 64;
            const uint32_t tpos = hpos[idx];
            const uint32_t tfp = hfp[idx];
            if (vis) {
                hit = skey == key;
                cand = spos;
            } else {
                cand = tpos;
                hit = false;
                if (probe && tfp == ph) {
                    // found_match :259-265, and a head start on find_copy_length :61-72
                    const uint32_t c0 = ld_le32(b, cand, last_word);
                    const uint32_t c1 = ld_le32(b, cand + 4, last_word);
                    hit = bswap32(c0) == key;
                    const uint32_t x = bswap32(c1) ^ nkey;
                    if (nkey_ok && x)
                        ext4 = (uint32_t)__clz((int)x) >> 3; // big-endian: leading equal bytes
                }
            }
        } else {
            grp = __match_any_sync(kFull, key);
            const unsigned vis = grp & vis_mask;
            const int src = vis ? __ffs((int)vis) - 1 : 0; // first occurrence wins (insert-if-absent)
            const uint32_t spos = __shfl_sync(kFull, ev_pos, src);
            uint32_t tpos = 0;
            if (!end_j)
                (void)et.find(b, last_word, key, in_table, tpos);
            hit = in_table || vis != 0;
            cand = in_table ? tpos : spos;
        }

        const unsigned H = __ballot_sync(kFull, probe && hit);
        const unsigned E = __ballot_sync(kFull, odd && end_j);
        const unsigned HE = H | E;
        // ---- commit the misses before the cut (the cut probe's own p-1 event is not one)
        const int f = HE ? __ffs((int)HE) - 1 : 33;
        const unsigned cm = f >= 33 ? kFull : (1u << (f - 1)) - 1u;
        const unsigned g = grp & cm;
        if (MODE == 0) {
            // update_hash_table :303-307: in program order the last writer of a slot wins
            if (g && 31 - __clz((int)g) == (int)lane) {
                hpos[idx] = (uint16_t)ev_pos;
                hfp[idx] = (uint8_t)ph;
            }
        } else {
            // insert-if-absent, src/BST.c:30-43: the first occurrence of a new key is kept
            const bool ins = g && !in_table && __ffs((int)g) - 1 == (int)lane;
            if (ins)
                et.insert_absent(key, ev_pos);
            n_keys += __popc(__ballot_sync(kFull, ins));
        }

        if (HE == 0) {
            pos += 16 * q + (16 > k1 ? 16 - k1 : 0u); // 16 x append_literal :283-287
            skip += 16 * C;
        } else if (!((H >> f) & 1u)) {
            break; // the end-of-block test fired first
        } else {
            __syncwarp();
            const uint32_t p = __shfl_sync(kFull, ev_pos, f);
            const uint32_t c = __shfl_sync(kFull, cand, f);
            if (MODE == 0) {
                if ((int)lane == f) { // emit_copy :327
                    hpos[idx] = (uint16_t)ev_pos;
                    hfp[idx] = (uint8_t)ph;
                }
            } else {
                if ((int)lane == f) { // tree.c:221: the found node now points at this position
                    bool fnd;
                    uint32_t tp;
                    const uint32_t s = et.find(b, last_word, key, fnd, tp);
                    et.set(s, key, ev_pos);
                }
            }
            const uint32_t e4 = __shfl_sync(kFull, ext4, f);
            const uint32_t len = e4 < 4 ? 4 + e4 : match_extend(b, p, c, n, last_word, lane);
            if (lane == (nh & 31u))
                rec = make_uint2(p | ((p - c) << 16), len | ((p - prev_end) << 16));
            ++nh;
            if ((nh & 31u) == 0)
                my_recs[nh - 32 + lane] = rec;
            pos = p + len;
            prev_end = pos;
            skip = 32; // start_new_literal :271-274
            narrow = true;
            __syncwarp();
        }

        if (MODE == 1 && !FINAL && n_keys > (ExactTable<LOG_SLOTS, GLOBAL>::kSlots * 3) / 4) {
            if (lane == 0)
                nrec[blk] = kAbortMark;
            return;
        }
    }
    if (lane < (nh & 31u))
        my_recs[(nh & ~31u) + lane] = rec;
    if (lane == 0)
        nrec[blk] = nh;
}

// The big exact tiers with the table in shared memory, one CTA per block: only the blocks an earlier tier gave up on.
template <int LOG_SLOTS, bool FINAL>
__global__ void __launch_bounds__(32) k_parse(const uint8_t *__restrict__ in, uint64_t n_bytes,
                                              uint2 *__restrict__ recs, uint32_t *__restrict__ nrec)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const uint64_t blk = blockIdx.x;
    if (nrec[blk] != kAbortMark)
        return;
    parse_block<1, LOG_SLOTS, FINAL>(in, n_bytes, recs, nrec, blk, smem_raw);
}

// The big exact tier: 2^16 slots (128 KiB) per chain do not fit many times into shared memory
// (1 chain per SM), and a chain is bound by latency, not by bandwidth -- so the tables go to global
// memory (the blocks' output slots, which nothing uses before k_emit) and every SM runs as many
// chains as it can hold warps for.  Persistent CTAs: each owns one table and takes marked blocks
// from a counter.
constexpr int kGlobalTierLog = 16;
template <int LOG_SLOTS, bool FINAL>
__global__ void __launch_bounds__(32) k_parse_exact_global(const uint8_t *__restrict__ in, uint64_t n_bytes,
                                                           uint64_t n_blocks, uint2 *__restrict__ recs,
                                                           uint32_t *__restrict__ nrec, uint8_t *__restrict__ tables,
                                                           uint32_t *__restrict__ counter, int only_marked)
{
    uint8_t *table = tables + (size_t)blockIdx.x * ((size_t)4 << LOG_SLOTS); // 32-bit entries (position + fingerprint)
    for (;;) {
        uint32_t blk = 0;
        if (threadIdx.x == 0)
            blk = atomicAdd(counter, 1u);
        blk = __shfl_sync(kFull, blk, 0);
        if (blk >= n_blocks)
            return;
        if (only_marked && nrec[blk] != kAbortMark)
            continue;
        parse_block<1, LOG_SLOTS, FINAL, true>(in, n_bytes, recs, nrec, blk, table);
        __syncwarp();
    }
}

// Hash mode with the two table arrays (12 KiB per chain) in global memory: persistent one-warp CTAs,
// 32 per SM, each with its own tables, taking blocks from a counter.  With nothing in shared
// memory the SM's whole 256 KB is L1, which keeps the hot part of the tables close, and 32
// latency-bound chains per SM beat the 17-18 that 12 KiB shared-memory tables allow (measured:
// 16.0 -> 14.0 ms per GiB of the mixed corpus, DESIGN.md §4).
__global__ void __launch_bounds__(32) k_parse_hash_global(const uint8_t *__restrict__ in, uint64_t n_bytes,
                                                          uint64_t n_blocks, uint2 *__restrict__ recs,
                                                          uint32_t *__restrict__ nrec, uint8_t *__restrict__ tables,
                                                          uint32_t *__restrict__ counter)
{
    uint8_t *table = tables + (size_t)blockIdx.x * (size_t)(3 * SNAPPY_B200_HTABLE_SIZE);
    __shared__ __align__(16) uint8_t fp_smem[SNAPPY_B200_HTABLE_SIZE];
    for (;;) {
        uint32_t blk = 0;
        if (threadIdx.x == 0)
            blk = atomicAdd(counter, 1u);
        blk = __shfl_sync(kFull, blk, 0);
        if (blk >= n_blocks)
            return;
        parse_block<0, 12, true, true>(in, n_bytes, recs, nrec, blk, table, fp_smem);
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------- emission
constexpr int kEmitThreads = 128;
constexpr uint32_t kCoopLiteral = 48; // literals at least this long are copied by the whole CTA

// reference: write_literal :95-120 -- header bytes for a literal of len (>0) bytes
__device__ __forceinline__ uint32_t literal_header(uint32_t len, uint8_t *__restrict__ o)
{
    const uint32_t m = len - 1;
    if (m < 60) {
        o[0] = (uint8_t)(m << 2);
        return 1;
    }
    if (m < 256) {
        o[0] = 60u << 2;
        o[1] = (uint8_t)m;
        return 2;
    }
    o[0] = 61u << 2; // m <= 65535 inside a 64 KiB block
    o[1] = (uint8_t)m;
    o[2] = (uint8_t)(m >> 8);
    return 3;
}

__device__ __forceinline__ uint32_t literal_size(uint32_t len)
{
    return len == 0 ? 0 : len + (len <= 60 ? 1 : (len <= 256 ? 2 : 3));
}

// reference: write_copy :153-165 / write_single_copy :131-145
__device__ __forceinline__ uint32_t copy_size(uint32_t len, uint32_t off)
{
    const uint32_t n64 = len > 68 ? (len - 5) / 64 : 0; // "while (len > 68) emit 64"
    uint32_t rem = len - 64 * n64, sz = 3 * n64;
    if (rem > 64) { // 64 < rem <= 68: emit 60 so that at least 4 remain
        sz += 3;
        rem -= 60;
    }
    return sz + ((rem < 12 && off < 2048) ? 2 : 3);
}

__device__ __forceinline__ void copy_emit(uint32_t len, uint32_t off, uint8_t *__restrict__ o)
{
    const uint32_t n64 = len > 68 ? (len - 5) / 64 : 0;
    uint32_t rem = len - 64 * n64;
    for (uint32_t k = 0; k < n64; ++k) {
        o[0] = 0xfe; // ((64-1) << 2) | 2
        o[1] = (uint8_t)off;
        o[2] = (uint8_t)(off >> 8);
        o += 3;
    }
    if (rem > 64) {
        o[0] = 0xee; // ((60-1) << 2) | 2
        o[1] = (uint8_t)off;
        o[2] = (uint8_t)(off >> 8);
        o += 3;
        rem -= 60;
    }
    if (rem < 12 && off < 2048) {
        o[0] = (uint8_t)(((off >> 8) << 5) + ((rem - 4) << 2) + 1);
        o[1] = (uint8_t)off;
    } else {
        o[0] = (uint8_t)(((rem - 1) << 2) | 2);
        o[1] = (uint8_t)off;
        o[2] = (uint8_t)(off >> 8);
    }
}

__global__ void __launch_bounds__(kEmitThreads) k_emit(const uint8_t *__restrict__ in, uint64_t n_bytes,
                                                       const uint2 *__restrict__ recs,
                                                       const uint32_t *__restrict__ nrec,
                                                       uint8_t *__restrict__ scratch, uint32_t *__restrict__ sizes)
{
    __shared__ uint32_t warp_sum[kEmitThreads / 32 + 1];
    __shared__ uint32_t q_src[kEmitThreads], q_dst[kEmitThreads], q_len[kEmitThreads];
    __shared__ uint32_t q_n;
    const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint64_t blk = blockIdx.x;
    const uint8_t *__restrict__ b = in + blk * (uint64_t)kBlock;
    const uint64_t left = n_bytes - blk * (uint64_t)kBlock;
    const uint32_t n = left < kBlock ? (uint32_t)left : kBlock;
    const uint2 *__restrict__ my_recs = recs + blk * (uint64_t)kMaxRecords;
    uint8_t *__restrict__ out = scratch + blk * (uint64_t)kSlot;
    const uint32_t nr = nrec[blk];

    uint32_t carry = 0;    // bytes emitted by earlier chunks
    uint32_t last_end = 0; // end of the last copy: where the tail literal starts
    for (uint32_t base = 0; base < nr; base += kEmitThreads) {
        if (tid == 0)
            q_n = 0;
        const uint32_t i = base + tid;
        uint32_t p = 0, off = 0, len = 0, lit = 0, sz = 0;
        if (i < nr) {
            const uint2 rc = my_recs[i];
            p = rc.x & 0xffffu, off = rc.x >> 16, len = rc.y & 0xffffu, lit = rc.y >> 16;
            sz = literal_size(lit) + copy_size(len, off);
        }
        // exclusive scan of sz over the CTA
        uint32_t incl = sz;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(kFull, incl, d);
            if ((int)lane >= d)
                incl += t;
        }
        if (lane == 31)
            warp_sum[wid] = incl;
        __syncthreads();
        if (tid == 0) {
            uint32_t run = 0;
#pragma unroll
            for (int w = 0; w < kEmitThreads / 32; ++w) {
                const uint32_t t = warp_sum[w];
                warp_sum[w] = run;
                run += t;
            }
            warp_sum[kEmitThreads / 32] = run;
        }
        __syncthreads();
        uint32_t o = carry + warp_sum[wid] + (incl - sz);
        const uint32_t chunk_total = warp_sum[kEmitThreads / 32];
        if (i < nr) {
            if (lit) { // emit_literal :313-316
                const uint32_t hdr = literal_header(lit, out + o);
                const uint32_t src = p - lit;
                if (lit >= kCoopLiteral) {
                    const uint32_t slot = atomicAdd(&q_n, 1u);
                    q_src[slot] = src, q_dst[slot] = o + hdr, q_len[slot] = lit;
                } else {
                    for (uint32_t k = 0; k < lit; ++k)
                        out[o + hdr + k] = __ldg(b + src + k);
                }
                o += hdr + lit;
            }
            copy_emit(len, off, out + o); // emit_copy :323-329
            if (i == nr - 1)
                last_end = p + len;
        }
        __syncthreads();
        const uint32_t nq = q_n;
        for (uint32_t k = 0; k < nq; ++k)
            coop_copy_ro(out + q_dst[k], b + q_src[k], q_len[k], tid, kEmitThreads);
        carry += chunk_total;
        __syncthreads();
    }
    // tail literal: exhaust_input :292-297 + emit_literal :401-402
    if (nr) {
        // last_end lives in the thread that handled record nr-1
        __shared__ uint32_t s_last;
        if ((nr - 1) % kEmitThreads == tid)
            s_last = last_end;
        __syncthreads();
        last_end = s_last;
    }
    const uint32_t tail = n - last_end;
    uint32_t hdr = 0;
    if (tail) {
        __shared__ uint32_t s_hdr;
        if (tid == 0)
            s_hdr = literal_header(tail, out + carry);
        __syncthreads();
        hdr = s_hdr;
        coop_copy_ro(out + carry + hdr, b + last_end, tail, tid, kEmitThreads);
    }
    if (tid == 0)
        sizes[blk] = carry + hdr + tail;
}

// ------------------------------------------------------------------------------- launchers
cudaError_t launch_parallel_parse(const uint8_t *, uint64_t, uint64_t, uint16_t *, uint8_t *, uint2 *, uint32_t *,
                                  cudaStream_t, uint64_t *); // compress_parallel.cu

// d_cand: SNAPPY_B200_MODE_PARALLEL's candidate offsets (a u16 per input byte); not used by the other modes.
cudaError_t launch_compress(const uint8_t *d_in, uint64_t n_bytes, int mode, uint8_t *d_scratch, uint32_t *d_sizes,
                            uint2 *d_recs, uint32_t *d_nrec, uint16_t *d_cand, cudaStream_t st, uint64_t *launches)
{
    const uint64_t nb = (n_bytes + kBlock - 1) / kBlock;
    if (nb == 0)
        return cudaSuccess;
    if (nb > 0x7fffffffull)
        return cudaErrorInvalidValue;
    const dim3 grid((unsigned)nb), cta(32);
    // Tables in global memory: carved out of the blocks' output slots, which nothing uses before
    // k_emit; the last 256 bytes of that area hold the work counters of the persistent kernels.
    int n_sm = 0, dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        n_sm <= 0)
        n_sm = 148;
    const uint64_t chains = std::min<uint64_t>(nb, (uint64_t)n_sm * 32); // one-warp CTAs: 32 per SM
    const uint64_t area = nb * (uint64_t)kSlot - 256;
    uint32_t *counters = reinterpret_cast<uint32_t *>(d_scratch + area);
    cudaError_t e = cudaMemsetAsync(counters, 0, 16, st);
    if (e != cudaSuccess)
        return e;
    if (mode == SNAPPY_B200_MODE_HASH) {
        k_parse_hash_global<<<(unsigned)chains, cta, 0, st>>>(d_in, n_bytes, nb, d_recs, d_nrec, d_scratch, counters);
        *launches += 1;
    } else if (mode == SNAPPY_B200_MODE_PARALLEL) {
        e = launch_parallel_parse(d_in, n_bytes, nb, d_cand, d_scratch, d_recs, d_nrec, st, launches);
        if (e != cudaSuccess)
            return e;
    } else {
        // exact mode: 8 Ki slots (16 KiB), then 64 Ki slots (128 KiB) for the blocks that outgrow them
        // (> 6144 distinct keys: text)
        // (the opt-in to > 48 KiB of dynamic shared memory is per device: once per device, thread-safe)
        static std::once_flag attr_once[64];
        std::call_once(attr_once[dev & 63], [&] {
            e = cudaFuncSetAttribute(k_parse<15, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (1 << 15) * 2);
            if (e == cudaSuccess)
                e = cudaFuncSetAttribute(k_parse<16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (1 << 16) * 2);
        });
        if (e != cudaSuccess)
            return e;
        k_parse_exact_global<13, false><<<(unsigned)chains, cta, 0, st>>>(d_in, n_bytes, nb, d_recs, d_nrec, d_scratch,
                                                                          counters + 1, 0);
        const uint64_t n_big = std::min<uint64_t>(area / ((uint64_t)4 << kGlobalTierLog), chains);
        if (n_big >= 1) {
            k_parse_exact_global<kGlobalTierLog, true><<<(unsigned)n_big, cta, 0, st>>>(d_in, n_bytes, nb, d_recs, d_nrec,
                                                                                     d_scratch, counters + 2, 1);
            *launches += 2;
        } else { // 1 to 3 blocks: the output slots cannot hold one 256 KiB table, so the big tiers go to shared memory
            k_parse<15, false><<<grid, cta, (1 << 15) * 2, st>>>(d_in, n_bytes, d_recs, d_nrec);
            k_parse<16, true><<<grid, cta, (1 << 16) * 2, st>>>(d_in, n_bytes, d_recs, d_nrec);
            *launches += 3;
        }
    }
    k_emit<<<grid, kEmitThreads, 0, st>>>(d_in, n_bytes, d_recs, d_nrec, d_scratch, d_sizes);
    *launches += 1;
    return cudaGetLastError();
}

size_t compress_records_bytes(uint64_t n_blocks) { return n_blocks * (size_t)kMaxRecords * sizeof(uint2); }

} // namespace sb200
