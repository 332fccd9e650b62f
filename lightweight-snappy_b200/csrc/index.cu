// index.cu -- K0: where does every 64 KiB output block start inside an index-less stream?
//
// The reference discovers this implicitly by walking the elements one after another
// (src/snappy_decompression.c:353-356): block boundaries are not recorded in the format
// (src/snappy_compression.c:334-336 just appends blocks).  A sequential tag walk over a
// gigabyte is hopeless on a GPU, so the walk is made parallel by speculation:
//
//   A  k_index_spec    the stream body is cut into 128-byte segments, one thread each.  Every
//                      thread walks elements from the first byte of its segment as if an
//                      element started there, remembers the visited offsets in a 128-bit map
//                      and the offset at which it leaves the segment.  Snappy streams
//                      re-synchronise within a few elements, so most of these walks merge
//                      into the true element chain long before the segment ends.
//   B  k_group_*       the segments are taken 64 at a time (8 KiB "groups"), one warp per group.
//                      Inside a group the chain is resolved by a relaxation over its 64 segments
//                      (group_resolve): every segment publishes the exit of its current walk to
//                      the segment it lands in, a live segment marks the segments a long
//                      element jumps over as "dead" (holding no element start), a segment that
//                      was itself marked dead keeps publishing its exit at low priority, the
//                      lowest source wins, and a segment whose entry changed re-walks from the
//                      new entry until it meets its recorded path.  The entry of one segment is
//                      known, every other segment is claimed or marked by a live predecessor, so
//                      the beliefs are correct on a prefix that grows every round, and a round
//                      that changes nothing is the unique fixed point = the chain.  (ASCII text
//                      makes mis-speculated walks take ~27-byte strides, so about half of the
//                      128-byte walks do NOT merge by themselves: lanes re-walk different
//                      segments in parallel here instead of one serial chase per group.)
//                      The groups themselves are resolved by the same relaxation one level up
//                      (k_group_scatter / k_group_apply in round 0, then one fused k_group_apply32
//                      per round; group 0's entry is known).  Keeping dead groups talking
//                      matters: when a mis-speculated "long literal" wrongly kills a run of
//                      groups they all come back in the round after it is corrected instead of
//                      one per round.
//                      Runs of incompressible blocks are chains of maximal literals that can
//                      only be found one from the other; scatter_group looks 24 of them ahead.
//                      An adversarial stream degrades to sequential but stays correct.
//   C  (k_group_final) every live segment sums the output bytes of its elements and stores the
//                      exact bit map of its element starts (for the segment-driven decoder)
//      k_scan_*        exclusive scan -> output offset of every segment
//   D  k_index_blocks  every live segment walks once more and records the stream offset of
//                      each element that starts a 64 KiB output block; elements that straddle
//                      a block boundary (legal raw Snappy, never produced by this framing) are
//                      reported as SNAPPY_B200_ST_FRAMING.
#include <algorithm>
#include <atomic>

#include "common.cuh"

namespace sb200 {

constexpr uint32_t kSeg = 128;          // bytes of stream per segment
constexpr uint32_t kDead = 0x80u;       // entry[t] bit 7: no element starts here (bits 0-6 keep the last entry)
constexpr uint32_t kMark = 0xffu;       // claim payload: "a literal jumps over you"
constexpr unsigned long long kLowPrio = 1ull << 63;
constexpr unsigned long long kNone = ~0ull;
constexpr uint64_t kMaxLiteralElemBytes = 3 + (uint64_t)SNAPPY_B200_BLOCK_SIZE; // "f4 ff ff" + 65 536 bytes

struct Elem {
    uint64_t size; // bytes of stream this element occupies (header + literal payload)
    uint64_t out;  // bytes of output it produces
    bool ok;       // header fits in the body
};

// Decodes the element header at body offset e (reference: decompressor :290-333, do_literal
// :193-224).  Bytes past the end of the body read as zero and clear `ok`.
// LDG: read through the read-only global path; otherwise plain loads (body may then be a view of
// a shared-memory copy: body + e must be a valid address for every e that is touched).
template <bool LDG = true>
__device__ __forceinline__ Elem decode_at(const uint8_t *__restrict__ body, uint64_t body_len, uint64_t e)
{
    // Written with selects instead of branches: the threads of a warp walk different segments, and every
    // branch on the element kind would split the warp (the walks are issue bound: k_index_spec ran at 91 %
    // issue utilisation with 14 of 32 lanes active).  Only the 1..4 length bytes of a long literal, which are
    // rare, sit behind a branch.
    Elem r;
    const uint32_t tag = LDG ? __ldg(body + e) : body[e];
    const uint32_t type = tag & 3u, m = tag >> 2;
    const bool lit = type == 0;
    const bool longlit = lit && m >= 60;
    const uint32_t extra = lit ? (longlit ? m - 59u : 0u) : ((0x4210u >> (type * 4u)) & 0xfu); // header bytes after the tag
    r.ok = e + 1 + extra <= body_len;
    uint32_t raw = m;
    if (longlit) {
        raw = 0;
        if (r.ok)
            for (uint32_t k = 0; k < extra; ++k)
                raw |= (uint32_t)(LDG ? __ldg(body + e + 1 + k) : body[e + 1 + k]) << (8 * k);
    }
    const uint64_t len = lit ? (uint64_t)raw + 1 : 0;      // payload bytes that follow the header
    r.size = 1 + extra + len;
    r.out = lit ? len : (uint64_t)(type == 1 ? (m & 7u) + 4u : m + 1u);
    return r;
}

struct Path {
    uint32_t bits[4];
    __device__ __forceinline__ void clear() { bits[0] = bits[1] = bits[2] = bits[3] = 0; }
    __device__ __forceinline__ void set(uint32_t i)
    {
        const uint32_t b = 1u << (i & 31), w = i >> 5;
        bits[0] |= w == 0 ? b : 0u;
        bits[1] |= w == 1 ? b : 0u;
        bits[2] |= w == 2 ? b : 0u;
        bits[3] |= w == 3 ? b : 0u;
    }
    __device__ __forceinline__ bool test(uint32_t i) const
    {
        const uint32_t w = i >> 5;
        const uint32_t v = w == 0 ? bits[0] : (w == 1 ? bits[1] : (w == 2 ? bits[2] : bits[3]));
        return (v >> (i & 31)) & 1u;
    }
};

// Walks from e until the segment [seg_lo, seg_hi) is left, or (when `old` is given) until an
// offset already on the old path is met.  Visited offsets are recorded in `fresh`.
template <bool LDG = true>
__device__ __forceinline__ uint64_t walk(const uint8_t *__restrict__ body, uint64_t body_len, uint64_t seg_lo,
                                         uint64_t seg_hi, uint64_t e, const Path *old, Path &fresh, bool &merged)
{
    merged = false;
    while (e < seg_hi) {
        const uint32_t rel = (uint32_t)(e - seg_lo);
        if (old && old->test(rel)) {
            merged = true;
            return e;
        }
        fresh.set(rel);
        const Elem el = decode_at<LDG>(body, body_len, e);
        e += el.size; // seg_hi <= body_len, sizes < 2^33: no overflow
    }
    return e;
}

__global__ void __launch_bounds__(256) k_index_spec(const uint8_t *__restrict__ body, uint64_t body_len, uint64_t nseg,
                                                    uint4 *__restrict__ paths, uint64_t *__restrict__ exits)
{
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= nseg)
        return;
    const uint64_t lo = t * kSeg;
    const uint64_t hi = min(lo + kSeg, body_len);
    Path p;
    p.clear();
    bool merged;
    const uint64_t x = walk(body, body_len, lo, hi, lo, nullptr, p, merged);
    paths[t] = make_uint4(p.bits[0], p.bits[1], p.bits[2], p.bits[3]);
    exits[t] = x;
}

// ---- groups of kGroup segments ------------------------------------------------------------
constexpr uint32_t kGroup = 64;                   // segments per group
constexpr uint64_t kGroupBytes = kGroup * kSeg;   // 8 KiB of stream
constexpr uint32_t kGDead = 0x80000000u;          // g_entry bit 31: no element starts in this group
constexpr uint32_t kGMark = 0xffffffu;            // claim payload: "a literal jumps over you"

// One warp works on one group.  The group's per-segment records (path map + exit) are staged
// in shared memory with coalesced loads; the chase itself is a short dependent chain that all
// lanes execute redundantly on the staged copy.
constexpr int kGroupCta = 128;                 // 4 warps = 4 groups per CTA
struct GroupStage {
    uint4 paths[kGroup];
    uint64_t exits[kGroup];
    uint32_t claim[kGroup];
    uint8_t entry[kGroup];
};

// Stages the per-segment records of group g.
__device__ __forceinline__ void group_stage(GroupStage &sm, uint64_t g, uint64_t nseg, const uint4 *__restrict__ paths,
                                            const uint64_t *__restrict__ exits)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t s0 = g * kGroup;
#pragma unroll
    for (uint32_t k = lane; k < kGroup; k += 32) {
        const bool ok = s0 + k < nseg;
        sm.paths[k] = ok ? paths[s0 + k] : make_uint4(0, 0, 0, 0);
        sm.exits[k] = ok ? exits[s0 + k] : 0;
    }
    __syncwarp();
}

// Writes the (possibly improved) per-segment records back, so that later passes find the chain
// on the recorded paths.
// `entries` keeps the entry offset of every segment on the chain just resolved (kDead: none), so that the
// last pass does not have to resolve the group once more.
__device__ __forceinline__ void group_unstage(const GroupStage &sm, uint64_t g, uint64_t nseg, uint4 *__restrict__ paths,
                                              uint64_t *__restrict__ exits, uint8_t *__restrict__ entries)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t s0 = g * kGroup;
#pragma unroll
    for (uint32_t k = lane; k < kGroup; k += 32)
        if (s0 + k < nseg) {
            paths[s0 + k] = sm.paths[k];
            exits[s0 + k] = sm.exits[k];
            entries[s0 + k] = sm.entry[k];
        }
}

// Makes `rel` the entry of staged segment k (global index t): if it is not on the recorded path
// the tags are walked from it until the path is met (the exit stands, the path grows) or the
// segment is left (a different chain: path and exit are replaced).
__device__ __forceinline__ void segment_enter(const uint8_t *__restrict__ body, uint64_t body_len, GroupStage &sm,
                                              uint32_t k, uint64_t t, uint32_t rel)
{
    const uint4 pv = sm.paths[k];
    Path p;
    p.bits[0] = pv.x, p.bits[1] = pv.y, p.bits[2] = pv.z, p.bits[3] = pv.w;
    if (p.test(rel))
        return;
    Path fresh;
    fresh.clear();
    bool merged;
    const uint64_t lo = t * kSeg, hi = min(lo + kSeg, body_len);
    const uint64_t x = walk(body, body_len, lo, hi, lo + rel, &p, fresh, merged);
    if (merged) {
#pragma unroll
        for (int w = 0; w < 4; ++w)
            fresh.bits[w] |= p.bits[w];
    } else {
        sm.exits[k] = x;
    }
    sm.paths[k] = make_uint4(fresh.bits[0], fresh.bits[1], fresh.bits[2], fresh.bits[3]);
}

// Resolves the element chain of group g from body offset e0 (which lies in the group) to the
// end of the group: the same relaxation as between groups, but over the 64 staged segments and
// inside one warp -- lane l owns segments l and l+32, so the tag walks of different segments run
// in parallel instead of one after the other.  Every segment publishes the exit of its current
// walk to the segment it lands in and (if live) marks the segments a long element jumps over
// as dead; dead segments keep publishing at low priority; the lowest source wins.  The segment
// that holds e0 is known, so the correct prefix grows every round and the fixed point is the
// chain.  Leaves the entry of every segment in sm.entry (kDead where no element starts), sets
// vis to the live segments and returns the offset at which the chain leaves the group.
__device__ __forceinline__ uint64_t group_resolve(const uint8_t *__restrict__ body, uint64_t body_len, uint64_t nseg,
                                                  GroupStage &sm, uint64_t g, uint64_t e0, uint64_t &vis)
{
    constexpr uint32_t kNoClaim = 0xffffffffu, kLow = 0x80000000u;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t s0 = g * kGroup;
    const uint32_t nk = (uint32_t)(min(s0 + kGroup, nseg) - s0); // segments in this group
    const uint64_t g_hi = min((s0 + nk) * kSeg, body_len);
    const uint32_t k0 = (uint32_t)(e0 / kSeg - s0);
    const uint32_t rel0 = (uint32_t)(e0 - (s0 + k0) * kSeg);
    // initial beliefs: the segment of e0 is known, later ones start out at the first offset of
    // their recorded path (any offset on it leads to the recorded exit), earlier ones hold nothing
    for (uint32_t k = lane; k < kGroup; k += 32) {
        const uint4 pv = sm.paths[k];
        const uint32_t first = pv.x   ? __ffs((int)pv.x) - 1
                               : pv.y ? 32 + __ffs((int)pv.y) - 1
                               : pv.z ? 64 + __ffs((int)pv.z) - 1
                               : pv.w ? 96 + __ffs((int)pv.w) - 1
                                      : 0;
        sm.entry[k] = (uint8_t)(k < k0 || k >= nk ? kDead : (k == k0 ? rel0 : first));
        if (k == k0 && k < nk)
            segment_enter(body, body_len, sm, k, s0 + k, rel0);
    }
    __syncwarp();
    for (uint32_t round = 0; round < kGroup + 2; ++round) {
        for (uint32_t k = lane; k < kGroup; k += 32)
            sm.claim[k] = kNoClaim;
        __syncwarp();
        for (uint32_t k = lane; k < nk; k += 32) {
            if (k < k0)
                continue;
            const bool dead = sm.entry[k] & kDead;
            const uint64_t x = sm.exits[k];
            const uint64_t u64 = x / kSeg - s0; // staged index of the landing segment (>= k + 1)
            const uint32_t u = u64 < kGroup ? (uint32_t)u64 : kGroup;
            if (!dead) {
                for (uint32_t v = k + 1; v < min(u, nk); ++v)
                    atomicMin(&sm.claim[v], (k << 8) | kMark);
                if (u < nk && x >= body_len)
                    atomicMin(&sm.claim[u], (k << 8) | kMark);
            }
            if (u < nk && x < body_len)
                atomicMin(&sm.claim[u], (dead ? kLow : 0u) | (k << 8) | (uint32_t)(x - (s0 + u) * kSeg));
        }
        __syncwarp();
        bool changed = false;
        for (uint32_t k = lane; k < nk; k += 32) {
            if (k <= k0)
                continue;
            const uint32_t c = sm.claim[k];
            const uint32_t old = sm.entry[k];
            const uint32_t payload = c & 0xffu;
            const uint32_t ne = (c == kNoClaim || payload == kMark) ? ((old & 0x7fu) | kDead) : payload;
            if (ne == old)
                continue;
            changed = true;
            sm.entry[k] = (uint8_t)ne;
            if (!(ne & kDead))
                segment_enter(body, body_len, sm, k, s0 + k, ne); // (returns at once if ne is on the path)
        }
        __syncwarp();
        if (!__any_sync(kFull, changed))
            break;
    }
    // live segments, and the exit of the last one
    const bool live0 = lane < nk && !(sm.entry[lane] & kDead);
    const bool live1 = lane + 32 < nk && !(sm.entry[lane + 32] & kDead);
    const unsigned m0 = __ballot_sync(kFull, live0), m1 = __ballot_sync(kFull, live1);
    vis = (uint64_t)m0 | ((uint64_t)m1 << 32);
    const uint32_t last = m1 ? 32 + (31 - __clz((int)m1)) : (m0 ? 31 - __clz((int)m0) : k0);
    (void)g_hi;
    return sm.exits[last];
}

// Initial state: every group believes an element starts at its first byte.
__global__ void __launch_bounds__(kGroupCta) k_group_init(const uint8_t *__restrict__ body, uint64_t body_len,
                                                          uint64_t nseg, uint64_t ngroup, uint4 *__restrict__ paths,
                                                          uint64_t *__restrict__ exits,
                                                          uint32_t *__restrict__ g_entry, uint64_t *__restrict__ g_exit,
                                                          uint64_t *__restrict__ g_vis,
                                                          unsigned long long *__restrict__ g_claim,
                                                          uint8_t *__restrict__ entries, int literal_scan)
{
    __shared__ GroupStage stage[kGroupCta / 32];
    const uint64_t g = blockIdx.x * (uint64_t)(kGroupCta / 32) + (threadIdx.x >> 5);
    if (g >= ngroup)
        return;
    GroupStage &sm = stage[threadIdx.x >> 5];
    group_stage(sm, g, nseg, paths, exits);
    // First belief about where the chain enters this group.  "At its first byte" is right one time in four
    // on text; the speculative walks of the segments just before the group are a free run-up: follow their
    // exits (exit of segment s, landing on the recorded path of the segment it falls in, that segment's exit,
    // ...) from up to three segments back into the group.  Every hop that lands on a recorded path halves the
    // chance that the walk is still off the true chain.  Only table look-ups, no tag walk; any value read here
    // is a guess that the relaxation corrects (a neighbour may be rewriting its records meanwhile).
    uint64_t e0 = g * kGroupBytes;
    // Incompressible blocks are maximal literals, "f4 ff ff" + 65 536 bytes, and the payload in between
    // tells nothing: a group that lies right after such a literal looks 65 539 bytes back for the header that
    // would end inside it.  A hit is strong evidence (24 bits) for an element start, and it turns the chain of
    // literals of a run of incompressible blocks, which the relaxation can only follow 24 per round, into
    // local knowledge of every group (random data: 32 -> 10 rounds, K0 4.9 -> 3.1 ms).  The 8 KiB are read
    // with coalesced word loads, every lane checks the four byte positions of its word against the word after
    // it.  Reading the stream once more costs 0.15 ms per GiB of mixed data, where it finds nothing: the scan is
    // only switched on for streams that are mostly incompressible (run_index).
    uint64_t lit_end = kNone;
    if (literal_scan && g * kGroupBytes >= kMaxLiteralElemBytes) {
        const uint64_t g_lo = g * kGroupBytes, g_hi = min(g_lo + kGroupBytes, body_len);
        const uint32_t lane = threadIdx.x & 31;
        const uint32_t n = (uint32_t)(g_hi - g_lo); // header positions src .. src + n
        const uint8_t *src = body + (g_lo - kMaxLiteralElemBytes);
        const uint32_t a = (uint32_t)reinterpret_cast<uintptr_t>(src) & 3u;
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(src - a);
        const uint32_t nw = (a + n + 3u) >> 2; // words that hold a candidate position (<= 2049)
        uint32_t first = 0xffffffffu;         // position (relative to src) of the first header found by this lane
#pragma unroll 4
        for (uint32_t i = lane; i < nw; i += 32) {
            const uint32_t w0 = __ldg(wp + i), w1 = __ldg(wp + i + 1); // (w1: at most 4 bytes past the last position, still before g_lo)
#pragma unroll
            for (uint32_t k = 0; k < 4; ++k) {
                const uint32_t off = 4u * i + k - a; // wraps below 0 for the bytes before src
                if ((__funnelshift_r(w0, w1, 8u * k) & 0xffffffu) == 0xfffff4u && off < n)
                    first = min(first, off);
            }
        }
        const uint32_t best = __reduce_min_sync(kFull, first);
        if (best != 0xffffffffu)
            lit_end = g_lo + best;
    }
    if (lit_end != kNone) {
        e0 = lit_end;
    } else if (g > 0) {
        const uint64_t g_lo = g * kGroupBytes, g_hi = min(g_lo + kGroupBytes, body_len);
        const uint64_t s_last = g * kGroup - 1;
        for (int back = 2; back >= 0; --back) {
            if (s_last < (uint64_t)back)
                continue;
            uint64_t x = exits[s_last - back];
            bool ok = true;
            for (int hop = 0; ok && x < g_lo && hop < 4; ++hop) {
                const uint64_t sx = x / kSeg;
                const uint4 pv = paths[sx];
                Path p;
                p.bits[0] = pv.x, p.bits[1] = pv.y, p.bits[2] = pv.z, p.bits[3] = pv.w;
                ok = p.test((uint32_t)(x - sx * kSeg));
                if (ok)
                    x = exits[sx];
            }
            if (ok && x >= g_lo) {
                if (x < g_hi)
                    e0 = x;
                break; // (a chain that jumps over the whole group keeps the default)
            }
        }
    }
    uint64_t vis;
    const uint64_t x = group_resolve(body, body_len, nseg, sm, g, e0, vis);
    group_unstage(sm, g, nseg, paths, exits, entries);
    if ((threadIdx.x & 31) == 0) {
        g_exit[g] = x;
        g_vis[g] = vis;
        g_entry[g] = (uint32_t)(e0 - g * kGroupBytes);
        g_claim[g] = kNone;
    }
}

// Runs of incompressible 64 KiB blocks are chains of maximal literals, "f4 ff ff" + 65536 bytes,
// each of which can only be found through the one before: one hop per round.  When a live
// group's chain leaves through such a literal, the positions of the next kLookahead headers are
// guessed (65539 apart), fetched all at once, and the confirmed prefix of the run is published
// in the same round.
constexpr uint32_t kLookahead = 24;
constexpr uint64_t kMaxLiteralElem = 3 + (uint64_t)kBlock; // header + payload of a maximal literal

__device__ __forceinline__ bool is_max_literal(const uint8_t *__restrict__ body, uint64_t body_len, uint64_t q)
{
    return q + kMaxLiteralElem <= body_len && __ldg(body + q) == 0xf4 && __ldg(body + q + 1) == 0xff &&
           __ldg(body + q + 2) == 0xff;
}

// What group g tells the groups after it (one round of the relaxation between groups).
__device__ __forceinline__ void scatter_group(const uint8_t *__restrict__ body, uint64_t body_len, uint64_t ngroup,
                                              uint64_t g, uint32_t entry, uint64_t x,
                                              unsigned long long *__restrict__ g_claim)
{
    const bool dead = entry & kGDead;
    const unsigned long long prio = dead ? kLowPrio : 0ull;
    const uint64_t u = x / kGroupBytes; // group the chain lands in
    if (!dead) {
        // Groups jumped over hold no element start (only a live source may say so: a dead
        // group's chase is pure speculation).  An element of this framing never spans more than
        // one 64 KiB block (+ header), which bounds the work a mis-speculated literal can cause;
        // a true element that long is reported as SNAPPY_B200_ST_FRAMING by k_group_final.
        const uint64_t vmax = min(min(u, ngroup), g + 2 + (kBlock + 1024) / kGroupBytes);
        for (uint64_t v = g + 1; v < vmax; ++v)
            atomicMin(g_claim + v, (unsigned long long)((g << 24) | kGMark));
        if (u < ngroup && x >= body_len) // the chain ends inside the last group: nothing starts there
            atomicMin(g_claim + u, (unsigned long long)((g << 24) | kGMark));
    }
    if (u < ngroup && x < body_len)
        atomicMin(g_claim + u, prio | (unsigned long long)((g << 24) | (x - u * kGroupBytes)));
    if (!dead && u > g + 1 && x < body_len) {
        // left through a long literal: look ahead along a possible run of maximal literals
        bool ok[kLookahead];
#pragma unroll
        for (uint32_t k = 0; k < kLookahead; ++k)
            ok[k] = is_max_literal(body, body_len, x + k * kMaxLiteralElem);
        uint64_t q = x;
#pragma unroll
        for (uint32_t k = 0; k < kLookahead; ++k) {
            if (!ok[k])
                break;
            // the element at q is a maximal literal: the chain continues at q + 65539
            const uint64_t qn = q + kMaxLiteralElem;
            const uint64_t uq = q / kGroupBytes, un = qn / kGroupBytes;
            for (uint64_t v = uq + 1; v < un && v < ngroup; ++v)
                atomicMin(g_claim + v, (unsigned long long)((g << 24) | kGMark));
            if (un < ngroup) {
                if (qn < body_len)
                    atomicMin(g_claim + un, (unsigned long long)((g << 24) | (qn - un * kGroupBytes)));
                else
                    atomicMin(g_claim + un, (unsigned long long)((g << 24) | kGMark));
            }
            q = qn;
        }
    }
}

__global__ void __launch_bounds__(128) k_group_scatter(const uint8_t *__restrict__ body, uint64_t body_len,
                                                       uint64_t ngroup, const uint32_t *__restrict__ g_entry,
                                                       const uint64_t *__restrict__ g_exit,
                                                       unsigned long long *__restrict__ g_claim)
{
    const uint64_t g = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (g >= ngroup)
        return;
    scatter_group(body, body_len, ngroup, g, g_entry[g], g_exit[g], g_claim);
}

__global__ void __launch_bounds__(kGroupCta) k_group_apply(const uint8_t *__restrict__ body, uint64_t body_len,
                                                           uint64_t nseg, uint64_t ngroup, uint4 *__restrict__ paths,
                                                           uint64_t *__restrict__ exits,
                                                           uint32_t *__restrict__ g_entry,
                                                           uint64_t *__restrict__ g_exit, uint64_t *__restrict__ g_vis,
                                                           unsigned long long *__restrict__ g_claim,
                                                           uint32_t *__restrict__ changed, uint8_t *__restrict__ entries)
{
    __shared__ GroupStage stage[kGroupCta / 32];
    const uint64_t g = blockIdx.x * (uint64_t)(kGroupCta / 32) + (threadIdx.x >> 5);
    if (g >= ngroup)
        return;
    const uint32_t lane = threadIdx.x & 31;
    const unsigned long long c = g_claim[g]; // every lane reads the same words (broadcast)
    const uint32_t old = g_entry[g];
    __syncwarp();
    if (lane == 0)
        g_claim[g] = kNone; // ready for the next round
    const uint32_t payload = (uint32_t)(c & 0xffffffu);
    uint32_t ne;
    if (g == 0)
        ne = 0; // the body starts with an element
    else if (c == kNone || payload == kGMark)
        ne = (old & ~kGDead) | kGDead;
    else
        ne = payload;
    if (ne == old)
        return;
    if (lane == 0) {
        g_entry[g] = ne;
        atomicOr(changed, 1u);
    }
    if ((ne & kGDead) || ne == (old & ~kGDead))
        return; // dead, or revived with the entry it already chased from
    // does the new entry lie on the old chain?  (it does if the old chain entered that segment on
    // the segment's recorded path and the new entry is on that path too)
    const uint64_t e = g * kGroupBytes + ne;
    const uint64_t sg = e / kSeg;
    const uint4 pv = paths[sg];
    Path p;
    p.bits[0] = pv.x, p.bits[1] = pv.y, p.bits[2] = pv.z, p.bits[3] = pv.w;
    if (((g_vis[g] >> (sg - g * kGroup)) & 1ull) && p.test((uint32_t)(e - sg * kSeg)))
        return; // same exit, and everything the old chain recorded still holds from here on
    GroupStage &sm = stage[threadIdx.x >> 5];
    group_stage(sm, g, nseg, paths, exits);
    uint64_t vis;
    const uint64_t x = group_resolve(body, body_len, nseg, sm, g, e, vis);
    group_unstage(sm, g, nseg, paths, exits, entries);
    if (lane == 0) {
        g_exit[g] = x;
        g_vis[g] = vis;
    }
}

// The same step with one LANE per group for the part every group goes through (two loads and,
// for nearly all groups after the first round, the finding that nothing changed); the few groups
// whose new entry is off their known chain are then re-resolved one after the other by the
// whole warp.  Lane l of warp w takes group l * n_warps + w, so that neighbouring groups -- which
// tend to need work together -- land in different warps.  32x fewer warps than k_group_apply.
__global__ void __launch_bounds__(kGroupCta) k_group_apply32(const uint8_t *__restrict__ body, uint64_t body_len,
                                                             uint64_t nseg, uint64_t ngroup, uint4 *__restrict__ paths,
                                                             uint64_t *__restrict__ exits,
                                                             uint32_t *__restrict__ g_entry,
                                                             uint64_t *__restrict__ g_exit,
                                                             uint64_t *__restrict__ g_vis,
                                                             unsigned long long *__restrict__ g_claim,
                                                             uint32_t *__restrict__ changed,
                                                             const uint32_t *__restrict__ prev_changed,
                                                             uint8_t *__restrict__ entries,
                                                             unsigned long long *__restrict__ claim_out)
{
    __shared__ GroupStage stage[kGroupCta / 32];
    if (prev_changed && *prev_changed == 0)
        return; // fixed point reached earlier in this batch
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t n_warps = (uint64_t)gridDim.x * (kGroupCta / 32);
    const uint64_t w = blockIdx.x * (uint64_t)(kGroupCta / 32) + (threadIdx.x >> 5);
    const uint64_t g = lane * n_warps + w;
    bool moved = false, heavy = false;
    uint64_t e = 0;
    if (g < ngroup) {
        const unsigned long long c = g_claim[g];
        const uint32_t old = g_entry[g];
        g_claim[g] = kNone; // ready for the next round
        const uint32_t payload = (uint32_t)(c & 0xffffffu);
        uint32_t ne;
        if (g == 0)
            ne = 0; // the body starts with an element
        else if (c == kNone || payload == kGMark)
            ne = (old & ~kGDead) | kGDead;
        else
            ne = payload;
        if (ne != old) {
            moved = true;
            g_entry[g] = ne;
            if (!(ne & kGDead) && ne != (old & ~kGDead)) { // (else: dead, or revived with the entry it already chased from)
                e = g * kGroupBytes + ne; // does the new entry lie on the old chain?
                const uint64_t sg = e / kSeg;
                const uint4 pv = paths[sg];
                Path p;
                p.bits[0] = pv.x, p.bits[1] = pv.y, p.bits[2] = pv.z, p.bits[3] = pv.w;
                heavy = !(((g_vis[g] >> (sg - g * kGroup)) & 1ull) && p.test((uint32_t)(e - sg * kSeg)));
            }
        }
    }
    if (__any_sync(kFull, moved) && lane == 0)
        atomicOr(changed, 1u);
    unsigned H = __ballot_sync(kFull, heavy);
    GroupStage &sm = stage[threadIdx.x >> 5];
    while (H) {
        const int src = __ffs((int)H) - 1;
        H &= H - 1;
        const uint64_t gg = (uint64_t)src * n_warps + w;
        const uint64_t ee = __shfl_sync(kFull, e, src);
        group_stage(sm, gg, nseg, paths, exits);
        uint64_t vis;
        const uint64_t x = group_resolve(body, body_len, nseg, sm, gg, ee, vis);
        group_unstage(sm, gg, nseg, paths, exits, entries);
        if (lane == 0) {
            g_exit[gg] = x;
            g_vis[gg] = vis;
        }
        __syncwarp();
    }
    // Fused: what this group tells the next round goes straight into the other claim buffer (the claims this
    // round read are in g_claim, which every group has just reset for the round after next): one kernel per
    // round instead of two.
    if (g < ngroup) {
        __syncwarp(); // (lane 0's g_exit of a re-resolved group is visible to the lane that owns the group)
        scatter_group(body, body_len, ngroup, g, *reinterpret_cast<volatile uint32_t *>(g_entry + g),
                      *reinterpret_cast<volatile uint64_t *>(g_exit + g), claim_out);
    }
}

// Last pass over the tags.  Every live group chases once more from its true entry, which gives
// the entry of each of its segments; every live segment is then walked from that entry (C): the
// output bytes of the elements that start in it are summed, and the (speculative) path map is
// replaced by the exact map of element starts -- what the segment-driven decoder consumes.
__global__ void __launch_bounds__(256) k_group_final(const uint8_t *__restrict__ body, uint64_t body_len, uint64_t nseg,
                                                     uint64_t ngroup, uint4 *__restrict__ paths,
                                                     const uint32_t *__restrict__ g_entry,
                                                     const uint8_t *__restrict__ entries, uint64_t *__restrict__ outlen,
                                                     uint32_t *__restrict__ status, int open_end)
{
    // One thread per segment.  The entry of the segment comes from the last resolution of its group (stored
    // by group_unstage): the group's final entry always lies on that chain (a group is re-resolved whenever
    // its entry leaves the chain), so the stored entries hold from the final entry's segment onwards;
    // segments before it belonged to a speculative prefix and hold nothing.
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= nseg)
        return;
    const uint64_t g = t / kGroup;
    const uint32_t ge = g_entry[g];
    const uint32_t k = (uint32_t)(t - g * kGroup);
    uint32_t en = kDead;
    if (!(ge & kGDead)) {
        const uint32_t k0 = ge / kSeg;
        if (k == k0)
            en = ge - k0 * kSeg;
        else if (k > k0)
            en = entries[t];
    }
    uint64_t sum = 0;
    Path p;
    p.clear();
    if (!(en & kDead)) {
        const uint64_t lo = t * kSeg, hi = min(lo + kSeg, body_len);
        uint64_t e = lo + en;
        while (e < hi) {
            const Elem el = decode_at<true>(body, body_len, e);
            if (!el.ok || e + el.size > body_len) {
                // the element runs past the bytes we have: an error for a whole stream, the
                // normal end of a partial one (open_end: the rest has not been uploaded yet)
                if (!open_end)
                    atomicOr(status, SNAPPY_B200_ST_CORRUPT);
                break;
            }
            if (el.out > kBlock)
                atomicOr(status, SNAPPY_B200_ST_FRAMING);
            p.set((uint32_t)(e - lo));
            sum += el.out;
            e += el.size;
        }
    }
    outlen[t] = sum;
    paths[t] = make_uint4(p.bits[0], p.bits[1], p.bits[2], p.bits[3]);
}

// Exclusive scan of a u64 array (one entry per 128 stream bytes, so millions of entries): tile
// sums, a one-CTA scan of the tile sums, then a per-tile scan seeded with its tile offset.
constexpr int kScanTile = 4096;   // elements per CTA
constexpr int kScanCta = 512;     // threads per CTA, 8 elements each

__device__ __forceinline__ uint64_t cta_exclusive_scan_u64(uint64_t v, uint64_t *warp_sum, uint64_t &total)
{
    const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    uint64_t incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint64_t s = __shfl_up_sync(kFull, incl, d);
        if ((int)lane >= d)
            incl += s;
    }
    if (lane == 31)
        warp_sum[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        const uint32_t nw = blockDim.x >> 5;
        const uint64_t w = lane < nw ? warp_sum[lane] : 0;
        uint64_t wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint64_t s = __shfl_up_sync(kFull, wi, d);
            if ((int)lane >= d)
                wi += s;
        }
        if (lane < nw)
            warp_sum[lane] = wi - w;
        if (lane == 31)
            warp_sum[32] = wi;
    }
    __syncthreads();
    total = warp_sum[32];
    const uint64_t r = warp_sum[wid] + (incl - v);
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(kScanCta) k_scan_tile_sums(const uint64_t *__restrict__ in, uint64_t n,
                                                             uint64_t *__restrict__ tile_sums)
{
    __shared__ uint64_t warp_sum[33];
    const uint64_t i0 = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * 8;
    uint64_t sum = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k)
        sum += i0 + k < n ? in[i0 + k] : 0;
    uint64_t total;
    (void)cta_exclusive_scan_u64(sum, warp_sum, total);
    if (threadIdx.x == 0)
        tile_sums[blockIdx.x] = total;
}

// One CTA: exclusive scan of the tile sums in place (loops when there are more than 4096).
__global__ void __launch_bounds__(kScanCta) k_scan_tiles(uint64_t *__restrict__ tile_sums, uint64_t n_tiles,
                                                         uint64_t *__restrict__ total_out)
{
    __shared__ uint64_t warp_sum[33];
    uint64_t carry = 0;
    for (uint64_t start = 0; start < n_tiles; start += kScanTile) {
        const uint64_t i0 = start + (uint64_t)threadIdx.x * 8;
        uint64_t v[8], sum = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            v[k] = i0 + k < n_tiles ? tile_sums[i0 + k] : 0;
            sum += v[k];
        }
        uint64_t total;
        uint64_t run = carry + cta_exclusive_scan_u64(sum, warp_sum, total);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (i0 + k < n_tiles)
                tile_sums[i0 + k] = run;
            run += v[k];
        }
        carry += total;
    }
    if (threadIdx.x == 0)
        *total_out = carry;
}

__global__ void __launch_bounds__(kScanCta) k_scan_apply(const uint64_t *__restrict__ in, uint64_t n,
                                                         const uint64_t *__restrict__ tile_offsets,
                                                         uint64_t *__restrict__ out)
{
    __shared__ uint64_t warp_sum[33];
    const uint64_t i0 = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * 8;
    uint64_t v[8], sum = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        v[k] = i0 + k < n ? in[i0 + k] : 0;
        sum += v[k];
    }
    uint64_t total;
    uint64_t run = tile_offsets[blockIdx.x] + cta_exclusive_scan_u64(sum, warp_sum, total);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (i0 + k < n)
            out[i0 + k] = run;
        run += v[k];
    }
}

// D: stream offset of the element that opens each 64 KiB output block: one thread per block.  The
// segment is found by binary search over the output offsets (the last segment whose first
// element starts at or before the block boundary), the element by walking that segment's
// starts.  A boundary that falls inside an element (legal raw Snappy, never produced by this
// framing) is reported as SNAPPY_B200_ST_FRAMING.
__global__ void __launch_bounds__(256) k_index_blocks(const uint8_t *__restrict__ body, uint64_t body_len, uint64_t nseg,
                                                      const uint4 *__restrict__ starts,
                                                      const uint64_t *__restrict__ outoff,
                                                      const uint64_t *__restrict__ total, uint64_t body_offset,
                                                      uint64_t n_blocks, uint64_t *__restrict__ block_offsets,
                                                      uint32_t *__restrict__ status, int open_end)
{
    const uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (b >= n_blocks)
        return;
    const uint64_t target = b * (uint64_t)kBlock;
    if (target > *total || (target == *total && !open_end))
        return; // beyond what the stream produces (k_index_finish reports a wrong total)
    // last segment t with outoff[t] <= target
    uint64_t lo = 0, hi = nseg; // invariant: outoff[lo] <= target (outoff[0] == 0), answer in [lo, hi)
    while (hi - lo > 1) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (outoff[mid] <= target)
            lo = mid;
        else
            hi = mid;
    }
    const uint64_t t = lo;
    const uint4 sv = starts[t];
    const uint32_t R[4] = {sv.x, sv.y, sv.z, sv.w};
    uint64_t op = outoff[t];
    const uint64_t seg_lo = t * kSeg;
    bool found = false;
    for (uint32_t w = 0; w < 4 && !found && op <= target; ++w) {
        uint32_t bits = R[w];
        while (bits) {
            const uint32_t bit = (uint32_t)__ffs((int)bits) - 1;
            bits &= bits - 1;
            const uint64_t e = seg_lo + 32 * w + bit;
            if (op == target) {
                block_offsets[b] = body_offset + e;
                found = true;
                break;
            }
            if (op > target)
                break;
            op += decode_at(body, body_len, e).out;
        }
    }
    if (found)
        return;
    if (op == target && open_end) {
        // open-ended region: the element that opens the block is the one cut off by the end of
        // the bytes we have.  The chain reaches its start (right after the last complete element
        // of the segment), but an incomplete element has no bit in the map.
        for (int w = 3; w >= 0; --w)
            if (R[w]) {
                const uint64_t e = seg_lo + 32 * w + (31 - __clz((int)R[w]));
                const uint64_t e_end = e + decode_at(body, body_len, e).size;
                if (e_end < body_len)
                    block_offsets[b] = body_offset + e_end;
                break;
            }
        return; // (if it is not known yet the host pipeline does not use this entry)
    }
    atomicOr(status, SNAPPY_B200_ST_FRAMING);
}

__global__ void k_index_finish(const uint64_t *__restrict__ total, uint64_t total_out, uint64_t stream_bytes,
                               uint64_t n_blocks, uint64_t *__restrict__ block_offsets, uint32_t *__restrict__ status,
                               int open_end, const uint32_t *__restrict__ last_changed)
{
    // the last relaxation round that was run still moved a group: the chain is not resolved, nothing
    // built on it may be trusted (the decode kernels return at once on a non-zero status)
    if (threadIdx.x == 0 && blockIdx.x == 0 && last_changed && *last_changed != 0)
        atomicOr(status, SNAPPY_B200_ST_UNRESOLVED);
    if (threadIdx.x == 0 && blockIdx.x == 0 && !open_end) {
        block_offsets[n_blocks] = stream_bytes;
        if (*total != total_out)
            atomicOr(status, SNAPPY_B200_ST_CORRUPT);
    }
}

__global__ void __launch_bounds__(256) k_fill_u64(unsigned long long *p, uint64_t n, unsigned long long v)
{
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < n)
        p[i] = v;
}

// ------------------------------------------------------------------------------- host side
struct IndexWorkspace {
    uint4 *paths;
    uint64_t *exits;
    unsigned long long *claim;
    uint64_t *outlen;
    uint64_t *outoff;
    uint64_t *total;
    uint64_t *tile_sums;
    uint32_t *changed;
    uint8_t *entry;
    uint32_t *g_entry;
    uint64_t *g_exit;
    uint64_t *g_vis;
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

size_t index_workspace_bytes(uint64_t stream_bytes)
{
    const uint64_t nseg = (stream_bytes + kSeg - 1) / kSeg + 1;
    const uint64_t ntile = (nseg + kScanTile - 1) / kScanTile + 1;
    const uint64_t ngroup = (nseg + kGroup - 1) / kGroup + 1;
    return align_up(nseg * 16, 256) + 3 * align_up(nseg * 8, 256) + align_up(std::max<uint64_t>(nseg, 128) * 8, 256) +
           align_up(ntile * 8, 256) + 256 + 256 +
           align_up(nseg, 256) + align_up(ngroup * 4, 256) + 2 * align_up(ngroup * 8, 256) + 256;
}

static IndexWorkspace carve(void *ws, uint64_t stream_bytes)
{
    const uint64_t nseg = (stream_bytes + kSeg - 1) / kSeg + 1;
    uint8_t *p = static_cast<uint8_t *>(ws);
    IndexWorkspace w;
    w.paths = reinterpret_cast<uint4 *>(p), p += align_up(nseg * 16, 256);
    w.exits = reinterpret_cast<uint64_t *>(p), p += align_up(nseg * 8, 256);
    // (two claim buffers of one entry per GROUP live here: at least 128 entries, see run_index)
    w.claim = reinterpret_cast<unsigned long long *>(p), p += align_up(std::max<uint64_t>(nseg, 128) * 8, 256);
    w.outlen = reinterpret_cast<uint64_t *>(p), p += align_up(nseg * 8, 256);
    w.outoff = reinterpret_cast<uint64_t *>(p), p += align_up(nseg * 8, 256);
    w.total = reinterpret_cast<uint64_t *>(p), p += 256;
    w.tile_sums = reinterpret_cast<uint64_t *>(p), p += align_up(((nseg + kScanTile - 1) / kScanTile + 1) * 8, 256);
    w.changed = reinterpret_cast<uint32_t *>(p), p += 256; // 64 round flags
    w.entry = p, p += align_up(nseg, 256);
    const uint64_t ngroup = (nseg + kGroup - 1) / kGroup + 1;
    w.g_entry = reinterpret_cast<uint32_t *>(p), p += align_up(ngroup * 4, 256);
    w.g_exit = reinterpret_cast<uint64_t *>(p), p += align_up(ngroup * 8, 256);
    w.g_vis = reinterpret_cast<uint64_t *>(p);
    return w;
}

// The exact element-start maps k_group_final leaves behind (one uint4 per 128-byte segment).
const uint4 *index_starts(void *d_ws, uint64_t stream_bytes) { return carve(d_ws, stream_bytes).paths; }
// Output offset of the first element that starts in each segment (exclusive scan of the segment output lengths).
const uint64_t *index_outoff(void *d_ws, uint64_t stream_bytes) { return carve(d_ws, stream_bytes).outoff; }

static std::atomic<uint64_t> g_last_rounds{0}; // diagnostic only (last call on any thread)
uint64_t index_last_rounds() { return g_last_rounds; }

// Synchronises the stream between relaxation rounds (it has to read the "changed" flag).
// The total output length the last run_index counted (device scalar in the workspace).
const uint64_t *index_total(void *d_ws, uint64_t stream_bytes) { return carve(d_ws, stream_bytes).total; }

// open_end: the bytes are the beginning of a longer stream (the host pipeline decodes while the
// rest is still being uploaded).  The element cut off by the end is not an error then, the
// total is not checked, and at most n_blocks_cap block starts are recorded.
//
// The relaxation rounds end on the device: every round reads the "changed" flag of the round before and
// returns at once when it is clear, so a batch of rounds can be enqueued blind.
//   fixed_rounds == 0  adaptive: batches of 16, 48, 64, ... rounds, the flags read back after each batch
//                      (synchronises the stream), until a round changes nothing.  A chain over ngroup groups is
//                      resolved after at most ngroup rounds and one more shows that nothing moves, so every
//                      valid stream converges within max_rounds = ngroup + 2 + one batch; an adversarial one
//                      (tests/k0gen.py: every speculative walk misses the chain) needs about ngroup rounds, which
//                      costs time linear in the stream, the order of the sequential walk of the general decoder.
//                      ST_UNRESOLVED from this mode can only mean a bug in K0.
//   fixed_rounds  > 0  asynchronous: exactly one batch of min(fixed_rounds, 64) rounds, no read-back, no
//                      synchronisation (graph-capturable); ST_UNRESOLVED if its last round still moved.
constexpr uint32_t kMaxBatch = 64;

cudaError_t run_index(const uint8_t *d_stream, uint64_t stream_bytes, uint64_t body_offset, uint64_t total_out,
                      uint64_t *d_block_offsets, uint32_t *d_status, void *d_ws, cudaStream_t st, uint64_t *launches,
                      bool open_end, uint64_t n_blocks_cap, uint32_t fixed_rounds)
{
    const uint64_t n_blocks = open_end ? n_blocks_cap : (total_out + kBlock - 1) / kBlock;
    const uint64_t body_len = stream_bytes - body_offset;
    const uint8_t *body = d_stream + body_offset;
    const uint64_t nseg = (body_len + kSeg - 1) / kSeg;
    IndexWorkspace w = carve(d_ws, stream_bytes);
    cudaError_t e;
    if (nseg == 0) {
        if ((e = cudaMemsetAsync(w.total, 0, 8, st)) != cudaSuccess)
            return e;
        k_index_finish<<<1, 32, 0, st>>>(w.total, total_out, stream_bytes, n_blocks, d_block_offsets, d_status,
                                         open_end, nullptr);
        *launches += 1;
        return cudaGetLastError();
    }
    const unsigned grid = (unsigned)((nseg + 255) / 256);
    const uint64_t ngroup = (nseg + kGroup - 1) / kGroup;
    const unsigned ggrid = (unsigned)((ngroup + 127) / 128);                       // one thread per group
    const unsigned wgrid = (unsigned)((ngroup + kGroupCta / 32 - 1) / (kGroupCta / 32)); // one warp per group
    const unsigned wgrid32 = (unsigned)((ngroup + kGroupCta - 1) / kGroupCta);           // one lane per group
    k_index_spec<<<grid, 256, 0, st>>>(body, body_len, nseg, w.paths, w.exits);
    k_group_init<<<wgrid, kGroupCta, 0, st>>>(body, body_len, nseg, ngroup, w.paths, w.exits, w.g_entry, w.g_exit, w.g_vis,
                                        w.claim, w.entry,
                                        // mostly incompressible (stream >= 80 % of the output): chains of maximal literals
                                        !open_end && stream_bytes / 4 >= total_out / 5);
    *launches += 2;
    const uint64_t max_rounds = ngroup + 2 + kMaxBatch;
    const uint32_t *unresolved = nullptr; // flag of the last round run, when nothing proves convergence
    uint32_t batch = fixed_rounds ? std::min<uint32_t>(fixed_rounds, kMaxBatch) : 16;
    // a chain over ngroup groups is resolved after at most ngroup rounds (one more shows that nothing moves):
    // small streams do not pay for a full batch of launches
    batch = (uint32_t)std::min<uint64_t>(batch, ngroup + 1);
    // Two claim buffers: round 0 is scatter + k_group_apply (one warp per group: the first round moves most
    // groups) + scatter of the claims of round 1; from round 1 on one fused kernel per round applies the claims of
    // one buffer and scatters those of the next round into the other.
    unsigned long long *claim[2] = {w.claim, w.claim + align_up(ngroup + 1, 32)};
    if ((e = cudaMemsetAsync(claim[1], 0xff, (ngroup + 1) * 8, st)) != cudaSuccess) // kNone
        return e;
    int cur = 0; // buffer that holds the claims of the next round to apply (from round 1 on)
    for (uint64_t round = 0;;) {
        if ((e = cudaMemsetAsync(w.changed, 0, 4 * kMaxBatch, st)) != cudaSuccess)
            return e;
        for (uint32_t k = 0; k < batch; ++k) {
            const uint32_t *prev = k ? w.changed + k - 1 : nullptr;
            if (round + k == 0) {
                k_group_scatter<<<ggrid, 128, 0, st>>>(body, body_len, ngroup, w.g_entry, w.g_exit, claim[0]);
                k_group_apply<<<wgrid, kGroupCta, 0, st>>>(body, body_len, nseg, ngroup, w.paths, w.exits, w.g_entry,
                                                           w.g_exit, w.g_vis, claim[0], w.changed + k, w.entry);
                k_group_scatter<<<ggrid, 128, 0, st>>>(body, body_len, ngroup, w.g_entry, w.g_exit, claim[0]);
                *launches += 3;
            } else {
                k_group_apply32<<<wgrid32, kGroupCta, 0, st>>>(body, body_len, nseg, ngroup, w.paths, w.exits,
                                                               w.g_entry, w.g_exit, w.g_vis, claim[cur], w.changed + k,
                                                               prev, w.entry, claim[cur ^ 1]);
                cur ^= 1;
                *launches += 1;
            }
        }
        if (fixed_rounds) {
            unresolved = w.changed + batch - 1;
            break;
        }
        uint32_t *changed = thread_pinned_scratch(); // >= kMaxBatch words
        if (!changed)
            return cudaErrorMemoryAllocation;
        if ((e = peek_u32(changed, w.changed, batch, st)) != cudaSuccess || (e = cudaStreamSynchronize(st)) != cudaSuccess)
            return e;
        g_last_rounds = round + batch;
        bool converged = false;
        for (uint32_t k = 0; k < batch; ++k)
            if (!changed[k]) { // a round without change is the fixed point
                g_last_rounds = round + k + 1;
                converged = true;
                break;
            }
        if (converged)
            break;
        round += batch;
        if (round >= max_rounds) {
            unresolved = w.changed + batch - 1; // (still set: the finish kernel raises ST_UNRESOLVED)
            break;
        }
        batch = std::min<uint32_t>(batch * 3, kMaxBatch);
    }
    k_group_final<<<grid, 256, 0, st>>>(body, body_len, nseg, ngroup, w.paths, w.g_entry, w.entry, w.outlen, d_status,
                                        open_end);
    const uint64_t ntile = (nseg + kScanTile - 1) / kScanTile;
    k_scan_tile_sums<<<(unsigned)ntile, kScanCta, 0, st>>>(w.outlen, nseg, w.tile_sums);
    k_scan_tiles<<<1, kScanCta, 0, st>>>(w.tile_sums, ntile, w.total);
    k_scan_apply<<<(unsigned)ntile, kScanCta, 0, st>>>(w.outlen, nseg, w.tile_sums, w.outoff);
    if (n_blocks)
        k_index_blocks<<<(unsigned)((n_blocks + 255) / 256), 256, 0, st>>>(body, body_len, nseg, w.paths, w.outoff,
                                                                          w.total, body_offset, n_blocks,
                                                                          d_block_offsets, d_status, open_end);
    k_index_finish<<<1, 32, 0, st>>>(w.total, total_out, stream_bytes, n_blocks, d_block_offsets, d_status, open_end,
                                     unresolved);
    *launches += 6;
    return cudaGetLastError();
}

} // namespace sb200
