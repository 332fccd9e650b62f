/* parallel_parse.c -- CPU model of SNAPPY_B200_MODE_PARALLEL: the definition the kernels of
 * csrc/compress_parallel.cu are held to, byte for byte (tests/test_parallel_compress.py).
 *
 * The parse is described in csrc/parallel_parse.h, whose constants both sides include.  The element
 * encodings are the reference's (src/snappy_compression.c:95-165), as k_emit writes them.
 *
 *   uint64_t oracle_compress_parallel(const uint8_t *in, uint64_t n, uint8_t *out, uint32_t *block_sizes)
 *     writes varint(n) and the blocks to out (capacity: 10 + n + 1010 per block) and, when block_sizes is
 *     not NULL, the compressed size of every block; returns the stream length (0 for n == 0).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "parallel_parse.h"

#define BLOCK 65536u

static uint32_t ld32(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }
static uint32_t hash_of(uint32_t key) { return (key * 0x1e35a7bdu) >> (32 - SB200_PAR_TABLE_LOG); }

static uint8_t *put_literal(uint8_t *o, const uint8_t *src, uint32_t len)
{
    const uint32_t m = len - 1;
    if (m < 60) {
        *o++ = (uint8_t)(m << 2);
    } else if (m < 256) {
        *o++ = 60u << 2;
        *o++ = (uint8_t)m;
    } else {
        *o++ = 61u << 2;
        *o++ = (uint8_t)m;
        *o++ = (uint8_t)(m >> 8);
    }
    memcpy(o, src, len);
    return o + len;
}

static uint8_t *put_one_copy(uint8_t *o, uint32_t len, uint32_t off)
{
    if (len < 12 && off < 2048) {
        *o++ = (uint8_t)(((off >> 8) << 5) + ((len - 4) << 2) + 1);
        *o++ = (uint8_t)off;
    } else {
        *o++ = (uint8_t)(((len - 1) << 2) | 2);
        *o++ = (uint8_t)off;
        *o++ = (uint8_t)(off >> 8);
    }
    return o;
}

static uint8_t *put_copy(uint8_t *o, uint32_t len, uint32_t off)
{
    while (len > 68) {
        o = put_one_copy(o, 64, off);
        len -= 64;
    }
    if (len > 64) {
        o = put_one_copy(o, 60, off);
        len -= 60;
    }
    return put_one_copy(o, len, off);
}

/* equal bytes of b[c + 4 ..] and b[p + 4 ..], at most 4 * SB200_PAR_CMP_WORDS and not past n */
static uint32_t head_match(const uint8_t *b, uint32_t n, uint32_t p, uint32_t c)
{
    uint32_t k = 0;
    while (k < 4u * SB200_PAR_CMP_WORDS && p + 4 + k < n && b[c + 4 + k] == b[p + 4 + k])
        ++k;
    return k;
}

/* step 1: offset of the chosen candidate of every position (0 = none); T: the table, position + 1 (0 = empty) */
static void candidates(const uint8_t *b, uint32_t n, uint16_t *off, uint32_t *T)
{
    memset(T, 0, sizeof(uint32_t) << SB200_PAR_TABLE_LOG);
    const uint32_t np = n >= 4 ? n - 3 : 0;
    uint32_t misses = 0, skip = 0; /* steps in a row without a candidate; steps still to skip */
    int64_t pending = -1;          /* candidates of the last step looked up, not counted yet */
    for (uint32_t g0 = 0; g0 < np; g0 += SB200_PAR_STEP) {
        const uint32_t g1 = g0 + SB200_PAR_STEP < np ? g0 + SB200_PAR_STEP : np;
        if (skip) {
            --skip;
            for (uint32_t p = g0; p < g1; ++p)
                off[p] = 0;
            continue;
        }
        if (pending == 0) {
            ++misses;
            skip = misses - 1 < 31 && (1u << (misses - 1)) < SB200_PAR_SKIP_MAX ? 1u << (misses - 1) : SB200_PAR_SKIP_MAX;
        } else if (pending > 0) {
            misses = 0;
        }
        uint32_t hits = 0;
        for (uint32_t p = g0; p < g1; ++p) {
            const uint32_t key = ld32(b + p), h = hash_of(key);
            int64_t c1 = (int64_t)T[h] - 1, c2 = -1;
            for (int64_t q = (int64_t)p - 1; q >= (int64_t)(p & ~(uint32_t)(SB200_PAR_GROUP - 1)); --q)
                if (hash_of(ld32(b + q)) == h) {
                    c2 = q;
                    break;
                }
            const int v1 = c1 >= 0 && ld32(b + c1) == key, v2 = c2 >= 0 && ld32(b + c2) == key;
            int64_t c = -1;
            if (v1 && v2)
                c = head_match(b, n, p, (uint32_t)c2) >= head_match(b, n, p, (uint32_t)c1) ? c2 : c1;
            else if (v1)
                c = c1;
            else if (v2)
                c = c2;
            off[p] = c >= 0 ? (uint16_t)(p - c) : 0;
            hits += c >= 0;
        }
        for (uint32_t p = g0; p < g1; ++p) {
            const uint32_t h = hash_of(ld32(b + p));
            if (p + 1 > T[h])
                T[h] = p + 1;
        }
        pending = hits;
    }
}

/* step 2: the walk; writes the elements when out is not NULL, returns the bytes the copies cover */
static uint32_t walk(const uint8_t *b, uint32_t n, const uint16_t *off, uint8_t **out)
{
    uint8_t *o = out ? *out : NULL;
    uint32_t lit = 0; /* start of the pending literal run */
    uint32_t covered = 0;
    for (uint32_t s0 = 0; s0 < n; s0 += SB200_PAR_SLICE) {
        const uint32_t s1 = s0 + SB200_PAR_SLICE < n ? s0 + SB200_PAR_SLICE : n;
        uint32_t p = s0;
        while (p + 4 <= s1) {
            if (!off[p]) {
                ++p;
                continue;
            }
            const uint32_t c = p - off[p];
            uint32_t len = 4;
            while (p + len < s1 && b[c + len] == b[p + len])
                ++len;
            if (o && p > lit)
                o = put_literal(o, b + lit, p - lit);
            if (o)
                o = put_copy(o, len, off[p]);
            covered += len;
            p += len;
            lit = p;
        }
    }
    if (o && n > lit)
        o = put_literal(o, b + lit, n - lit);
    if (out)
        *out = o;
    return covered;
}

/* one block: returns the bytes written */
static uint32_t compress_block(const uint8_t *b, uint32_t n, uint8_t *out, uint16_t *off, uint32_t *T)
{
    candidates(b, n, off, T);
    uint8_t *o = out;
    if (walk(b, n, off, NULL) < SB200_PAR_MIN_COVER) /* step 3 */
        o = put_literal(o, b, n);
    else
        walk(b, n, off, &o);
    return (uint32_t)(o - out);
}

uint64_t oracle_compress_parallel(const uint8_t *in, uint64_t n, uint8_t *out, uint32_t *block_sizes)
{
    if (n == 0)
        return 0;
    uint64_t o = 0;
    for (uint64_t v = n; ; v >>= 7) {
        out[o++] = (uint8_t)((v & 0x7f) | (v >= 0x80 ? 0x80 : 0));
        if (v < 0x80)
            break;
    }
    uint16_t *off = malloc(BLOCK * sizeof(uint16_t));
    uint32_t *T = malloc(sizeof(uint32_t) << SB200_PAR_TABLE_LOG);
    if (!off || !T) {
        free(off);
        free(T);
        return 0;
    }
    for (uint64_t b0 = 0, blk = 0; b0 < n; b0 += BLOCK, ++blk) {
        const uint32_t len = n - b0 < BLOCK ? (uint32_t)(n - b0) : BLOCK;
        const uint32_t sz = compress_block(in + b0, len, out + o, off, T);
        if (block_sizes)
            block_sizes[blk] = sz;
        o += sz;
    }
    free(off);
    free(T);
    return o;
}
