/* parallel_parse.h -- the constants that define the parse of SNAPPY_B200_MODE_PARALLEL.
 *
 * Shared, as the one definition, by the kernels (csrc/compress_parallel.cu) and the CPU model the tests
 * hold them to byte for byte (tests/parallel_parse.c).  Plain C: the model is compiled by gcc.
 *
 * For one 64 KiB block b[0..n), with key(p) = the little-endian 32 bits at p (p + 4 <= n) and
 * h(p) = (key(p) * 0x1e35a7bd) >> (32 - SB200_PAR_TABLE_LOG):
 *   1. Candidates, in steps of SB200_PAR_STEP positions.  Position p of a step has two candidates:
 *      the table entry T[h(p)] as it was when the step began (the latest earlier step's position with that
 *      hash), and the latest q < p of the same aligned SB200_PAR_GROUP positions with h(q) == h(p).
 *      After the candidates are read, every position of the step goes into T (the larger position wins).
 *      A candidate counts only if its key equals key(p).  When both count, the one whose match goes on
 *      for more of the next 4 * SB200_PAR_CMP_WORDS bytes (inside the block) wins; a tie goes to the
 *      in-group one, which is nearer.  The result is an offset per position (0 = none).
 *      Steps in which no position has a candidate make later steps be skipped, so that incompressible data is
 *      passed over (as the reference's parse skips ahead after misses): when a step is about to be looked
 *      up, the previous looked-up step is counted -- a step with a candidate resets m, the m-th step in a row
 *      without one makes the min(2^(m-1), SB200_PAR_SKIP_MAX) steps after the one about to be looked up be
 *      skipped.  A skipped step is neither looked up nor entered into T and has no candidates.
 *   2. Walk: the block is cut into slices of SB200_PAR_SLICE bytes, each parsed greedily on its own:
 *      at p, with p + 4 <= slice end and a candidate c, emit a copy from c that is extended byte by byte
 *      up to the slice end and continue after it; otherwise p + 1.  Literal runs are what lies between the
 *      copies, across slice boundaries, so a block with no copy is one literal.
 *   3. A block whose copies cover fewer than SB200_PAR_MIN_COVER bytes in all is one literal as well: random
 *      data holds a few chance 4-byte matches per block, which save nothing worth having and would keep the
 *      decoder's boundary search from taking the block as one maximal literal.
 */
#ifndef SB200_PARALLEL_PARSE_H
#define SB200_PARALLEL_PARSE_H

#define SB200_PAR_TABLE_LOG 14 /* 2^14 table slots */
#define SB200_PAR_STEP 1024    /* positions per table snapshot (= threads of the candidate kernel) */
#define SB200_PAR_GROUP 32     /* aligned positions searched for an in-group predecessor (= one warp) */
#define SB200_PAR_SLICE 2048   /* bytes parsed independently (= 65536 / 32: one lane per slice) */
#define SB200_PAR_CMP_WORDS 1  /* words compared after the key to choose between two candidates */
#define SB200_PAR_MIN_COVER 64 /* fewer bytes covered by copies: the block is one literal */
#define SB200_PAR_SKIP_MAX 8   /* most steps skipped after a step without a candidate */

#endif
