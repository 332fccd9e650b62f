/* cli.c -- `snappy [-c|-b|-d] [-r] infile outfile`, the reference's command line
 * (src/cmd.c:19-28, :56-105) in front of libsnappy_b200.so.  Same options and defaults;
 * -r reports wall-clock time and throughput on the UNCOMPRESSED size for both directions
 * (the reference used CPU time and the compressed size, SURVEY.md Q9).                   */
#define _POSIX_C_SOURCE 200809L
#include <errno.h>
#include <getopt.h>
#include <stdio.h>
#include <unistd.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "snappy_b200.h"
#include "snappy_compression.h"
#include "snappy_compression_tree.h"
#include "snappy_decompression.h"

static void usage(void)
{
    fprintf(stderr, "snappy [-c|-d|-b] [-r] [-i|-f] [infile] [outfile]\n"
                    "-c compress (hash table)\n"
                    "-b compress (exact-key / BST match finder)\n"
                    "-d decompress\n"
                    "-r print sizes, ratio, time and throughput\n"
                    "-i side index: compress also writes <outfile>.idx (block offsets; the stream is\n"
                    "   unchanged), decompress reads <infile>.idx and skips the boundary search\n"
                    "-f the Snappy framing format (.sz: stream identifier, CRC-32C-checked chunks) instead of\n"
                    "   the reference's stream; the input of -d may be a pipe\n");
    exit(EXIT_FAILURE);
}

static unsigned long long file_size(FILE *f)
{
    fseek(f, 0, SEEK_END);
    unsigned long long s = (unsigned long long)ftell(f);
    fseek(f, 0, SEEK_SET);
    return s;
}

static double now(void)
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec + 1e-9 * ts.tv_nsec;
}

int main(int argc, char *argv[])
{
    enum { COMPRESS, COMPRESS_BST, UNCOMPRESS } mode = COMPRESS;
    int report = 0, use_index = 0, framed = 0, opt;
    if (argc < 4)
        usage();
    while ((opt = getopt(argc, argv, "cbdrif")) != -1) {
        switch (opt) {
        case 'c': mode = COMPRESS; break;
        case 'b': mode = COMPRESS_BST; break;
        case 'd': mode = UNCOMPRESS; break;
        case 'r': report = 1; break;
        case 'i': use_index = 1; break;
        case 'f': framed = 1; break;
        default: usage();
        }
    }
    if (framed && use_index) {
        fprintf(stderr, "-f and -i cannot be combined: the chunk headers of a framed stream are its index\n");
        usage();
    }
    const char *in_name = argv[argc - 2], *out_name = argv[argc - 1];
    FILE *in = fopen(in_name, "rb");
    if (!in) {
        fprintf(stderr, "cannot open %s: %s\n", in_name, strerror(errno));
        return EXIT_FAILURE;
    }
    FILE *out = fopen(out_name, "wb");
    if (!out) {
        fprintf(stderr, "cannot open %s: %s\n", out_name, strerror(errno));
        fclose(in);
        return EXIT_FAILURE;
    }
    const unsigned long long in_size = framed && mode == UNCOMPRESS ? 0 : file_size(in); /* (-f -d: may be a pipe) */
    int rc = 0;
    FILE *idx = NULL;
    if (use_index) {
        char idx_name[4096];
        snprintf(idx_name, sizeof idx_name, "%s.idx", mode == UNCOMPRESS ? in_name : out_name);
        idx = fopen(idx_name, mode == UNCOMPRESS ? "rb" : "wb");
        if (!idx) {
            fprintf(stderr, "cannot open %s: %s\n", idx_name, strerror(errno));
            fclose(in);
            fclose(out);
            return EXIT_FAILURE;
        }
    }
    const double t0 = now();
    if (framed && mode == UNCOMPRESS)
        rc = snappy_b200_frame_decompress_file(in, out);
    else if (framed)
        rc = snappy_b200_frame_compress_file(in, out, mode == COMPRESS ? SNAPPY_B200_MODE_HASH : SNAPPY_B200_MODE_BST);
    else if (idx && mode == UNCOMPRESS)
        rc = snappy_b200_decompress_file_indexed(in, idx, out);
    else if (idx)
        rc = snappy_b200_compress_file_indexed(in, in_size, mode == COMPRESS ? SNAPPY_B200_MODE_HASH : SNAPPY_B200_MODE_BST,
                                               out, idx);
    else if (mode == COMPRESS)
        snappy_compress(in, in_size, out);
    else if (mode == COMPRESS_BST)
        rc = snappy_compress_bst(in, in_size, out);
    else
        rc = snappy_decompress(in, out);
    const double dt = now() - t0;
    if (idx)
        fclose(idx);
    fclose(in);
    fflush(out);
    const unsigned long long out_size = (unsigned long long)ftell(out);
    fclose(out);
    if (rc != 0 || snappy_b200_last_error()[0]) {
        fprintf(stderr, "snappy: failed: %s\n", snappy_b200_last_error());
        return EXIT_FAILURE;
    }
    if (report) {
        const unsigned long long unc = mode == UNCOMPRESS ? out_size : in_size;
        const unsigned long long cmp = mode == UNCOMPRESS ? in_size : out_size;
        printf("uncompressed = %llu bytes\ncompressed   = %llu bytes\nratio        = %.3f\n", unc, cmp,
               cmp ? (double)unc / (double)cmp : 0.0);
        printf("time         = %.6f s (wall)\nthroughput   = %.1f MB/s (uncompressed)\n", dt, dt > 0 ? unc / dt / 1e6 : 0.0);
    }
    /* Everything is written and closed.  Leave without tearing the CUDA context down piece by piece
     * (unlocking the page-locked rings and freeing GiB of device memory takes about a second and helps nobody). */
    fflush(stdout);
    fflush(stderr);
    _exit(EXIT_SUCCESS);
}
