/*
 * snappy_b200.h -- C-ABI of libsnappy_b200.so, the B200-native (sm_100a) Snappy block
 * codec that sits behind the C API of tturturiello/lightweight-snappy.
 *
 * Three layers, all `extern "C"`, plain pointers and sizes:
 *
 *   1. device-level batched API   (this file; DEVICE pointers, asynchronous on a stream)
 *   2. host-buffer API            (this file; HOST pointers, staging + copies inside)
 *   3. the reference's own symbols (snappy_compression.h, snappy_compression_tree.h,
 *      snappy_decompression.h, varint.h, buffer_compression.h in this directory):
 *      same names, signatures and stream format as the reference headers, so cmd.c-style
 *      callers relink unchanged.
 *
 * What each entry point replaces in the reference (paths relative to the reference repo):
 *   snappy_b200_compress_device / _host, MODE_HASH -> the per-block loop of
 *        src/snappy_compression.c:384-403 driven by snappy_compress :414-428
 *   snappy_b200_compress_device / _host, MODE_BST  -> src/snappy_compression_tree.c:269-288
 *        driven by snappy_compress_bst :291-306 (exact-key dictionary of src/BST.c)
 *   snappy_b200_decompress_device[_indexed] / _host -> src/snappy_decompression.c:345-363
 *        (element loop :290-333, literal :193-239, copy :253-280)
 *   snappy_b200_index_device                        -> the block boundaries that the
 *        sequential loop at src/snappy_decompression.c:353-356 discovers implicitly
 *   varint preamble                                 -> src/varint.c:12-20 / :28-58
 *
 * Stream format (identical to the reference): LEB128(total uncompressed bytes) followed
 * by the compressed 64 KiB blocks, concatenated with no framing.  An empty input gives an
 * empty stream (the reference never flushes the varint, SURVEY.md 8c).
 *
 * There is no CPU fallback: every call fails with SNAPPY_B200_ERR_CUDA when no usable
 * sm_100 device / driver is present.
 */
#ifndef SNAPPY_B200_H
#define SNAPPY_B200_H

#include <stddef.h>
#include <stdio.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNAPPY_B200_BLOCK_SIZE 65536u  /* MAX_BLOCK_SIZE, src/snappy_compression.c:9 */
#define SNAPPY_B200_HTABLE_SIZE 4096u  /* MAX_HTABLE_SIZE, src/snappy_compression.c:10 */
#define SNAPPY_B200_SLOT_STRIDE 66560u /* per-block scratch slot: 65536 + 1010 (+pad), :180-190 */

#define SNAPPY_B200_MODE_HASH 0 /* src/snappy_compression.c */
#define SNAPPY_B200_MODE_BST 1  /* src/snappy_compression_tree.c */

#define SNAPPY_B200_OK 0
#define SNAPPY_B200_ERR_CUDA (-1)     /* CUDA runtime / driver error, or no device */
#define SNAPPY_B200_ERR_ARG (-2)      /* bad argument (null, misaligned, too small) */
#define SNAPPY_B200_ERR_CAPACITY (-3) /* output buffer too small */
#define SNAPPY_B200_ERR_CORRUPT (-4)  /* malformed compressed stream */
#define SNAPPY_B200_ERR_FRAMING (-5)  /* valid Snappy, but an element straddles a 64 KiB block */
#define SNAPPY_B200_ERR_IO (-6)       /* FILE* read/write failed (drop-in layer) */
#define SNAPPY_B200_ERR_CHECKSUM (-7) /* framed stream: a chunk's CRC-32C does not match its data */

/* Status word written by the device kernels (bit set; 0 = clean). */
#define SNAPPY_B200_ST_CAPACITY 1u
#define SNAPPY_B200_ST_CORRUPT 2u
#define SNAPPY_B200_ST_FRAMING 4u
#define SNAPPY_B200_ST_UNRESOLVED 8u /* async decode only: the element chain did not resolve within max_rounds */
#define SNAPPY_B200_ST_CHECKSUM 16u  /* framed stream: a chunk's CRC-32C does not match (CORRUPT takes precedence) */

/* Message of the last failing call on this thread (never NULL). */
const char *snappy_b200_last_error(void);
/* Number of CUDA devices visible, or a negative SNAPPY_B200_ERR_CUDA. */
int snappy_b200_device_count(void);
/* How many kernels this library has launched in this process (bench.py's gpu_launches). */
uint64_t snappy_b200_launch_count(void);
/* Relaxation rounds the last snappy_b200_index_device call needed (diagnostic). */
uint64_t snappy_b200_index_rounds(void);

/* Upper bound of the stream for n input bytes: 10 + n + 1010 per block (src :180-190). */
uint64_t snappy_b200_max_compressed_bytes(uint64_t n_bytes);
uint64_t snappy_b200_block_count(uint64_t n_bytes);

/* ---------------------------------------------------------------- 1. device-level API
 * All pointers are device pointers on the current device, 16-byte aligned unless noted.
 * `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls only enqueue
 * work; results (including *d_status) are valid after the stream is synchronised.       */

size_t snappy_b200_compress_workspace_bytes(uint64_t n_bytes, int mode);

/* Compresses n_bytes at d_in into one reference-format stream at d_out.
 *   d_out_bytes      [1]  total stream length (varint + blocks)
 *   d_block_offsets  [n_blocks+1] (optional, may be NULL) stream offset of every block --
 *                    the side index a later indexed decode can reuse; entry n_blocks =
 *                    stream length
 *   d_status         [1]  SNAPPY_B200_ST_* bits (CAPACITY when out_capacity was too small) */
int snappy_b200_compress_device(const uint8_t *d_in, uint64_t n_bytes, int mode, uint8_t *d_out,
                                uint64_t out_capacity, uint64_t *d_out_bytes, uint64_t *d_block_offsets,
                                uint32_t *d_status, void *d_workspace, size_t workspace_bytes, void *stream);

/* Decodes n_blocks blocks whose stream offsets are given (d_block_offsets[n_blocks+1]);
 * block i produces bytes [i*65536, min(total_out, (i+1)*65536)) of d_out.  Valid raw Snappy the block
 * decoder does not take (see snappy_b200_decompress_host_indexed) gives SNAPPY_B200_ST_FRAMING.  *d_status is
 * OR-ed into, not reset: the caller zeroes it, and a non-zero status on entry (e.g. left by
 * a failed snappy_b200_index_device on the same stream) turns the call into a no-op.     */
int snappy_b200_decompress_device_indexed(const uint8_t *d_stream, const uint64_t *d_block_offsets,
                                          uint64_t n_blocks, uint64_t total_out, uint8_t *d_out,
                                          uint32_t *d_status, void *stream);

size_t snappy_b200_index_workspace_bytes(uint64_t stream_bytes);

/* Finds the block boundaries of an index-less stream body (the bytes after the varint):
 * d_block_offsets[n_blocks+1] receives offsets relative to d_stream (which must point at
 * the start of the whole stream; body_offset = length of the varint).                   */
int snappy_b200_index_device(const uint8_t *d_stream, uint64_t stream_bytes, uint64_t body_offset,
                             uint64_t total_out, uint64_t *d_block_offsets, uint32_t *d_status,
                             void *d_workspace, size_t workspace_bytes, void *stream);

/* The segment-driven decoder on its own: requires the workspace exactly as
 * snappy_b200_index_device left it for this stream (it holds the element maps) and the
 * block offsets that call produced.                                                      */
int snappy_b200_decode_segments_device(const uint8_t *d_stream, uint64_t stream_bytes, uint64_t body_offset,
                                       uint64_t total_out, uint8_t *d_out, const uint64_t *d_block_offsets,
                                       uint32_t *d_status, void *d_workspace, size_t workspace_bytes,
                                       void *stream);

/* Decodes an index-less stream: K0 followed by the segment-driven decoder (the decode kernel
 * runs on a library-owned second stream that is joined back into `stream` before the call
 * returns).  d_block_offsets [n_blocks+1] (optional) is filled as a by-product.
 * Workspace: snappy_b200_decompress_workspace_bytes.  Synchronises `stream` between K0
 * rounds; the last decode is only enqueued.  K0 here (and in snappy_b200_index_device, the
 * host-buffer and FILE* calls) runs rounds until the element chain is resolved, which every
 * valid stream is after at most one round per 8 KiB of stream (adversarial input needs about
 * that many; ordinary streams a few dozen): these calls never give SNAPPY_B200_ST_UNRESOLVED,
 * which only snappy_b200_decompress_device_async reports.                                  */
size_t snappy_b200_decompress_workspace_bytes(uint64_t stream_bytes, uint64_t total_out);
int snappy_b200_decompress_device(const uint8_t *d_stream, uint64_t stream_bytes, uint64_t body_offset,
                                  uint64_t total_out, uint8_t *d_out, uint64_t *d_block_offsets,
                                  uint32_t *d_status, void *d_workspace, size_t workspace_bytes, void *stream);

/* The same decode as a purely ASYNCHRONOUS call: K0 runs a fixed batch of max_rounds (<= 64; 0 = 64)
 * relaxation rounds that end themselves on the device as soon as the chain is resolved, then the block
 * decode follows on the same stream.  Nothing is read back, nothing synchronises, no lock is taken and
 * nothing is allocated, so the call may be captured into a CUDA graph and replayed.  If the stream needs
 * more rounds than were enqueued (measured: text 5, low-entropy 4, mixed 10, random 38) *d_status gets
 * SNAPPY_B200_ST_UNRESOLVED and nothing is decoded: use snappy_b200_decompress_device for such input.
 * d_block_offsets (optional) as above.  *d_status is OR-ed into; the caller zeroes it.              */
size_t snappy_b200_decompress_async_workspace_bytes(uint64_t stream_bytes, uint64_t total_out);
int snappy_b200_decompress_device_async(const uint8_t *d_stream, uint64_t stream_bytes, uint64_t body_offset,
                                        uint64_t total_out, uint8_t *d_out, uint64_t *d_block_offsets,
                                        uint32_t *d_status, void *d_workspace, size_t workspace_bytes,
                                        unsigned max_rounds, void *stream);

/* ---------------------------------------------------------------- 2. host-buffer API
 * Synchronous.  Host pointers (pageable or pinned); staging through pinned buffers and
 * the host<->device copies happen inside.                                               */
int snappy_b200_compress_host(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                              uint64_t *out_bytes);
int snappy_b200_uncompressed_length(const void *stream, uint64_t stream_bytes, uint64_t *n_bytes);
int snappy_b200_decompress_host(const void *stream, uint64_t stream_bytes, void *out, uint64_t out_capacity,
                                uint64_t *out_bytes);
/* The same two calls with the optional side index (SURVEY.md 8f-4): block_offsets[b] is the
 * stream offset at which the b-th 64 KiB block starts, block_offsets[snappy_b200_block_count(n)]
 * the stream length.  The stream itself is unchanged (byte-identical to the reference); a decoder
 * that is handed the index does not have to discover the block boundaries (no K0).  The
 * indexed decoder checks the index against the stream and reports SNAPPY_B200_ERR_CORRUPT when
 * they disagree.  Valid raw Snappy that the block decoders do not take -- elements that straddle
 * a block, copies into an earlier block, blocks longer than 2 * 65536 stream bytes (non-minimal
 * encodings) -- is decoded by the general decoder, as snappy_b200_decompress_host does.  A stream
 * may be up to 6 bytes per output byte long (1-byte literals with a 4-byte length) plus the
 * varint; only a longer one is rejected before it is decoded.                              */
int snappy_b200_compress_host_indexed(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                                      uint64_t *out_bytes, uint64_t *block_offsets);
int snappy_b200_decompress_host_indexed(const void *stream, uint64_t stream_bytes, const uint64_t *block_offsets,
                                        uint64_t n_blocks, void *out, uint64_t out_capacity, uint64_t *out_bytes);
/* One range of a longer input, for callers that stream (the FILE* layer does): n_bytes must be whole
 * 64 KiB blocks except for the last range.  varint_value != 0: the range opens the stream, and the preamble
 * carries that value (the length of the WHOLE input: src/snappy_compression.c:417 writes the declared size);
 * varint_value == 0: blocks only.  Concatenating the outputs of consecutive ranges gives exactly the stream
 * of one call over the whole input.  block_offsets (optional) are relative to this range's output.        */
int snappy_b200_compress_host_range(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                                    uint64_t *out_bytes, uint64_t *block_offsets, uint64_t varint_value);
int snappy_b200_compress_host_multi_range(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                                          uint64_t *out_bytes, uint64_t *block_offsets, int n_devices,
                                          uint64_t varint_value);
/* The same calls over the first n_devices GPUs of the box (SURVEY.md 8e): contiguous block ranges per device,
 * one worker thread and one arena per device, no collective and no peer copy -- the only cross-device datum
 * is the compressed size of every partition (an exclusive scan on the host places the partitions).  The
 * stream is byte-identical to the one-device stream.  The index-less decode first runs K0 over the whole
 * stream on the current device.  The plain calls above forward here when SNAPPY_B200_DEVICES=N (N > 1) is set,
 * more than one device is present and the data is at least 64 MiB.  Streams the block decoders do not take go
 * to the general decoder on the current device, as in the one-device calls.                               */
int snappy_b200_compress_host_multi(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                                    uint64_t *out_bytes, uint64_t *block_offsets, int n_devices);
int snappy_b200_decompress_host_multi(const void *stream, uint64_t stream_bytes, void *out, uint64_t out_capacity,
                                      uint64_t *out_bytes, int n_devices);
int snappy_b200_decompress_host_indexed_multi(const void *stream, uint64_t stream_bytes, const uint64_t *block_offsets,
                                              uint64_t n_blocks, void *out, uint64_t out_capacity, uint64_t *out_bytes,
                                              int n_devices);
/* FILE*-level versions for the command line (`snappy -i`): the index is written to / read from its
 * own file next to the unchanged stream -- "SNPIDX1\0", u64 uncompressed bytes, u64 n_blocks,
 * then n_blocks + 1 u64 stream offsets, all little-endian.  Same FILE* ownership rules as the
 * drop-in calls (caller opens and closes).                                                */
int snappy_b200_compress_file_indexed(FILE *in, unsigned long long input_size, int mode, FILE *out, FILE *index_out);
int snappy_b200_decompress_file_indexed(FILE *in, FILE *index_in, FILE *out);
/* FILE* -> FILE* decompression with the stream and the output device-resident and only a ring of three
 * page-locked 32 MiB chunks on the host (fread -> H2D, K0 + decode, D2H -> fwrite).  Returns 1 (nothing read,
 * nothing written) when `in` is not seekable or the data does not fit the device: decode whole buffers then. */
int snappy_b200_decompress_file(FILE *in, FILE *out);
/* ---------------------------------------------------------------- framing format
 * The Snappy framing format of google/snappy framing_format.txt (".sz" files; what golang/snappy, the Rust `snap`
 * crate and python-snappy read and write): the stream identifier ff 06 00 00 "sNaPpY", then chunks of a 1-byte type
 * and a 3-byte little-endian length.  A data chunk carries at most 65536 uncompressed bytes and the masked CRC-32C
 * (Castagnoli; ((c >> 15) | (c << 17)) + 0xa282ead8, little-endian) of them: 0x00 = a raw Snappy buffer
 * varint(n) || elements whose copies stay inside the chunk, 0x01 = the bytes themselves.  0xff repeats the
 * identifier, 0xfe (padding) and 0x80-0xfd are skipped, 0x02-0x7f are an error.  Every CRC is checked on decode.
 *
 * The writer emits the identifier, then one chunk per 64 KiB block of input (the last may be shorter): compressed
 * when the raw payload varint(n_b) + the block's elements is shorter than n_b - n_b / 8, uncompressed otherwise
 * (golang/snappy's rule).  The compressed payload of a block is exactly what snappy_b200_compress_host gives for
 * that block alone, in either mode.  An empty input gives the identifier alone; an empty buffer decodes as an empty
 * stream.  SNAPPY_B200_DEVICES does not apply: the framed calls run on the current device.                        */

/* Upper bound of a framed stream for n input bytes: 10 + n + 8 * ceil(n / 65536). */
uint64_t snappy_b200_frame_max_compressed_bytes(uint64_t n_bytes);
size_t snappy_b200_frame_compress_workspace_bytes(uint64_t n_bytes, int mode);
/* Device-level framed compression: d_in / d_out / d_workspace as for snappy_b200_compress_device (16-byte
 * aligned; the workspace is required, also for n_bytes == 0).  *d_out_bytes receives the stream length, *d_status
 * SNAPPY_B200_ST_* bits (CAPACITY when out_capacity was too small).  Enqueue only: no read-back, no lock, no
 * allocation, so the call may be captured into a CUDA graph.                                                      */
int snappy_b200_frame_compress_device(const uint8_t *d_in, uint64_t n_bytes, int mode, uint8_t *d_out,
                                      uint64_t out_capacity, uint64_t *d_out_bytes, uint32_t *d_status,
                                      void *d_workspace, size_t workspace_bytes, void *stream);
/* Host buffers, synchronous, like snappy_b200_compress_host (128 MiB chunks, uploads and downloads overlapped). */
int snappy_b200_frame_compress_host(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                                    uint64_t *out_bytes);
/* Host only, no device needed: walks the chunk headers and checks every rule above except the compressed payloads
 * and the CRCs; *n_bytes = the total uncompressed length.  SNAPPY_B200_ERR_CORRUPT names the offset of the first
 * bad chunk.                                                                                                     */
int snappy_b200_frame_uncompressed_length(const void *stream, uint64_t stream_bytes, uint64_t *n_bytes);
/* Decodes a framed stream from host memory: the chunk headers are walked on the host, the stream goes up in
 * pieces cut at chunk boundaries, every piece is decoded (one warp per chunk, no K0) and checked (CRC-32C of every
 * chunk) while the next one is in flight.  SNAPPY_B200_ERR_CORRUPT for a malformed stream,
 * SNAPPY_B200_ERR_CHECKSUM when the stream is well formed but a chunk's data does not match its CRC.            */
int snappy_b200_frame_decompress_host(const void *stream, uint64_t stream_bytes, void *out, uint64_t out_capacity,
                                      uint64_t *out_bytes);
/* FILE* -> FILE* (the command line's `-f`; caller opens and closes).  Compression reads the input in chunks of
 * whole blocks through a ring of page-locked buffers (reader thread -> GPU -> writer thread), as the drop-in
 * snappy_compress does; an empty input gives the identifier alone.  Decompression needs no seekable input: it
 * reads 32 MiB windows, decodes the chunks that are complete in each (at most 32 MiB of output at a time) and
 * carries the incomplete tail into the next window, so page-locked and device memory are bounded by the window
 * size, not by the file size.                                                                                    */
int snappy_b200_frame_compress_file(FILE *in, FILE *out, int mode);
int snappy_b200_frame_decompress_file(FILE *in, FILE *out);

/* Releases the cached device/pinned buffers of the host-buffer API. */
void snappy_b200_release(void);
/* Page-locked host memory for the buffers handed to the host-buffer API (what the reference's
 * IO_utils.c / Buffer allocations become on this path: with page-locked buffers the copies
 * overlap with the kernels).  Returns NULL when no device is usable.                       */
void *snappy_b200_host_alloc(size_t bytes);
void snappy_b200_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* SNAPPY_B200_H */
