// abi.cu -- the C-ABI of libsnappy_b200.so (see include/snappy_b200.h): argument checks,
// workspace carving, kernel sequencing, and the synchronous host-buffer entry points.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>

#include "common.cuh"

namespace sb200 {
cudaError_t launch_compress(const uint8_t *, uint64_t, int, uint8_t *, uint32_t *, uint2 *, uint32_t *, uint16_t *,
                            cudaStream_t, uint64_t *);
size_t compress_records_bytes(uint64_t);
size_t parallel_cand_bytes(uint64_t);
cudaError_t launch_compact(const uint8_t *, const uint32_t *, uint64_t, uint64_t, uint64_t, int, uint8_t *, uint64_t,
                           uint64_t *, uint64_t *, uint32_t *, cudaStream_t, uint64_t *);
cudaError_t launch_decode(const uint8_t *, const uint64_t *, uint64_t, uint64_t, uint8_t *, uint32_t *, cudaStream_t,
                          uint64_t *);
cudaError_t launch_decode_seg(const uint8_t *, uint64_t, const uint64_t *, const uint4 *, const uint64_t *, uint64_t,
                              uint64_t, uint8_t *, uint32_t *, uint64_t, cudaStream_t, uint64_t *);
const uint4 *index_starts(void *, uint64_t);
const uint64_t *index_outoff(void *, uint64_t);
size_t index_workspace_bytes(uint64_t);
cudaError_t run_index(const uint8_t *, uint64_t, uint64_t, uint64_t, uint64_t *, uint32_t *, void *, cudaStream_t,
                      uint64_t *, bool, uint64_t, uint32_t fixed_rounds = 0);
uint32_t host_varint_len(uint64_t);
uint64_t index_last_rounds();
cudaError_t launch_frame_compact(const uint8_t *, uint64_t, const uint8_t *, const uint32_t *, uint32_t *, uint32_t *, int,
                                 uint8_t *, uint64_t, uint64_t *, uint64_t *, uint32_t *, cudaStream_t, uint64_t *);

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

static int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

static int cuda_fail(cudaError_t e, const char *what)
{
    return fail(SNAPPY_B200_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

struct CompressWorkspace {
    uint8_t *scratch;   // one 66560-byte slot per block: the block's compressed bytes
    uint2 *recs;        // one 8-byte record per copy, 16384 per block
    uint32_t *sizes;    // compressed size of every block
    uint32_t *nrec;     // records of every block
    uint64_t *offsets;  // stream offset of every block (when the caller does not want them)
    uint16_t *cand;     // SNAPPY_B200_MODE_PARALLEL only: the candidate offset of every input byte
};

static size_t compress_ws_bytes(uint64_t n_bytes, int mode)
{
    const uint64_t nb = (n_bytes + kBlock - 1) / kBlock;
    const size_t base = align_up(nb * (size_t)kSlot + 64, 256) + align_up(compress_records_bytes(nb) + 64, 256) +
                        2 * align_up(nb * 4 + 4, 256) + align_up((nb + 1) * 8, 256);
    return mode == SNAPPY_B200_MODE_PARALLEL ? base + align_up(parallel_cand_bytes(nb), 256) : base;
}

static CompressWorkspace carve_compress(void *ws, uint64_t n_bytes, int mode)
{
    const uint64_t nb = (n_bytes + kBlock - 1) / kBlock;
    uint8_t *p = static_cast<uint8_t *>(ws);
    CompressWorkspace w;
    w.scratch = p, p += align_up(nb * (size_t)kSlot + 64, 256);
    w.recs = reinterpret_cast<uint2 *>(p), p += align_up(compress_records_bytes(nb) + 64, 256);
    w.sizes = reinterpret_cast<uint32_t *>(p), p += align_up(nb * 4 + 4, 256);
    w.nrec = reinterpret_cast<uint32_t *>(p), p += align_up(nb * 4 + 4, 256);
    w.offsets = reinterpret_cast<uint64_t *>(p), p += align_up((nb + 1) * 8, 256);
    w.cand = mode == SNAPPY_B200_MODE_PARALLEL ? reinterpret_cast<uint16_t *>(p) : nullptr;
    return w;
}

// The framed compressor's workspace: the raw compressor's, then the masked CRC and the chunk size of every block.
static size_t frame_ws_bytes(uint64_t n_bytes, int mode)
{
    const uint64_t nb = (n_bytes + kBlock - 1) / kBlock;
    return compress_ws_bytes(n_bytes, mode) + 2 * align_up(nb * 4 + 4, 256);
}

static void carve_frame(void *ws, uint64_t n_bytes, int mode, uint32_t **crcs, uint32_t **fsizes)
{
    const uint64_t nb = (n_bytes + kBlock - 1) / kBlock;
    uint8_t *p = static_cast<uint8_t *>(ws) + compress_ws_bytes(n_bytes, mode);
    *crcs = reinterpret_cast<uint32_t *>(p);
    *fsizes = reinterpret_cast<uint32_t *>(p + align_up(nb * 4 + 4, 256));
}

static int status_to_error(uint32_t st)
{
    // FRAMING first: once an element leaves the 64 KiB framing the blocks after it may look malformed to the
    // block-parallel decoders although the stream is valid; the general decoder is the arbiter then
    if (st & SNAPPY_B200_ST_FRAMING)
        return fail(SNAPPY_B200_ERR_FRAMING,
                    "the stream is not framed in 64 KiB blocks (an element straddles a block or reaches into an "
                    "earlier one; device status 0x%x)", st);
    if (st & SNAPPY_B200_ST_CORRUPT)
        return fail(SNAPPY_B200_ERR_CORRUPT, "malformed compressed stream (device status 0x%x)", st);
    if (st & SNAPPY_B200_ST_CHECKSUM)
        return fail(SNAPPY_B200_ERR_CHECKSUM, "a chunk's CRC-32C does not match its data (device status 0x%x)", st);
    if (st & SNAPPY_B200_ST_UNRESOLVED)
        return fail(SNAPPY_B200_ERR_CORRUPT,
                    "the element chain of the stream did not resolve within the relaxation rounds allowed "
                    "(device status 0x%x): adversarial input, or max_rounds too small for the asynchronous call",
                    st);
    if (st & SNAPPY_B200_ST_CAPACITY)
        return fail(SNAPPY_B200_ERR_CAPACITY, "output buffer too small (device status 0x%x)", st);
    if (st)
        return fail(SNAPPY_B200_ERR_CORRUPT, "device status 0x%x", st);
    return SNAPPY_B200_OK;
}

int fail_msg(int code, const char *msg) { return fail(code, "%s", msg); }
// The one place that decides which compression modes exist: SNAPPY_B200_OK, or SNAPPY_B200_ERR_ARG with the message set.
int check_mode(int mode)
{
    if (mode == SNAPPY_B200_MODE_HASH || mode == SNAPPY_B200_MODE_BST || mode == SNAPPY_B200_MODE_PARALLEL)
        return SNAPPY_B200_OK;
    return fail(SNAPPY_B200_ERR_ARG, "unknown mode %d", mode);
}
void clear_error() { g_err[0] = 0; } // every public entry point starts clean: a stale message is never reported twice
int cuda_fail_msg(cudaError_t e, const char *what) { return cuda_fail(e, what); }
int status_error(uint32_t st) { return status_to_error(st); }
size_t compress_workspace_bytes_internal(uint64_t n_bytes, bool framed, int mode)
{
    return framed ? frame_ws_bytes(n_bytes, mode) : compress_ws_bytes(n_bytes, mode);
}
void add_launches(uint64_t n) { g_launches += n; }

// Small device -> host read-backs (sizes, flags, status words).  A cudaMemcpyAsync would queue
// on the D2H copy engine behind whatever bulk download is in flight (measured: K0 of the next
// piece waited 6 ms for a 330 MiB download); a one-CTA kernel that stores straight into pinned
// host memory does not.
__global__ void k_peek(uint32_t *__restrict__ dst, const uint32_t *__restrict__ src, uint32_t n)
{
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x)
        dst[i] = src[i];
}

cudaError_t peek_u32(uint32_t *h_pinned_dst, const void *d_src, uint32_t n_u32, cudaStream_t st)
{
    k_peek<<<1, 64, 0, st>>>(h_pinned_dst, static_cast<const uint32_t *>(d_src), n_u32);
    g_launches += 1;
    return cudaGetLastError();
}

// 1 KiB of pinned host memory per calling thread (kept for the life of the process).
uint32_t *thread_pinned_scratch()
{
    thread_local uint32_t *p = nullptr;
    if (!p && cudaHostAlloc(reinterpret_cast<void **>(&p), 1024, cudaHostAllocDefault) != cudaSuccess) {
        (void)cudaGetLastError();
        p = nullptr;
    }
    return p;
}

// One chunk of a longer input: blocks only, or (varint_value != 0: the chunk opens the stream) the varint of the
// WHOLE input followed by blocks.  framed: data chunks of the framing format instead of bare blocks (varint_value
// is not used), with the stream identifier in front when `identifier` is set.  Same kernels as
// snappy_b200_compress_device / snappy_b200_frame_compress_device.
cudaError_t compress_chunk(const uint8_t *d_in, uint64_t chunk_bytes, uint64_t varint_value, int mode, bool framed,
                           bool identifier, uint8_t *d_out, uint64_t out_capacity, uint64_t *d_out_bytes,
                           uint32_t *d_status, void *d_workspace, cudaStream_t st)
{
    const uint64_t nb = (chunk_bytes + kBlock - 1) / kBlock;
    CompressWorkspace w = carve_compress(d_workspace, chunk_bytes, mode);
    uint64_t launches = 0;
    cudaError_t e =
        launch_compress(d_in, chunk_bytes, mode, w.scratch, w.sizes, w.recs, w.nrec, w.cand, st, &launches);
    if (e == cudaSuccess && framed) {
        uint32_t *crcs, *fsizes;
        carve_frame(d_workspace, chunk_bytes, mode, &crcs, &fsizes);
        e = launch_frame_compact(d_in, chunk_bytes, w.scratch, w.sizes, crcs, fsizes, identifier ? 1 : 0, d_out,
                                 out_capacity, w.offsets, d_out_bytes, d_status, st, &launches);
    } else if (e == cudaSuccess) {
        e = launch_compact(w.scratch, w.sizes, nb, varint_value, varint_value ? host_varint_len(varint_value) : 0,
                           varint_value ? 1 : 0, d_out, out_capacity, w.offsets, d_out_bytes, d_status, st, &launches);
    }
    g_launches += launches;
    return e;
}

// The block offsets (relative to the chunk's output) compress_chunk left in its workspace: nb + 1 entries.
const uint64_t *compress_chunk_offsets(void *d_workspace, uint64_t chunk_bytes)
{
    return carve_compress(d_workspace, chunk_bytes, SNAPPY_B200_MODE_HASH).offsets; // (the same for every mode)
}

} // namespace sb200

using namespace sb200;

extern "C" {

const char *snappy_b200_last_error(void) { return g_err; }

int snappy_b200_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess)
        return cuda_fail(e, "cudaGetDeviceCount");
    return n;
}

uint64_t snappy_b200_launch_count(void) { return g_launches.load(); }

uint64_t snappy_b200_index_rounds(void) { return index_last_rounds(); }

uint64_t snappy_b200_block_count(uint64_t n_bytes) { return (n_bytes + kBlock - 1) / kBlock; }

uint64_t snappy_b200_max_compressed_bytes(uint64_t n_bytes)
{
    return n_bytes ? 10 + n_bytes + snappy_b200_block_count(n_bytes) * 1010 : 0;
}

size_t snappy_b200_compress_workspace_bytes(uint64_t n_bytes, int mode)
{
    return compress_ws_bytes(n_bytes, mode);
}

int snappy_b200_compress_device(const uint8_t *d_in, uint64_t n_bytes, int mode, uint8_t *d_out, uint64_t out_capacity,
                                uint64_t *d_out_bytes, uint64_t *d_block_offsets, uint32_t *d_status,
                                void *d_workspace, size_t workspace_bytes, void *stream)
{
    clear_error();
    if (check_mode(mode) != SNAPPY_B200_OK)
        return SNAPPY_B200_ERR_ARG;
    if (!d_out_bytes || !d_status || (n_bytes && (!d_in || !d_out || !d_workspace)))
        return fail(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (!aligned16(d_in) || !aligned16(d_out) || !aligned16(d_workspace))
        return fail(SNAPPY_B200_ERR_ARG, "d_in, d_out and d_workspace must be 16-byte aligned");
    if (workspace_bytes < compress_ws_bytes(n_bytes, mode))
        return fail(SNAPPY_B200_ERR_ARG, "workspace too small: %zu < %zu", workspace_bytes,
                    compress_ws_bytes(n_bytes, mode));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const uint64_t nb = (n_bytes + kBlock - 1) / kBlock;
    cudaError_t e = cudaMemsetAsync(d_status, 0, sizeof(uint32_t), st);
    if (e != cudaSuccess)
        return cuda_fail(e, "cudaMemsetAsync(status)");
    if (nb == 0) { // reference: an empty input gives an empty stream (SURVEY.md 8c)
        e = cudaMemsetAsync(d_out_bytes, 0, sizeof(uint64_t), st);
        if (e == cudaSuccess && d_block_offsets)
            e = cudaMemsetAsync(d_block_offsets, 0, sizeof(uint64_t), st);
        return e == cudaSuccess ? SNAPPY_B200_OK : cuda_fail(e, "cudaMemsetAsync");
    }
    CompressWorkspace w = carve_compress(d_workspace, n_bytes, mode);
    uint64_t launches = 0;
    e = launch_compress(d_in, n_bytes, mode, w.scratch, w.sizes, w.recs, w.nrec, w.cand, st, &launches);
    if (e == cudaSuccess)
        e = launch_compact(w.scratch, w.sizes, nb, n_bytes, host_varint_len(n_bytes), 1, d_out, out_capacity,
                           d_block_offsets ? d_block_offsets : w.offsets, d_out_bytes, d_status, st, &launches);
    g_launches += launches;
    if (e != cudaSuccess)
        return cuda_fail(e, "compress launch");
    return SNAPPY_B200_OK;
}

uint64_t snappy_b200_frame_max_compressed_bytes(uint64_t n_bytes)
{
    return 10 + n_bytes + 8 * snappy_b200_block_count(n_bytes);
}

size_t snappy_b200_frame_compress_workspace_bytes(uint64_t n_bytes, int mode)
{
    return frame_ws_bytes(n_bytes, mode);
}

int snappy_b200_frame_compress_device(const uint8_t *d_in, uint64_t n_bytes, int mode, uint8_t *d_out,
                                      uint64_t out_capacity, uint64_t *d_out_bytes, uint32_t *d_status,
                                      void *d_workspace, size_t workspace_bytes, void *stream)
{
    clear_error();
    if (check_mode(mode) != SNAPPY_B200_OK)
        return SNAPPY_B200_ERR_ARG;
    if (!d_out_bytes || !d_status || !d_out || !d_workspace || (n_bytes && !d_in))
        return fail(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (!aligned16(d_in) || !aligned16(d_out) || !aligned16(d_workspace))
        return fail(SNAPPY_B200_ERR_ARG, "d_in, d_out and d_workspace must be 16-byte aligned");
    if (workspace_bytes < frame_ws_bytes(n_bytes, mode))
        return fail(SNAPPY_B200_ERR_ARG, "workspace too small: %zu < %zu", workspace_bytes, frame_ws_bytes(n_bytes, mode));
    if ((n_bytes + kBlock - 1) / kBlock > 0x7fffffffull)
        return fail(SNAPPY_B200_ERR_ARG, "input too large");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(d_status, 0, sizeof(uint32_t), st);
    if (e != cudaSuccess)
        return cuda_fail(e, "cudaMemsetAsync(status)");
    e = compress_chunk(d_in, n_bytes, 0, mode, true, true, d_out, out_capacity, d_out_bytes, d_status, d_workspace, st);
    if (e != cudaSuccess)
        return cuda_fail(e, "framed compress launch");
    return SNAPPY_B200_OK;
}

int snappy_b200_decompress_device_indexed(const uint8_t *d_stream, const uint64_t *d_block_offsets, uint64_t n_blocks,
                                          uint64_t total_out, uint8_t *d_out, uint32_t *d_status, void *stream)
{
    clear_error();
    if (!d_status || (n_blocks && (!d_stream || !d_block_offsets || !d_out)))
        return fail(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (n_blocks != (total_out + kBlock - 1) / kBlock)
        return fail(SNAPPY_B200_ERR_ARG, "n_blocks does not match total_out");
    uint64_t launches = 0;
    cudaError_t e = launch_decode(d_stream, d_block_offsets, n_blocks, total_out, d_out, d_status,
                                  static_cast<cudaStream_t>(stream), &launches);
    g_launches += launches;
    if (e != cudaSuccess)
        return cuda_fail(e, "decode launch");
    return SNAPPY_B200_OK;
}

size_t snappy_b200_index_workspace_bytes(uint64_t stream_bytes) { return index_workspace_bytes(stream_bytes); }

int snappy_b200_index_device(const uint8_t *d_stream, uint64_t stream_bytes, uint64_t body_offset, uint64_t total_out,
                             uint64_t *d_block_offsets, uint32_t *d_status, void *d_workspace, size_t workspace_bytes,
                             void *stream)
{
    clear_error();
    if (!d_stream || !d_block_offsets || !d_status || !d_workspace)
        return fail(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (body_offset > stream_bytes || stream_bytes >= (1ull << 40))
        return fail(SNAPPY_B200_ERR_ARG, "bad stream size / body offset");
    if (workspace_bytes < index_workspace_bytes(stream_bytes))
        return fail(SNAPPY_B200_ERR_ARG, "workspace too small");
    uint64_t launches = 0;
    cudaError_t e = run_index(d_stream, stream_bytes, body_offset, total_out, d_block_offsets, d_status, d_workspace,
                              static_cast<cudaStream_t>(stream), &launches, false, 0);
    g_launches += launches;
    if (e != cudaSuccess)
        return cuda_fail(e, "index launch");
    return SNAPPY_B200_OK;
}

int snappy_b200_decode_segments_device(const uint8_t *d_stream, uint64_t stream_bytes, uint64_t body_offset,
                                       uint64_t total_out, uint8_t *d_out, const uint64_t *d_block_offsets,
                                       uint32_t *d_status, void *d_workspace, size_t workspace_bytes, void *stream)
{
    clear_error();
    if (!d_stream || !d_block_offsets || !d_status || !d_workspace || (!d_out && total_out))
        return fail(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (workspace_bytes < index_workspace_bytes(stream_bytes))
        return fail(SNAPPY_B200_ERR_ARG, "workspace too small");
    uint64_t launches = 0;
    cudaError_t e = launch_decode_seg(d_stream, body_offset, d_block_offsets, index_starts(d_workspace, stream_bytes),
                                      index_outoff(d_workspace, stream_bytes), (total_out + kBlock - 1) / kBlock,
                                      total_out, d_out, d_status, 0, static_cast<cudaStream_t>(stream), &launches);
    g_launches += launches;
    if (e != cudaSuccess)
        return cuda_fail(e, "decode launch");
    return SNAPPY_B200_OK;
}

// ---- asynchronous index-less decode: K0 with a fixed number of relaxation rounds (ended on the device)
// followed by the block decode, all enqueued on `stream`: no host read-back, no synchronisation, no lock,
// no allocation -- the call can be captured into a CUDA graph.
size_t snappy_b200_decompress_async_workspace_bytes(uint64_t stream_bytes, uint64_t total_out)
{
    const uint64_t nb = (total_out + kBlock - 1) / kBlock;
    return align_up(index_workspace_bytes(stream_bytes), 256) + align_up((nb + 2) * 8, 256);
}

int snappy_b200_decompress_device_async(const uint8_t *d_stream, uint64_t stream_bytes, uint64_t body_offset,
                                        uint64_t total_out, uint8_t *d_out, uint64_t *d_block_offsets, uint32_t *d_status,
                                        void *d_workspace, size_t workspace_bytes, unsigned max_rounds, void *stream)
{
    clear_error();
    if (!d_stream || !d_status || !d_workspace || (!d_out && total_out))
        return fail(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (body_offset > stream_bytes || stream_bytes >= (1ull << 40))
        return fail(SNAPPY_B200_ERR_ARG, "bad stream size / body offset");
    if (workspace_bytes < snappy_b200_decompress_async_workspace_bytes(stream_bytes, total_out))
        return fail(SNAPPY_B200_ERR_ARG, "workspace too small (see snappy_b200_decompress_async_workspace_bytes)");
    if (total_out == 0)
        return stream_bytes == body_offset ? SNAPPY_B200_OK
                                           : fail(SNAPPY_B200_ERR_CORRUPT, "trailing bytes after an empty stream");
    const uint64_t nb = (total_out + kBlock - 1) / kBlock;
    uint64_t *offs = d_block_offsets
                         ? d_block_offsets
                         : reinterpret_cast<uint64_t *>(static_cast<uint8_t *>(d_workspace) +
                                                        align_up(index_workspace_bytes(stream_bytes), 256));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint64_t launches = 0;
    cudaError_t e = run_index(d_stream, stream_bytes, body_offset, total_out, offs, d_status, d_workspace, st, &launches,
                              false, 0, max_rounds ? max_rounds : 64u);
    if (e == cudaSuccess)
        e = launch_decode_seg(d_stream, body_offset, offs, index_starts(d_workspace, stream_bytes),
                              index_outoff(d_workspace, stream_bytes), nb, total_out, d_out, d_status, 0, st, &launches);
    g_launches += launches;
    if (e != cudaSuccess)
        return cuda_fail(e, "asynchronous decompress launch");
    return SNAPPY_B200_OK;
}

} // extern "C"

