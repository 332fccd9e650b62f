// host_pipeline.cu -- the host-buffer entry points (include/snappy_b200.h, layer 2): the
// batched block scheduler that sits where the reference's Buffer / fread / fwrite loop was
// (src/snappy_compression.c:414-428, src/snappy_decompression.c:345-363).
//
// The input is framed into chunks of whole 64 KiB blocks and streamed through the GPU on three
// CUDA streams so that the upload of chunk j+1, the kernels of chunk j and the download of
// chunk j-1 overlap (PCIe is full duplex):
//   compress    chunk = 2048 blocks (128 MiB), four chunks in flight, each on its own stream: the
//               parse is a latency-bound chain per block, so the GPU only fills up when
//               thousands of blocks are resident at once.  Each chunk is compressed into bare
//               blocks (the first one also carries the varint of the whole input); its size is
//               read back, which tells where the chunk goes in the caller's buffer, and its
//               bytes follow on the download stream.
//   decompress  the stream is uploaded in pieces that grow from 16 to 128 MiB (measured best on PCIe 5
//               x16; SNAPPY_B200_PIECE_START_MIB / _GROWTH / _MIB override).  Whenever a piece has landed, K0 runs
//               on the not-yet-decoded tail of what is on the device ("open-ended": the
//               element cut off by the end of the piece is not an error); every block that is
//               complete is decoded by the segment-driven decoder on a second stream (so it
//               overlaps K0 of the next piece) and downloaded while later pieces are still in
//               flight; the incomplete last block is taken up again with the next piece.
// Host buffers may be pageable or page-locked; with page-locked buffers (cudaHostAlloc /
// cudaHostRegister, torch pin_memory) the copies are truly asynchronous.
#include <algorithm>
#include <functional>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"

namespace sb200 {
int decompress_host_general(const void *stream, uint64_t stream_bytes, void *out, uint64_t *out_bytes);
int fail_msg(int code, const char *msg);
void clear_error();
int cuda_fail_msg(cudaError_t e, const char *what);
int status_error(uint32_t st);
size_t compress_workspace_bytes_internal(uint64_t n_bytes, bool framed, int mode);
int check_mode(int mode);
void add_launches(uint64_t n);
cudaError_t compress_chunk(const uint8_t *, uint64_t, uint64_t, int, bool, bool, uint8_t *, uint64_t, uint64_t *, uint32_t *,
                           void *, cudaStream_t);
cudaError_t launch_frame_decode(const uint8_t *, uint64_t, const FrameChunk *, uint64_t, uint8_t *, uint32_t *,
                                cudaStream_t, uint64_t *);
int frame_decompress_buffer(const void *, uint64_t, void *, uint64_t, uint64_t *, bool);
cudaError_t launch_frame_check(const uint8_t *, const FrameChunk *, uint64_t, uint32_t *, cudaStream_t, uint64_t *);
size_t index_workspace_bytes(uint64_t);
cudaError_t run_index(const uint8_t *, uint64_t, uint64_t, uint64_t, uint64_t *, uint32_t *, void *, cudaStream_t,
                      uint64_t *, bool, uint64_t, uint32_t fixed_rounds = 0);
const uint4 *index_starts(void *, uint64_t);
const uint64_t *index_total(void *, uint64_t);
const uint64_t *compress_chunk_offsets(void *, uint64_t);
cudaError_t launch_decode(const uint8_t *, const uint64_t *, uint64_t, uint64_t, uint8_t *, uint32_t *, cudaStream_t,
                          uint64_t *);
cudaError_t launch_decode_sequential(const uint8_t *, uint64_t, uint64_t, uint64_t, uint8_t *, uint32_t *, cudaStream_t,
                                     uint64_t *);
const uint64_t *index_outoff(void *, uint64_t);
cudaError_t launch_decode_seg(const uint8_t *, uint64_t, const uint64_t *, const uint4 *, const uint64_t *, uint64_t, uint64_t, uint8_t *,
                              uint32_t *, uint64_t, cudaStream_t, uint64_t *);

namespace {

constexpr int kSlots = 4; // compress chunks in flight

// Chunk sizes in MiB; SNAPPY_B200_CHUNK_MIB / SNAPPY_B200_PIECE_MIB override them (tests use
// small values to exercise many chunks on small inputs).
uint64_t env_mib(const char *name, uint64_t dflt)
{
    const char *v = getenv(name);
    const long long x = v ? atoll(v) : 0;
    return (uint64_t)(x > 0 ? x : (long long)dflt) << 20;
}
#define kCompressChunk env_mib("SNAPPY_B200_CHUNK_MIB", 128) /* input bytes per compress chunk (whole blocks) */
#define kUploadPiece env_mib("SNAPPY_B200_PIECE_MIB", 128)   /* stream bytes per upload piece (host path) */

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

inline uint64_t max_compressed(uint64_t n)
{
    return n ? 10 + n + ((n + kBlock - 1) / kBlock) * 1010 : 0;
}

// The longest valid encoding of `total` output bytes: one 1-byte literal with a 4-byte length (6 stream bytes)
// per output byte.  Streams between max_compressed(total) and this are valid raw Snappy that no compressor
// emits; they are decoded (by the general decoder when their blocks are too long for the block decoders).
inline bool longer_than_any_encoding(uint64_t stream_bytes, uint64_t hdr, uint64_t total)
{
    return (stream_bytes - hdr + 5) / 6 > total;
}

unsigned host_varint_decode(const uint8_t *p, uint64_t avail, uint64_t *out)
{
    uint64_t v = 0;
    unsigned shift = 0;
    for (unsigned k = 0; k < avail && k < 10; ++k) {
        v |= (uint64_t)(p[k] & 0x7fu) << shift;
        shift += 7;
        if (!(p[k] & 0x80u)) {
            *out = v;
            return k + 1;
        }
    }
    return 0;
}

// ---- framing format (include/snappy_b200.h): the chunk headers are walked on the host
const uint8_t kStreamId[10] = {0xff, 0x06, 0x00, 0x00, 's', 'N', 'a', 'P', 'p', 'Y'};

int frame_fail(int code, uint64_t at, const char *what)
{
    char msg[160];
    snprintf(msg, sizeof msg, "framed stream, chunk at offset %llu: %s", (unsigned long long)at, what);
    return fail_msg(code, msg);
}

// Checks every rule of the framing format except the compressed payloads and the CRCs; *total = the uncompressed
// length; `chunks` (optional) receives one descriptor per data chunk, in stream order.  opens_stream: the buffer is
// a whole stream (it must begin with the identifier); otherwise it is a run of whole chunks from inside a stream.
int frame_walk(const uint8_t *p, uint64_t n, bool opens_stream, std::vector<FrameChunk> *chunks, uint64_t *total)
{
    *total = 0;
    if (n == 0)
        return SNAPPY_B200_OK; // an empty buffer is an empty stream, as for the raw calls
    if (opens_stream && (n < sizeof kStreamId || memcmp(p, kStreamId, sizeof kStreamId) != 0))
        return frame_fail(SNAPPY_B200_ERR_CORRUPT, 0, "the stream does not start with the stream identifier");
    uint64_t at = opens_stream ? sizeof kStreamId : 0, out = 0;
    while (at < n) {
        if (n - at < 4)
            return frame_fail(SNAPPY_B200_ERR_CORRUPT, at, "truncated chunk header");
        const uint32_t type = p[at], L = p[at + 1] | (uint32_t)p[at + 2] << 8 | (uint32_t)p[at + 3] << 16;
        if (L > n - at - 4)
            return frame_fail(SNAPPY_B200_ERR_CORRUPT, at, "the chunk runs past the end of the stream");
        const uint8_t *body = p + at + 4;
        if (type == kChunkCompressed || type == kChunkUncompressed) {
            if (L < 4)
                return frame_fail(SNAPPY_B200_ERR_CORRUPT, at, "data chunk shorter than its checksum");
            FrameChunk c;
            c.type = type;
            c.crc = body[0] | (uint32_t)body[1] << 8 | (uint32_t)body[2] << 16 | (uint32_t)body[3] << 24;
            if (type == kChunkCompressed) {
                uint64_t len = 0;
                const unsigned vl = host_varint_decode(body + 4, L - 4, &len);
                if (!vl)
                    return frame_fail(SNAPPY_B200_ERR_CORRUPT, at, "bad varint in a compressed chunk");
                if (len > kBlock)
                    return frame_fail(SNAPPY_B200_ERR_CORRUPT, at, "compressed chunk of more than 65536 bytes");
                c.in_off = at + 8 + vl, c.in_len = L - 4 - vl, c.out_len = (uint32_t)len;
            } else {
                if (L - 4 > kBlock)
                    return frame_fail(SNAPPY_B200_ERR_CORRUPT, at, "uncompressed chunk of more than 65536 bytes");
                c.in_off = at + 8, c.in_len = L - 4, c.out_len = L - 4;
            }
            c.out_off = out;
            out += c.out_len;
            if (chunks)
                chunks->push_back(c);
        } else if (type == 0xff) {
            if (L != 6 || memcmp(body, kStreamId + 4, 6) != 0)
                return frame_fail(SNAPPY_B200_ERR_CORRUPT, at, "bad stream identifier");
        } else if (type < 0x80) {
            return frame_fail(SNAPPY_B200_ERR_CORRUPT, at, "reserved unskippable chunk type");
        } // 0x80-0xfd reserved skippable, 0xfe padding
        at += 4 + (uint64_t)L;
    }
    *total = out;
    return SNAPPY_B200_OK;
}

// Cached per-process resources of the synchronous host-buffer entry points.
struct HostCtx {
    static constexpr int kBufs = 16;
    std::mutex mu;
    cudaStream_t s_up = nullptr, s_run = nullptr, s_down = nullptr, s_dec = nullptr;
    cudaStream_t s_slot[kSlots] = {};
    void *buf[kBufs] = {};
    size_t cap[kBufs] = {};
    uint64_t *h_small = nullptr; // pinned scratch for small read-backs
    cudaEvent_t ev[32] = {};
    static constexpr int kFileSlots = 3;
    uint8_t *h_file[kFileSlots] = {}; // page-locked chunk ring of the FILE* decompressor
    size_t h_file_cap = 0;
    cudaError_t need_file_ring(size_t bytes)
    {
        if (h_file_cap >= bytes)
            return cudaSuccess;
        for (auto &p : h_file) {
            if (p)
                cudaFreeHost(p);
            p = nullptr;
        }
        h_file_cap = 0;
        for (auto &p : h_file) {
            const cudaError_t e = cudaHostAlloc(reinterpret_cast<void **>(&p), bytes, cudaHostAllocDefault);
            if (e != cudaSuccess)
                return e;
        }
        h_file_cap = bytes;
        return cudaSuccess;
    }

    cudaError_t need(int i, size_t bytes)
    {
        bytes = align_up(bytes + 256, 1 << 20);
        if (cap[i] >= bytes)
            return cudaSuccess;
        if (buf[i])
            cudaFree(buf[i]);
        buf[i] = nullptr;
        cap[i] = 0;
        cudaError_t e = cudaMalloc(&buf[i], bytes);
        if (e == cudaSuccess)
            cap[i] = bytes;
        return e;
    }
    int device = -1;
    cudaError_t init()
    {
        int dev = -1;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess)
            return e;
        if (device != -1 && dev != device)
            release(); // the cached streams / buffers belong to another device
        device = dev;
        for (cudaStream_t *s : {&s_up, &s_run, &s_down, &s_dec, &s_slot[0], &s_slot[1], &s_slot[2], &s_slot[3]})
            if (e == cudaSuccess && !*s)
                e = cudaStreamCreateWithFlags(s, cudaStreamNonBlocking);
        if (e == cudaSuccess && !h_small)
            e = cudaHostAlloc(reinterpret_cast<void **>(&h_small), 256, cudaHostAllocDefault);
        for (auto &x : ev)
            if (e == cudaSuccess && !x)
                e = cudaEventCreateWithFlags(&x, cudaEventDisableTiming);
        return e;
    }
    void release()
    {
        device = -1;
        for (int i = 0; i < kBufs; ++i) {
            if (buf[i])
                cudaFree(buf[i]);
            buf[i] = nullptr;
            cap[i] = 0;
        }
        if (h_small)
            cudaFreeHost(h_small);
        h_small = nullptr;
        for (auto &p : h_file) {
            if (p)
                cudaFreeHost(p);
            p = nullptr;
        }
        h_file_cap = 0;
        for (auto &x : ev) {
            if (x)
                cudaEventDestroy(x);
            x = nullptr;
        }
        for (cudaStream_t *s : {&s_up, &s_run, &s_down, &s_dec, &s_slot[0], &s_slot[1], &s_slot[2], &s_slot[3]}) {
            if (*s)
                cudaStreamDestroy(*s);
            *s = nullptr;
        }
    }
};

// One context per device (streams, events and cached buffers belong to a device), each behind its own lock:
// calls on different devices run concurrently, calls on the same device take turns.
constexpr int kMaxDevices = 64;
HostCtx g_ctx_pool[kMaxDevices];

// SNAPPY_B200_DEVICES=N (N > 1): the host-buffer calls shard block ranges over the first N devices
// (csrc/multi_device.cu) for inputs of at least 64 MiB.  Default 1 = the current device only: under a
// one-process-per-GPU launcher every rank must stay on its own device.
int env_devices()
{
    const char *v = getenv("SNAPPY_B200_DEVICES");
    const int n = v ? atoi(v) : 1;
    return n < 1 ? 1 : n;
}
// Devices a decompress call would shard over: SNAPPY_B200_DEVICES, at most the devices present.  The decode
// forwards to the multi-device calls only when this is above 1: with a single device those calls come back
// to the one-device path.
int decode_devices()
{
    const int want = env_devices();
    int n = 0;
    if (want < 2)
        return 1;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 1;
    }
    return std::min(want, n);
}
constexpr uint64_t kMultiMin = 64ull << 20;

HostCtx &current_ctx()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) {
        (void)cudaGetLastError();
        dev = 0;
    }
    return g_ctx_pool[(unsigned)dev % kMaxDevices];
}

// SNAPPY_B200_TRACE=1: timeline of a host call (milliseconds since its first enqueue) on stderr.
struct Trace {
    bool on = getenv("SNAPPY_B200_TRACE") != nullptr;
    cudaEvent_t t0 = nullptr;
    std::vector<std::pair<std::string, cudaEvent_t>> marks;
    void start(cudaStream_t s)
    {
        if (!on)
            return;
        cudaEventCreate(&t0);
        cudaEventRecord(t0, s);
    }
    void mark(const std::string &what, cudaStream_t s)
    {
        if (!on)
            return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, s);
        marks.emplace_back(what, e);
    }
    void dump()
    {
        if (!on)
            return;
        cudaDeviceSynchronize();
        for (auto &m : marks) {
            float ms = 0;
            cudaEventElapsedTime(&ms, t0, m.second);
            fprintf(stderr, "[trace] %8.3f ms  %s\n", ms, m.first.c_str());
            cudaEventDestroy(m.second);
        }
        cudaEventDestroy(t0);
        marks.clear();
    }
};

// Adds `add` to n offsets (K0 reports them relative to the region it was given).
__global__ void k_rebase_offsets(uint64_t *__restrict__ dst, const uint64_t *__restrict__ src, uint64_t n, uint64_t add)
{
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < n)
        dst[i] = src[i] + add;
}

struct PieceHooks {
    // enqueue on s_run whatever makes stream bytes of piece p resident (host path: wait for its upload)
    std::function<cudaError_t(uint64_t p, cudaStream_t s_run)> before_piece;
    // output bytes [first, first + bytes) are final once `done` (recorded on the decode stream) fires
    std::function<cudaError_t(uint64_t first, uint64_t bytes, cudaEvent_t done)> after_decode;
    Trace *trace = nullptr;
};

struct PieceResources {
    void *ws[2];           // K0 workspaces, index_workspace_bytes(region_cap) each
    uint64_t *offs[2];     // region-relative block offsets, blocks + 2 entries each
    cudaStream_t s_run, s_dec;
    cudaEvent_t ev_k0[2], ev_dec[2];
    uint64_t *h_small;     // pinned, >= 4 words
};

uint64_t piece_region_cap(uint64_t stream_bytes, uint64_t piece)
{
    return std::min<uint64_t>(stream_bytes, piece + 2 * (uint64_t)kBlock + 4096);
}

// Decodes a device-resident stream piece by piece: K0 on the not-yet-decoded tail of pieces
// 0..p ("open-ended" except for the last piece), then the segment-driven decoder for every
// block that is complete, on a second stream so that it overlaps K0 of the next piece.
// Returns a SNAPPY_B200_* code; the last decode may still be in flight on r.s_dec.
int decode_pieces(const uint8_t *d_stream, uint64_t stream_bytes, uint64_t hdr, uint64_t total, uint8_t *d_out,
                  uint64_t *d_abs_offsets, uint32_t *d_status, const std::vector<uint64_t> &piece_end,
                  uint64_t region_cap, const PieceResources &r, const PieceHooks &hooks)
{
#define CUP(call, what)                                                                                                \
    do {                                                                                                               \
        cudaError_t e__ = (call);                                                                                      \
        if (e__ != cudaSuccess) {                                                                                      \
            cudaDeviceSynchronize();                                                                                   \
            add_launches(launches);                                                                                    \
            return cuda_fail_msg(e__, what);                                                                           \
        }                                                                                                              \
    } while (0)
    const uint64_t nb = (total + kBlock - 1) / kBlock;
    const uint64_t n_pieces = piece_end.size();
    uint64_t rs = hdr; // stream offset of the first block that is not decoded yet
    uint64_t ob = 0;   // blocks decoded so far
    uint64_t launches = 0, used = 0;
    for (uint64_t p = 0; p < n_pieces; ++p) {
        const bool last = p + 1 == n_pieces;
        const uint64_t hi = piece_end[p];
        if (hooks.before_piece)
            CUP(hooks.before_piece(p, r.s_run), "stream wait");
        if (hi <= rs)
            continue;
        const uint64_t region = hi - rs;
        if (region > region_cap) {
            cudaDeviceSynchronize();
            add_launches(launches);
            return fail_msg(SNAPPY_B200_ERR_FRAMING, "a block of the stream is larger than any 64 KiB block can be");
        }
        const int s = (int)(used & 1);
        if (used >= 2) // the decode that last read this workspace must be done
            CUP(cudaStreamWaitEvent(r.s_run, r.ev_dec[s], 0), "stream wait");
        const uint64_t blocks_left = nb - ob;
        const uint64_t out_left = total - ob * kBlock;
        // K0 on the not-yet-decoded tail; offsets come out relative to d_stream + rs
        CUP(run_index(d_stream + rs, region, 0, last ? out_left : 0, r.offs[s], d_status, r.ws[s], r.s_run, &launches,
                      !last, blocks_left),
            "index launch");
        CUP(cudaEventRecord(r.ev_k0[s], r.s_run), "event record");
        if (hooks.trace)
            hooks.trace->mark("K0 done, piece " + std::to_string(p), r.s_run);
        CUP(peek_u32(reinterpret_cast<uint32_t *>(r.h_small), index_total(r.ws[s], region), 2, r.s_run), "read-back");
        CUP(peek_u32(reinterpret_cast<uint32_t *>(r.h_small + 1), d_status, 1, r.s_run), "read-back");
        CUP(cudaStreamSynchronize(r.s_run), "index");
        const uint32_t status = (uint32_t)r.h_small[1];
        if (status) {
            cudaDeviceSynchronize();
            add_launches(launches);
            return status_error(status);
        }
        const uint64_t produced = r.h_small[0];
        // complete blocks: all of their elements are on the device and the start of the next
        // block is known (it is an element start inside the region)
        uint64_t kdone = last ? blocks_left : produced / kBlock;
        if (!last && kdone > 0 && produced == kdone * kBlock)
            --kdone; // the start of block kdone may lie just beyond the region: wait for more bytes
        if (kdone > blocks_left)
            kdone = blocks_left;
        if (kdone == 0)
            continue;
        ++used;
        const uint64_t out_bytes_now = last ? out_left : kdone * kBlock;
        CUP(peek_u32(reinterpret_cast<uint32_t *>(r.h_small + 2), r.offs[s] + kdone, 2, r.s_run), "read-back");
        if (d_abs_offsets) {
            k_rebase_offsets<<<(unsigned)((kdone + 1 + 255) / 256), 256, 0, r.s_run>>>(d_abs_offsets + ob, r.offs[s],
                                                                                      kdone + 1, rs);
            ++launches;
        }
        // decode on its own stream: K0 of the next piece does not wait for it
        CUP(cudaStreamWaitEvent(r.s_dec, r.ev_k0[s], 0), "stream wait");
        CUP(launch_decode_seg(d_stream + rs, 0, r.offs[s], index_starts(r.ws[s], region), index_outoff(r.ws[s], region),
                              kdone, out_bytes_now, d_out + ob * kBlock, d_status, ob, r.s_dec, &launches),
            "decode launch");
        CUP(cudaEventRecord(r.ev_dec[s], r.s_dec), "event record");
        if (hooks.trace)
            hooks.trace->mark("decode done, piece " + std::to_string(p) + " (" + std::to_string(out_bytes_now >> 20) + " MiB out)", r.s_dec);
        if (hooks.after_decode)
            CUP(hooks.after_decode(ob * kBlock, out_bytes_now, r.ev_dec[s]), "D2H copy");
        CUP(cudaStreamSynchronize(r.s_run), "read-back");
        rs += r.h_small[2];
        ob += kdone;
    }
    add_launches(launches);
    if (ob != nb) {
        cudaDeviceSynchronize();
        return fail_msg(SNAPPY_B200_ERR_CORRUPT, "the stream ends before its declared length is reached");
    }
    return SNAPPY_B200_OK;
#undef CUP
}

#define CU(call, what)                                                                                                 \
    do {                                                                                                               \
        cudaError_t e__ = (call);                                                                                      \
        if (e__ != cudaSuccess) {                                                                                      \
            cudaDeviceSynchronize();                                                                                   \
            return cuda_fail_msg(e__, what);                                                                           \
        }                                                                                                              \
    } while (0)

} // namespace
} // namespace sb200

using namespace sb200;

extern "C" {

int snappy_b200_compress_host(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                              uint64_t *out_bytes)
{
    return snappy_b200_compress_host_indexed(in, n_bytes, mode, out, out_capacity, out_bytes, nullptr);
}

int snappy_b200_compress_host_indexed(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                                      uint64_t *out_bytes, uint64_t *block_offsets)
{
    return snappy_b200_compress_host_range(in, n_bytes, mode, out, out_capacity, out_bytes, block_offsets, n_bytes);
}

} // extern "C"

// The chunk loop of the host-buffer compressors: n_bytes > 0 of input, raw blocks (after the varint of
// varint_value) or, framed, the chunks of the framing format (after the stream identifier when `identifier` is
// set).  Arguments checked.
static int compress_host_chunks(const void *in, uint64_t n_bytes, int mode, bool framed, bool identifier, void *out,
                                uint64_t out_capacity, uint64_t *out_bytes, uint64_t *block_offsets,
                                uint64_t varint_value)
{
    HostCtx &g_ctx = current_ctx();
    std::lock_guard<std::mutex> lock(g_ctx.mu);
    CU(g_ctx.init(), "context init");
    const uint64_t chunk = std::min<uint64_t>(kCompressChunk, align_up(n_bytes, kBlock));
    const uint64_t n_chunks = (n_bytes + chunk - 1) / chunk;
    const uint64_t out_cap_chunk = framed ? snappy_b200_frame_max_compressed_bytes(chunk) : max_compressed(chunk);
    const size_t ws_bytes = compress_workspace_bytes_internal(chunk, framed, mode);
    const int slots = (int)std::min<uint64_t>(kSlots, n_chunks);
    // buffers: s input, 4+s output, 8+s workspace, 12 small
    for (int s = 0; s < slots; ++s) {
        CU(g_ctx.need(0 + s, chunk), "cudaMalloc");
        CU(g_ctx.need(4 + s, out_cap_chunk), "cudaMalloc");
        CU(g_ctx.need(8 + s, ws_bytes), "cudaMalloc");
    }
    CU(g_ctx.need(12, 256), "cudaMalloc");
    uint64_t *d_small = static_cast<uint64_t *>(g_ctx.buf[12]); // per slot: [4s] out_bytes, [4s+1] status
    cudaEvent_t *ev_up = g_ctx.ev, *ev_run = g_ctx.ev + 4, *ev_down = g_ctx.ev + 8, *ev_size = g_ctx.ev + 12;
    const uint8_t *src = static_cast<const uint8_t *>(in);
    uint8_t *dst = static_cast<uint8_t *>(out);

    Trace trace;
    trace.start(g_ctx.s_up);
    // Enqueues everything chunk j needs up to (and including) the read-back of its size.
    auto issue = [&](uint64_t j) -> cudaError_t {
        const int s = (int)(j % slots);
        const uint64_t lo = j * chunk, len = std::min(chunk, n_bytes - lo);
        cudaStream_t st = g_ctx.s_slot[s];
        cudaError_t e = cudaSuccess;
        if (j >= (uint64_t)slots) // the kernels of the previous user of this slot are done with its input
            e = cudaStreamWaitEvent(g_ctx.s_up, ev_run[s], 0);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(g_ctx.buf[0 + s], src + lo, len, cudaMemcpyHostToDevice, g_ctx.s_up);
        if (e == cudaSuccess)
            e = cudaEventRecord(ev_up[s], g_ctx.s_up);
        trace.mark("upload done, chunk " + std::to_string(j), g_ctx.s_up);
        if (e == cudaSuccess)
            e = cudaStreamWaitEvent(st, ev_up[s], 0);
        if (e == cudaSuccess && j >= (uint64_t)slots) // ... and its download has left the output buffer
            e = cudaStreamWaitEvent(st, ev_down[s], 0);
        uint64_t *d_bytes = d_small + 4 * s;
        uint32_t *d_status = reinterpret_cast<uint32_t *>(d_small + 4 * s + 1);
        if (e == cudaSuccess)
            e = cudaMemsetAsync(d_bytes, 0, 16, st);
        if (e == cudaSuccess)
            e = compress_chunk(static_cast<const uint8_t *>(g_ctx.buf[0 + s]), len, j == 0 ? varint_value : 0, mode,
                               framed, identifier && j == 0, static_cast<uint8_t *>(g_ctx.buf[4 + s]), out_cap_chunk, d_bytes, d_status,
                               g_ctx.buf[8 + s], st);
        if (e == cudaSuccess)
            e = cudaEventRecord(ev_run[s], st);
        trace.mark("kernels done, chunk " + std::to_string(j), st);
        if (e == cudaSuccess)
            e = peek_u32(reinterpret_cast<uint32_t *>(g_ctx.h_small + 4 * s), d_bytes, 4, st);
        if (e == cudaSuccess)
            e = cudaEventRecord(ev_size[s], st);
        return e;
    };

    uint64_t off = 0, issued = 0;
    std::vector<uint64_t> chunk_off(n_chunks); // where each chunk landed in the caller's buffer
    for (uint64_t j = 0; j < n_chunks; ++j) {
        while (issued < n_chunks && issued < j + (uint64_t)slots)
            CU(issue(issued++), "compress launch");
        const int s = (int)(j % slots);
        CU(cudaEventSynchronize(ev_size[s]), "compress");
        const uint64_t clen = g_ctx.h_small[4 * s];
        const uint32_t status = (uint32_t)g_ctx.h_small[4 * s + 1];
        if (status) {
            cudaDeviceSynchronize();
            return status_error(status);
        }
        if (off + clen > out_capacity) {
            cudaDeviceSynchronize();
            return fail_msg(SNAPPY_B200_ERR_CAPACITY, "output buffer too small for the compressed stream");
        }
        CU(cudaStreamWaitEvent(g_ctx.s_down, ev_run[s], 0), "stream wait");
        CU(cudaMemcpyAsync(dst + off, g_ctx.buf[4 + s], clen, cudaMemcpyDeviceToHost, g_ctx.s_down), "D2H copy");
        if (block_offsets) { // the chunk's offsets, chunk-relative for now (entry nb of chunk j = entry 0 of chunk j+1)
            const uint64_t lo = j * chunk, len = std::min(chunk, n_bytes - lo);
            CU(cudaMemcpyAsync(block_offsets + lo / kBlock, compress_chunk_offsets(g_ctx.buf[8 + s], len),
                               ((len + kBlock - 1) / kBlock + 1) * 8, cudaMemcpyDeviceToHost, g_ctx.s_down),
               "D2H copy");
        }
        chunk_off[j] = off;
        CU(cudaEventRecord(ev_down[s], g_ctx.s_down), "event record");
        trace.mark("download done, chunk " + std::to_string(j) + " (" + std::to_string(clen >> 20) + " MiB)", g_ctx.s_down);
        off += clen;
    }
    CU(cudaStreamSynchronize(g_ctx.s_down), "D2H copy");
    trace.dump();
    if (block_offsets) {
        for (uint64_t j = 0; j < n_chunks; ++j) {
            const uint64_t b0 = j * chunk / kBlock, b1 = std::min((j + 1) * chunk, align_up(n_bytes, kBlock)) / kBlock;
            for (uint64_t b = b0; b < b1; ++b)
                block_offsets[b] += chunk_off[j];
        }
        block_offsets[(n_bytes + kBlock - 1) / kBlock] = off;
    }
    *out_bytes = off;
    return SNAPPY_B200_OK;
}

extern "C" {

int snappy_b200_compress_host_range(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                                    uint64_t *out_bytes, uint64_t *block_offsets, uint64_t varint_value)
{
    clear_error();
    if (!out_bytes || (n_bytes && (!in || !out)))
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (check_mode(mode) != SNAPPY_B200_OK)
        return SNAPPY_B200_ERR_ARG;
    *out_bytes = 0;
    if (n_bytes == 0)
        return SNAPPY_B200_OK; // reference: an empty input gives an empty stream
    if (env_devices() > 1 && n_bytes >= kMultiMin)
        return snappy_b200_compress_host_multi_range(in, n_bytes, mode, out, out_capacity, out_bytes, block_offsets,
                                                     env_devices(), varint_value);
    return compress_host_chunks(in, n_bytes, mode, false, false, out, out_capacity, out_bytes, block_offsets,
                                varint_value);
}

} // extern "C"

namespace sb200 {
// One range of a longer input as framed chunks, for callers that stream (the FILE* layer): n_bytes must be whole
// 64 KiB blocks except for the last range; `identifier`: the range opens the stream.
int frame_compress_host_range(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                              uint64_t *out_bytes, bool identifier)
{
    if (!out_bytes || !out || (n_bytes && !in))
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (check_mode(mode) != SNAPPY_B200_OK)
        return SNAPPY_B200_ERR_ARG;
    *out_bytes = 0;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev < 1) { // no CPU path, also for the empty input
        (void)cudaGetLastError();
        return fail_msg(SNAPPY_B200_ERR_CUDA, "no CUDA device");
    }
    if (n_bytes == 0) {
        if (!identifier)
            return SNAPPY_B200_OK;
        if (out_capacity < sizeof kStreamId)
            return fail_msg(SNAPPY_B200_ERR_CAPACITY, "output buffer too small for the stream identifier");
        memcpy(out, kStreamId, sizeof kStreamId);
        *out_bytes = sizeof kStreamId;
        return SNAPPY_B200_OK;
    }
    return compress_host_chunks(in, n_bytes, mode, true, identifier, out, out_capacity, out_bytes, nullptr, 0);
}
} // namespace sb200

extern "C" {

int snappy_b200_frame_compress_host(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                                    uint64_t *out_bytes)
{
    clear_error();
    return frame_compress_host_range(in, n_bytes, mode, out, out_capacity, out_bytes, true);
}

int snappy_b200_uncompressed_length(const void *stream, uint64_t stream_bytes, uint64_t *n_bytes)
{
    clear_error();
    if (!n_bytes)
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    *n_bytes = 0;
    if (stream_bytes == 0)
        return SNAPPY_B200_OK; // the reference's empty stream
    if (!host_varint_decode(static_cast<const uint8_t *>(stream), stream_bytes, n_bytes))
        return fail_msg(SNAPPY_B200_ERR_CORRUPT, "bad varint preamble");
    return SNAPPY_B200_OK;
}

static int decompress_host_framed(const void *stream, uint64_t stream_bytes, void *out, uint64_t out_capacity,
                                  uint64_t *out_bytes)
{
    clear_error();
    HostCtx &g_ctx = current_ctx();
    if (!out_bytes || (stream_bytes && !stream))
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    *out_bytes = 0;
    if (stream_bytes == 0)
        return SNAPPY_B200_OK;
    uint64_t total = 0;
    const unsigned hdr = host_varint_decode(static_cast<const uint8_t *>(stream), stream_bytes, &total);
    if (!hdr)
        return fail_msg(SNAPPY_B200_ERR_CORRUPT, "bad varint preamble");
    if (total > out_capacity)
        return fail_msg(SNAPPY_B200_ERR_CAPACITY, "output buffer too small for the decompressed data");
    if (total == 0)
        return stream_bytes == hdr ? SNAPPY_B200_OK
                                   : fail_msg(SNAPPY_B200_ERR_CORRUPT, "trailing bytes after an empty stream");
    if (!out)
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (longer_than_any_encoding(stream_bytes, hdr, total))
        return fail_msg(SNAPPY_B200_ERR_CORRUPT, "stream is longer than any encoding of its declared length");
    if (decode_devices() > 1 && total >= kMultiMin)
        return snappy_b200_decompress_host_multi(stream, stream_bytes, out, out_capacity, out_bytes, decode_devices());

    std::lock_guard<std::mutex> lock(g_ctx.mu);
    CU(g_ctx.init(), "context init");
    const uint64_t nb = (total + kBlock - 1) / kBlock;
    // pieces grow from 1/8 of the full size: the first download starts early, the later pieces are
    // large enough to amortise K0's fixed cost and to fill the GPU.  All the small read-backs of
    // the loop go through peek_u32 so that they never queue behind a download.
    const uint64_t piece = kUploadPiece;
    std::vector<uint64_t> piece_end;
    const uint64_t growth = std::max<uint64_t>(env_mib("SNAPPY_B200_PIECE_GROWTH", 2) >> 20, 1);
    for (uint64_t at = 0, len = std::min(piece, env_mib("SNAPPY_B200_PIECE_START_MIB", std::max<uint64_t>(piece >> 23, 1)));
         at < stream_bytes; len = std::min(len * growth, piece)) {
        at = std::min(at + len, stream_bytes);
        piece_end.push_back(at);
    }
    const uint64_t n_pieces = piece_end.size();
    // a K0 region is at most one piece plus the carried-over incomplete block
    const uint64_t region_cap = piece_region_cap(stream_bytes, piece);
    // buffers: 0 stream, 1 output, 2/3 K0 workspace (alternating), 4/5 block offsets, 6 small
    CU(g_ctx.need(0, stream_bytes + 64), "cudaMalloc");
    CU(g_ctx.need(1, total), "cudaMalloc");
    for (int s = 0; s < 2; ++s) {
        CU(g_ctx.need(2 + s, index_workspace_bytes(region_cap)), "cudaMalloc");
        CU(g_ctx.need(4 + s, (nb + 2) * 8), "cudaMalloc");
    }
    CU(g_ctx.need(6, 256), "cudaMalloc");
    uint8_t *d_stream = static_cast<uint8_t *>(g_ctx.buf[0]);
    uint8_t *d_out = static_cast<uint8_t *>(g_ctx.buf[1]);
    uint32_t *d_status = static_cast<uint32_t *>(g_ctx.buf[6]);
    const uint8_t *src = static_cast<const uint8_t *>(stream);
    uint8_t *dst = static_cast<uint8_t *>(out);
    cudaEvent_t *ev_up = g_ctx.ev; // 8, round robin
    PieceResources r;
    for (int s = 0; s < 2; ++s) {
        r.ws[s] = g_ctx.buf[2 + s];
        r.offs[s] = static_cast<uint64_t *>(g_ctx.buf[4 + s]);
        r.ev_k0[s] = g_ctx.ev[8 + s];
        r.ev_dec[s] = g_ctx.ev[10 + s];
    }
    r.s_run = g_ctx.s_run, r.s_dec = g_ctx.s_dec, r.h_small = g_ctx.h_small;

    CU(cudaMemsetAsync(d_status, 0, 4, g_ctx.s_run), "memset");
    Trace trace;
    trace.start(g_ctx.s_run);
    uint64_t issued = 0; // pieces whose upload has been enqueued (at most 8 ahead of the consumer)
    auto issue_upload = [&]() -> cudaError_t {
        const uint64_t q = issued++;
        const uint64_t lo = q ? piece_end[q - 1] : 0, len = piece_end[q] - lo;
        cudaError_t e = cudaMemcpyAsync(d_stream + lo, src + lo, len, cudaMemcpyHostToDevice, g_ctx.s_up);
        if (e == cudaSuccess)
            e = cudaEventRecord(ev_up[q & 7], g_ctx.s_up);
        trace.mark("upload done, piece " + std::to_string(q) + " (" + std::to_string(len >> 20) + " MiB)", g_ctx.s_up);
        return e;
    };
    while (issued < n_pieces && issued < 8)
        CU(issue_upload(), "H2D copy");

    PieceHooks hooks;
    hooks.before_piece = [&](uint64_t p, cudaStream_t s_run) -> cudaError_t {
        cudaError_t e = cudaStreamWaitEvent(s_run, ev_up[p & 7], 0);
        if (e == cudaSuccess && issued < n_pieces) // keep the upload queue full (the event slot is free again)
            e = issue_upload();
        return e;
    };
    hooks.after_decode = [&](uint64_t first, uint64_t bytes, cudaEvent_t done) -> cudaError_t {
        cudaError_t e = cudaStreamWaitEvent(g_ctx.s_down, done, 0);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(dst + first, d_out + first, bytes, cudaMemcpyDeviceToHost, g_ctx.s_down);
        trace.mark("download done, " + std::to_string(bytes >> 20) + " MiB", g_ctx.s_down);
        return e;
    };
    hooks.trace = &trace;
    const int rc = decode_pieces(d_stream, stream_bytes, hdr, total, d_out, nullptr, d_status, piece_end, region_cap, r,
                                 hooks);
    if (rc != SNAPPY_B200_OK)
        return rc;
    CU(cudaStreamSynchronize(g_ctx.s_dec), "decode");
    CU(peek_u32(reinterpret_cast<uint32_t *>(g_ctx.h_small + 1), d_status, 1, g_ctx.s_run), "read-back");
    CU(cudaStreamSynchronize(g_ctx.s_run), "decode");
    CU(cudaStreamSynchronize(g_ctx.s_down), "D2H copy");
    trace.dump();
    const uint32_t status = (uint32_t)g_ctx.h_small[1];
    if (status)
        return status_error(status);
    *out_bytes = total;
    return SNAPPY_B200_OK;
}

} // extern "C"

namespace sb200 {
// Valid raw Snappy that is not framed in 64 KiB blocks (straddling elements, copies into earlier blocks, blocks
// longer than the block decoders take): decoded like the reference does, one element after the other
// (k_decode_sequential).  The caller has checked the arguments and that the output fits.
int decompress_host_general(const void *stream, uint64_t stream_bytes, void *out, uint64_t *out_bytes)
{
    HostCtx &g_ctx = current_ctx();
    uint64_t total = 0;
    const unsigned hdr = host_varint_decode(static_cast<const uint8_t *>(stream), stream_bytes, &total);
    std::lock_guard<std::mutex> lock(g_ctx.mu);
    CU(g_ctx.init(), "context init");
    CU(g_ctx.need(0, stream_bytes + 64), "cudaMalloc");
    CU(g_ctx.need(1, total), "cudaMalloc");
    CU(g_ctx.need(6, 256), "cudaMalloc");
    uint32_t *d_status = static_cast<uint32_t *>(g_ctx.buf[6]);
    uint64_t launches = 0;
    CU(cudaMemcpyAsync(g_ctx.buf[0], stream, stream_bytes, cudaMemcpyHostToDevice, g_ctx.s_run), "H2D copy");
    CU(cudaMemsetAsync(d_status, 0, 4, g_ctx.s_run), "memset");
    CU(launch_decode_sequential(static_cast<const uint8_t *>(g_ctx.buf[0]), stream_bytes, hdr, total,
                                static_cast<uint8_t *>(g_ctx.buf[1]), d_status, g_ctx.s_run, &launches),
       "decode launch");
    add_launches(launches);
    CU(cudaMemcpyAsync(out, g_ctx.buf[1], total, cudaMemcpyDeviceToHost, g_ctx.s_run), "D2H copy");
    CU(peek_u32(reinterpret_cast<uint32_t *>(g_ctx.h_small + 1), d_status, 1, g_ctx.s_run), "read-back");
    CU(cudaStreamSynchronize(g_ctx.s_run), "decode");
    const uint32_t status = (uint32_t)g_ctx.h_small[1];
    if (status)
        return status_error(status);
    *out_bytes = total;
    return SNAPPY_B200_OK;
}
} // namespace sb200

extern "C" {

int snappy_b200_decompress_host(const void *stream, uint64_t stream_bytes, void *out, uint64_t out_capacity,
                                uint64_t *out_bytes)
{
    const int rc = decompress_host_framed(stream, stream_bytes, out, out_capacity, out_bytes);
    if (rc != SNAPPY_B200_ERR_FRAMING)
        return rc;
    clear_error();
    return decompress_host_general(stream, stream_bytes, out, out_bytes); // (all arguments were checked above)
}

// ---- FILE* -> FILE* decompression (what snappy_decompress, src/snappy_decompression.c:345-363, becomes).
// The reference reads the stream through a 128 KiB window and holds the whole output in memory until one
// final fwrite (:349, :359).  Here the whole stream and the whole output live in DEVICE memory; the host
// only ever holds a ring of three page-locked chunks (32 MiB each, kept for the life of the process):
//   fread chunk -> H2D   (the upload of chunk i overlaps the fread of chunk i+1)
//   K0 + block decode on the device-resident stream (or the general decoder for unframed streams)
//   D2H chunk -> fwrite  (the download of chunk i+1 overlaps the fwrite of chunk i)
// Returns 1 when the stream cannot be handled this way (not seekable, or too large for the device): the
// caller then falls back to whole-buffer decoding.
int snappy_b200_decompress_file(FILE *in, FILE *out)
{
    clear_error();
    if (!in || !out)
        return fail_msg(SNAPPY_B200_ERR_IO, "null FILE*");
    const long at = ftell(in);
    if (at < 0 || fseek(in, 0, SEEK_END) != 0)
        return 1;
    const long end = ftell(in);
    if (end < at || fseek(in, at, SEEK_SET) != 0)
        return 1;
    const uint64_t L = (uint64_t)(end - at);
    if (L == 0)
        return SNAPPY_B200_OK; // the reference's empty stream
    uint8_t head[16];
    const size_t got_head = fread(head, 1, std::min<uint64_t>(L, sizeof head), in);
    if (fseek(in, at, SEEK_SET) != 0)
        return fail_msg(SNAPPY_B200_ERR_IO, "seek failed");
    uint64_t total = 0;
    const unsigned hdr = host_varint_decode(head, got_head, &total);
    if (!hdr)
        return fail_msg(SNAPPY_B200_ERR_CORRUPT, "bad varint preamble");
    if (total == 0)
        return L == hdr ? SNAPPY_B200_OK : fail_msg(SNAPPY_B200_ERR_CORRUPT, "trailing bytes after an empty stream");
    if (longer_than_any_encoding(L, hdr, total))
        return fail_msg(SNAPPY_B200_ERR_CORRUPT, "stream is longer than any encoding of its declared length");
    if (total >= (1ull << 40))
        return 1;
    HostCtx &g_ctx = current_ctx();
    std::lock_guard<std::mutex> lock(g_ctx.mu);
    CU(g_ctx.init(), "context init");
    constexpr size_t kFileChunk = 32u << 20;
    const uint64_t nb = (total + kBlock - 1) / kBlock;
    if (g_ctx.need(0, L + 64) != cudaSuccess || g_ctx.need(1, total) != cudaSuccess ||
        g_ctx.need(2, index_workspace_bytes(L)) != cudaSuccess || g_ctx.need(4, (nb + 2) * 8) != cudaSuccess ||
        g_ctx.need(6, 256) != cudaSuccess) {
        (void)cudaGetLastError();
        return 1; // does not fit this device: the piecewise host path needs far less device memory
    }
    CU(g_ctx.need_file_ring(kFileChunk), "cudaHostAlloc");
    uint8_t *d_stream = static_cast<uint8_t *>(g_ctx.buf[0]);
    uint8_t *d_out = static_cast<uint8_t *>(g_ctx.buf[1]);
    uint64_t *d_offs = static_cast<uint64_t *>(g_ctx.buf[4]);
    uint32_t *d_status = static_cast<uint32_t *>(g_ctx.buf[6]);
    cudaEvent_t *ev = g_ctx.ev + 21; // three slots
    // ---- up
    uint64_t k = 0;
    for (uint64_t off = 0; off < L; off += kFileChunk, ++k) {
        const int slot = (int)(k % HostCtx::kFileSlots);
        const uint64_t len = std::min<uint64_t>(kFileChunk, L - off);
        if (k >= (uint64_t)HostCtx::kFileSlots)
            CU(cudaEventSynchronize(ev[slot]), "H2D copy");
        if (fread(g_ctx.h_file[slot], 1, len, in) != len) {
            cudaDeviceSynchronize();
            return fail_msg(SNAPPY_B200_ERR_IO, "reading the compressed stream failed");
        }
        CU(cudaMemcpyAsync(d_stream + off, g_ctx.h_file[slot], len, cudaMemcpyHostToDevice, g_ctx.s_run), "H2D copy");
        CU(cudaEventRecord(ev[slot], g_ctx.s_run), "event record");
    }
    // ---- decode
    uint64_t launches = 0;
    CU(cudaMemsetAsync(d_status, 0, 4, g_ctx.s_run), "memset");
    CU(run_index(d_stream, L, hdr, total, d_offs, d_status, g_ctx.buf[2], g_ctx.s_run, &launches, false, 0), "index launch");
    CU(launch_decode_seg(d_stream, hdr, d_offs, index_starts(g_ctx.buf[2], L), index_outoff(g_ctx.buf[2], L), nb, total,
                         d_out, d_status, 0, g_ctx.s_run, &launches),
       "decode launch");
    CU(peek_u32(reinterpret_cast<uint32_t *>(g_ctx.h_small + 1), d_status, 1, g_ctx.s_run), "read-back");
    CU(cudaStreamSynchronize(g_ctx.s_run), "decode");
    uint32_t status = (uint32_t)g_ctx.h_small[1];
    if (status & SNAPPY_B200_ST_FRAMING) { // valid raw Snappy, but not framed in 64 KiB blocks: the general decoder
        CU(cudaMemsetAsync(d_status, 0, 4, g_ctx.s_run), "memset");
        CU(launch_decode_sequential(d_stream, L, hdr, total, d_out, d_status, g_ctx.s_run, &launches), "decode launch");
        CU(peek_u32(reinterpret_cast<uint32_t *>(g_ctx.h_small + 1), d_status, 1, g_ctx.s_run), "read-back");
        CU(cudaStreamSynchronize(g_ctx.s_run), "decode");
        status = (uint32_t)g_ctx.h_small[1];
    }
    add_launches(launches);
    if (status)
        return status_error(status);
    // ---- down
    const uint64_t n_chunks = (total + kFileChunk - 1) / kFileChunk;
    auto issue_down = [&](uint64_t c) -> cudaError_t {
        const int slot = (int)(c % HostCtx::kFileSlots);
        const uint64_t off = c * kFileChunk, len = std::min<uint64_t>(kFileChunk, total - off);
        cudaError_t e = cudaMemcpyAsync(g_ctx.h_file[slot], d_out + off, len, cudaMemcpyDeviceToHost, g_ctx.s_down);
        if (e == cudaSuccess)
            e = cudaEventRecord(ev[slot], g_ctx.s_down);
        return e;
    };
    CU(issue_down(0), "D2H copy");
    if (n_chunks > 1)
        CU(issue_down(1), "D2H copy");
    for (uint64_t c = 0; c < n_chunks; ++c) {
        const int slot = (int)(c % HostCtx::kFileSlots);
        const uint64_t off = c * kFileChunk, len = std::min<uint64_t>(kFileChunk, total - off);
        CU(cudaEventSynchronize(ev[slot]), "D2H copy");
        if (c + 2 < n_chunks) // (its slot was written out two chunks ago)
            CU(issue_down(c + 2), "D2H copy");
        if (fwrite(g_ctx.h_file[slot], 1, len, out) != len) {
            cudaDeviceSynchronize();
            return fail_msg(SNAPPY_B200_ERR_IO, "short write of the output");
        }
    }
    return SNAPPY_B200_OK;
}

// ---- decode with the side index: no K0.  The stream goes up in pieces cut at block boundaries
// (growing like the index-less path's), every piece is decoded by the window decoder as soon as it
// has landed and downloaded while the next one is in flight.
static int decompress_host_indexed_blocks(const void *stream, uint64_t stream_bytes, const uint64_t *block_offsets,
                                          uint64_t n_blocks, void *out, uint64_t out_capacity, uint64_t *out_bytes)
{
    clear_error();
    HostCtx &g_ctx = current_ctx();
    if (!out_bytes || (stream_bytes && !stream) || !block_offsets)
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    *out_bytes = 0;
    if (stream_bytes == 0)
        return SNAPPY_B200_OK;
    uint64_t total = 0;
    const unsigned hdr = host_varint_decode(static_cast<const uint8_t *>(stream), stream_bytes, &total);
    if (!hdr)
        return fail_msg(SNAPPY_B200_ERR_CORRUPT, "bad varint preamble");
    if (total > out_capacity)
        return fail_msg(SNAPPY_B200_ERR_CAPACITY, "output buffer too small for the decompressed data");
    if (n_blocks != (total + kBlock - 1) / kBlock || n_blocks >= (1ull << 31))
        return fail_msg(SNAPPY_B200_ERR_ARG, "the index does not have one entry per 64 KiB block of the declared length");
    if (total == 0)
        return stream_bytes == hdr ? SNAPPY_B200_OK
                                   : fail_msg(SNAPPY_B200_ERR_CORRUPT, "trailing bytes after an empty stream");
    if (!out)
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (block_offsets[0] != hdr || block_offsets[n_blocks] != stream_bytes)
        return fail_msg(SNAPPY_B200_ERR_CORRUPT, "the index does not span the stream");
    for (uint64_t b = 0; b < n_blocks; ++b)
        if (block_offsets[b + 1] <= block_offsets[b])
            return fail_msg(SNAPPY_B200_ERR_CORRUPT, "the index is not increasing");
    for (uint64_t b = 0; b < n_blocks; ++b)
        if (block_offsets[b + 1] - block_offsets[b] > 2u * kBlock)
            return fail_msg(SNAPPY_B200_ERR_FRAMING, "a block is longer than the block decoders take (2 * 65536 stream bytes)");
    if (decode_devices() > 1 && total >= kMultiMin)
        return snappy_b200_decompress_host_indexed_multi(stream, stream_bytes, block_offsets, n_blocks, out, out_capacity,
                                                         out_bytes, decode_devices());

    std::lock_guard<std::mutex> lock(g_ctx.mu);
    CU(g_ctx.init(), "context init");
    CU(g_ctx.need(0, stream_bytes + 64), "cudaMalloc");
    CU(g_ctx.need(1, total), "cudaMalloc");
    CU(g_ctx.need(4, (n_blocks + 2) * 8), "cudaMalloc");
    CU(g_ctx.need(6, 256), "cudaMalloc");
    uint8_t *d_stream = static_cast<uint8_t *>(g_ctx.buf[0]);
    uint8_t *d_out = static_cast<uint8_t *>(g_ctx.buf[1]);
    uint64_t *d_offs = static_cast<uint64_t *>(g_ctx.buf[4]);
    uint32_t *d_status = static_cast<uint32_t *>(g_ctx.buf[6]);
    const uint8_t *src = static_cast<const uint8_t *>(stream);
    uint8_t *dst = static_cast<uint8_t *>(out);
    CU(cudaMemsetAsync(d_status, 0, 4, g_ctx.s_up), "memset");
    CU(cudaMemcpyAsync(d_offs, block_offsets, (n_blocks + 1) * 8, cudaMemcpyHostToDevice, g_ctx.s_up), "H2D copy");
    uint64_t launches = 0;
    const uint64_t piece = kUploadPiece;
    uint64_t b0 = 0, want = std::max<uint64_t>(piece / 8, 1 << 20);
    int k = 0;
    while (b0 < n_blocks) {
        // blocks [b0, b1): about `want` stream bytes
        uint64_t b1 = std::upper_bound(block_offsets + b0, block_offsets + n_blocks, block_offsets[b0] + want) - block_offsets;
        b1 = std::min(std::max(b1, b0 + 1), n_blocks);
        const uint64_t lo = b0 ? block_offsets[b0] : 0, hi = block_offsets[b1];
        cudaEvent_t ev_up = g_ctx.ev[k & 7], ev_dec = g_ctx.ev[8 + (k & 7)];
        CU(cudaMemcpyAsync(d_stream + lo, src + lo, hi - lo, cudaMemcpyHostToDevice, g_ctx.s_up), "H2D copy");
        CU(cudaEventRecord(ev_up, g_ctx.s_up), "event record");
        CU(cudaStreamWaitEvent(g_ctx.s_dec, ev_up, 0), "stream wait");
        const uint64_t out_lo = b0 * kBlock, out_n = std::min(total, b1 * (uint64_t)kBlock) - out_lo;
        CU(launch_decode(d_stream, d_offs + b0, b1 - b0, out_n, d_out + out_lo, d_status, g_ctx.s_dec, &launches),
           "decode launch");
        CU(cudaEventRecord(ev_dec, g_ctx.s_dec), "event record");
        CU(cudaStreamWaitEvent(g_ctx.s_down, ev_dec, 0), "stream wait");
        CU(cudaMemcpyAsync(dst + out_lo, d_out + out_lo, out_n, cudaMemcpyDeviceToHost, g_ctx.s_down), "D2H copy");
        b0 = b1;
        want = std::min(want * 2, piece);
        ++k;
    }
    add_launches(launches);
    CU(cudaStreamSynchronize(g_ctx.s_dec), "decode");
    CU(peek_u32(reinterpret_cast<uint32_t *>(g_ctx.h_small + 1), d_status, 1, g_ctx.s_dec), "read-back");
    CU(cudaStreamSynchronize(g_ctx.s_dec), "decode");
    CU(cudaStreamSynchronize(g_ctx.s_down), "D2H copy");
    const uint32_t status = (uint32_t)g_ctx.h_small[1];
    if (status)
        return status_error(status);
    *out_bytes = total;
    return SNAPPY_B200_OK;
}

int snappy_b200_decompress_host_indexed(const void *stream, uint64_t stream_bytes, const uint64_t *block_offsets,
                                        uint64_t n_blocks, void *out, uint64_t out_capacity, uint64_t *out_bytes)
{
    const int rc = decompress_host_indexed_blocks(stream, stream_bytes, block_offsets, n_blocks, out, out_capacity,
                                                  out_bytes);
    if (rc != SNAPPY_B200_ERR_FRAMING)
        return rc;
    clear_error();
    return decompress_host_general(stream, stream_bytes, out, out_bytes); // (all arguments were checked above)
}

// ---- framed streams: the chunk headers are walked on the host (the framing is the block index: no K0); the
// stream goes up in pieces cut at chunk boundaries, growing like the indexed path's, and every piece is decoded
// (k_frame_decode), checked (k_crc32c_chunks) and downloaded while the next one is in flight.
int snappy_b200_frame_uncompressed_length(const void *stream, uint64_t stream_bytes, uint64_t *n_bytes)
{
    clear_error();
    if (!n_bytes || (stream_bytes && !stream))
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    return frame_walk(static_cast<const uint8_t *>(stream), stream_bytes, true, nullptr, n_bytes);
}

int snappy_b200_frame_decompress_host(const void *stream, uint64_t stream_bytes, void *out, uint64_t out_capacity,
                                      uint64_t *out_bytes)
{
    clear_error();
    return frame_decompress_buffer(stream, stream_bytes, out, out_capacity, out_bytes, true);
}

} // extern "C"

namespace sb200 {
// A whole framed stream (opens_stream) or, for the FILE* layer, a run of whole chunks from inside one.
int frame_decompress_buffer(const void *stream, uint64_t stream_bytes, void *out, uint64_t out_capacity,
                            uint64_t *out_bytes, bool opens_stream)
{
    if (!out_bytes || (stream_bytes && !stream))
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    *out_bytes = 0;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev < 1) { // no CPU path, also for streams without data
        (void)cudaGetLastError();
        return fail_msg(SNAPPY_B200_ERR_CUDA, "no CUDA device");
    }
    std::vector<FrameChunk> chunks;
    uint64_t total = 0;
    const int rc = frame_walk(static_cast<const uint8_t *>(stream), stream_bytes, opens_stream, &chunks, &total);
    if (rc != SNAPPY_B200_OK)
        return rc;
    if (total > out_capacity)
        return fail_msg(SNAPPY_B200_ERR_CAPACITY, "output buffer too small for the decompressed data");
    if (total == 0) { // only empty data chunks (or none): each must be empty and carry the CRC of no bytes
        for (const FrameChunk &c : chunks) // (a malformed chunk takes precedence over a checksum, as on the device)
            if (c.in_len != 0)
                return fail_msg(SNAPPY_B200_ERR_CORRUPT, "framed stream: an empty chunk with a non-empty body");
        for (const FrameChunk &c : chunks)
            if (c.crc != 0xa282ead8u) // mask(CRC-32C of no bytes = 0)
                return fail_msg(SNAPPY_B200_ERR_CHECKSUM, "framed stream: a chunk's CRC-32C does not match its data");
        return SNAPPY_B200_OK;
    }
    if (!out)
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    HostCtx &g_ctx = current_ctx();
    std::lock_guard<std::mutex> lock(g_ctx.mu);
    CU(g_ctx.init(), "context init");
    const uint64_t nc = chunks.size();
    CU(g_ctx.need(0, stream_bytes + 64), "cudaMalloc");
    CU(g_ctx.need(1, total), "cudaMalloc");
    CU(g_ctx.need(4, nc * sizeof(FrameChunk)), "cudaMalloc");
    CU(g_ctx.need(6, 256), "cudaMalloc");
    uint8_t *d_stream = static_cast<uint8_t *>(g_ctx.buf[0]);
    uint8_t *d_out = static_cast<uint8_t *>(g_ctx.buf[1]);
    FrameChunk *d_chunks = static_cast<FrameChunk *>(g_ctx.buf[4]);
    uint32_t *d_status = static_cast<uint32_t *>(g_ctx.buf[6]);
    const uint8_t *src = static_cast<const uint8_t *>(stream);
    uint8_t *dst = static_cast<uint8_t *>(out);
    CU(cudaMemsetAsync(d_status, 0, 4, g_ctx.s_up), "memset");
    CU(cudaMemcpyAsync(d_chunks, chunks.data(), nc * sizeof(FrameChunk), cudaMemcpyHostToDevice, g_ctx.s_up),
       "H2D copy");
    uint64_t launches = 0;
    const uint64_t piece = kUploadPiece;
    uint64_t c0 = 0, lo = 0, want = std::max<uint64_t>(piece / 8, 1 << 20);
    int k = 0;
    while (c0 < nc) {
        // chunks [c0, c1): about `want` stream bytes; the last piece takes the rest of the stream
        uint64_t c1 = c0 + 1;
        while (c1 < nc && chunks[c1].in_off + chunks[c1].in_len - lo <= want)
            ++c1;
        const uint64_t hi = c1 == nc ? stream_bytes : chunks[c1 - 1].in_off + chunks[c1 - 1].in_len;
        cudaEvent_t ev_up = g_ctx.ev[k & 7], ev_dec = g_ctx.ev[8 + (k & 7)];
        CU(cudaMemcpyAsync(d_stream + lo, src + lo, hi - lo, cudaMemcpyHostToDevice, g_ctx.s_up), "H2D copy");
        CU(cudaEventRecord(ev_up, g_ctx.s_up), "event record");
        CU(cudaStreamWaitEvent(g_ctx.s_dec, ev_up, 0), "stream wait");
        CU(launch_frame_decode(d_stream, stream_bytes, d_chunks + c0, c1 - c0, d_out, d_status, g_ctx.s_dec, &launches),
           "decode launch");
        CU(launch_frame_check(d_out, d_chunks + c0, c1 - c0, d_status, g_ctx.s_dec, &launches), "checksum launch");
        CU(cudaEventRecord(ev_dec, g_ctx.s_dec), "event record");
        CU(cudaStreamWaitEvent(g_ctx.s_down, ev_dec, 0), "stream wait");
        const uint64_t out_lo = chunks[c0].out_off, out_hi = chunks[c1 - 1].out_off + chunks[c1 - 1].out_len;
        CU(cudaMemcpyAsync(dst + out_lo, d_out + out_lo, out_hi - out_lo, cudaMemcpyDeviceToHost, g_ctx.s_down),
           "D2H copy");
        c0 = c1, lo = hi;
        want = std::min(want * 2, piece);
        ++k;
    }
    add_launches(launches);
    CU(cudaStreamSynchronize(g_ctx.s_dec), "decode");
    CU(peek_u32(reinterpret_cast<uint32_t *>(g_ctx.h_small + 1), d_status, 1, g_ctx.s_dec), "read-back");
    CU(cudaStreamSynchronize(g_ctx.s_dec), "decode");
    CU(cudaStreamSynchronize(g_ctx.s_down), "D2H copy");
    const uint32_t status = (uint32_t)g_ctx.h_small[1];
    if (status)
        return status_error(status);
    *out_bytes = total;
    return SNAPPY_B200_OK;
}
} // namespace sb200

extern "C" {

// ---- device-level index-less decode (include/snappy_b200.h): the piecewise loop of the host path on a
// device-resident stream, with a library-owned second stream for the decode kernels.
// A device-resident stream is decoded as ONE piece: K0 has about 2 ms of latency-bound fixed cost
// per call (measured, profiles/), so splitting only pays when there is a transfer to hide.
// The workspace has room for two piece slots (K0 workspace + block offsets); one piece uses the first.
size_t snappy_b200_decompress_workspace_bytes(uint64_t stream_bytes, uint64_t total_out)
{
    const uint64_t nb = (total_out + kBlock - 1) / kBlock;
    const size_t per_slot = align_up(index_workspace_bytes(stream_bytes), 256) + align_up((nb + 2) * 8, 256);
    return 2 * per_slot + 256;
}

int snappy_b200_decompress_device(const uint8_t *d_stream, uint64_t stream_bytes, uint64_t body_offset,
                                  uint64_t total_out, uint8_t *d_out, uint64_t *d_block_offsets, uint32_t *d_status,
                                  void *d_workspace, size_t workspace_bytes, void *stream)
{
    clear_error();
    HostCtx &g_ctx = current_ctx();
    if (!d_stream || !d_status || !d_workspace || (!d_out && total_out))
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (body_offset > stream_bytes || stream_bytes >= (1ull << 40))
        return fail_msg(SNAPPY_B200_ERR_ARG, "bad stream size / body offset");
    if (workspace_bytes < snappy_b200_decompress_workspace_bytes(stream_bytes, total_out))
        return fail_msg(SNAPPY_B200_ERR_ARG, "workspace too small (see snappy_b200_decompress_workspace_bytes)");
    if (total_out == 0)
        return stream_bytes == body_offset ? SNAPPY_B200_OK
                                           : fail_msg(SNAPPY_B200_ERR_CORRUPT, "trailing bytes after an empty stream");
    std::lock_guard<std::mutex> lock(g_ctx.mu);
    CU(g_ctx.init(), "context init");
    const uint64_t nb = (total_out + kBlock - 1) / kBlock;
    const size_t ws_slot = align_up(index_workspace_bytes(stream_bytes), 256);
    const size_t off_slot = align_up((nb + 2) * 8, 256);
    uint8_t *w = static_cast<uint8_t *>(d_workspace);
    PieceResources r;
    for (int s = 0; s < 2; ++s) {
        r.ws[s] = w + s * (ws_slot + off_slot);
        r.offs[s] = reinterpret_cast<uint64_t *>(w + s * (ws_slot + off_slot) + ws_slot);
        r.ev_k0[s] = g_ctx.ev[16 + s];
        r.ev_dec[s] = g_ctx.ev[18 + s];
    }
    r.s_run = static_cast<cudaStream_t>(stream);
    r.s_dec = g_ctx.s_dec;
    r.h_small = g_ctx.h_small + 8;
    PieceHooks hooks; // nothing to wait for, nothing to download
    const std::vector<uint64_t> piece_end = {stream_bytes}; // one piece, the whole stream
    const int rc = decode_pieces(d_stream, stream_bytes, body_offset, total_out, d_out, d_block_offsets, d_status,
                                 piece_end, stream_bytes, r, hooks);
    if (rc != SNAPPY_B200_OK)
        return rc;
    // join: work the caller enqueues next on `stream` sees the decoded output
    CU(cudaEventRecord(g_ctx.ev[20], g_ctx.s_dec), "event record");
    CU(cudaStreamWaitEvent(r.s_run, g_ctx.ev[20], 0), "stream wait");
    return SNAPPY_B200_OK;
}

void *snappy_b200_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    return p;
}

void snappy_b200_host_free(void *p)
{
    if (p)
        cudaFreeHost(p);
}

void snappy_b200_release(void)
{
    int keep = 0;
    const bool have = cudaGetDevice(&keep) == cudaSuccess;
    for (int d = 0; d < kMaxDevices; ++d) {
        HostCtx &c = g_ctx_pool[d];
        std::lock_guard<std::mutex> lock(c.mu);
        if (c.device < 0)
            continue;
        if (cudaSetDevice(c.device) == cudaSuccess)
            c.release();
    }
    if (have)
        cudaSetDevice(keep);
    (void)cudaGetLastError();
}

} // extern "C"
