// multi_device.cu -- the host-buffer API over several GPUs of one box (SURVEY.md 8e).
//
// reference: blocks are compressed and decoded independently (src/snappy_compression.c:419-425 resets the
// table and the buffers per block), so contiguous block ranges go to different devices and nothing crosses
// between them: no collective, no peer copy.  The only cross-device datum is the compressed size of every
// partition (an exclusive scan on the host places the partitions in the one output stream).
//
//   compress    phase 1: every device uploads its block range chunk by chunk and compresses it into its own
//               memory; phase 2 (after the host scan of the sizes): every device downloads straight to the
//               final offsets of the caller's buffer.  The stream is byte-identical to the one-device stream.
//   decompress  with the side index the block ranges are dealt out directly; without it device 0 first finds
//               the block boundaries of the whole stream (K0), then the same indexed path runs.
// One worker thread per device; every device has its own arena (buffers + stream) behind its own lock.
#include <algorithm>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"

namespace sb200 {
int decompress_host_general(const void *stream, uint64_t stream_bytes, void *out, uint64_t *out_bytes);
int fail_msg(int code, const char *msg);
int cuda_fail_msg(cudaError_t e, const char *what);
int status_error(uint32_t st);
void clear_error();
void add_launches(uint64_t n);
size_t compress_workspace_bytes_internal(uint64_t n_bytes, bool framed);
cudaError_t compress_chunk(const uint8_t *, uint64_t, uint64_t, int, bool, bool, uint8_t *, uint64_t, uint64_t *, uint32_t *, void *,
                           cudaStream_t);
const uint64_t *compress_chunk_offsets(void *, uint64_t);
size_t index_workspace_bytes(uint64_t);
cudaError_t run_index(const uint8_t *, uint64_t, uint64_t, uint64_t, uint64_t *, uint32_t *, void *, cudaStream_t,
                      uint64_t *, bool, uint64_t, uint32_t fixed_rounds = 0);
cudaError_t launch_decode(const uint8_t *, const uint64_t *, uint64_t, uint64_t, uint8_t *, uint32_t *, cudaStream_t,
                          uint64_t *);

namespace {

constexpr uint64_t kChunk = 256ull << 20; // input bytes per compress chunk / output bytes per decode chunk
constexpr int kMaxDev = 64;

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline uint64_t max_compressed(uint64_t n) { return n ? 10 + n + ((n + kBlock - 1) / kBlock) * 1010 : 0; }

struct Arena {
    std::mutex mu;
    void *buf[5] = {};
    size_t cap[5] = {};
    cudaStream_t st = nullptr;
    uint64_t *h_small = nullptr; // pinned
    cudaError_t need(int i, size_t bytes)
    {
        bytes = align_up(bytes + 256, 1 << 20);
        if (cap[i] >= bytes)
            return cudaSuccess;
        if (buf[i])
            cudaFree(buf[i]);
        buf[i] = nullptr, cap[i] = 0;
        const cudaError_t e = cudaMalloc(&buf[i], bytes);
        if (e == cudaSuccess)
            cap[i] = bytes;
        return e;
    }
    cudaError_t init()
    {
        cudaError_t e = cudaSuccess;
        if (!st)
            e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
        if (e == cudaSuccess && !h_small)
            e = cudaHostAlloc(reinterpret_cast<void **>(&h_small), 256, cudaHostAllocDefault);
        return e;
    }
};
Arena g_arena[kMaxDev];

struct Result {
    int rc = SNAPPY_B200_OK;
    cudaError_t cuda = cudaSuccess;
    const char *what = "";
    uint32_t status = 0;
};

int finish(const std::vector<Result> &res)
{
    for (const Result &r : res) {
        if (r.cuda != cudaSuccess)
            return cuda_fail_msg(r.cuda, r.what);
        if (r.status)
            return status_error(r.status);
        if (r.rc != SNAPPY_B200_OK)
            return fail_msg(r.rc, r.what);
    }
    return SNAPPY_B200_OK;
}

#define W(call, msg)                                                                                                   \
    do {                                                                                                               \
        const cudaError_t e__ = (call);                                                                                \
        if (e__ != cudaSuccess) {                                                                                      \
            r.cuda = e__, r.what = msg;                                                                                \
            return;                                                                                                    \
        }                                                                                                              \
    } while (0)

int usable_devices(int wanted)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return std::max(0, std::min(std::min(n, kMaxDev), wanted));
}

template <class F> void run_workers(int G, F f)
{
    std::vector<std::thread> th;
    for (int g = 1; g < G; ++g)
        th.emplace_back(f, g);
    f(0);
    for (auto &t : th)
        t.join();
}

} // namespace
} // namespace sb200

using namespace sb200;

extern "C" {

int snappy_b200_compress_host_multi(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                                    uint64_t *out_bytes, uint64_t *block_offsets, int n_devices)
{
    return snappy_b200_compress_host_multi_range(in, n_bytes, mode, out, out_capacity, out_bytes, block_offsets, n_devices,
                                                 n_bytes);
}

int snappy_b200_compress_host_multi_range(const void *in, uint64_t n_bytes, int mode, void *out, uint64_t out_capacity,
                                          uint64_t *out_bytes, uint64_t *block_offsets, int n_devices,
                                          uint64_t varint_value)
{
    clear_error();
    if (!out_bytes || (n_bytes && (!in || !out)))
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    if (mode != SNAPPY_B200_MODE_HASH && mode != SNAPPY_B200_MODE_BST)
        return fail_msg(SNAPPY_B200_ERR_ARG, "unknown mode");
    *out_bytes = 0;
    if (n_bytes == 0)
        return SNAPPY_B200_OK;
    const uint64_t nb = (n_bytes + kBlock - 1) / kBlock;
    const int G = (int)std::min<uint64_t>(usable_devices(n_devices), nb);
    if (G < 1)
        return fail_msg(SNAPPY_B200_ERR_CUDA, "no usable CUDA device");
    int home = 0;
    cudaGetDevice(&home);
    const uint8_t *src = static_cast<const uint8_t *>(in);
    uint8_t *dst = static_cast<uint8_t *>(out);
    struct Part {
        uint64_t b0, b1;                     // block range
        std::vector<uint64_t> csize, cdev;   // per chunk: compressed bytes, offset inside the device output buffer
        uint64_t total = 0, base = 0;        // compressed bytes of the partition, its offset in the stream
    };
    std::vector<Part> part(G);
    std::vector<Result> res(G);
    for (int g = 0; g < G; ++g)
        part[g].b0 = nb * g / G, part[g].b1 = nb * (g + 1) / G;

    for (int g = 0; g < G; ++g)
        g_arena[g].mu.lock(); // (always in device order: no deadlock between concurrent calls)
    // ---- phase 1: upload + compress, the compressed chunks stay on the device
    run_workers(G, [&](int g) {
        Result &r = res[g];
        Part &p = part[g];
        W(cudaSetDevice(g), "cudaSetDevice");
        Arena &a = g_arena[g];
        const uint64_t lo = p.b0 * kBlock, hi = std::min(n_bytes, p.b1 * kBlock);
        const uint64_t chunk = std::min<uint64_t>(kChunk, align_up(hi - lo, kBlock));
        const uint64_t n_chunks = (hi - lo + chunk - 1) / chunk;
        W(a.init(), "arena init");
        W(a.need(0, 2 * chunk), "cudaMalloc");                                            // two input slots
        W(a.need(1, max_compressed(hi - lo) + 32 * n_chunks + 64), "cudaMalloc");        // all compressed chunks
        W(a.need(2, compress_workspace_bytes_internal(chunk, false)), "cudaMalloc");
        W(a.need(3, 256), "cudaMalloc");
        uint8_t *d_in = static_cast<uint8_t *>(a.buf[0]);
        uint8_t *d_out = static_cast<uint8_t *>(a.buf[1]);
        uint64_t *d_small = static_cast<uint64_t *>(a.buf[3]);
        uint64_t doff = 0;
        for (uint64_t c = 0; c < n_chunks; ++c) {
            const uint64_t clo = lo + c * chunk, len = std::min(chunk, hi - clo);
            uint8_t *slot = d_in + (c & 1) * chunk;
            W(cudaMemcpyAsync(slot, src + clo, len, cudaMemcpyHostToDevice, a.st), "H2D copy");
            W(cudaMemsetAsync(d_small, 0, 16, a.st), "memset");
            W(compress_chunk(slot, len, (g == 0 && c == 0) ? varint_value : 0, mode, false, false, d_out + doff, max_compressed(len), d_small,
                             reinterpret_cast<uint32_t *>(d_small + 1), a.buf[2], a.st),
              "compress launch");
            W(cudaMemcpyAsync(a.h_small, d_small, 16, cudaMemcpyDeviceToHost, a.st), "read-back");
            if (block_offsets) // chunk-relative for now (one entry per block: neighbours never write the same word)
                W(cudaMemcpyAsync(block_offsets + clo / kBlock, compress_chunk_offsets(a.buf[2], len),
                                  ((len + kBlock - 1) / kBlock) * 8, cudaMemcpyDeviceToHost, a.st),
                  "D2H copy");
            W(cudaStreamSynchronize(a.st), "compress");
            if ((uint32_t)a.h_small[1]) {
                r.status = (uint32_t)a.h_small[1];
                return;
            }
            p.csize.push_back(a.h_small[0]);
            p.cdev.push_back(doff);
            p.total += a.h_small[0];
            doff = align_up(doff + a.h_small[0], 16);
        }
    });
    int rc = finish(res);
    // ---- the scan of the partition sizes
    uint64_t off = 0;
    for (int g = 0; g < G; ++g) {
        part[g].base = off;
        off += part[g].total;
    }
    if (rc == SNAPPY_B200_OK && off > out_capacity)
        rc = fail_msg(SNAPPY_B200_ERR_CAPACITY, "output buffer too small for the compressed stream");
    // ---- phase 2: every device downloads to the final offsets
    if (rc == SNAPPY_B200_OK) {
        run_workers(G, [&](int g) {
            Result &r = res[g];
            Part &p = part[g];
            W(cudaSetDevice(g), "cudaSetDevice");
            Arena &a = g_arena[g];
            const uint8_t *d_out = static_cast<const uint8_t *>(a.buf[1]);
            uint64_t at = p.base;
            const uint64_t lo = p.b0 * kBlock, hi = std::min(n_bytes, p.b1 * kBlock);
            const uint64_t chunk = std::min<uint64_t>(kChunk, align_up(hi - lo, kBlock));
            for (size_t c = 0; c < p.csize.size(); ++c) {
                W(cudaMemcpyAsync(dst + at, d_out + p.cdev[c], p.csize[c], cudaMemcpyDeviceToHost, a.st), "D2H copy");
                if (block_offsets) { // rebase this chunk's offsets (entries [first, last)); the host owns them by now
                    const uint64_t first = (lo + c * chunk) / kBlock;
                    const uint64_t last = std::min<uint64_t>(p.b1, first + chunk / kBlock);
                    for (uint64_t b = first; b < last; ++b)
                        block_offsets[b] += at;
                }
                at += p.csize[c];
            }
            W(cudaStreamSynchronize(a.st), "D2H copy");
        });
        rc = finish(res);
    }
    for (int g = 0; g < G; ++g)
        g_arena[g].mu.unlock();
    cudaSetDevice(home);
    if (rc != SNAPPY_B200_OK)
        return rc;
    if (block_offsets)
        block_offsets[nb] = off;
    *out_bytes = off;
    return SNAPPY_B200_OK;
}

static int decompress_host_indexed_multi_blocks(const void *stream, uint64_t stream_bytes, const uint64_t *block_offsets,
                                                uint64_t n_blocks, void *out, uint64_t out_capacity, uint64_t *out_bytes,
                                                int n_devices)
{
    clear_error();
    if (!out_bytes || (stream_bytes && !stream) || !block_offsets)
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    *out_bytes = 0;
    if (stream_bytes == 0)
        return SNAPPY_B200_OK;
    uint64_t total = 0;
    unsigned hdr = 0;
    {
        const uint8_t *p = static_cast<const uint8_t *>(stream);
        unsigned shift = 0;
        for (unsigned k = 0; k < stream_bytes && k < 10; ++k) {
            total |= (uint64_t)(p[k] & 0x7fu) << shift;
            shift += 7;
            if (!(p[k] & 0x80u)) {
                hdr = k + 1;
                break;
            }
        }
    }
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
    const int G = (int)std::min<uint64_t>(usable_devices(n_devices), n_blocks);
    if (G < 1)
        return fail_msg(SNAPPY_B200_ERR_CUDA, "no usable CUDA device");
    int home = 0;
    cudaGetDevice(&home);
    const uint8_t *src = static_cast<const uint8_t *>(stream);
    uint8_t *dst = static_cast<uint8_t *>(out);
    std::vector<Result> res(G);
    run_workers(G, [&](int g) {
        Result &r = res[g];
        W(cudaSetDevice(g), "cudaSetDevice");
        Arena &a = g_arena[g];
        std::lock_guard<std::mutex> lock(a.mu);
        W(a.init(), "arena init");
        const uint64_t b0 = n_blocks * g / G, b1 = n_blocks * (g + 1) / G;
        const uint64_t per = kChunk / kBlock; // blocks per chunk
        std::vector<uint64_t> rel(per + 1);
        uint64_t launches = 0;
        W(a.need(3, 256), "cudaMalloc");
        uint32_t *d_status = static_cast<uint32_t *>(a.buf[3]);
        W(cudaMemsetAsync(d_status, 0, 4, a.st), "memset");
        for (uint64_t c0 = b0; c0 < b1; c0 += per) {
            const uint64_t c1 = std::min(b1, c0 + per), k = c1 - c0;
            const uint64_t s0 = block_offsets[c0], s1 = block_offsets[c1];
            const uint64_t out_lo = c0 * kBlock, out_n = std::min(total, c1 * kBlock) - out_lo;
            W(a.need(0, s1 - s0 + 64), "cudaMalloc");
            W(a.need(1, out_n), "cudaMalloc");
            W(a.need(2, (per + 2) * 8), "cudaMalloc");
            W(cudaStreamSynchronize(a.st), "decode"); // (rel[] and the buffers of the chunk before are free again)
            for (uint64_t i = 0; i <= k; ++i)
                rel[i] = block_offsets[c0 + i] - s0;
            W(cudaMemcpyAsync(a.buf[0], src + s0, s1 - s0, cudaMemcpyHostToDevice, a.st), "H2D copy");
            W(cudaMemcpyAsync(a.buf[2], rel.data(), (k + 1) * 8, cudaMemcpyHostToDevice, a.st), "H2D copy");
            W(launch_decode(static_cast<const uint8_t *>(a.buf[0]), static_cast<const uint64_t *>(a.buf[2]), k, out_n,
                            static_cast<uint8_t *>(a.buf[1]), d_status, a.st, &launches),
              "decode launch");
            W(cudaMemcpyAsync(dst + out_lo, a.buf[1], out_n, cudaMemcpyDeviceToHost, a.st), "D2H copy");
        }
        W(cudaMemcpyAsync(a.h_small, d_status, 4, cudaMemcpyDeviceToHost, a.st), "read-back");
        W(cudaStreamSynchronize(a.st), "decode");
        r.status = (uint32_t)a.h_small[0];
        add_launches(launches);
    });
    cudaSetDevice(home);
    const int rc = finish(res);
    if (rc != SNAPPY_B200_OK)
        return rc;
    *out_bytes = total;
    return SNAPPY_B200_OK;
}

int snappy_b200_decompress_host_indexed_multi(const void *stream, uint64_t stream_bytes, const uint64_t *block_offsets,
                                              uint64_t n_blocks, void *out, uint64_t out_capacity, uint64_t *out_bytes,
                                              int n_devices)
{
    const int rc = decompress_host_indexed_multi_blocks(stream, stream_bytes, block_offsets, n_blocks, out, out_capacity,
                                                        out_bytes, n_devices);
    if (rc != SNAPPY_B200_ERR_FRAMING)
        return rc;
    // valid raw Snappy the block decoders do not take: the general decoder on the current device
    clear_error();
    return decompress_host_general(stream, stream_bytes, out, out_bytes); // (all arguments were checked above)
}

int snappy_b200_decompress_host_multi(const void *stream, uint64_t stream_bytes, void *out, uint64_t out_capacity,
                                      uint64_t *out_bytes, int n_devices)
{
    clear_error();
    if (!out_bytes || (stream_bytes && !stream))
        return fail_msg(SNAPPY_B200_ERR_ARG, "null pointer argument");
    *out_bytes = 0;
    if (stream_bytes == 0)
        return SNAPPY_B200_OK;
    uint64_t total = 0;
    int rc = snappy_b200_uncompressed_length(stream, stream_bytes, &total);
    if (rc != SNAPPY_B200_OK)
        return rc;
    const uint64_t nb = (total + kBlock - 1) / kBlock;
    if (total == 0 || usable_devices(n_devices) < 2 || nb < 2)
        return snappy_b200_decompress_host(stream, stream_bytes, out, out_capacity, out_bytes);
    if (total > out_capacity)
        return fail_msg(SNAPPY_B200_ERR_CAPACITY, "output buffer too small for the decompressed data");
    // ---- K0 over the whole stream on the current device: where does every block start?
    int home = 0;
    cudaGetDevice(&home);
    std::vector<uint64_t> offs(nb + 1);
    {
        Arena &a = g_arena[(unsigned)home % kMaxDev];
        std::lock_guard<std::mutex> lock(a.mu);
        Result r;
        auto k0 = [&]() {
            W(a.init(), "arena init");
            W(a.need(0, stream_bytes + 64), "cudaMalloc");
            W(a.need(2, (nb + 2) * 8), "cudaMalloc");
            W(a.need(3, 256), "cudaMalloc");
            W(a.need(4, index_workspace_bytes(stream_bytes)), "cudaMalloc");
            uint32_t *d_status = static_cast<uint32_t *>(a.buf[3]);
            unsigned hdr = 0;
            while (static_cast<const uint8_t *>(stream)[hdr++] & 0x80u) {
            }
            uint64_t launches = 0;
            W(cudaMemcpyAsync(a.buf[0], stream, stream_bytes, cudaMemcpyHostToDevice, a.st), "H2D copy");
            W(cudaMemsetAsync(d_status, 0, 4, a.st), "memset");
            W(run_index(static_cast<const uint8_t *>(a.buf[0]), stream_bytes, hdr, total, static_cast<uint64_t *>(a.buf[2]),
                        d_status, a.buf[4], a.st, &launches, false, 0),
              "index launch");
            W(cudaMemcpyAsync(offs.data(), a.buf[2], (nb + 1) * 8, cudaMemcpyDeviceToHost, a.st), "D2H copy");
            W(cudaMemcpyAsync(a.h_small, d_status, 4, cudaMemcpyDeviceToHost, a.st), "read-back");
            W(cudaStreamSynchronize(a.st), "index");
            r.status = (uint32_t)a.h_small[0];
            add_launches(launches);
        };
        k0();
        rc = finish(std::vector<Result>{r});
    }
    if (rc == SNAPPY_B200_ERR_FRAMING) { // an element straddles a block: the general decoder on the current device
        clear_error();
        return decompress_host_general(stream, stream_bytes, out, out_bytes);
    }
    if (rc != SNAPPY_B200_OK)
        return rc;
    return snappy_b200_decompress_host_indexed_multi(stream, stream_bytes, offs.data(), nb, out, out_capacity, out_bytes,
                                                     n_devices);
}

} // extern "C"
