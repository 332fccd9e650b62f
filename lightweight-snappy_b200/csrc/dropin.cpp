// dropin.cpp -- the reference's own entry points (include/snappy_compression.h,
// snappy_compression_tree.h, snappy_decompression.h, varint.h, buffer_compression.h) on top
// of the host-buffer API.  Same symbol names, signatures, FILE* ownership rules and stream
// bytes as the reference (SURVEY.md 8b); the work happens on the GPU.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include <algorithm>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>
#include <vector>

#include "buffer_compression.h"
#include "snappy_b200.h"
#include "snappy_compression.h"
#include "snappy_compression_tree.h"
#include "snappy_decompression.h"
#include "varint.h"

namespace sb200 {
int fail_msg(int code, const char *msg); // abi.cu: records the thread's last error
int check_mode(int mode);                // abi.cu: SNAPPY_B200_OK, or SNAPPY_B200_ERR_ARG for an unknown mode
void clear_error();
int frame_compress_host_range(const void *, uint64_t, int, void *, uint64_t, uint64_t *, bool); // host_pipeline.cu
int frame_decompress_buffer(const void *, uint64_t, void *, uint64_t, uint64_t *, bool);          // host_pipeline.cu
} // namespace sb200

namespace {

int io_fail(const char *what) { return sb200::fail_msg(SNAPPY_B200_ERR_IO, what); }

// Page-locking is expensive (measured on the B200 box: 85 ms for 64 MiB, 410 ms for 1 GiB), so buffers that
// are given back are kept for the next call of the process instead of being unlocked (up to 1 GiB in total).
struct PinnedPool {
    struct Item {
        void *p;
        size_t cap;
    };
    std::mutex mu;
    std::vector<Item> items;
    size_t bytes = 0;
    void *take(size_t want, size_t &cap)
    {
        std::lock_guard<std::mutex> l(mu);
        for (size_t i = 0; i < items.size(); ++i)
            if (items[i].cap >= want && items[i].cap <= 2 * want + (1u << 20)) {
                void *p = items[i].p;
                cap = items[i].cap;
                bytes -= cap;
                items.erase(items.begin() + (long)i);
                return p;
            }
        return nullptr;
    }
    bool give(void *p, size_t cap)
    {
        std::lock_guard<std::mutex> l(mu);
        if (bytes + cap > (1ull << 30))
            return false;
        items.push_back({p, cap});
        bytes += cap;
        return true;
    }
};
PinnedPool &pinned_pool()
{
    static PinnedPool *pool = new PinnedPool; // (never destroyed: the CUDA runtime may be gone by then)
    return *pool;
}

// A growable byte buffer in page-locked host memory (plain malloc when no device is usable, so
// that error paths still work): what the reference's Buffer / IO_utils allocations become.
struct PinnedBuf {
    uint8_t *p = nullptr;
    size_t cap = 0, n = 0;
    bool pinned = false;
    ~PinnedBuf() { drop(); }
    void drop()
    {
        if (p) {
            if (pinned) {
                if (!pinned_pool().give(p, cap))
                    snappy_b200_host_free(p);
            } else {
                free(p);
            }
        }
        p = nullptr;
        cap = n = 0;
    }
    bool reserve(size_t want)
    {
        if (want <= cap)
            return true;
        size_t got_cap = want;
        void *q = pinned_pool().take(want, got_cap);
        if (!q)
            q = snappy_b200_host_alloc(want);
        bool qp = q != nullptr;
        if (!q)
            q = malloc(want);
        if (!q)
            return false;
        if (n)
            memcpy(q, p, n);
        const size_t keep = n;
        drop();
        p = static_cast<uint8_t *>(q);
        cap = qp ? got_cap : want;
        n = keep;
        pinned = qp;
        return true;
    }
    uint8_t *data() { return p; }
    size_t size() const { return n; }
    bool empty() const { return n == 0; }
};

// Reads from the current position to EOF (the reference's fread loop, src/snappy_compression.c:210-213).
bool read_all(FILE *f, uint64_t hint, PinnedBuf &buf)
{
    size_t cap = hint ? hint + 1 : (1u << 20);
    buf.n = 0;
    for (;;) {
        if (!buf.reserve(cap))
            return false;
        const size_t got = fread(buf.p + buf.n, 1, cap - buf.n, f);
        buf.n += got;
        if (buf.n < cap) {
            if (ferror(f))
                return false;
            break;
        }
        cap *= 2;
    }
    return true;
}

const char kIndexMagic[8] = {'S', 'N', 'P', 'I', 'D', 'X', '1', 0};

// The streaming compressor behind snappy_compress / snappy_compress_bst.  The reference works through the file
// 64 KiB at a time (src/snappy_compression.c:210-213, :419-425); here the unit is a chunk of whole blocks
// (32 MiB per device in use): a reader thread fills page-locked input buffers, the calling thread runs the
// GPU pipeline on one chunk while the next is being read, a writer thread appends the finished chunks.
// Three chunks are in flight, so page-locked memory is bounded by the chunk size, not by the file size.
struct ChunkQueue { // hands slot numbers from one thread to the next
    std::mutex mu;
    std::condition_variable cv;
    std::deque<int> q;
    void push(int v)
    {
        {
            std::lock_guard<std::mutex> l(mu);
            q.push_back(v);
        }
        cv.notify_one();
    }
    int pop()
    {
        std::unique_lock<std::mutex> l(mu);
        cv.wait(l, [&] { return !q.empty(); });
        const int v = q.front();
        q.pop_front();
        return v;
    }
};

uint64_t stream_chunk_bytes(unsigned long long declared)
{
    uint64_t mib = 32; // (page-locking costs ~45 ms per 32 MiB buffer and there are six: a cold command line pays it)
    if (const char *v = getenv("SNAPPY_B200_FILE_CHUNK_MIB"))
        mib = (uint64_t)std::max(1ll, atoll(v));
    uint64_t dev = 1;
    if (const char *v = getenv("SNAPPY_B200_DEVICES"))
        dev = (uint64_t)std::max(1ll, atoll(v));
    uint64_t chunk = (mib << 20) * dev;
    const uint64_t whole = ((uint64_t)declared + 65535) / 65536 * 65536;
    if (declared && whole < chunk)
        chunk = whole; // a small file: one chunk of its own size (if the file is longer than declared, more follow)
    return chunk;
}

// framed: the framing format (stream identifier, then CRC-checked chunks) instead of the reference's stream;
// `declared` only sizes the chunks then.
int compress_file(FILE *in, unsigned long long declared, FILE *out, int mode, FILE *index_out = nullptr,
                  bool framed = false)
{
    sb200::clear_error();
    if (!in || !out)
        return io_fail("null FILE*");
    constexpr int kInFlight = 3;
    const uint64_t chunk = stream_chunk_bytes(declared);
    const uint64_t out_cap =
        framed ? snappy_b200_frame_max_compressed_bytes(chunk) : snappy_b200_max_compressed_bytes(chunk);
    PinnedBuf ibuf[kInFlight], obuf[kInFlight];
    uint64_t ilen[kInFlight] = {}, olen[kInFlight] = {};
    ChunkQueue free_in, filled, to_write, free_out;
    bool read_error = false, write_error = false;
    int rc = SNAPPY_B200_OK;

    // reader: fills input slots until EOF (a slot with 0 bytes marks the end)
    std::thread reader([&] {
        for (;;) {
            const int s = free_in.pop();
            if (s < 0)
                return; // the caller gave up
            const int c = fgetc(in); // (no page-locked buffer is set up just to find the end of the file)
            if (c == EOF) {
                if (ferror(in))
                    read_error = true;
                ilen[s] = 0;
                filled.push(s);
                return;
            }
            ungetc(c, in);
            if (!ibuf[s].reserve(chunk)) {
                read_error = true;
                ilen[s] = 0;
                filled.push(s);
                return;
            }
            uint64_t got = 0;
            while (got < chunk) {
                const size_t k = fread(ibuf[s].p + got, 1, chunk - got, in);
                if (k == 0)
                    break;
                got += k;
            }
            if (ferror(in))
                read_error = true;
            ilen[s] = read_error ? 0 : got;
            filled.push(s);
            if (got < chunk)
                return;
        }
    });
    // writer: appends finished chunks in order (a negative slot ends it)
    std::thread writer([&] {
        for (;;) {
            const int s = to_write.pop();
            if (s < 0)
                return;
            if (!write_error && fwrite(obuf[s].p, 1, olen[s], out) != olen[s])
                write_error = true;
            free_out.push(s);
        }
    });
    for (int s = 0; s < kInFlight; ++s) {
        free_in.push(s);
        free_out.push(s);
    }
    std::vector<uint64_t> index; // stream offset of every block, when an index file is wanted
    std::vector<uint64_t> offs;
    uint64_t n_in = 0, n_out = 0;
    bool first = true, ended = false;
    while (!ended) {
        const int s = filled.pop();
        const uint64_t n = ilen[s];
        if (n < chunk)
            ended = true; // the last chunk (possibly empty)
        if (n == 0 && !(framed && first)) { // (an empty input still gets the stream identifier when framed)
            free_in.push(s);
            break;
        }
        const int o = free_out.pop();
        if (rc == SNAPPY_B200_OK && !obuf[o].reserve(out_cap))
            rc = io_fail("out of host memory for the compressed stream");
        uint64_t got = 0;
        const uint64_t nb = snappy_b200_block_count(n);
        if (index_out)
            offs.resize(nb + 1);
        if (rc == SNAPPY_B200_OK && framed)
            rc = sb200::frame_compress_host_range(ibuf[s].p, n, mode, obuf[o].p, obuf[o].cap, &got, first);
        else if (rc == SNAPPY_B200_OK)
            // the reference writes the DECLARED size into the preamble (src/snappy_compression.c:417) and then
            // whatever the file really holds: keep that even when the two disagree
            rc = snappy_b200_compress_host_range(ibuf[s].p, n, mode, obuf[o].p, obuf[o].cap, &got,
                                                 index_out ? offs.data() : nullptr,
                                                 first ? (declared ? declared : ~0ull) : 0);
        if (rc == SNAPPY_B200_OK && !framed && first && declared == 0) {
            // (a declared size of 0 still needs its one-byte preamble "00": ask for any value, then patch it)
            unsigned char tmp[10];
            const unsigned k = parse_to_varint(~0ull, tmp);
            memmove(obuf[o].p + 1, obuf[o].p + k, got - k);
            obuf[o].p[0] = 0;
            for (uint64_t b = 0; index_out && b <= nb; ++b)
                offs[b] -= k - 1;
            got -= k - 1;
        }
        if (rc == SNAPPY_B200_OK && index_out)
            for (uint64_t b = 0; b < nb; ++b)
                index.push_back(n_out + offs[b]);
        first = false;
        olen[o] = rc == SNAPPY_B200_OK ? got : 0;
        n_in += n;
        n_out += olen[o];
        to_write.push(o);
        free_in.push(s); // (the reader blocks in pop() at most once more; it returns on the -1 below)
    }
    free_in.push(-1);
    to_write.push(-1);
    reader.join();
    writer.join();
    if (rc != SNAPPY_B200_OK)
        return rc;
    if (read_error)
        return io_fail("reading the input failed (read error or out of host memory)");
    if (write_error)
        return io_fail("short write of the compressed stream");
    if (index_out && n_in) {
        index.push_back(n_out);
        const uint64_t head[2] = {n_in, (uint64_t)index.size() - 1};
        if (fwrite(kIndexMagic, 1, 8, index_out) != 8 || fwrite(head, 8, 2, index_out) != 2 ||
            fwrite(index.data(), 8, index.size(), index_out) != index.size())
            return io_fail("short write of the block index");
    }
    return SNAPPY_B200_OK; // (an empty input leaves an empty output, like the reference: SURVEY.md 8c)
}

// Framed FILE* -> FILE* decompression with bounded memory and no seek: 32 MiB windows are read into a page-locked
// buffer, the chunks that are complete in it (at most 32 MiB of output at a time) are decoded by the host-buffer
// path and written out, and the incomplete tail is carried into the next window.  A chunk is shorter than
// 16 MiB + 4 bytes, so a window always completes at least one.
int decompress_file_framed(FILE *in, FILE *out)
{
    sb200::clear_error();
    if (!in || !out)
        return io_fail("null FILE*");
    constexpr uint64_t kWindow = 32u << 20, kMaxOut = 32u << 20;
    PinnedBuf ib, ob;
    if (!ib.reserve(kWindow) || !ob.reserve(kMaxOut))
        return io_fail("out of host memory for the window buffers");
    uint64_t have = 0;
    bool eof = false, first = true;
    for (;;) {
        while (!eof && have < kWindow) {
            const size_t k = fread(ib.p + have, 1, kWindow - have, in);
            have += k;
            if (k == 0) {
                if (ferror(in))
                    return io_fail("reading the compressed stream failed");
                eof = true;
            }
        }
        // the complete chunks at the front, at most kMaxOut bytes of output (but always at least one chunk)
        uint64_t at = 0, produced = 0;
        while (at + 4 <= have) {
            const uint8_t *h = ib.p + at;
            const uint64_t L = h[1] | (uint64_t)h[2] << 8 | (uint64_t)h[3] << 16;
            if (at + 4 + L > have)
                break;
            // (an upper bound of the chunk's output: the decode checks the chunk itself)
            const uint64_t o = (h[0] == 0x00 || h[0] == 0x01) ? 65536 : 0;
            if (at > 0 && produced + o > kMaxOut)
                break;
            produced += o;
            at += 4 + L;
        }
        if (at == 0 && eof)
            at = have; // a truncated chunk (or nothing at all): the decode reports it
        uint64_t got = 0;
        const int rc = sb200::frame_decompress_buffer(ib.p, at, ob.p, ob.cap, &got, first);
        if (rc != SNAPPY_B200_OK)
            return rc;
        if (got && fwrite(ob.p, 1, got, out) != got)
            return io_fail("short write of the output");
        first = false;
        memmove(ib.p, ib.p + at, have - at);
        have -= at;
        if (eof && have == 0)
            return SNAPPY_B200_OK;
    }
}

} // namespace

extern "C" {

int snappy_b200_frame_compress_file(FILE *in, FILE *out, int mode)
{
    sb200::clear_error();
    if (sb200::check_mode(mode) != SNAPPY_B200_OK)
        return SNAPPY_B200_ERR_ARG;
    return compress_file(in, 0, out, mode, nullptr, true);
}

int snappy_b200_frame_decompress_file(FILE *in, FILE *out) { return decompress_file_framed(in, out); }

int snappy_b200_compress_file_indexed(FILE *in, unsigned long long input_size, int mode, FILE *out, FILE *index_out)
{
    sb200::clear_error();
    if (sb200::check_mode(mode) != SNAPPY_B200_OK)
        return SNAPPY_B200_ERR_ARG;
    return compress_file(in, input_size, out, mode, index_out);
}

int snappy_b200_decompress_file_indexed(FILE *in, FILE *index_in, FILE *out)
{
    PinnedBuf stream, data;
    sb200::clear_error();
    if (!in || !index_in || !out || !read_all(in, 0, stream))
        return io_fail("reading the compressed stream failed");
    char magic[8];
    uint64_t head[2];
    if (fread(magic, 1, 8, index_in) != 8 || memcmp(magic, kIndexMagic, 8) != 0 || fread(head, 8, 2, index_in) != 2 ||
        head[1] != snappy_b200_block_count(head[0]) || head[1] >= (1ull << 31)) {
        return sb200::fail_msg(SNAPPY_B200_ERR_CORRUPT, "not a block index file");
    }
    uint64_t *offsets = static_cast<uint64_t *>(malloc((head[1] + 1) * 8));
    if (!offsets)
        return io_fail("out of host memory for the block index");
    int rc = SNAPPY_B200_OK;
    if (fread(offsets, 8, head[1] + 1, index_in) != head[1] + 1)
        rc = sb200::fail_msg(SNAPPY_B200_ERR_CORRUPT, "truncated block index file");
    uint64_t n = 0;
    if (rc == SNAPPY_B200_OK && head[0] && !data.reserve(head[0]))
        rc = io_fail("out of host memory for the output");
    if (rc == SNAPPY_B200_OK && head[0]) {
        rc = snappy_b200_decompress_host_indexed(stream.data(), stream.size(), offsets, head[1], data.data(), data.cap, &n);
        if (rc == SNAPPY_B200_OK && n != head[0])
            rc = sb200::fail_msg(SNAPPY_B200_ERR_CORRUPT, "the index file declares another length than the stream");
        if (rc == SNAPPY_B200_OK && fwrite(data.data(), 1, n, out) != n)
            rc = io_fail("short write of the output");
    }
    free(offsets);
    return rc;
}

void snappy_compress(FILE *file_input, unsigned long long input_size, FILE *file_compressed)
{
    (void)compress_file(file_input, input_size, file_compressed, SNAPPY_B200_MODE_HASH);
}

int snappy_compress_bst(FILE *file_input, unsigned long long input_size, FILE *file_compressed)
{
    return compress_file(file_input, input_size, file_compressed, SNAPPY_B200_MODE_BST);
}

int snappy_decompress(FILE *file_input, FILE *file_decompressed)
{
    PinnedBuf stream, out;
    sb200::clear_error();
    if (!file_input || !file_decompressed)
        return io_fail("null FILE*");
    // the streamed path (stream and output device-resident, three page-locked chunks on the host) ...
    const int streamed = snappy_b200_decompress_file(file_input, file_decompressed);
    if (streamed != 1)
        return streamed;
    // ... or, for a pipe or a stream too large for one device, whole host buffers and the piecewise pipeline
    if (!read_all(file_input, 0, stream))
        return io_fail("reading the compressed stream failed");
    uint64_t total = 0;
    int rc = snappy_b200_uncompressed_length(stream.data(), stream.size(), &total);
    if (rc == SNAPPY_B200_OK && total) {
        if (!out.reserve(total))
            return io_fail("out of host memory for the output");
        uint64_t n = 0;
        rc = snappy_b200_decompress_host(stream.data(), stream.size(), out.data(), out.cap, &n);
        if (rc == SNAPPY_B200_OK && fwrite(out.data(), 1, n, file_decompressed) != n)
            rc = io_fail("short write of the output");
    }
    return rc;
}

// ---- varint.h (reference src/varint.c) ---------------------------------------------------
unsigned int parse_to_varint(unsigned long long n, unsigned char *varint)
{
    unsigned int k = 0;
    while (n >= 0x80u) {
        varint[k++] = (unsigned char)(n | 0x80u);
        n >>= 7;
    }
    varint[k++] = (unsigned char)n;
    return k;
}

int str_varint_to_dim_(unsigned char *varint)
{
    // the reference accumulates in an int (src/varint.c:44-58): keep its wrap-around
    unsigned int result = 0, mult = 1;
    unsigned char b;
    do {
        b = *varint++;
        result += (unsigned int)(b & 0x7fu) * mult;
        mult *= 128u;
    } while (b & 0x80u);
    return (int)result;
}

int varint_to_dim(FILE *source)
{
    unsigned int result = 0, mult = 1;
    unsigned char b = 0;
    do {
        if (fread(&b, 1, 1, source) != 1)
            break;
        result += (unsigned int)(b & 0x7fu) * mult;
        mult *= 128u;
    } while (b & 0x80u);
    return (int)result;
}

// ---- buffer_compression.h (reference src/buffer_compression.c) ----------------------------
void init_Buffer(Buffer *bf, unsigned int buffer_size)
{
    bf->current = (char *)calloc(buffer_size, 1);
    bf->beginning = bf->current;
    bf->bytes_left = buffer_size;
}

void move_current(Buffer *bf, unsigned int offset)
{
    bf->current += offset;
    bf->bytes_left -= offset;
}

void reset(Buffer *bf) { bf->current = bf->beginning; }

} // extern "C"
